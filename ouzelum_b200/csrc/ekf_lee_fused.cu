// Fused estimator + controller of the EKFLeeLanded task: ONE kernel per control step, one env per thread, replaces the
// chain apply_resets -> get_state -> sensor_frontend -> ekf_set_q -> ekf_update -> pv_reset -> pv_step -> waypoint ->
// lee_wrench (8 launches + AoS gathers).  Reference: isaacgymenvs/tasks/ekf_lee_landed.py:308-530.
//   * reads the true root state straight from the env handle's SoA planes (no AoS gather); envs flagged for reset are
//     re-spawned in registers with the same draws ozl_step will make (reset_idx runs first, :312-314)
//   * the step index, warm-up flag and the shared sensor-trigger counters come from the env's DEVICE step counter, so the
//     whole task step (vehicle kernel, this kernel, step kernel) takes no host-changing argument: CUDA-graph capturable
//   * traffic per env: root 72 B + EKF 2x160 B + PV 2x360 B + ~100 B of glue  (config 3: ~1.3 KB / env-step with the step kernel;
//     L2-resident in steady state at 65536 envs)
// (the counter-RNG draws stay inline: one out-of-line copy shared by the ~22 draw sites of this kernel is 20 KB less code but
//  measured slower on B200, 28.2 vs 27.1 us per 65536-env step)
#include "internal.h"
#include "bulk_copy.cuh"
#include "quad_io.cuh"
#include "targets.cuh"
#include "filters.cuh"
#include "glue.cuh"
#include "lee_control.cuh"
#include "tile_chain.cuh"

constexpr int kEkfSmemRows = 81 + 12;                      // covariance tile + the cooperative fixes' scratch columns, floats per env
constexpr int kWarpTile = kEkfSmemRows * 32;                // floats of shared memory per WARP: [81][32] tile + [12][32] scratch

namespace ozl {

struct EkfLeeArgs {
    int64_t n, n_total;                   // envs of this handle / of the whole job (all ranks): trigger index = step * n_total + global env
    double* ekf_q;  double* ekf_P;        // [4][n], [16][n]
    float* pv_x;    float* pv_P;          // [9][n], [81][n]
    float* prev_linvel;                   // [n,3]
    float* waypoint;                      // [n,3]
    const float* target;                  // [n,3]
    const int64_t* reset;                 // [n]
    float4* wrench;                       // [n] out
    float* est13;   float4* cmd4;         // optional debug outputs
    float dt, dt2, inv_dt, mg, hover;
    int64_t convergence;
    FaultCfg f;                           // mode / probabilities / seed (step filled in-kernel)
    uint32_t pos_period, pos_phase, vel_period, vel_phase;
    int per_env_triggers;
    float acc_var[3], pos_var[3];
    double ekf_Dt, ekf_g_noise;
    LeeGains g;
};

// Envs per CTA: 96 (5 CTAs per SM at 128 registers per thread; 64-env CTAs fit 8, 128 fit 4, 256 fit 2, 512 fit 1).  Measured on B200 at config 3
// (65536 envs, one wave): 96 -> 27.1 us, 128 -> 28.4 us, 64 -> 29.4 us, 256 -> +0.1 us over 128, 512 -> +1.3 us.  (Final kernel, warp-private
// tiles: 96 -> 23.8 us, 64 -> 24.3 us, 128 -> 24.7 us, 32 -> 26.5 us.)  65536 envs
// are 443 envs per SM: with 128-env CTAs the SMs hold 3 or 4 of them (12 or 16 warps) and the launch lasts as long as the SMs
// with 16; 96-env CTAs spread the same envs as 4 or 5 CTAs (12 or 15 warps).
constexpr int kEkfLeeBlock = 96;
constexpr int kEkfLeeMinBlocks = 5;

// Layout of the work inside a CTA (one env per thread, kEkfBlock envs per CTA, shared memory WARP-PRIVATE):
//   * each warp's [81][32] slice of the PV covariance planes is brought into its own shared-memory tile by ONE 2-D tensor-map copy
//     (cp.async.bulk.tensor.2d on the warp's mbarrier; the caller's [81][N] planes are described by a CUtensorMap with an [81][32]
//     box) before anything else: the loads fly while every thread runs the vehicle, the sensor front-end and the float64 attitude
//     EKF out of registers.  (81 separate 1-D bulk copies per CTA compiled to an elect / broadcast loop per warp: 24.95 -> 23.9 us)
//   * each stage's loads are issued before the previous stage's arithmetic.  (Round 2 also prefetched everything the later stages
//     read into L2 at the top; with the state L2-resident in steady state -- profiles/r02q_steady_state_dram_traffic.json -- the
//     ~40 prefetch instructions per thread only cost L2 bandwidth: 26.15 -> 25.92 us without them)
//   * the PV filter then works in place on the thread's column of that tile with rolled loops (filters.cuh, PVShared<32>); the
//     gated fixes are shared by the lanes of the warp (pv_correct_coop)
//   * the updated tile leaves through one tensor-map store per warp while the threads run the waypoint logic and the Lee controller
//   * after the step-index broadcast nothing needs a block barrier (measured equal to the block-wide tile: 23.7 vs 23.6 us; kept
//     because the box no longer depends on the CTA size)
//   * N % 4 != 0 (plane rows not 16-byte aligned) or no tensor map: the same tile is filled / drained with plain coalesced loads / stores
// WITH_STEP = true is the WHOLE EKFLeeLanded control step in one launch (ozl_ekf_lee_landed_step): the ground vehicle that
// carries the target runs first (targets.cuh), and after the controller the same thread applies its wrench to its env --
// env_step(ACT_WRENCH) with the vehicle's target, sensor-fault epilogue on the observation, stores, episode statistics and
// the step-counter retirement of quad_step_kernel (quad_io.cuh).  Each warp stages its [32][13] observation rows in its covariance
// tile once the drain has read it.  Replaces three launches (husky_step, ekf_lee_fused, quad_step) and their re-reads.
struct StepIo {
    float* obs; float* rew; int64_t* reset; int64_t* progress; uint8_t* timeout; float* ep_ret;
};

template <int kEkfBlock, bool WITH_STEP>
__global__ void __launch_bounds__(kEkfBlock, kEkfLeeMinBlocks)
ekf_lee_fused_kernel(const __grid_constant__ DevCfg c, const Planes pl, const EkfLeeArgs a, const int use_tma, const HuskyArgs h, const StepIo io,
                     const int chain, const __grid_constant__ CUtensorMap tmap) {
    static_assert(kEkfBlock % 32 == 0, "whole warps");
    // Shared memory is WARP-PRIVATE: warp w owns [81][32] floats of covariance tile (+ [12][32] of scratch for the cooperative
    // fixes), its own mbarrier, and later stages its [32][13] observation rows in the same tile.  Nothing after the step-index
    // broadcast needs a block barrier: the tile comes and goes through per-warp tensor-map copies, the fixes are intra-warp.
    extern __shared__ __align__(128) float s_all[];
    __shared__ __align__(8) uint64_t s_bars[kEkfBlock / 32];
    __shared__ uint64_t s_step;
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    float* const s_P = s_all + warp * kWarpTile;             // this warp's tile, element (k, lane) at s_P[k * 32 + lane]
    uint64_t* const s_bar = &s_bars[warp];
    const int64_t base = (int64_t)blockIdx.x * kEkfBlock;
    const int64_t i = base + tid;
    const bool valid = i < a.n;
    const int n_here = (a.n - base) < kEkfBlock ? (int)(a.n - base) : kEkfBlock;
    // valid lanes of this warp (a prefix): the participants of the warp-cooperative PV fixes
    const int wl = n_here - (tid & ~31);
    const unsigned wmask = wl >= 32 ? 0xffffffffu : (wl > 0 ? (1u << wl) - 1u : 0u);
    if (lane == 0 && use_tma) mbar_init(s_bar, 1);
    // tile-chained launches (tile_chain.cuh): chained == this launch does NOT wait for the previous grid, only for its own tile
    // chain: -1 classic launch (no tile words touched), 0 first launch of a chain, 1 chained
    const bool chained = WITH_STEP && chain > 0;
    const bool chain_words = WITH_STEP && chain >= 0;
    unsigned long long* const seq = pl.tile_seq + 2 * (size_t)blockIdx.x;
    if (!chained) {
        griddep_wait();                // PDL (bulk_copy.cuh): everything below reads what the previous launch wrote
        if (!chain_words) griddep_launch_dependents();
        if (tid == 0) {
            const uint64_t s0 = read_step(pl.ctrl);
            s_step = s0;
            if (chain_words) { seq[0] = s0 + 1ull; __threadfence(); }   // visible before this CTA's launch trigger
        }
    } else if (tid == 0) {
        s_step = atomicAdd(seq, 1ull);                                  // returned before this CTA's launch trigger
    }
    // ---- stage-0 loads (registers)
    bool rst = false;
    float4 d0 = make_float4(0.f, 0.f, 0.f, 0.f), d1 = d0, d2 = d0;
    float wz0 = 0.f, pvl[3] = {0.f, 0.f, 0.f}, wp[3] = {0.f, 0.f, 0.f};
    float4 hpose = d0;
    int2 hidx = make_int2(0, 0);
    auto stage0_loads = [&]() {
        rst = a.reset[i] != 0;
        if (WITH_STEP) { hpose = h.pose[i]; hidx = h.idx[i]; }
        d0 = *plane4_ptr(pl, 0, i); d1 = *plane4_ptr(pl, 1, i); d2 = *plane4_ptr(pl, 2, i);
        wz0 = plane4_ptr(pl, 3, i)->x;
#pragma unroll
        for (int j = 0; j < 3; ++j) { pvl[j] = a.prev_linvel[i * 3 + j]; wp[j] = a.waypoint[i * 3 + j]; }
    };
    if (valid) {
        if (!chained) stage0_loads();  // in flight while the block waits for its leader's read of the step record
    }
    __syncthreads();                   // the mbarrier is initialised, the step index is published
    if (chain_words) griddep_launch_dependents();   // after the tile's `started` word is final: the next launch's CTAs read it in launch order
    if (chained) {
        if (tid == 0) tile_chain_wait(seq, s_step);     // the tile's previous step has been released (acquire)
        __syncthreads();
        if (valid) stage0_loads();
        fence_proxy_async_all();       // the bulk loads below (async proxy) are ordered behind the acquire
    }
    const int64_t wbase = base + warp * 32;                  // first env of this warp
    if (use_tma) {
        // ONE 2-D tensor-map copy per warp brings its [81][32] box in (columns beyond N are zero-filled and still counted)
        if (lane == 0 && wbase < a.n) {
            mbar_expect_tx(s_bar, 81u * 32u * 4u);
            tma_load_2d(s_P, &tmap, (int32_t)wbase, 0, s_bar);
        }
    } else if (valid) {
#pragma unroll 3          // fallback path (N % 4 != 0 or no tensor map): kept small, this kernel is instruction-fetch bound
        for (int k = 0; k < 81; ++k) s_P[k * 32 + lane] = a.pv_P[(int64_t)k * a.n + i];
    }
    const uint64_t step = s_step;
    const bool warm = (int64_t)step < a.convergence;                                     // :339
    const uint32_t genv = c.env_id_base + (uint32_t)i;
    // live across the block barrier that precedes the drain of the covariance tile: controller inputs
    float q[4], w[3], est_p[3], est_v[3], cmd[4];
    float tgt[3] = {0.f, 0.f, 0.f};
    if (valid) {
        if (WITH_STEP) husky_step_env(h, i, step, tgt, hpose, hidx);     // landing target for this step (landing.py:373-374)
        // ---- true root state (post reset_idx)
        float p[3], v[3];
        if (rst) {
            const uint4 r = draw_cold(c.seed, genv, step, P_SPAWN);
            p[0] = c.spawn_base[0] + (c.spawn_range[0] * u01(r.x) + c.spawn_lo[0]);
            p[1] = c.spawn_base[1] + (c.spawn_range[1] * u01(r.y) + c.spawn_lo[1]);
            p[2] = c.spawn_base[2] + (c.spawn_range[2] * u01(r.z) + c.spawn_lo[2]);
            q[0] = q[1] = q[2] = 0.f; q[3] = 1.f;
            for (int j = 0; j < 3; ++j) { v[j] = 0.f; w[j] = 0.f; }
        } else {
            p[0] = d0.x; p[1] = d0.y; p[2] = d0.z; q[0] = d0.w; q[1] = d1.x; q[2] = d1.y; q[3] = d1.z;
            v[0] = d1.w; v[1] = d2.x; v[2] = d2.y; w[0] = d2.z; w[1] = d2.w; w[2] = wz0;
        }
        // ---- attitude-EKF state: loads issued here (L2 hits), consumed after the sensor front-end
        EKF4 s;
        if (warm || rst) { s.q[0] = q[3]; s.q[1] = q[0]; s.q[2] = q[1]; s.q[3] = q[2]; }
        else { for (int k = 0; k < 4; ++k) s.q[k] = a.ekf_q[(int64_t)k * a.n + i]; }
        for (int k = 0; k < 16; ++k) s.P[k / 4][k % 4] = a.ekf_P[(int64_t)k * a.n + i];
        // ---- sensor front-end (:345-346,366-375,397-406)
        FaultCfg f = a.f;
        f.step = step;
        if (warm) f.mode = 0;
        float acc[3], gyr[3], ang[4], pos[3], vel[3];
        for (int j = 0; j < 3; ++j) {
            acc[j] = (v[j] - pvl[j]) * a.inv_dt;     // :345-346: `dv / dt` on a CUDA tensor = multiplication by the float32 reciprocal
            gyr[j] = w[j]; pos[j] = p[j]; vel[j] = v[j];
            a.prev_linvel[i * 3 + j] = v[j];                                              // :454
        }
        acc[2] = acc[2] + 9.8f;
        for (int j = 0; j < 4; ++j) ang[j] = q[j];
        sensor_fault(f, genv, 1, false, gyr, 3);
        sensor_fault(f, genv, 3, true, ang, 4);
        sensor_fault(f, genv, 4, false, acc, 3);
        sensor_fault(f, genv, 5, false, pos, 3);
        sensor_fault(f, genv, 6, false, vel, 3);
        // ---- PV state: loads issued before the EKF arithmetic, consumed after it
        PVShared<32> pvs;
        pvs.P = s_P + lane;
        for (int k = 0; k < 9; ++k) pvs.x[k] = a.pv_x[(int64_t)k * a.n + i];
        // ---- attitude EKF (:348-352,378-391), float64 in registers
        float q32[4];
        {
            const double gd[3] = {(double)gyr[0], (double)gyr[1], (double)gyr[2]};
            const double ad[4] = {(double)ang[3], (double)ang[0], (double)ang[1], (double)ang[2]};
            ekf_update(s, gd, ad, a.ekf_Dt, a.ekf_g_noise, 0.0000001);
            for (int k = 0; k < 4; ++k) { a.ekf_q[(int64_t)k * a.n + i] = s.q[k]; q32[k] = (float)s.q[k]; }
            for (int k = 0; k < 16; ++k) a.ekf_P[(int64_t)k * a.n + i] = s.P[k / 4][k % 4];
        }
        // ---- PV filter (:353-358,397-444) on the shared-memory covariance tile
        {
            if (rst) { for (int k = 0; k < 3; ++k) { pvs.x[k] = p[k]; pvs.x[3 + k] = v[k]; pvs.x[6 + k] = 0.f; } }
            const float qt[4] = {q[3], q[0], q[1], q[2]};
            if (use_tma) mbar_wait(s_bar, 0);                    // the covariance tile has landed
            pv_predict(pvs, acc, warm ? qt : q32, a.dt, a.dt2, a.acc_var);
            // shared sensor-trigger counters (:425-440): the reference advances them once per env-iteration, i.e. the k-th
            // iteration overall is step * N_total + GLOBAL env id (invariant to how the envs are sharded over GPUs)
            const uint64_t k = a.per_env_triggers ? step : step * (uint64_t)a.n_total + (uint64_t)genv;
            const bool fix_pos = a.pos_period && (k % a.pos_period) == a.pos_phase;
            const bool fix_vel = a.vel_period && (k % a.vel_period) == a.vel_phase;
            const float zero3[3] = {0.f, 0.f, 0.f};                                                  // gps_var=None => R = 0
            // warp-cooperative fixes (filters.cuh): first fix of every env, then the velocity fix of the envs that had both
            float* const scr = s_P + 81 * 32 + lane;
            pv_correct_coop(pvs, scr, wmask, lane, fix_pos ? 0 : (fix_vel ? 3 : -1), fix_pos ? pos : vel, a.pos_var, zero3);
            pv_correct_coop(pvs, scr, wmask, lane, (fix_pos && fix_vel) ? 3 : -1, vel, a.pos_var, zero3);
            for (int kk = 0; kk < 9; ++kk) a.pv_x[(int64_t)kk * a.n + i] = pvs.x[kk];
            for (int kk = 0; kk < 3; ++kk) { est_p[kk] = pvs.x[kk]; est_v[kk] = pvs.x[3 + kk]; }
        }
        if (!use_tma) {
#pragma unroll 3
            for (int k = 0; k < 81; ++k) a.pv_P[(int64_t)k * a.n + i] = s_P[k * 32 + lane];
        }
        // (the TMA drain of the tile is issued below, after the block barrier, and overlaps the controller)
        // ---- waypoint + controller (:458-529)
        float t[3];
        if (WITH_STEP) { t[0] = tgt[0]; t[1] = tgt[1]; t[2] = tgt[2]; }
        else { t[0] = a.target[i * 3]; t[1] = a.target[i * 3 + 1]; t[2] = a.target[i * 3 + 2]; }
        waypoint_update(p, t, wp, warm);
        for (int j = 0; j < 3; ++j) a.waypoint[i * 3 + j] = wp[j];
        if (a.est13) {
            float* e = a.est13 + i * 13;
            for (int j = 0; j < 3; ++j) { e[j] = warm ? p[j] : est_p[j]; e[7 + j] = warm ? v[j] : est_v[j]; e[10 + j] = w[j]; }
            for (int j = 0; j < 4; ++j) e[3 + j] = q[j];
        }
        if (a.cmd4) a.cmd4[i] = make_float4(wp[0], wp[1], wp[2], 0.0f);
        cmd[0] = wp[0] * a.g.scale[0]; cmd[1] = wp[1] * a.g.scale[1]; cmd[2] = wp[2] * a.g.scale[2]; cmd[3] = 0.0f;
    }
    if (use_tma) {
        // drain: the warp's filter writes are made visible to the async proxy, then its leader issues one tensor-map store
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && wbase < a.n) tma_store_2d(&tmap, (int32_t)wbase, 0, s_P);
    }
    // the env's remaining planes for the step below: loads issued before the controller arithmetic (L2 hits by now)
    Loaded L;
    int64_t prog = 0;
    if (WITH_STEP && valid) {
        load_env(pl, i, L);
        prog = io.progress[i];
    }
    float4 wr = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
        if (warm) {
            wr = make_float4(a.hover, 0.f, 0.f, 0.f);                                     // :526-528
        } else {
            float th, tq[3];
            lee_control(LEE_POSITION, est_p, q, est_v, w, cmd, a.g, th, tq);               // :493-499
            wr = make_float4(a.mg * th, tq[0], tq[1], tq[2]);                              // :504-505
        }
        a.wrench[i] = wr;
    }
    if (use_tma && lane == 0) bulk_wait_read_all();     // the tile must stay alive until the bulk store has read it
    if (!WITH_STEP) return;

    // ---- the env step itself (quad_step_kernel's body, wrench actuation, target from the vehicle)
    StepOut o;
    o.rew = 0.0f; o.ep_ret_done = 0.0f; o.prog = 0;
    o.reset = o.timeout = o.did_reset = o.static_dirty = o.fault_active = o.crash_dist = o.crash_z = o.landed_episode = false;
    float* s_obs = s_P;                                  // reused: the warp's [32][13] observation rows
    __syncwarp();                                        // every lane is done with its covariance column, the drain has read the tile
    if (valid) {
        Env e;
        unpack(L, e);
        const float act[4] = {wr.x, wr.y, wr.z, wr.w};
        env_step(e, act, prog, rst, genv, step, c, o, ACT_WRENCH, tgt);
        obs_epilogue(o.obs, genv, step, flicker_blackout(step, c), c);
        store_dynamic(pl, i, e);
        store_static(pl, i, e);
        io.rew[i] = o.rew;
        io.reset[i] = o.reset ? 1 : 0;
        io.progress[i] = o.prog;
        if (io.timeout) io.timeout[i] = o.timeout ? 1 : 0;
        if (io.ep_ret) io.ep_ret[i] = o.ep_ret_done;
#pragma unroll
        for (int j = 0; j < 13; ++j) s_obs[lane * 13 + j] = o.obs[j];
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (wl > 0) {
        float* dst = io.obs + wbase * 13;                // 32 x 13 x 4 B per warp: every warp's slice starts on a 16-byte boundary
        const int nflt = (wl < 32 ? wl : 32) * 13;
        if ((nflt & 3) == 0) {
            if (lane == 0) bulk_store_s2g(dst, s_obs, (uint32_t)nflt * 4u);
        } else {
#pragma unroll 1
            for (int k = lane; k < nflt; k += 32) dst[k] = s_obs[k];
        }
    }
    // step counter: the launch retires one unit per 128-env tile in total -- block b accounts for the tiles that END in its env range
    const unsigned long long units = (unsigned long long)((base + n_here + kTile - 1) / kTile - (base + kTile - 1) / kTile);
    block_epilogue<kEkfBlock>(c, pl, valid, o, n_here, units + (blockIdx.x == 0 ? (unsigned long long)c.step_pad : 0ull));
    // release the tile (tile_chain.cuh): every bulk store of this CTA has completed, every thread's plain stores are ordered
    // before the barrier, then one fence + release store by the leader
    if (!chain_words) {
        if (lane == 0) bulk_wait_read_all();
        return;
    }
    if (lane == 0) { bulk_wait_all(); fence_proxy_async_all(); }
    __syncthreads();
    if (tid == 0) { __threadfence(); st_release_u64(seq + 1, step + 1ull); }
}

}  // namespace ozl

using namespace ozl;

// 2-D tensor map over the caller's [81][N] covariance planes, box = [81][32] = one warp's envs (cached in the handle: the pointer is
// fixed per task).
// Returns 0 when env->pv_tmap is valid for P.
static int ozl_encode_pv_tmap(ozl_env* env, const float* P, int64_t n) {
    if (env->pv_tmap_ptr == P) return 0;
    if (n < 32) return 1;
    const PFN_cuTensorMapEncodeTiled fn = tensor_map_encoder();
    if (!fn) return 1;
    const cuuint64_t gdim[2] = {(cuuint64_t)n, 81ull};
    const cuuint64_t gstr[1] = {(cuuint64_t)n * sizeof(float)};
    const cuuint32_t box[2] = {32u, 81u};
    const cuuint32_t estr[2] = {1u, 1u};
    if (fn(reinterpret_cast<CUtensorMap*>(env->pv_tmap), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(P), gdim, gstr, box, estr,
           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
        env->pv_tmap_ptr = nullptr;
        return 1;
    }
    env->pv_tmap_ptr = P;
    return 0;
}

static int launch_ekf_lee(ozl_env* env, const ozl_ekf_lee_args* in, const ozl_husky_args* husky, const StepIo io, void* stream) {
    if (!env || !in) return set_error("ozl_ekf_lee_step: NULL argument");
    if (!in->ekf_q4xN || !in->ekf_P16xN || !in->pv_x9xN || !in->pv_P81xN || !in->prev_linvel3 || !in->waypoint3 || !in->target3 ||
        !in->reset || !in->wrench4 || !in->gains16)
        return set_error("ozl_ekf_lee_step: NULL buffer");
    if (((uintptr_t)in->wrench4 & 15) || ((uintptr_t)in->cmd4 & 15)) return set_error("ozl_ekf_lee_step: wrench4/cmd4 must be 16-byte aligned");
    if (in->pomdp_mode < 0 || in->pomdp_mode > 3) return set_error("pomdp was not in ['flicker', 'random_noise', 'flickering_and_random_noise']!");
    EkfLeeArgs a;
    a.n = env->cfg.num_envs;
    a.n_total = in->num_envs_total > 0 ? in->num_envs_total : env->cfg.num_envs;
    a.ekf_q = in->ekf_q4xN; a.ekf_P = in->ekf_P16xN; a.pv_x = in->pv_x9xN; a.pv_P = in->pv_P81xN;
    a.prev_linvel = in->prev_linvel3; a.waypoint = in->waypoint3; a.target = in->target3; a.reset = in->reset;
    a.wrench = (float4*)in->wrench4; a.est13 = in->est13; a.cmd4 = (float4*)in->cmd4;
    a.dt = in->dt; a.dt2 = (float)((double)in->dt * (double)in->dt); a.inv_dt = 1.0f / in->dt; a.mg = in->mg; a.hover = in->hover_force;
    a.convergence = in->convergence_steps;
    a.f.mode = in->pomdp_mode;
    a.f.flicker_p = (in->pomdp_mode == 3) ? 0.1f : in->pomdp_prob;
    const float lo = (float)(1.0 - (double)in->pomdp_prob), hi = (float)(1.0 + (double)in->pomdp_prob);
    a.f.noise_lo = lo; a.f.noise_range = hi - lo;
    a.f.seed = env->cfg.seed; a.f.step = 0;
    a.pos_period = in->pos_period; a.pos_phase = in->pos_phase; a.vel_period = in->vel_period; a.vel_phase = in->vel_phase;
    a.per_env_triggers = in->per_env_triggers;
    for (int j = 0; j < 3; ++j) { a.acc_var[j] = in->acc_var[j]; a.pos_var[j] = in->pos_var[j]; }
    a.ekf_Dt = in->ekf_Dt; a.ekf_g_noise = in->ekf_g_noise;
    for (int k = 0; k < 3; ++k) { a.g.kP[k] = in->gains16[k]; a.g.kV[k] = in->gains16[3 + k]; a.g.kR[k] = in->gains16[6 + k]; a.g.kO[k] = in->gains16[9 + k]; }
    for (int k = 0; k < 4; ++k) a.g.scale[k] = in->gains16[12 + k];
    // TMA path: every [k][N] plane slice of a block must start on a 16-byte boundary and be a multiple of 16 bytes long
    int use_tma = 0;                                                        // 1: per-warp tensor-map copies of the covariance tile
    HuskyArgs h{};
    if (husky) {
        if (ozl_fill_husky_args(husky, h, "ozl_ekf_lee_landed_step")) return 1;
        if (!h.tables) return set_error("ozl_ekf_lee_landed_step: tables204x2 is NULL");
        if (h.n != a.n) return set_error("ozl_ekf_lee_landed_step: vehicle count %lld != env count %lld", (long long)h.n, (long long)a.n);
        if (!io.obs || !io.rew || !io.reset || !io.progress) return set_error("ozl_ekf_lee_landed_step: NULL buffer");
        if ((uintptr_t)io.obs & 15) return set_error("ozl_ekf_lee_landed_step: obs must be 16-byte aligned");
        if (io.reset != a.reset || (h.reset && h.reset != a.reset))
            return set_error("ozl_ekf_lee_landed_step: the estimator, the vehicle and the step must see the same reset buffer");
    }
    // tile-chained launches (tile_chain.cuh): chain only behind the previous chained launch of this handle in the SAME stream
    // capture, with nothing captured in between (the stream's one dependency is that launch's node)
    // Chaining pays when the grid is several waves long (262144 envs: 125 -> 110 us per step); a ONE-wave grid runs in lockstep
    // either way and only pays the protocol's latency (65536 envs: 27.2 -> 33 us), so it keeps the classic launch (chain = -1).
    const unsigned grid = (unsigned)((a.n + kEkfLeeBlock - 1) / kEkfLeeBlock);
    const size_t smem = (size_t)kEkfSmemRows * kEkfLeeBlock * sizeof(float);
    if ((a.n % 4 == 0) && (((uintptr_t)a.pv_P & 15) == 0) && ozl_encode_pv_tmap(env, a.pv_P, a.n) == 0) use_tma = 1;
    const long long slots = (long long)env->sm_count * kEkfLeeMinBlocks;
    const bool may_chain = husky && (env->chain_mode == 2 || (env->chain_mode == 1 && (long long)grid > slots));
    int chain = may_chain ? 0 : -1;
    if (may_chain && env->chain_last_node) {
        cudaStreamCaptureStatus cs; unsigned long long cid = 0; size_t nd = 0;
        const cudaGraphNode_t* deps = nullptr;
        if (cudaStreamGetCaptureInfo_v3((cudaStream_t)stream, &cs, &cid, nullptr, &deps, nullptr, &nd) == cudaSuccess) {
            if (cs == cudaStreamCaptureStatusActive && cid == env->chain_capture_id && nd == 1 && (void*)deps[0] == env->chain_last_node)
                chain = 1;
        } else {
            cudaGetLastError();
        }
    }
    static bool attr_set[2] = {false, false};         // per kernel: the dynamic shared memory exceeds the 48 KB default
    const auto kernel = husky ? ekf_lee_fused_kernel<kEkfLeeBlock, true> : ekf_lee_fused_kernel<kEkfLeeBlock, false>;
    if (!attr_set[husky != nullptr]) {
        if (check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute")) return 1;
        attr_set[husky != nullptr] = true;
    }
    if (launch_pdl_smem(kernel, dim3(grid), dim3(kEkfLeeBlock), smem, (cudaStream_t)stream, env->dev, env->pl, a, use_tma, h, io, chain,
                        *reinterpret_cast<const CUtensorMap*>(env->pv_tmap)))
        return check_cuda(cudaGetLastError(), "ekf_lee_fused_kernel");
    if (may_chain) {       // remember the node this launch became (if it was captured): the next launch may chain behind it
        cudaStreamCaptureStatus cs; unsigned long long cid = 0; size_t nd = 0;
        const cudaGraphNode_t* deps = nullptr;
        env->chain_last_node = nullptr;
        if (cudaStreamGetCaptureInfo_v3((cudaStream_t)stream, &cs, &cid, nullptr, &deps, nullptr, &nd) == cudaSuccess) {
            if (cs == cudaStreamCaptureStatusActive && nd == 1) { env->chain_capture_id = cid; env->chain_last_node = (void*)deps[0]; }
        } else {
            cudaGetLastError();
        }
    }
    return 0;
}

extern "C" int ozl_ekf_lee_step(ozl_env* env, const ozl_ekf_lee_args* in, void* stream) {
    return launch_ekf_lee(env, in, nullptr, StepIo{}, stream);
}

extern "C" int ozl_ekf_lee_landed_step(ozl_env* env, const ozl_ekf_lee_args* in, const ozl_husky_args* husky, float* obs,
                                       float* rew, int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret,
                                       void* stream) {
    if (!husky) return set_error("ozl_ekf_lee_landed_step: husky args are NULL");
    if (env && env->states)
        return set_error("ozl_ekf_lee_landed_step: a states output is registered (ozl_set_states_output) and the fused estimator step does not write it");
    if (env && env->scn)
        return set_error("ozl_ekf_lee_landed_step: a scenario table is registered (ozl_set_scenarios) and the fused estimator step does not apply it");
    if (env && env->log.rec)
        return set_error("ozl_ekf_lee_landed_step: an episode log is registered (ozl_set_episode_log) and the fused estimator step writes no records");
    if (env && env->cfg.fault_mode == 2)
        return set_error("ozl_ekf_lee_landed_step: cfg.fault_mode 2 (multi-rotor faults) does not apply to the wrench-actuated step");
    return launch_ekf_lee(env, in, husky, StepIo{obs, rew, reset, progress, timeout, ep_ret}, stream);
}

extern "C" int ozl_step_counter_ptr(ozl_env* env, const uint64_t** out) {
    if (!env || !out) return set_error("ozl_step_counter_ptr: NULL argument");
    *out = reinterpret_cast<const uint64_t*>(env->pl.ctrl);
    return 0;
}
