// K1 `quad_step`: the fused x500 env step, one env per thread, for sm_100a.
// Host-side twin of the arithmetic: oracle/quad_step.py.  Layout + roofline: DESIGN.md.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <cmath>
#include "internal.h"
#include "bulk_copy.cuh"
#include "quad_io.cuh"
#include "targets.cuh"
#include "lee_control.cuh"

namespace ozl {

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
int set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}
int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return 0;
    return set_error("%s: %s", what, cudaGetErrorString(e));
}
PFN_cuTensorMapEncodeTiled tensor_map_encoder() {
    static const PFN_cuTensorMapEncodeTiled fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            return (PFN_cuTensorMapEncodeTiled)p;
        cudaGetLastError();
        return (PFN_cuTensorMapEncodeTiled)nullptr;
    }();
    return fn;
}

// ------------------------------------------------------------------------------------------------ K1
constexpr int kStepMinBlocks = 7;      // 128-env CTAs resident per SM (the one-wave limit behind tma_min_tiles)
// FRONT selects what runs in front of the env step inside the same thread (one launch per control step for every task):
//   FRONT_NONE     nothing: Ouzelum, Lando, the tracking / wrench variants fed from caller buffers
//   FRONT_VEHICLE  the waypoint-following ground vehicle that carries the target (targets.cuh): Landing, Landed
//   FRONT_LEE      vehicle + Lee position controller on the TRUE state after reset_idx, wrench actuation, landing detector
//                  on the controller target: LeeLanded (lee_landed.py:263-330)
enum { FRONT_NONE = 0, FRONT_VEHICLE = 1, FRONT_LEE = 2 };
struct FrontArgs {
    HuskyArgs h;
    LeeGains g;
    float cmd[4];        // controller target (x, y, z, yaw), lee_landed.py:299-302
    float mg;            // thrust scale 2 * 9.81, lee_landed.py:296
    float4* wrench_out;  // optional [N] debug output
};

// One env's row of the [kTile, OZL_STATES_WIDTH] states tile in shared memory, laid out as CU_TENSOR_MAP_SWIZZLE_128B expects
// (16-byte chunk k of row r sits at chunk k ^ (r & 7); the tile is 1024-byte aligned): the eight 16-byte stores of a quarter-warp
// land in eight different bank groups, where plain 128-byte rows would put all of them in the same four banks (8-way conflict).
// The tensor-map store un-swizzles the tile into the caller's row-major [N, 32] buffer.
__device__ __forceinline__ void stage_states_row(float* tile, int r, const float clean[13], const Env& e, const StepOut& o,
                                                 const DevCfg& c) {
    float s[OZL_STATES_WIDTH];
    states_row(s, clean, e, o, c);
    float4* row = reinterpret_cast<float4*>(tile + r * OZL_STATES_WIDTH);
#pragma unroll
    for (int k = 0; k < OZL_STATES_WIDTH / 4; ++k) row[k ^ (r & 7)] = make_float4(s[4 * k], s[4 * k + 1], s[4 * k + 2], s[4 * k + 3]);
}

// STATES: also write the privileged critic state (ozl_set_states_output) through `states_map`; the STATES = false instantiations
// are the kernels without that output.  SCN: lay the scenario table `scn` (ozl_set_scenarios) over the reset draws; the body
// is instantiated by two kernels, quad_step_kernel (no table, `scn` unused) and quad_step_scn_kernel.
#define OZL_STEP_PARAMS                                                                                                         \
    const DevCfg c, const Planes pl, const float4* __restrict__ actions, float* __restrict__ obs, float* __restrict__ rew,       \
        int64_t* __restrict__ reset, int64_t* __restrict__ progress, uint8_t* __restrict__ timeout, float* __restrict__ ep_ret_out, \
        const float* __restrict__ target_in, const int act_mode, uint8_t* __restrict__ done_u8, int64_t* __restrict__ reset_mirror, \
        const int obs_bulk, const int64_t env0, const FrontArgs fa, volatile unsigned int* host_done, const unsigned int host_seq
#define OZL_STEP_ARGS c, pl, actions, obs, rew, reset, progress, timeout, ep_ret_out, target_in, act_mode, done_u8, reset_mirror, \
                      obs_bulk, env0, fa, host_done, host_seq, states_map, scn
template <int BLOCK, int FRONT, bool STATES, bool SCN>
__device__ __forceinline__ void quad_step_body(OZL_STEP_PARAMS, const CUtensorMap& states_map, const float* __restrict__ scn) {
    __shared__ __align__(16) float s_obs[BLOCK * 13];
    __shared__ __align__(1024) float s_states[STATES ? BLOCK * OZL_STATES_WIDTH : 4];
    __shared__ uint64_t s_step;

    const int64_t base = env0 + (int64_t)blockIdx.x * BLOCK;
    const int64_t i = base + threadIdx.x;
    const bool valid = i < c.num_envs;
    griddep_wait();                    // PDL: everything below reads what the previous launch on the stream wrote
    griddep_launch_dependents();       // ... and the next launch may be staged behind this one from here on
    if (threadIdx.x == 0) s_step = read_step(pl.ctrl);     // one request per block (all of them hit the same L2 slice)

    StepOut o;
    o.rew = 0.0f; o.ep_ret_done = 0.0f; o.prog = 0;
    o.reset = o.timeout = o.did_reset = o.static_dirty = o.fault_active = o.crash_dist = o.crash_z = o.landed_episode = false;

    // all loads issued up front: 9 x 128-bit + 2 x 64-bit per env in flight while the block waits for the step index
    Loaded L;
    float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
    int64_t prog = 0;
    bool rst = false;
    if (valid) {
        load_env(pl, i, L);
        if (FRONT != FRONT_LEE) a4 = __ldg(actions + i);
        prog = progress[i];
        rst = reset[i] != 0;
    }
    __syncthreads();
    const uint64_t step = s_step;
    if (valid) {
        Env e;
        unpack(L, e);
        float tnew[3];
        const float* tptr = nullptr;
        if (FRONT != FRONT_NONE) {   // the vehicle moves first; its top plate is this step's target (landing.py:373-374)
            husky_step_env(fa.h, i, step, tnew);
            tptr = tnew;
        } else if (target_in) {      // externally driven target (caller buffer)
            tnew[0] = target_in[i * 3]; tnew[1] = target_in[i * 3 + 1]; tnew[2] = target_in[i * 3 + 2];
            tptr = tnew;
        }
        float act[4] = {a4.x, a4.y, a4.z, a4.w};
        const uint32_t genv = c.env_id_base + (uint32_t)i;
        const float* scn_row = SCN ? scn + i * OZL_SCENARIO_WIDTH : nullptr;
        if (FRONT == FRONT_LEE) {
            const int64_t prog1 = env_reset_phase<SCN>(e, prog, rst, genv, step, c, o, scn_row);
            const float cmd[4] = {fa.cmd[0] * fa.g.scale[0], fa.cmd[1] * fa.g.scale[1], fa.cmd[2] * fa.g.scale[2], fa.cmd[3] * fa.g.scale[3]};
            float th, tq[3];
            lee_control(LEE_POSITION, e.p, e.q, e.v, e.w, cmd, fa.g, th, tq);                  // lee_landed.py:311
            act[0] = fa.mg * th; act[1] = tq[0]; act[2] = tq[1]; act[3] = tq[2];                 // :313-314
            if (fa.wrench_out) fa.wrench_out[i] = make_float4(act[0], act[1], act[2], act[3]);
            env_act_phase(e, act, prog1, rst, genv, step, c, o, ACT_WRENCH, tptr, fa.cmd);       // detector on the controller target, :305,318-322
        } else {
            env_step<SCN>(e, act, prog, rst, genv, step, c, o, act_mode, tptr, scn_row);
        }
        if constexpr (STATES) stage_states_row(s_states, threadIdx.x, o.obs, e, o, c);
        obs_epilogue(o.obs, genv, step, flicker_blackout(step, c), c);

        store_dynamic(pl, i, e);
        if (o.static_dirty || tptr) store_static(pl, i, e);
        rew[i] = o.rew;
        reset[i] = o.reset ? 1 : 0;
        progress[i] = o.prog;
        if (timeout) timeout[i] = o.timeout ? 1 : 0;
        if (ep_ret_out) ep_ret_out[i] = o.ep_ret_done;
        if (done_u8) done_u8[i] = o.reset ? 1 : 0;
        if (reset_mirror) reset_mirror[i] = o.reset ? 1 : 0;      // reset_buf with the reference's dtype, for a host consumer
#pragma unroll
        for (int j = 0; j < 13; ++j) s_obs[threadIdx.x * 13 + j] = o.obs[j];   // stride 13: conflict-free
    }
    fence_proxy_async_smem();          // make the generic-proxy smem writes visible to the bulk-copy (async) proxy
    __syncthreads();
    // [N,13] row-major observation tile of this block is contiguous: write it with full 16-byte lanes
    const int64_t remaining = c.num_envs - base;
    const int n_here = remaining < BLOCK ? (int)remaining : BLOCK;
    {
        float* dst = obs + base * 13;
        const int nflt = n_here * 13;
        if ((nflt & 3) == 0) {   // base*13*4 bytes is 16-byte aligned whenever BLOCK % 4 == 0
            if (obs_bulk) {
                if (threadIdx.x == 0) bulk_store_s2g(dst, s_obs, (uint32_t)nflt * 4u);
            } else {
                float4* d4p = reinterpret_cast<float4*>(dst);
                const float4* s4 = reinterpret_cast<const float4*>(s_obs);
                for (int k = threadIdx.x; k < nflt / 4; k += BLOCK) d4p[k] = s4[k];
            }
        } else {
            for (int k = threadIdx.x; k < nflt; k += BLOCK) dst[k] = s_obs[k];
        }
    }
    // [BLOCK, 32] states tile: one tensor-map store (rows at and beyond num_envs are clipped)
    if constexpr (STATES) {
        if (threadIdx.x == 0) tma_store_2d(&states_map, 0, (int32_t)base, s_states);
    }
    // one work unit per block; block 0 of the full-range launch also retires the padding (env0 != 0: ragged-tail launch
    // behind the TMA kernel, which has retired the padding already)
    block_epilogue<BLOCK>(c, pl, valid, o, n_here, 1ull + ((blockIdx.x == 0 && env0 == 0) ? (unsigned long long)c.step_pad : 0ull));
    if (threadIdx.x == 0) bulk_wait_read_all();   // s_obs (and s_states) must stay alive until the bulk copies have read them
    // Host consumer: completion word.  Every block orders its zero-copy result stores before a ticket (the barrier makes the
    // block's stores visible to thread 0, the system-scope fence orders them before the ticket); the block that draws the last
    // ticket writes the step's sequence number to pinned host memory, where the host is polling -- no stream synchronise, whose
    // driver path costs ~6 us per step.  (Only in host mode: the device-buffer steps keep their election-free epilogue.)
    if (host_done) {
        __syncthreads();
        if (threadIdx.x == 0) {
            if constexpr (STATES) bulk_wait_all();     // the states tile has reached memory before the ticket
            __threadfence_system();
            const unsigned long long t = atomicAdd(pl.ctrl + 6, 1ull);
            if (t == (unsigned long long)gridDim.x - 1ull) {
                pl.ctrl[6] = 0ull;
                __threadfence_system();
                *host_done = host_seq;
            }
        }
    }
}

template <int BLOCK, int FRONT, bool STATES>
__global__ void __launch_bounds__(BLOCK, kStepMinBlocks)
quad_step_kernel(OZL_STEP_PARAMS, const __grid_constant__ CUtensorMap states_map, const float* __restrict__ scn) {
    quad_step_body<BLOCK, FRONT, STATES, false>(OZL_STEP_ARGS);
}
template <int BLOCK, int FRONT, bool STATES>
__global__ void __launch_bounds__(BLOCK, kStepMinBlocks)
quad_step_scn_kernel(OZL_STEP_PARAMS, const __grid_constant__ CUtensorMap states_map, const float* __restrict__ scn) {
    quad_step_body<BLOCK, FRONT, STATES, true>(OZL_STEP_ARGS);
}

// ------------------------------------------------------------------------------------------------ K1, TMA-pipelined
// Persistent variant for large N (rotor-action mode, stored target): one CTA per (SM x 8) slot loops over tiles of
// kTile = 128 envs.  Thanks to the tiled state layout a tile's whole state is ONE contiguous 15 KiB region, so thread 0
// brings a tile in with four TMA bulk copies (state, actions, progress, reset -> shared memory, completion on an mbarrier)
// and issues the loads of tile t+1 as soon as every thread has copied tile t from shared memory into registers: the load
// latency of the next tile is hidden behind the ~1100-instruction step of the current one regardless of occupancy.
// Stores stay plain coalesced STG (fire and forget); the [128,13] observation tile leaves through a TMA bulk store.
// Metrics are accumulated in registers over all tiles of the CTA and reduced once.
// SASS evidence: UBLKCP (bulk copies), SYNCS (mbarrier).
constexpr int kTmaStateBytes = kTileBytes;                        // 15360
constexpr int kTmaActOff = kTmaStateBytes;                        // actions  [128] float4   2048 B
constexpr int kTmaProgOff = kTmaActOff + kTile * 16;              // progress [128] int64    1024 B
constexpr int kTmaRstOff = kTmaProgOff + kTile * 8;               // reset    [128] int64    1024 B
constexpr int kTmaStageBytes = kTmaRstOff + kTile * 8;            // 19456

constexpr int kTmaMinBlocks = 5;       // CTAs per SM of the TMA kernel, and its persistent grid's slots per SM
#define OZL_TMA_PARAMS                                                                                                          \
    const DevCfg c, const Planes pl, const float4* __restrict__ actions, float* __restrict__ obs, float* __restrict__ rew,       \
        int64_t* __restrict__ reset, int64_t* __restrict__ progress, uint8_t* __restrict__ timeout, float* __restrict__ ep_ret_out, \
        const int64_t full_tiles
#define OZL_TMA_ARGS c, pl, actions, obs, rew, reset, progress, timeout, ep_ret_out, full_tiles, states_map, scn
template <bool STATES, bool SCN>
__device__ __forceinline__ void quad_step_tma_body(OZL_TMA_PARAMS, const CUtensorMap& states_map, const float* __restrict__ scn) {
    __shared__ __align__(128) unsigned char s_stage[kTmaStageBytes];
    __shared__ __align__(16) float s_obs[kTile * 13];
    __shared__ __align__(1024) float s_states[STATES ? kTile * OZL_STATES_WIDTH : 4];   // 16 KB: 5 CTAs/SM still fit
    __shared__ __align__(8) uint64_t s_bar;
    __shared__ double s_m[kTile / 32][11];
    const int tid = threadIdx.x;
    __shared__ uint64_t s_step;
    __shared__ long long s_next;

    auto issue = [&](int64_t tile) {            // thread 0 only
        mbar_expect_tx(&s_bar, kTmaStageBytes);
        bulk_load_g2s(s_stage, pl.base + tile * kTileBytes, kTmaStateBytes, &s_bar);
        bulk_load_g2s(s_stage + kTmaActOff, actions + tile * kTile, kTile * 16, &s_bar);
        bulk_load_g2s(s_stage + kTmaProgOff, progress + tile * kTile, kTile * 8, &s_bar);
        bulk_load_g2s(s_stage + kTmaRstOff, reset + tile * kTile, kTile * 8, &s_bar);
    };
    // dynamic tile scheduler: the first tile of a CTA is its block index, further tiles come from a device counter (ctrl[4]);
    // thread 0 requests the index one iteration ahead so the atomic's round trip never sits on the critical path
    // Prologue order: the first tile's loads go out before anything else, the step index (one L2 round trip) is read behind them.
    int64_t tile = blockIdx.x;
    long long nxt = 0;
    if (tid == 0) mbar_init(&s_bar, 1);
    griddep_wait();                    // PDL: see quad_step_kernel
    griddep_launch_dependents();
    // The scheduler counter is MONOTONIC: a launch makes exactly full_tiles requests in total (every CTA makes one per tile it
    // processes), so the counter stands at a whole multiple of full_tiles between launches and a CTA's first request -- made
    // before the CTA has contributed its own share -- always returns a value inside the current multiple: no re-arming, hence
    // no last-CTA election at the tail of the kernel.
    unsigned long long tile_base = 0;
    if (tid == 0) {
        if (tile < full_tiles) issue(tile);
        const unsigned long long v = atomicAdd(pl.ctrl + 4, 1ull);
        tile_base = (v / (unsigned long long)full_tiles) * (unsigned long long)full_tiles;
        nxt = (long long)gridDim.x + (long long)(v - tile_base);
        s_step = read_step(pl.ctrl);
    }
    __syncthreads();
    const uint64_t step = s_step;
    const bool blackout = flicker_blackout(step, c);

    // metric accumulators over all tiles of this CTA (per-thread counts packed 16 bits each; the host keeps the average number of
    // tiles per CTA below 8192, and the dynamic scheduler spreads them evenly)
    double m_rew = 0.0, m_ret = 0.0;
    int m_len = 0;
    uint32_t m_pk0 = 0, m_pk1 = 0, m_pk2 = 0, m_pk3 = 0;   // done|timeout, crash_dist|crash_z, fault_active|resets, landed|tiles
    uint32_t phase = 0;
    while (tile < full_tiles) {
        mbar_wait(&s_bar, phase);
        phase ^= 1u;
        // shared -> registers (LDS.128, conflict-free: consecutive lanes, 16-byte stride)
        Loaded L;
        const float4* s4 = reinterpret_cast<const float4*>(s_stage);
        L.d0 = s4[tid]; L.d1 = s4[128 + tid]; L.d2 = s4[256 + tid]; L.d3 = s4[384 + tid];
        L.d4 = reinterpret_cast<const float2*>(s_stage + 8192)[tid];
        L.s0 = s4[576 + tid]; L.s1 = s4[704 + tid]; L.s2 = s4[832 + tid];
        const float4 a4 = reinterpret_cast<const float4*>(s_stage + kTmaActOff)[tid];
        const int64_t prog = reinterpret_cast<const int64_t*>(s_stage + kTmaProgOff)[tid];
        const bool rst = reinterpret_cast<const int64_t*>(s_stage + kTmaRstOff)[tid] != 0;
        if (tid == 0) {
            bulk_wait_read_all();                // previous tile's observation (and states) stores have finished reading s_obs
            s_next = nxt;
        }
        __syncthreads();                         // everyone has copied the stage out, s_obs is free, s_next is published
        const int64_t next = s_next;
        if (tid == 0) {
            if (next < full_tiles) {
                issue(next);
                nxt = (long long)gridDim.x + (long long)(atomicAdd(pl.ctrl + 4, 1ull) - tile_base);
            }
        }

        const int64_t i = tile * kTile + tid;
        Env e;
        unpack(L, e);
        const float act[4] = {a4.x, a4.y, a4.z, a4.w};
        const uint32_t genv = c.env_id_base + (uint32_t)i;
        StepOut o;
        env_step<SCN>(e, act, prog, rst, genv, step, c, o, ACT_ROTORS, nullptr, SCN ? scn + i * OZL_SCENARIO_WIDTH : nullptr);
        if constexpr (STATES) stage_states_row(s_states, tid, o.obs, e, o, c);
        obs_epilogue(o.obs, genv, step, blackout, c);
        store_dynamic(pl, i, e);
        if (o.static_dirty) store_static(pl, i, e);
        rew[i] = o.rew;
        reset[i] = o.reset ? 1 : 0;
        progress[i] = o.prog;
        if (timeout) timeout[i] = o.timeout ? 1 : 0;
        if (ep_ret_out) ep_ret_out[i] = o.ep_ret_done;
#pragma unroll
        for (int j = 0; j < 13; ++j) s_obs[tid * 13 + j] = o.obs[j];
        fence_proxy_async_smem();
        __syncthreads();
        if (tid == 0) bulk_store_s2g(obs + tile * (kTile * 13), s_obs, kTile * 13 * 4);
        if constexpr (STATES) {
            if (tid == 0) tma_store_2d(&states_map, 0, (int32_t)(tile * kTile), s_states);
        }
        // metrics
        m_rew += (double)o.rew;
        if (o.reset) { m_ret += (double)o.ep_ret_done; m_len += (int)o.prog; }
        m_pk0 += (uint32_t)o.reset | ((uint32_t)o.timeout << 16);
        m_pk1 += (uint32_t)o.crash_dist | ((uint32_t)o.crash_z << 16);
        m_pk2 += (uint32_t)o.fault_active | ((uint32_t)o.did_reset << 16);
        m_pk3 += (uint32_t)o.landed_episode | (1u << 16);
        tile = next;
    }
    const int m_done = m_pk0 & 0xFFFF, m_to = m_pk0 >> 16, m_cd = m_pk1 & 0xFFFF, m_cz = m_pk1 >> 16;
    const int m_fa = m_pk2 & 0xFFFF, m_rs = m_pk2 >> 16, m_ld = m_pk3 & 0xFFFF, m_valid = m_pk3 >> 16;
    // ---- one reduction per CTA
    if (c.collect_metrics) {
        const int lane = tid & 31, warp = tid >> 5;
        const double srew = warp_sum(m_rew), sret = warp_sum(m_ret);
        const int v[9] = {m_valid, m_done, m_len, m_to, m_cd, m_cz, m_fa, m_rs, m_ld};
        int r[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) r[k] = __reduce_add_sync(0xffffffffu, v[k]);
        if (lane == 0) {
            s_m[warp][0] = srew; s_m[warp][1] = sret;
#pragma unroll
            for (int k = 0; k < 9; ++k) s_m[warp][2 + k] = r[k];
        }
        __syncthreads();
        if (tid < 11) {
            double acc = 0.0;
#pragma unroll
            for (int wv = 0; wv < kTile / 32; ++wv) acc += s_m[wv][tid];
            const int idx = tid < 2 ? tid : (tid == 10 ? 2 : tid + 6);
            if (acc != 0.0) atomicAdd(pl.metrics + (blockIdx.x % kMetricSlots) * kMetricStride + idx, acc);
        }
    }
    if (tid == 0) {
        bulk_wait_read_all();
        // step counter: one work unit per tile processed (+ the padding, CTA 0); a ragged tail is retired by the one-block
        // launch of quad_step_kernel that follows on the stream
        retire_units(pl.ctrl, (unsigned long long)m_valid + (blockIdx.x == 0 ? (unsigned long long)c.step_pad : 0ull));
    }
}

template <bool STATES>
__global__ void __launch_bounds__(kTile, kTmaMinBlocks)
quad_step_tma_kernel(OZL_TMA_PARAMS, const __grid_constant__ CUtensorMap states_map, const float* __restrict__ scn) {
    quad_step_tma_body<STATES, false>(OZL_TMA_ARGS);
}
template <bool STATES>
__global__ void __launch_bounds__(kTile, kTmaMinBlocks)
quad_step_tma_scn_kernel(OZL_TMA_PARAMS, const __grid_constant__ CUtensorMap states_map, const float* __restrict__ scn) {
    quad_step_tma_body<STATES, true>(OZL_TMA_ARGS);
}

// ------------------------------------------------------------------------------------------------ mode B
// K steps per launch with the env in registers; actions a = 2u-1 from the counter RNG.
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK)
quad_rollout_kernel(const DevCfg c, const Planes pl, int K, float* __restrict__ obs, float* __restrict__ rew,
                    int64_t* __restrict__ reset, int64_t* __restrict__ progress) {
    const int64_t i = (int64_t)blockIdx.x * BLOCK + threadIdx.x;
    const bool valid = i < c.num_envs;
    __shared__ uint64_t s_step;
    if (threadIdx.x == 0) s_step = read_step(pl.ctrl);
    __syncthreads();
    const uint64_t step0 = s_step;
    StepOut o;
    o.rew = 0.0f; o.ep_ret_done = 0.0f; o.prog = 0;
    o.reset = o.timeout = o.did_reset = o.static_dirty = o.fault_active = o.crash_dist = o.crash_z = o.landed_episode = false;
    Env e;
    int64_t prog = 0;
    bool rst = false, dirty = false;
    const uint32_t genv = c.env_id_base + (uint32_t)i;
    if (valid) {
        Loaded L;
        load_env(pl, i, L);
        unpack(L, e);
        prog = progress[i];
        rst = reset[i] != 0;
    }
    for (int k = 0; k < K; ++k) {
        const uint64_t step = step0 + (uint64_t)k;
        if (valid) {
            const uint4 r = draw(c.seed, genv, step, P_ACTION);
            const float act[4] = {2.0f * u01(r.x) - 1.0f, 2.0f * u01(r.y) - 1.0f, 2.0f * u01(r.z) - 1.0f,
                                  2.0f * u01(r.w) - 1.0f};
            env_step(e, act, prog, rst, genv, step, c, o);
            prog = o.prog;
            rst = o.reset;
            dirty = dirty || o.static_dirty;
        }
        if (k + 1 < K && c.collect_metrics) {
            // metrics for the intermediate steps (the last step goes through block_epilogue)
            // -- same slots, landed episodes included, without the ticket
            const int lane = threadIdx.x & 31;
            const bool done = valid && o.reset;
            const double srew = warp_sum(valid ? (double)o.rew : 0.0);
            const double sret = warp_sum(done ? (double)o.ep_ret_done : 0.0);
            const int slen = __reduce_add_sync(0xffffffffu, done ? (int)o.prog : 0);
            const int cnt[7] = {__popc(__ballot_sync(0xffffffffu, valid)), __popc(__ballot_sync(0xffffffffu, done)), slen,
                                __popc(__ballot_sync(0xffffffffu, valid && o.timeout)),
                                __popc(__ballot_sync(0xffffffffu, valid && o.crash_dist)),
                                __popc(__ballot_sync(0xffffffffu, valid && o.crash_z)),
                                __popc(__ballot_sync(0xffffffffu, valid && o.fault_active))};
            const int n_rs = __popc(__ballot_sync(0xffffffffu, valid && o.did_reset));
            const int n_ld = __popc(__ballot_sync(0xffffffffu, valid && o.landed_episode));
            if (lane == 0) {
                double* m = pl.metrics + (blockIdx.x % kMetricSlots) * kMetricStride;
                if (srew != 0.0) atomicAdd(m + 0, srew);
                if (sret != 0.0) atomicAdd(m + 1, sret);
                if (n_ld) atomicAdd(m + 2, (double)n_ld);
#pragma unroll
                for (int j = 0; j < 7; ++j)
                    if (cnt[j]) atomicAdd(m + 8 + j, (double)cnt[j]);
                if (n_rs) atomicAdd(m + 15, (double)n_rs);
            }
        }
    }
    if (valid) {
        obs_epilogue(o.obs, genv, step0 + (uint64_t)(K - 1), flicker_blackout(step0 + (uint64_t)(K - 1), c), c);
        store_dynamic(pl, i, e);
        if (dirty) store_static(pl, i, e);
        rew[i] = o.rew;
        reset[i] = o.reset ? 1 : 0;
        progress[i] = o.prog;
#pragma unroll
        for (int j = 0; j < 13; ++j) obs[i * 13 + j] = o.obs[j];
    }
    // the launch retires ONE step's worth of units; the host adds the other K - 1 steps to the counter base afterwards
    __syncthreads();
    const int64_t remaining = c.num_envs - (int64_t)blockIdx.x * BLOCK;
    block_epilogue<BLOCK>(c, pl, valid, o, remaining < BLOCK ? (int)remaining : BLOCK,
                          1ull + (blockIdx.x == 0 ? (unsigned long long)c.step_pad : 0ull));
}

// ------------------------------------------------------------------------------------------------ state access
__global__ void get_state_kernel(const Planes pl, int64_t n, float* root13, float* thrust4, float* target3, float* ep_ret) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Loaded L;
    load_env(pl, i, L);
    Env e;
    unpack(L, e);
    if (root13) {
        float* r = root13 + i * 13;
        r[0] = e.p[0]; r[1] = e.p[1]; r[2] = e.p[2];
        r[3] = e.q[0]; r[4] = e.q[1]; r[5] = e.q[2]; r[6] = e.q[3];
        r[7] = e.v[0]; r[8] = e.v[1]; r[9] = e.v[2];
        r[10] = e.w[0]; r[11] = e.w[1]; r[12] = e.w[2];
    }
    if (thrust4) { float* t = thrust4 + i * 4; t[0] = e.T[0]; t[1] = e.T[1]; t[2] = e.T[2]; t[3] = e.T[3]; }
    if (target3) { float* t = target3 + i * 3; t[0] = e.tgt[0]; t[1] = e.tgt[1]; t[2] = e.tgt[2]; }
    if (ep_ret) ep_ret[i] = e.ep_ret;
}

__global__ void set_state_kernel(const Planes pl, int64_t n, const float* root13, const float* thrust4,
                                 const float* target3, const float* ep_ret) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Loaded L;
    load_env(pl, i, L);
    Env e;
    unpack(L, e);
    if (root13) {
        const float* r = root13 + i * 13;
        e.p[0] = r[0]; e.p[1] = r[1]; e.p[2] = r[2];
        e.q[0] = r[3]; e.q[1] = r[4]; e.q[2] = r[5]; e.q[3] = r[6];
        e.v[0] = r[7]; e.v[1] = r[8]; e.v[2] = r[9];
        e.w[0] = r[10]; e.w[1] = r[11]; e.w[2] = r[12];
    }
    if (thrust4) { const float* t = thrust4 + i * 4; e.T[0] = t[0]; e.T[1] = t[1]; e.T[2] = t[2]; e.T[3] = t[3]; }
    if (target3) { const float* t = target3 + i * 3; e.tgt[0] = t[0]; e.tgt[1] = t[1]; e.tgt[2] = t[2]; }
    if (ep_ret) e.ep_ret = ep_ret[i];
    store_dynamic(pl, i, e);
    store_static(pl, i, e);
}

__global__ void get_params_kernel(const Planes pl, int64_t n, float* params8, int32_t* fault2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Loaded L;
    load_env(pl, i, L);
    Env e;
    unpack(L, e);
    if (params8) {
        float* p = params8 + i * 8;
        p[0] = e.mass; p[1] = e.ixx; p[2] = e.iyy; p[3] = e.izz; p[4] = e.arm; p[5] = e.ks; p[6] = e.eff; p[7] = e.km;
    }
    // onset word: bits 0-28 onset, bit 31 = the env's landed flag (so that get -> set round-trips the whole fault word)
    if (fault2) { fault2[i * 2] = (int32_t)(e.fault & 3u); fault2[i * 2 + 1] = (int32_t)(((e.fault & ~LANDED_BIT) >> 2) | (e.fault & LANDED_BIT)); }
}

__global__ void set_params_kernel(const Planes pl, int64_t n, const float* params8, const int32_t* fault2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Loaded L;
    load_env(pl, i, L);
    Env e;
    unpack(L, e);
    if (params8) {
        const float* p = params8 + i * 8;
        // mass / inertia outside the normal range would break the range-check-free reciprocals of the step: keep the old value
        const float lo = 1.0e-30f, hi = 1.0e30f;
        if (p[0] > lo && p[0] < hi) e.mass = p[0];
        if (p[1] > lo && p[1] < hi) e.ixx = p[1];
        if (p[2] > lo && p[2] < hi) e.iyy = p[2];
        if (p[3] > lo && p[3] < hi) e.izz = p[3];
        e.arm = p[4]; e.ks = p[5]; e.eff = p[6]; e.km = p[7];
    }
    if (fault2) e.fault = ((uint32_t)fault2[i * 2] & 3u) | (((uint32_t)fault2[i * 2 + 1] & FAULT_NEVER) << 2) | ((uint32_t)fault2[i * 2 + 1] & LANDED_BIT);
    store_static(pl, i, e);
}

// reset phase only (see ozl_apply_resets): same draws as env_step, no physics, no bookkeeping; `scn`: the scenario table or NULL
__global__ void apply_resets_kernel(const DevCfg c, const Planes pl, const int64_t* __restrict__ reset, const float* __restrict__ scn) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c.num_envs || reset[i] == 0) return;
    const uint64_t step = read_step(pl.ctrl);
    Loaded L;
    load_env(pl, i, L);
    Env e;
    unpack(L, e);
    const uint32_t genv = c.env_id_base + (uint32_t)i;
    const uint32_t landed = e.fault & LANDED_BIT;
    if (!c.target_fixed) {
        const uint4 r = draw(c.seed, genv, step, P_TARGET);
        e.tgt[0] = u01(r.x) * c.target_scale[0] + c.target_off[0];
        e.tgt[1] = u01(r.y) * c.target_scale[1] + c.target_off[1];
        e.tgt[2] = u01(r.z) * c.target_scale[2] + c.target_off[2];
        if (scn) scn_target(e, scn + i * OZL_SCENARIO_WIDTH);
    }
    const uint4 r = draw(c.seed, genv, step, P_SPAWN);
    e.p[0] = c.spawn_base[0] + (c.spawn_range[0] * u01(r.x) + c.spawn_lo[0]);
    e.p[1] = c.spawn_base[1] + (c.spawn_range[1] * u01(r.y) + c.spawn_lo[1]);
    e.p[2] = c.spawn_base[2] + (c.spawn_range[2] * u01(r.z) + c.spawn_lo[2]);
    e.q[0] = e.q[1] = e.q[2] = 0.0f; e.q[3] = 1.0f;
    for (int j = 0; j < 3; ++j) { e.v[j] = 0.0f; e.w[j] = 0.0f; }
    if (c.fault_mode) {
        const uint4 f = draw(c.seed, genv, step, P_FAULT);
        e.fault = (f.x & 3u) | (__umulhi(f.y, (uint32_t)c.max_episode_length) << 2) | landed;
        e.eff = c.fault_eff_lo + c.fault_eff_range * u01(f.z);
    }
    if (c.dr_enable) dr_draw_all(e, genv, step, c);
    if (scn) scn_respawn(e, scn + i * OZL_SCENARIO_WIDTH);
    store_dynamic(pl, i, e);
    store_static(pl, i, e);
}

__global__ void init_state_kernel(const DevCfg c, const Planes pl) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        pl.ctrl[0] = step_word0_dev(0ull, c.step_shift); pl.ctrl[1] = 0ull;
        pl.ctrl[4] = 0ull; pl.ctrl[5] = 0ull; pl.ctrl[6] = 0ull;
    }
    if (i < kMetricSlots * kMetricStride) pl.metrics[i] = 0.0;
    if (i >= c.num_envs) return;
    Env e;
    e.p[0] = c.spawn_base[0]; e.p[1] = c.spawn_base[1]; e.p[2] = c.spawn_base[2];
    e.q[0] = e.q[1] = e.q[2] = 0.0f; e.q[3] = 1.0f;
    for (int j = 0; j < 3; ++j) { e.v[j] = 0.0f; e.w[j] = 0.0f; }
    for (int j = 0; j < 4; ++j) e.T[j] = 0.0f;
    e.ep_ret = 0.0f;
    e.tgt[0] = 0.0f; e.tgt[1] = 0.0f; e.tgt[2] = 1.0f;        // ouzelum.py:71-73
    e.eff = 1.0f;
    e.mass = c.mass; e.ixx = c.ixx; e.iyy = c.iyy; e.izz = c.izz; e.arm = c.arm; e.ks = 1.0f; e.km = c.yaw_km;
    e.fault = FAULT_NEVER << 2;
    store_dynamic(pl, i, e);
    store_static(pl, i, e);
}

// 16 warps, one per metric: lanes stride over the slots, then a warp reduction
__global__ void metrics_read_kernel(const Planes pl, double* out16, int clear) {
    // PDL: staged behind the step that precedes it on the stream, and the step that follows is staged behind this launch -- a
    // metrics read every 16 steps no longer breaks the chain of programmatic launches (it cost ~4 us per read: 4.2 -> 4.45 us per
    // 16384-env step at one read per 16 steps)
    griddep_wait();
    griddep_launch_dependents();
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double v = 0.0;
    for (int s = lane; s < kMetricSlots; s += 32) {
        v += pl.metrics[s * kMetricStride + j];
        if (clear) pl.metrics[s * kMetricStride + j] = 0.0;
    }
    v = warp_sum(v);
    if (lane == 0) out16[j] = v;
}

__global__ void set_step_kernel(const Planes pl, unsigned long long word0) { pl.ctrl[0] = word0; pl.ctrl[1] = 0ull; }
__global__ void add_steps_kernel(const Planes pl, unsigned long long k) { pl.ctrl[0] += k; }

}  // namespace ozl

using namespace ozl;

// ------------------------------------------------------------------------------------------------ host: cfg
static void derive_dev_cfg(const ozl_cfg& c, DevCfg& d) {
    memset(&d, 0, sizeof(d));
    d.num_envs = c.num_envs;
    d.seed = c.seed;
    d.env_id_base = (uint32_t)c.env_id_base;
    d.max_episode_length = c.max_episode_length;
    d.target_period = c.target_period;
    d.target_fixed = c.target_fixed;
    d.nsub = c.substeps * c.control_freq_inv;
    d.fault_mode = c.fault_mode;
    d.dr_enable = c.dr_enable;
    d.pomdp_mode = c.pomdp_mode;
    d.collect_metrics = c.collect_metrics;
    d.clip_actions = c.clip_actions; d.clip_obs = c.clip_obs;
    d.thrust_rate = c.thrust_rate; d.thrust_max = c.thrust_max;
    d.die_dist = c.die_dist; d.die_z = c.die_z; d.up_coef = c.up_coef;
    for (int j = 0; j < 3; ++j) {
        d.spawn_base[j] = c.spawn_base[j]; d.spawn_lo[j] = c.spawn_lo[j]; d.spawn_range[j] = c.spawn_range[j];
        d.target_scale[j] = c.target_scale[j]; d.target_off[j] = c.target_off[j];
    }
    d.mass = c.mass; d.ixx = c.ixx; d.iyy = c.iyy; d.izz = c.izz; d.arm = c.arm; d.com_z = c.com_z;
    d.max_angvel = c.max_angvel;
    d.max_angvel2 = (float)((double)c.max_angvel * (double)c.max_angvel);
    d.lin_drag = c.lin_drag; d.yaw_km = c.yaw_km; d.gravity_z = c.gravity_z;
    const double h = (double)c.dt / (double)c.substeps;
    d.h = (float)h;
    d.hh = (float)(0.5 * h);
    d.hh2 = d.hh * d.hh;
    d.fault_eff_lo = c.fault_eff_lo; d.fault_eff_range = c.fault_eff_range;
    d.land_cutoff = c.land_cutoff;
    d.plate_enable = c.plate_enable; d.plate_z = c.plate_z;
    d.plate_r2 = (float)((double)c.plate_radius * (double)c.plate_radius);
    d.wrench_warmup_steps = c.wrench_warmup_steps;
    const float nominal[OZL_DR_NUM] = {c.mass, c.ixx, c.iyy, c.izz, c.arm, 1.0f, c.yaw_km};
    for (int j = 0; j < OZL_DR_NUM; ++j) {
        const ozl_dr_param& s = c.dr[j];
        DrSpec& o = d.dr[j];
        o.dist = s.distribution; o.op = s.operation; o.sched = s.schedule; o.sched_steps = s.schedule_steps;
        o.a = s.range[0]; o.b = s.range[1]; o.nominal = nominal[j];
        o.inv_steps = s.schedule_steps > 0 ? 1.0f / (float)s.schedule_steps : 0.0f;          // "1 / sched_step * min(...)"  dr_utils.py:85
        if (s.distribution == OZL_DR_GAUSSIAN) d.dr_any_gauss = 1;
    }
    d.flicker_p = (c.pomdp_mode == OZL_POMDP_FLICKER_NOISE) ? 0.1f : c.pomdp_prob;      // POMDP.py:16-18
    const float lo = (float)(1.0 - (double)c.noise_sigma), hi = (float)(1.0 + (double)c.noise_sigma);
    d.noise_lo = lo;
    d.noise_range = hi - lo;
    d.inv3 = 1.0f / 3.0f;
    d.half = 1.0f / 2.0f;
    d.inv_pi = 1.0f / (float)M_PI;
    {   // n % d == n - ((n * magic) >> shift) * d for all 0 <= n < 2^31  (magic = ceil(2^(31+l) / d), l = ceil(log2 d))
        const uint32_t dd = (uint32_t)c.target_period;
        uint32_t l = 0;
        while ((1ull << l) < dd) ++l;
        d.period_shift = 31 + l;
        d.period_magic = (uint32_t)(((1ull << (31 + l)) + dd - 1) / dd);
    }
    {   // step counter (step_counter.cuh): one work unit per 128-env tile, padded to a power of two per step
        const uint64_t tiles = ((uint64_t)c.num_envs + kTile - 1) / kTile;
        uint32_t l = 0;
        while ((1ull << l) < tiles) ++l;
        d.step_shift = l;
        d.step_pad = (uint32_t)((1ull << l) - tiles);
    }
    d.sinc_c1 = (float)(-1.0 / 6.0); d.sinc_c2 = (float)(1.0 / 120.0);
    d.cos_c1 = -0.5f; d.cos_c2 = (float)(1.0 / 24.0); d.cos_c3 = (float)(-1.0 / 720.0);
}

extern "C" int ozl_abi_version(void) { return OZL_ABI_VERSION; }
extern "C" int ozl_cfg_size(void) { return (int)sizeof(ozl_cfg); }
extern "C" const char* ozl_last_error(void) { return g_err; }

extern "C" int ozl_cfg_default(ozl_cfg* c, int64_t num_envs) {
    if (!c) return set_error("ozl_cfg_default: cfg is NULL");
    memset(c, 0, sizeof(*c));
    c->abi_version = OZL_ABI_VERSION;
    c->num_envs = num_envs;
    c->max_episode_length = 2000;
    c->target_period = 500;
    c->substeps = 2;
    c->control_freq_inv = 1;
    c->dt = 0.01f;
    c->gravity_z = -9.81f;
    c->clip_actions = 1.0f; c->clip_obs = 5.0f;
    c->thrust_rate = (float)(0.01 * 2000); c->thrust_max = 2000.0f;
    c->die_dist = 8.0f; c->die_z = 0.5f; c->up_coef = 5.0f;
    const float sb[3] = {0.f, 0.f, 1.f}, sl[3] = {-1.5f, -1.5f, -0.2f};
    const float sr[3] = {(float)(1.5 - (-1.5)), (float)(1.5 - (-1.5)), (float)(1.5 - (-0.2))};
    const float ts[3] = {10.f, 10.f, 1.f}, to[3] = {-5.f, -5.f, 1.f};
    for (int j = 0; j < 3; ++j) {
        c->spawn_base[j] = sb[j]; c->spawn_lo[j] = sl[j]; c->spawn_range[j] = sr[j];
        c->target_scale[j] = ts[j]; c->target_off[j] = to[j];
    }
    // composite x500 body, derived from assets/x500/x500.urdf (see ouzelum_b200/x500.py for the derivation)
    const double m_b = 2.0, m_r = 0.016076923076923075, rz = 0.3, arm = 0.174;
    const double ib[3] = {0.02166666666666667, 0.02166666666666667, 0.04000000000000001};
    const double ir[3] = {3.8464910483993325e-07, 2.6115851691700804e-05, 2.649858234714004e-05};
    const double M = m_b + 4.0 * m_r, cz = 4.0 * m_r * rz / M, dz = rz - cz, irxy = 0.5 * (ir[0] + ir[1]);
    c->mass = (float)M;
    c->com_z = (float)cz;
    c->ixx = (float)(ib[0] + m_b * cz * cz + 4.0 * (irxy + m_r * (arm * arm + dz * dz)));
    c->iyy = (float)(ib[1] + m_b * cz * cz + 4.0 * (irxy + m_r * (arm * arm + dz * dz)));
    c->izz = (float)(ib[2] + 4.0 * (ir[2] + m_r * (2.0 * arm * arm)));
    c->arm = (float)arm;
    c->max_angvel = (float)(4.0 * M_PI);
    c->fault_eff_lo = 0.0f; c->fault_eff_range = 0.5f;
    for (int j = 0; j < OZL_DR_NUM; ++j) {       // isaacgymenvs/utils/dr_utils.py:121-130 (scaling, uniform); yaw_km: not randomised
        c->dr[j].distribution = j == OZL_DR_YAW_KM ? OZL_DR_NONE : OZL_DR_UNIFORM;
        c->dr[j].operation = OZL_DR_SCALING;
        c->dr[j].range[0] = 0.8f; c->dr[j].range[1] = 1.2f;
        c->dr[j].schedule = OZL_DR_SCHED_NONE; c->dr[j].schedule_steps = 0;
    }
    c->collect_metrics = 1;
    c->plate_enable = 0; c->plate_z = 0.377f; c->plate_radius = 0.35f; c->land_cutoff = 0.0f;
    return 0;
}

// ------------------------------------------------------------------------------------------------ host: lifecycle
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

extern "C" int ozl_create(const ozl_cfg* cfg, int device, ozl_env** out) {
    if (!cfg || !out) return set_error("ozl_create: NULL argument");
    if (cfg->abi_version != OZL_ABI_VERSION)
        return set_error("ozl_create: cfg.abi_version %d != library %d", cfg->abi_version, OZL_ABI_VERSION);
    if (cfg->num_envs <= 0 || cfg->num_envs > 0x7FFFFFFFll) return set_error("ozl_create: num_envs out of range");
    if (cfg->substeps <= 0 || cfg->control_freq_inv <= 0) return set_error("ozl_create: substeps/control_freq_inv must be > 0");
    if (cfg->max_episode_length <= 1 || cfg->max_episode_length >= (1 << 28))
        return set_error("ozl_create: max_episode_length out of range");
    if (cfg->target_period <= 0) return set_error("ozl_create: target_period must be > 0");
    if (cfg->pomdp_mode < 0 || cfg->pomdp_mode > 3) return set_error("ozl_create: unknown pomdp_mode %d", cfg->pomdp_mode);
    if (!(cfg->mass > 1e-30f && cfg->mass < 1e30f) || !(cfg->ixx > 1e-30f && cfg->ixx < 1e30f) ||
        !(cfg->iyy > 1e-30f && cfg->iyy < 1e30f) || !(cfg->izz > 1e-30f && cfg->izz < 1e30f))
        return set_error("ozl_create: mass and inertia must be positive normal floats");
    if (cfg->wrench_warmup_steps < 0) return set_error("ozl_create: wrench_warmup_steps must be >= 0");
    for (int j = 0; j < OZL_DR_NUM; ++j) {
        const ozl_dr_param& d = cfg->dr[j];
        if (d.distribution < OZL_DR_NONE || d.distribution > OZL_DR_GAUSSIAN) return set_error("ozl_create: dr[%d].distribution %d unknown", j, d.distribution);
        if (d.operation != OZL_DR_SCALING && d.operation != OZL_DR_ADDITIVE) return set_error("ozl_create: dr[%d].operation %d unknown", j, d.operation);
        if (d.schedule < OZL_DR_SCHED_NONE || d.schedule > OZL_DR_SCHED_CONSTANT) return set_error("ozl_create: dr[%d].schedule %d unknown", j, d.schedule);
        if (d.schedule != OZL_DR_SCHED_NONE && d.schedule_steps <= 0) return set_error("ozl_create: dr[%d].schedule_steps must be > 0", j);
        if (d.distribution == OZL_DR_LOGUNIFORM && !(d.range[0] > 0.f && d.range[1] > 0.f))
            return set_error("ozl_create: dr[%d]: loguniform needs a positive range", j);
    }
    int ndev = 0;
    if (check_cuda(cudaGetDeviceCount(&ndev), "cudaGetDeviceCount")) return 1;
    if (device < 0 || device >= ndev) return set_error("ozl_create: device %d not available (%d visible)", device, ndev);
    if (check_cuda(cudaSetDevice(device), "cudaSetDevice")) return 1;
    cudaDeviceProp prop;
    if (check_cuda(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties")) return 1;
    if (prop.major != 10)
        return set_error("ozl_create: this library is built for sm_100a (B200) only; device %d is sm_%d%d", device, prop.major, prop.minor);

    ozl_env* e = new ozl_env();
    e->cfg = *cfg;
    e->states = nullptr;
    memset(e->states_tmap, 0, sizeof(e->states_tmap));
    e->scn_buf = e->scn = nullptr;
    derive_dev_cfg(*cfg, e->dev);
    e->device = device;
    e->sm_count = prop.multiProcessorCount;
    {   // switch to the persistent TMA-pipelined kernel as soon as the generic kernel would need a second wave of CTAs (7 x 128-env
        // CTAs per SM are resident: 1036 tiles = 132608 envs on 148 SMs).
        // Measured on B200 with the round-2 kernels (profiles/r02at_sizes_*.jsonl; us per step, generic vs TMA):
        //   131072 envs  warm 8.09 vs 8.86, cold  9.78 vs  9.68      196608  warm 11.47 vs 11.16, cold 15.21 vs 11.98
        //   262144 envs  warm 13.7 vs 13.6, cold 18.33 vs 15.21      393216  warm 19.92 vs 18.38, cold 24.83 vs 21.96
        //   163840 envs (1280 tiles, a second generic wave of 244 CTAs): generic warm 10.29, cold 13.51; 180224 envs on the TMA kernel 10.34 / 11.16
        // (round 1's kernels crossed over at ~400k envs; the lighter integrator moved the crossover down)
        // (override: OZL_TMA_MIN_TILES, 0 = never)
        const char* ev = getenv("OZL_TMA_MIN_TILES");
        e->tma_min_tiles = ev ? atoll(ev) : (long long)kStepMinBlocks * prop.multiProcessorCount + 1;
    }
    const size_t n = (size_t)cfg->num_envs;
    const size_t tiles = (n + kTile - 1) / kTile;
    const size_t state = align_up(tiles * (size_t)kTileBytes, 256);
    const size_t ctrl = 256, metrics = align_up(sizeof(double) * kMetricSlots * kMetricStride, 256);
    const size_t tile_seq = align_up(tiles * 4 * sizeof(unsigned long long), 256);    // {started, done} per CTA of >= 64 envs
    e->arena_bytes = state + ctrl + metrics + tile_seq;
    if (check_cuda(cudaMalloc(&e->arena, e->arena_bytes), "cudaMalloc(state arena)")) { delete e; return 1; }
    if (check_cuda(cudaMemset(e->arena, 0, e->arena_bytes), "cudaMemset(state arena)")) { cudaFree(e->arena); delete e; return 1; }
    char* p = (char*)e->arena;
    e->pl.base = p;
    p += state;
    e->pl.ctrl = (unsigned long long*)p; p += ctrl;
    e->pl.metrics = (double*)p; p += metrics;
    e->pl.tile_seq = (unsigned long long*)p;
    {
        const char* cv = getenv("OZL_EKF_CHAIN");
        e->chain_mode = cv ? atoi(cv) : 1;
        e->chain_capture_id = 0;
        e->chain_last_node = nullptr;
        e->pv_tmap_ptr = nullptr;
    }
    {
        e->host_done = nullptr;
        e->host_seq = 0;
        void* hp = nullptr;
        if (cudaHostAlloc(&hp, 64, cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess) {
            memset(hp, 0, 64);
            e->host_done = (volatile unsigned int*)hp;
        } else {
            cudaGetLastError();        // no pinned word: host steps fall back to cudaStreamSynchronize
        }
    }
    *out = e;
    return ozl_reset_all(e, cfg->seed, nullptr);
}

extern "C" int ozl_destroy(ozl_env* env) {
    if (!env) return 0;
    cudaSetDevice(env->device);
    cudaFree(env->arena);
    if (env->scn_buf) cudaFree(env->scn_buf);
    if (env->host_done) cudaFreeHost((void*)env->host_done);
    delete env;
    return 0;
}

static inline unsigned blocks_for(int64_t n, int b) { return (unsigned)((n + b - 1) / b); }
#define OZL_ENV_CHECK(name)                                        \
    if (!env) return set_error(name ": env is NULL");              \
    cudaStream_t st = (cudaStream_t)stream;

extern "C" int ozl_reset_all(ozl_env* env, uint64_t seed, void* stream) {
    OZL_ENV_CHECK("ozl_reset_all");
    env->cfg.seed = seed;
    env->dev.seed = seed;
    int64_t n = env->cfg.num_envs;
    if (n < kMetricSlots * kMetricStride) n = kMetricSlots * kMetricStride;
    init_state_kernel<<<blocks_for(n, 256), 256, 0, st>>>(env->dev, env->pl);
    return check_cuda(cudaGetLastError(), "init_state_kernel");
}

// Block size: 128 threads keeps >= 1 block on every SM down to ~19k envs and lets 16k-env launches use 128 SMs.
constexpr int kStepBlock = 128;
static_assert(kStepBlock == kTile, "the step counter retires one work unit per 128-env tile == one block of the generic kernel");

// The states tensor map of the handle (zeros while no states buffer is registered: the STATES = false kernels never read it)
static inline const CUtensorMap& states_map(const ozl_env* env) { return *reinterpret_cast<const CUtensorMap*>(env->states_tmap); }

template <bool STATES, bool SCN>
static int launch_step_t(ozl_env* env, const float* actions, const float* target_in, int act_mode, float* obs, float* rew,
                         int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream, const char* who,
                         uint8_t* done_u8, int obs_bulk, int64_t* reset_mirror, int host_flag) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!actions || !obs || !rew || !reset || !progress) return set_error("%s: NULL buffer", who);
    if (((uintptr_t)actions & 15) || ((uintptr_t)obs & 15)) return set_error("%s: actions/obs must be 16-byte aligned", who);
    const int64_t n = env->cfg.num_envs;
    const int64_t full_tiles = n / kTile, tail = n % kTile;
    const int64_t resident = (int64_t)env->sm_count * kTmaMinBlocks;
    const bool plain = (target_in == nullptr) && act_mode == ACT_ROTORS && done_u8 == nullptr && reset_mirror == nullptr && obs_bulk;
    const auto tma_kernel = SCN ? quad_step_tma_scn_kernel<STATES> : quad_step_tma_kernel<STATES>;
    const auto kernel = SCN ? quad_step_scn_kernel<kStepBlock, FRONT_NONE, STATES> : quad_step_kernel<kStepBlock, FRONT_NONE, STATES>;
    if (plain && env->tma_min_tiles > 0 && full_tiles >= env->tma_min_tiles &&
        !(((uintptr_t)progress | (uintptr_t)reset) & 15)) {
        // large N: persistent TMA-pipelined kernel over the whole tiles, then one generic block for the ragged tail
        unsigned grid = (unsigned)(full_tiles < resident ? full_tiles : resident);
        while ((full_tiles + grid - 1) / grid > 8192) grid *= 2;     // 16-bit packed metric counters: keep tiles per CTA far below 65535
        if (launch_pdl(tma_kernel, dim3(grid), dim3(kTile), st, env->dev, env->pl, (const float4*)actions, obs, rew,
                       reset, progress, timeout, ep_ret, full_tiles, states_map(env), (const float*)env->scn))
            return check_cuda(cudaGetLastError(), "quad_step_tma_kernel");
        if (tail)
            kernel<<<1, kStepBlock, 0, st>>>(env->dev, env->pl, (const float4*)actions, obs, rew, reset, progress, timeout, ep_ret, nullptr,
                                             ACT_ROTORS, nullptr, nullptr, 1, full_tiles * kTile, FrontArgs{},
                                             (volatile unsigned int*)nullptr, 0u, states_map(env), (const float*)env->scn);
        return check_cuda(cudaGetLastError(), "quad_step_kernel(tail)");
    }
    if (launch_pdl(kernel, dim3(blocks_for(n, kStepBlock)), dim3(kStepBlock), st, env->dev,
                   env->pl, (const float4*)actions, obs, rew, reset, progress, timeout, ep_ret, target_in, act_mode, done_u8, reset_mirror,
                   obs_bulk, (int64_t)0, FrontArgs{}, (volatile unsigned int*)(host_flag ? env->host_done : nullptr),
                   host_flag ? ++env->host_seq : 0u, states_map(env), (const float*)env->scn))
        return check_cuda(cudaGetLastError(), "quad_step_kernel");
    return 0;
}

// The kernels with the states output run whenever the handle has a states buffer registered, the scenario kernels whenever it
// has a scenario table registered.
static int launch_step(ozl_env* env, const float* actions, const float* target_in, int act_mode, float* obs, float* rew,
                       int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream, const char* who,
                       uint8_t* done_u8 = nullptr, int obs_bulk = 1, int64_t* reset_mirror = nullptr, int host_flag = 0) {
    if (!env) return set_error("%s: env is NULL", who);
    auto* f = env->states ? (env->scn ? launch_step_t<true, true> : launch_step_t<true, false>)
                          : (env->scn ? launch_step_t<false, true> : launch_step_t<false, false>);
    return f(env, actions, target_in, act_mode, obs, rew, reset, progress, timeout, ep_ret, stream, who, done_u8, obs_bulk, reset_mirror,
             host_flag);
}

// Landing-family steps with the vehicle (and, for LeeLanded, the controller) in the same launch.
static int launch_front_step(ozl_env* env, int front, const float* actions, const ozl_husky_args* husky, const FrontArgs& fa_in,
                             float* obs, float* rew, int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream,
                             const char* who) {
    if (!env) return set_error("%s: env is NULL", who);
    if (!husky) return set_error("%s: husky args are NULL", who);
    if (!obs || !rew || !reset || !progress || (front == FRONT_VEHICLE && !actions)) return set_error("%s: NULL buffer", who);
    if (((uintptr_t)actions & 15) || ((uintptr_t)obs & 15)) return set_error("%s: actions/obs must be 16-byte aligned", who);
    FrontArgs fa = fa_in;
    if (ozl_fill_husky_args(husky, fa.h, who)) return 1;
    if (!fa.h.tables) return set_error("%s: tables204x2 is NULL", who);
    if (fa.h.n != env->cfg.num_envs) return set_error("%s: vehicle count %lld != env count %lld", who, (long long)fa.h.n, (long long)env->cfg.num_envs);
    if (fa.h.reset && fa.h.reset != reset) return set_error("%s: the vehicle and the step must see the same reset buffer", who);
    fa.h.reset = reset;
    fa.h.step_ptr = env->pl.ctrl;            // the vehicle follows the handle's device step counter (graph-capturable)
    const int64_t n = env->cfg.num_envs;
    cudaStream_t st = (cudaStream_t)stream;
#define OZL_LAUNCH_FRONT(F, S, MODE)                                                                                            \
    launch_pdl(env->scn ? quad_step_scn_kernel<kStepBlock, F, S> : quad_step_kernel<kStepBlock, F, S>, dim3(blocks_for(n, kStepBlock)), \
               dim3(kStepBlock), st, env->dev, env->pl, (const float4*)actions, obs, rew, reset, progress, timeout, ep_ret,          \
               (const float*)nullptr, (int)MODE, (uint8_t*)nullptr, (int64_t*)nullptr, 1, (int64_t)0, fa,                           \
               (volatile unsigned int*)nullptr, 0u, states_map(env), (const float*)env->scn)
    int rc;
    if (front == FRONT_VEHICLE)
        rc = env->states ? OZL_LAUNCH_FRONT(FRONT_VEHICLE, true, ACT_ROTORS) : OZL_LAUNCH_FRONT(FRONT_VEHICLE, false, ACT_ROTORS);
    else
        rc = env->states ? OZL_LAUNCH_FRONT(FRONT_LEE, true, ACT_WRENCH) : OZL_LAUNCH_FRONT(FRONT_LEE, false, ACT_WRENCH);
#undef OZL_LAUNCH_FRONT
    if (rc) return check_cuda(cudaGetLastError(), who);
    return 0;
}

extern "C" int ozl_landing_step(ozl_env* env, const float* actions, const ozl_husky_args* husky, float* obs, float* rew,
                                int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream) {
    return launch_front_step(env, FRONT_VEHICLE, actions, husky, FrontArgs{}, obs, rew, reset, progress, timeout, ep_ret, stream,
                             "ozl_landing_step");
}

extern "C" int ozl_lee_landed_step(ozl_env* env, const ozl_lee_landed_args* in, const ozl_husky_args* husky, float* obs, float* rew,
                                   int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream) {
    if (!in || !in->gains16) return set_error("ozl_lee_landed_step: NULL argument");
    if ((uintptr_t)in->wrench4 & 15) return set_error("ozl_lee_landed_step: wrench4 must be 16-byte aligned");
    FrontArgs fa{};
    for (int k = 0; k < 3; ++k) { fa.g.kP[k] = in->gains16[k]; fa.g.kV[k] = in->gains16[3 + k]; fa.g.kR[k] = in->gains16[6 + k]; fa.g.kO[k] = in->gains16[9 + k]; }
    for (int k = 0; k < 4; ++k) { fa.g.scale[k] = in->gains16[12 + k]; fa.cmd[k] = in->cmd[k]; }
    fa.mg = in->mg;
    fa.wrench_out = (float4*)in->wrench4;
    return launch_front_step(env, FRONT_LEE, nullptr, husky, fa, obs, rew, reset, progress, timeout, ep_ret, stream, "ozl_lee_landed_step");
}

extern "C" int ozl_step(ozl_env* env, const float* actions, float* obs, float* rew, int64_t* reset, int64_t* progress,
                        uint8_t* timeout, float* ep_ret, void* stream) {
    return launch_step(env, actions, nullptr, ACT_ROTORS, obs, rew, reset, progress, timeout, ep_ret, stream, "ozl_step");
}

static int step_host_impl(ozl_env* env, const float* actions_host, float* obs_host, float* rew_host, uint8_t* done_host,
                          int64_t* reset_host, int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream) {
    if (!done_host) return set_error("ozl_step_host: done_host is NULL");
    // host-mapped (pinned, UVA) buffers: plain coalesced stores over PCIe instead of the TMA bulk store (measured equal)
    return launch_step(env, actions_host, nullptr, ACT_ROTORS, obs_host, rew_host, reset, progress, timeout, ep_ret, stream,
                       "ozl_step_host", done_host, 0, reset_host, env && env->host_done);
}

// Wait for the last host step: poll the completion word (see quad_step_kernel); if it does not flip within ~2 s -- or the handle
// has no word because cudaHostAlloc failed -- synchronise the stream, which also surfaces any CUDA error.
static int host_step_wait(ozl_env* env, void* stream) {
    if (env->host_done) {
        const unsigned int want = env->host_seq;
        for (long spins = 0; spins < 400000000L; ++spins) {
            if (*env->host_done == want) { __atomic_thread_fence(__ATOMIC_ACQUIRE); return 0; }
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
    }
    return check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "cudaStreamSynchronize");
}
extern "C" int ozl_step_host(ozl_env* env, const float* actions_host, float* obs_host, float* rew_host, uint8_t* done_host,
                             int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream) {
    return step_host_impl(env, actions_host, obs_host, rew_host, done_host, nullptr, reset, progress, timeout, ep_ret, stream);
}

extern "C" int ozl_step_host_launch(ozl_env* env, const ozl_host_io* io, void* stream) {
    if (!io) return set_error("ozl_step_host_launch: io is NULL");
    return step_host_impl(env, io->actions_host, io->obs_host, io->rew_host, io->done_host, io->reset_host, io->reset, io->progress,
                          io->timeout, io->ep_ret, stream);
}

extern "C" int ozl_step_host_sync(ozl_env* env, const ozl_host_io* io, void* stream) {
    if (!io) return set_error("ozl_step_host_sync: io is NULL");
    if (ozl_step_host_launch(env, io, stream)) return 1;
    return host_step_wait(env, stream);
}

extern "C" int ozl_step_host_wait(ozl_env* env, void* stream) {
    if (!env) return set_error("ozl_step_host_wait: env is NULL");
    return host_step_wait(env, stream);
}

extern "C" int ozl_stream_sync(void* stream) {
    return check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "cudaStreamSynchronize");
}

extern "C" int ozl_step_tracking(ozl_env* env, const float* actions, const float* target3, float* obs, float* rew,
                                 int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream) {
    if (!target3) return set_error("ozl_step_tracking: target3 is NULL");
    return launch_step(env, actions, target3, ACT_ROTORS, obs, rew, reset, progress, timeout, ep_ret, stream, "ozl_step_tracking");
}

extern "C" int ozl_step_wrench(ozl_env* env, const float* wrench4, const float* target3, float* obs, float* rew,
                               int64_t* reset, int64_t* progress, uint8_t* timeout, float* ep_ret, void* stream) {
    return launch_step(env, wrench4, target3, ACT_WRENCH, obs, rew, reset, progress, timeout, ep_ret, stream, "ozl_step_wrench");
}

extern "C" int ozl_apply_resets(ozl_env* env, const int64_t* reset, void* stream) {
    OZL_ENV_CHECK("ozl_apply_resets");
    if (!reset) return set_error("ozl_apply_resets: reset is NULL");
    apply_resets_kernel<<<blocks_for(env->cfg.num_envs, 256), 256, 0, st>>>(env->dev, env->pl, reset, env->scn);
    return check_cuda(cudaGetLastError(), "apply_resets_kernel");
}

extern "C" int ozl_rollout(ozl_env* env, int32_t K, float* obs, float* rew, int64_t* reset, int64_t* progress, void* stream) {
    OZL_ENV_CHECK("ozl_rollout");
    if (K <= 0) return set_error("ozl_rollout: K must be > 0");
    if (env->states) return set_error("ozl_rollout: a states output is registered (ozl_set_states_output) and the K-step kernel does not write it");
    if (env->scn) return set_error("ozl_rollout: a scenario table is registered (ozl_set_scenarios) and the K-step kernel does not apply it");
    if (!obs || !rew || !reset || !progress) return set_error("ozl_rollout: NULL buffer");
    quad_rollout_kernel<kStepBlock><<<blocks_for(env->cfg.num_envs, kStepBlock), kStepBlock, 0, st>>>(
        env->dev, env->pl, K, obs, rew, reset, progress);
    if (check_cuda(cudaGetLastError(), "quad_rollout_kernel")) return 1;
    if (K > 1) add_steps_kernel<<<1, 1, 0, st>>>(env->pl, (unsigned long long)(K - 1));
    return check_cuda(cudaGetLastError(), "add_steps_kernel");
}

extern "C" int ozl_set_states_output(ozl_env* env, float* states, int32_t width) {
    if (!env) return set_error("ozl_set_states_output: env is NULL");
    if (width != OZL_STATES_WIDTH)
        return set_error("ozl_set_states_output: width %d != OZL_STATES_WIDTH (%d)", (int)width, (int)OZL_STATES_WIDTH);
    if (!states) {
        env->states = nullptr;
        memset(env->states_tmap, 0, sizeof(env->states_tmap));
        return 0;
    }
    if ((uintptr_t)states & 15) return set_error("ozl_set_states_output: states must be 16-byte aligned");
    const PFN_cuTensorMapEncodeTiled fn = tensor_map_encoder();
    if (!fn) return set_error("ozl_set_states_output: cuTensorMapEncodeTiled is not available from the driver");
    // [N][32] f32 rows of 128 bytes; box = one 128-env tile, 128-byte swizzle (stage_states_row writes the tile in that layout)
    const cuuint64_t gdim[2] = {(cuuint64_t)OZL_STATES_WIDTH, (cuuint64_t)env->cfg.num_envs};
    const cuuint64_t gstr[1] = {(cuuint64_t)OZL_STATES_WIDTH * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)OZL_STATES_WIDTH, (cuuint32_t)kTile};
    const cuuint32_t estr[2] = {1u, 1u};
    alignas(64) unsigned char m[sizeof(env->states_tmap)];
    const CUresult r = fn(reinterpret_cast<CUtensorMap*>(m), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, states, gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error("ozl_set_states_output: cuTensorMapEncodeTiled failed (%d)", (int)r);
    memcpy(env->states_tmap, m, sizeof(m));
    env->states = states;
    return 0;
}

// One scenario row against the rules of ozl_set_scenarios (include/ouzelum_b200.h); 0 = valid.
static int check_scenario_row(const ozl_cfg& cfg, const float* r, int64_t row) {
    static const struct { int first, count; const char* name; } groups[] = {
        {OZL_SCN_POS, 3, "position"}, {OZL_SCN_QUAT, 4, "attitude"}, {OZL_SCN_LINVEL, 3, "linear velocity"},
        {OZL_SCN_ANGVEL, 3, "angular velocity"}, {OZL_SCN_TARGET, 3, "target"}, {OZL_SCN_FAULT_ROTOR, 3, "fault"},
        {OZL_SCN_MASS, 1, "mass"}, {OZL_SCN_IXX, 1, "ixx"}, {OZL_SCN_IYY, 1, "iyy"}, {OZL_SCN_IZZ, 1, "izz"}, {OZL_SCN_ARM, 1, "arm"},
        {OZL_SCN_THRUST_SCALE, 1, "thrust_scale"}, {OZL_SCN_YAW_KM, 1, "yaw_km"}};
    const char* who = "ozl_set_scenarios";
    const long long k = (long long)row;
    for (int j = OZL_SCN_RESERVED; j < OZL_SCENARIO_WIDTH; ++j)
        if (!std::isnan(r[j])) return set_error("%s: row %lld: reserved slot %d must be NaN", who, k, j);
    for (const auto& g : groups) {
        int nan = 0;
        for (int j = g.first; j < g.first + g.count; ++j) {
            if (std::isnan(r[j])) ++nan;
            else if (!std::isfinite(r[j])) return set_error("%s: row %lld: %s group has a non-finite value in slot %d", who, k, g.name, j);
        }
        if (nan != 0 && nan != g.count) return set_error("%s: row %lld: %s group must be all NaN or all set", who, k, g.name);
    }
    const auto set = [&](int slot) { return !std::isnan(r[slot]); };
    if (set(OZL_SCN_QUAT)) {
        const double x = r[OZL_SCN_QUAT], y = r[OZL_SCN_QUAT + 1], z = r[OZL_SCN_QUAT + 2], w = r[OZL_SCN_QUAT + 3];
        if (!(std::fabs(x * x + y * y + z * z + w * w - 1.0) <= 1e-6))
            return set_error("%s: row %lld: attitude quaternion is not unit (|q|^2 - 1 must be within 1e-6)", who, k);
    }
    if (set(OZL_SCN_TARGET) && cfg.target_fixed)
        return set_error("%s: row %lld: target group set, but cfg.target_fixed is set (the target is driven by a vehicle or the caller)", who, k);
    if (set(OZL_SCN_FAULT_ROTOR)) {
        if (!cfg.fault_mode)
            return set_error("%s: row %lld: fault group set, but the handle has no rotor-fault model (cfg.fault_mode, rotorFault.enable)", who, k);
        const float rotor = r[OZL_SCN_FAULT_ROTOR], onset = r[OZL_SCN_FAULT_ONSET], eff = r[OZL_SCN_FAULT_EFF];
        if (!(rotor == -1.0f || rotor == 0.0f || rotor == 1.0f || rotor == 2.0f || rotor == 3.0f))
            return set_error("%s: row %lld: fault rotor %g is not one of -1, 0, 1, 2, 3", who, k, (double)rotor);
        if (!(onset >= 0.0f && onset < 16777216.0f && onset == std::floor(onset)))
            return set_error("%s: row %lld: fault onset %g is not an integer in [0, 2^24)", who, k, (double)onset);
        if (!(eff >= 0.0f && eff <= 1.0f)) return set_error("%s: row %lld: fault effectiveness %g is not in [0, 1]", who, k, (double)eff);
    }
    for (int j = OZL_SCN_MASS; j <= OZL_SCN_IZZ; ++j)
        if (set(j) && !(r[j] > 1e-30f && r[j] < 1e30f))
            return set_error("%s: row %lld: slot %d (mass / inertia) must be a positive normal float in (1e-30, 1e30)", who, k, j);
    if (set(OZL_SCN_ARM) && !(r[OZL_SCN_ARM] > 0.0f)) return set_error("%s: row %lld: arm must be > 0", who, k);
    if (set(OZL_SCN_THRUST_SCALE) && !(r[OZL_SCN_THRUST_SCALE] >= 0.0f)) return set_error("%s: row %lld: thrust_scale must be >= 0", who, k);
    return 0;
}

extern "C" int ozl_set_scenarios(ozl_env* env, const float* rows_host, int32_t width, void* stream) {
    OZL_ENV_CHECK("ozl_set_scenarios");
    if (width != OZL_SCENARIO_WIDTH)
        return set_error("ozl_set_scenarios: width %d != OZL_SCENARIO_WIDTH (%d)", (int)width, (int)OZL_SCENARIO_WIDTH);
    if (!rows_host) {
        env->scn = nullptr;
        return 0;
    }
    const int64_t n = env->cfg.num_envs;
    for (int64_t i = 0; i < n; ++i)
        if (check_scenario_row(env->cfg, rows_host + i * OZL_SCENARIO_WIDTH, i)) return 1;
    const size_t bytes = (size_t)n * OZL_SCENARIO_WIDTH * sizeof(float);
    if (!env->scn_buf && check_cuda(cudaMalloc(&env->scn_buf, bytes), "cudaMalloc(scenario table)")) {
        env->scn_buf = nullptr;
        return 1;
    }
    // stream-ordered behind any launch that still reads the old rows; synchronised so that the caller may free rows_host
    if (check_cuda(cudaMemcpyAsync(env->scn_buf, rows_host, bytes, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(scenario table)")) return 1;
    if (check_cuda(cudaStreamSynchronize(st), "cudaStreamSynchronize")) return 1;
    env->scn = env->scn_buf;
    return 0;
}

extern "C" int ozl_get_state(ozl_env* env, float* root13, float* thrust4, float* target3, float* ep_ret, void* stream) {
    OZL_ENV_CHECK("ozl_get_state");
    get_state_kernel<<<blocks_for(env->cfg.num_envs, 256), 256, 0, st>>>(env->pl, env->cfg.num_envs, root13, thrust4, target3, ep_ret);
    return check_cuda(cudaGetLastError(), "get_state_kernel");
}
extern "C" int ozl_set_state(ozl_env* env, const float* root13, const float* thrust4, const float* target3,
                             const float* ep_ret, void* stream) {
    OZL_ENV_CHECK("ozl_set_state");
    set_state_kernel<<<blocks_for(env->cfg.num_envs, 256), 256, 0, st>>>(env->pl, env->cfg.num_envs, root13, thrust4, target3, ep_ret);
    return check_cuda(cudaGetLastError(), "set_state_kernel");
}
extern "C" int ozl_get_params(ozl_env* env, float* params8, int32_t* fault2, void* stream) {
    OZL_ENV_CHECK("ozl_get_params");
    get_params_kernel<<<blocks_for(env->cfg.num_envs, 256), 256, 0, st>>>(env->pl, env->cfg.num_envs, params8, fault2);
    return check_cuda(cudaGetLastError(), "get_params_kernel");
}
extern "C" int ozl_set_params(ozl_env* env, const float* params8, const int32_t* fault2, void* stream) {
    OZL_ENV_CHECK("ozl_set_params");
    set_params_kernel<<<blocks_for(env->cfg.num_envs, 256), 256, 0, st>>>(env->pl, env->cfg.num_envs, params8, fault2);
    return check_cuda(cudaGetLastError(), "set_params_kernel");
}

extern "C" int ozl_get_step_count(ozl_env* env, uint64_t* out, void* stream) {
    OZL_ENV_CHECK("ozl_get_step_count");
    if (!out) return set_error("ozl_get_step_count: out is NULL");
    unsigned long long w[2] = {0, 0};
    if (check_cuda(cudaMemcpyAsync(w, env->pl.ctrl, sizeof(w), cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync")) return 1;
    if (check_cuda(cudaStreamSynchronize(st), "cudaStreamSynchronize")) return 1;
    *out = step_from_words(w);
    return 0;
}
extern "C" int ozl_set_step_count(ozl_env* env, uint64_t value, void* stream) {
    OZL_ENV_CHECK("ozl_set_step_count");
    if (value > kStepBaseMask) return set_error("ozl_set_step_count: value out of range");
    set_step_kernel<<<1, 1, 0, st>>>(env->pl, step_word0((unsigned long long)value, env->dev.step_shift));
    return check_cuda(cudaGetLastError(), "set_step_kernel");
}

extern "C" int ozl_metrics_read(ozl_env* env, double* out16, int32_t clear, void* stream) {
    OZL_ENV_CHECK("ozl_metrics_read");
    if (!out16) return set_error("ozl_metrics_read: out16 is NULL");
    if (launch_pdl(metrics_read_kernel, dim3(1), dim3(16 * 32), st, env->pl, out16, (int)clear))
        return check_cuda(cudaGetLastError(), "metrics_read_kernel");
    return 0;
}
