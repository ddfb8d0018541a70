// Batched estimators, one env per thread (kernels K2 and K3): attitude-EKF state in registers, PV covariance in shared memory.
//   K3  9-state position/velocity/accel-bias Kalman filter   CPU twin: oracle/pv_filter.py, exact twin: tests/filters_ref.c
//       reference: isaacgymenvs/PVFilter.py:25-64 (prediction_step), :67-110 (correction_step), :113-142
//   K2  4-state attitude EKF, float64                          CPU twin: oracle/ahrs_ekf.py, exact twin: tests/filters_ref.c
// The exact twin restates these functions operation for operation in C; the kernels must equal it bit for bit (any change here
// changes it too).
//       reference: isaacgymenvs/ahrs_ekf.py:1072-1158, 1280-1337 (the `ang` branch)
// The reference runs both as Python loops over envs (tasks/ekf_lee_landed.py:378-391, 417-444: N iterations of ~15 numpy
// calls / ~40 tiny CUDA launches per step).  Here one launch handles all envs; HBM traffic is the filter state once in,
// once out (SoA planes [k][N], coalesced across envs).
#pragma once
#include <math.h>

namespace ozl {

// ------------------------------------------------------------------------------------------------ K3: PV filter
// Arithmetic contract: every TU is compiled with -fmad=false; the fused multiply-adds below are explicit (fmaf), so the fused
// EKFLeeLanded kernel, the stand-alone pv_step_kernel and any other user of these functions produce IDENTICAL bits.
//
// The 9x9 covariance of the thread's env lives in SHARED memory -- element (r,c) of thread t at P[(r*9 + c) * STRIDE + t],
// conflict-free -- and the loops over columns / rows stay ROLLED (~250 instructions of loop body; the fully unrolled register
// form was ~2000 straight-line instructions at 168 registers and stalled on instruction fetch).

// quaternion_to_matrix of PVFilter.py:113-142 (normalises first), wxyz in
__device__ __forceinline__ void pv_quat_to_R(float r, float i, float j, float k, float R[3][3]) {
    const float n = sqrtf(fmaf(k, k, fmaf(j, j, fmaf(i, i, r * r))));
    r /= n; i /= n; j /= n; k /= n;
    const float two_s = 2.0f / fmaf(k, k, fmaf(j, j, fmaf(i, i, r * r)));
    R[0][0] = fmaf(-two_s, fmaf(k, k, j * j), 1.f); R[0][1] = two_s * fmaf(i, j, -(k * r)); R[0][2] = two_s * fmaf(i, k, j * r);
    R[1][0] = two_s * fmaf(i, j, k * r); R[1][1] = fmaf(-two_s, fmaf(k, k, i * i), 1.f); R[1][2] = two_s * fmaf(j, k, -(i * r));
    R[2][0] = two_s * fmaf(i, k, -(j * r)); R[2][1] = two_s * fmaf(j, k, i * r); R[2][2] = fmaf(-two_s, fmaf(j, j, i * i), 1.f);
}

#ifndef OZL_PV_UNROLL
#define OZL_PV_UNROLL 3     // unroll factor of the 9-iteration covariance loops (measured on B200, config 3: 1 -> 3: 27.1 -> 26.8 us)
#endif
#define OZL_PRAGMA_(x) _Pragma(#x)
#define OZL_PRAGMA(x) OZL_PRAGMA_(x)
#define OZL_PV_LOOP OZL_PRAGMA(unroll OZL_PV_UNROLL)

template <int STRIDE>
struct PVShared {
    float x[9];
    float* P;                              // this thread's column of the block's [81][STRIDE] covariance tile
    __device__ __forceinline__ float& at(int r, int c) { return P[(r * 9 + c) * STRIDE]; }
};

__device__ __forceinline__ float dot3(const float a0, const float a1, const float a2, const float b[3]) {
    return fmaf(a2, b[2], fmaf(a1, b[1], a0 * b[0]));
}

// prediction_step (PVFilter.py:25-64): x <- F x + G (a - b_a) ; P <- F P F^T + G diag(acc_var) G^T with the reference's
//   F = [[I, R dt, R dt^2/2], [0, R, R dt], [0, 0, I]],  G = F[:, 6:9] = [R dt^2/2; R dt; 0],  R = quaternion_to_matrix(q)^T
// (velocity block rotated every step, bias column reused as the input matrix -- the reference's quirks, reproduced).
// Evaluated through the common factor R: with rv = R p_v and rb = R p_b a column of F P is (p_p + dt rv + dt^2/2 rb,
// rv + dt rb, p_b) -- 27 instead of 36 multiply-adds per column, same for the rows of (F P) F^T; in the state update the bias
// terms of F x and G (a - b_a) cancel algebraically (G = F[:, 6:9]), leaving x_p + dt R x_v + dt^2/2 R a and R x_v + dt R a.
template <int STRIDE>
__device__ __forceinline__ void pv_predict(PVShared<STRIDE>& s, const float acc[3], const float q_wxyz[4], float dt, float dt2,
                                           const float acc_var[3]) {
    float Rq[3][3], R[3][3];
    pv_quat_to_R(q_wxyz[0], q_wxyz[1], q_wxyz[2], q_wxyz[3], Rq);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) R[i][j] = Rq[j][i];                // .T   (PVFilter.py:33-35)
    const float hdt2 = dt2 * 0.5f;
    // ---- state
    {
        const float xv[3] = {s.x[3], s.x[4], s.x[5]};
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float rv = dot3(R[i][0], R[i][1], R[i][2], xv), ra = dot3(R[i][0], R[i][1], R[i][2], acc);
            s.x[i] = fmaf(hdt2, ra, fmaf(dt, rv, s.x[i]));
            s.x[3 + i] = fmaf(dt, ra, rv);
        }
    }
    // ---- M = F P, one column per iteration
    OZL_PV_LOOP
    for (int c = 0; c < 9; ++c) {
        float pp[3], pv[3], pb[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) { pp[j] = s.at(j, c); pv[j] = s.at(3 + j, c); pb[j] = s.at(6 + j, c); }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float rv = dot3(R[i][0], R[i][1], R[i][2], pv), rb = dot3(R[i][0], R[i][1], R[i][2], pb);
            s.at(i, c) = fmaf(hdt2, rb, fmaf(dt, rv, pp[i]));
            s.at(3 + i, c) = fmaf(dt, rb, rv);
        }
    }
    // ---- process noise G Q G^T = [hdt2; dt] (R Q R^T) [hdt2; dt]^T on the p/v blocks: C = R Q R^T here, added to each entry right
    //      after the row of N it belongs to has been formed (same operation on the same value as a separate read-modify-write
    //      sweep over the 36 entries, without the 36 loads and stores)
    float C[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float rq[3] = {R[i][0] * acc_var[0], R[i][1] * acc_var[1], R[i][2] * acc_var[2]};
#pragma unroll
        for (int j = 0; j < 3; ++j) C[i][j] = dot3(rq[0], rq[1], rq[2], R[j]);
    }
    const float k_pp = hdt2 * hdt2, k_pv = hdt2 * dt, k_vv = dt * dt;
    // ---- N = M F^T, one row per iteration, rows in three groups (p, v, b); the group index is uniform
#pragma unroll 1
    for (int g = 0; g < 3; ++g) {
        const float kA = g == 0 ? k_pp : k_pv, kB = g == 0 ? k_pv : k_vv;      // (p,p)/(p,v) for the p rows, (v,p)/(v,v) for the v rows
#pragma unroll
        for (int ri = 0; ri < 3; ++ri) {
            const int r = g * 3 + ri;
            float mp[3], mv[3], mb[3];
#pragma unroll
            for (int j = 0; j < 3; ++j) { mp[j] = s.at(r, j); mv[j] = s.at(r, 3 + j); mb[j] = s.at(r, 6 + j); }
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const float rv = dot3(R[i][0], R[i][1], R[i][2], mv), rb = dot3(R[i][0], R[i][1], R[i][2], mb);
                float np = fmaf(hdt2, rb, fmaf(dt, rv, mp[i])), nv = fmaf(dt, rb, rv);
                if (g < 2) { np = fmaf(kA, C[ri][i], np); nv = fmaf(kB, C[ri][i], nv); }
                s.at(r, i) = np;
                s.at(r, 3 + i) = nv;
            }
        }
    }
}

// 3x3 inverse by the adjugate, evaluated in float64 and rounded to float32 once.  After the first fix P[H,H] is of the order of
// R = 1e-7 with strongly correlated entries; the float32 adjugate loses most of its digits to cancellation there (the reference's
// torch.linalg.inv is a pivoted LU), and the innovation gain inherits the error (measured against a float64 evaluation of the
// whole step: 1.7e-4 of the state scale with the float32 adjugate, 1e-7 for the reference).
__device__ __forceinline__ void pv_inverse3(const float S[3][3], float Si[3][3]) {
    const double s00 = S[0][0], s01 = S[0][1], s02 = S[0][2], s10 = S[1][0], s11 = S[1][1], s12 = S[1][2];
    const double s20 = S[2][0], s21 = S[2][1], s22 = S[2][2];
    const double c00 = fma(s11, s22, -(s12 * s21)), c01 = fma(s12, s20, -(s10 * s22)), c02 = fma(s10, s21, -(s11 * s20));
    const double id = 1.0 / fma(s02, c02, fma(s01, c01, s00 * c00));
    Si[0][0] = (float)(c00 * id); Si[1][0] = (float)(c01 * id); Si[2][0] = (float)(c02 * id);
    Si[0][1] = (float)(fma(s02, s21, -(s01 * s22)) * id);
    Si[1][1] = (float)(fma(s00, s22, -(s02 * s20)) * id);
    Si[2][1] = (float)(fma(s01, s20, -(s00 * s21)) * id);
    Si[0][2] = (float)(fma(s01, s12, -(s02 * s11)) * id);
    Si[1][2] = (float)(fma(s02, s10, -(s00 * s12)) * id);
    Si[2][2] = (float)(fma(s00, s11, -(s01 * s10)) * id);
}

// correction_step (PVFilter.py:67-110) on block H = [LO, LO+3):
//   K = P[:,H] inv(P[H,H] + diag(rvar)) ; x += K (z - x[H]) ; P = (I - K H) P   (full, non-symmetric update, as the reference)
template <int LO, int STRIDE>
__device__ __forceinline__ void pv_correct(PVShared<STRIDE>& s, const float z[3], const float rvar[3]) {
    // rows H of the OLD covariance (also S = P[H,H] + diag(rvar))
    float PH[3][9];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int j = 0; j < 9; ++j) PH[k][j] = s.at(LO + k, j);
    float S[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) S[i][j] = PH[i][LO + j] + (i == j ? rvar[i] : 0.f);
    // 3x3 inverse by the adjugate, evaluated in float64 and rounded to float32 once.  After the first fix P[H,H] is of the order
    // of R = 1e-7 with strongly correlated entries; the float32 adjugate loses most of its digits to cancellation there (the
    // reference's torch.linalg.inv is a pivoted LU), and the innovation gain inherits the error (measured against a float64
    // evaluation of the whole step: 1.7e-4 of the state scale with the float32 adjugate, 1e-7 for the reference).
    float Si[3][3];
    pv_inverse3(S, Si);
    const float inn[3] = {z[0] - s.x[LO], z[1] - s.x[LO + 1], z[2] - s.x[LO + 2]};     // from the OLD state, before any row updates x
    // one row of K, x and P per iteration: row i of K needs only row i of the old P, read before the row is overwritten.
    // Rows in three groups of three (p, v, b): the group index is uniform, so "is this row in H" and "which x entries does this
    // group update" are branches, not per-element selects.
#pragma unroll 1
    for (int g = 0; g < 3; ++g) {
        const bool inH = (g * 3 == LO);
        float dxg[3];
#pragma unroll
        for (int ii = 0; ii < 3; ++ii) {
            const int i = g * 3 + ii;
            float row[9];
#pragma unroll
            for (int j = 0; j < 9; ++j) row[j] = s.at(i, j);
            float K[3];
#pragma unroll
            for (int j = 0; j < 3; ++j) K[j] = fmaf(row[LO + 2], Si[2][j], fmaf(row[LO + 1], Si[1][j], row[LO] * Si[0][j]));
            dxg[ii] = fmaf(K[2], inn[2], fmaf(K[1], inn[1], K[0] * inn[0]));
            // P <- IKH @ P with IKH = I, IKH[:,H] -= K  (PVFilter.py:88-89 / 108-109)
            float w[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) w[k] = ((inH && ii == k) ? 1.0f : 0.0f) - K[k];
            if (inH) {
#pragma unroll
                for (int j = 0; j < 9; ++j) s.at(i, j) = fmaf(w[2], PH[2][j], fmaf(w[1], PH[1][j], w[0] * PH[0][j]));
            } else {
#pragma unroll
                for (int j = 0; j < 9; ++j) s.at(i, j) = row[j] + fmaf(w[2], PH[2][j], fmaf(w[1], PH[1][j], w[0] * PH[0][j]));
            }
        }
        if (g == 0) { s.x[0] += dxg[0]; s.x[1] += dxg[1]; s.x[2] += dxg[2]; }
        else if (g == 1) { s.x[3] += dxg[0]; s.x[4] += dxg[1]; s.x[5] += dxg[2]; }
        else { s.x[6] += dxg[0]; s.x[7] += dxg[1]; s.x[8] += dxg[2]; }
    }
}

// Warp-cooperative correction_step.  With the reference's SHARED trigger counters (ekf_lee_landed.py:425-440) the position fix
// fires for one env in 7 and the velocity fix for one in 3, so a warp that runs pv_correct<0> and pv_correct<3> one after the
// other works at 14 % and 33 % lane utilisation for ~1500 of its ~7000 instructions.  Here the lanes of a warp share the work:
//   * `job` per lane: -1 none, 0 position fix, 3 velocity fix (block H = [job, job + 3)); the caller makes two passes (first fix
//     of every env, then the velocity fix of the envs that had both);
//   * every job gets S = min(9, lanes / jobs) worker lanes; worker `sub` of a job updates rows sub, sub + S, ... of the OWNER's
//     covariance column in shared memory (rows are independent given the old rows of H, which every worker reads -- a broadcast --
//     before the warp barrier that precedes the first write) and leaves the row's state increment in a 9-float scratch column;
//   * the owner publishes its innovation z - x[H] in a 3-float scratch column before, and adds the increments to x after.
// The arithmetic of a row is exactly pv_correct<LO>'s (same fused operations on the same operands in the same order; LO becomes a
// per-lane value), so the cooperative and the per-thread form give identical bits.
// scr: [12][STRIDE] floats of shared memory (rows 0-2 innovation, 3-11 increments), indexed like the covariance tile.
template <int STRIDE>
__device__ __forceinline__ void pv_correct_coop(PVShared<STRIDE>& s, float* scr_col, const unsigned wmask, const int lane, const int job,
                                                const float z[3], const float rvar_pos[3], const float rvar_vel[3]) {
    const unsigned busy = __ballot_sync(wmask, job >= 0);
    if (busy == 0u) return;                                  // uniform
    const int njobs = __popc(busy), nl = __popc(wmask);
    // S = nl / njobs and jidx = wrank / S for operands <= 32: one MUFU reciprocal each (the +0.5 keeps exact multiples on the right
    // side of the floor; an integer division here compiles to a call into a helper at the far end of a 128 KB kernel image)
    int S = (int)__fdividef((float)nl + 0.5f, (float)njobs);
    S = S > 9 ? 9 : S;
    if (job >= 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) scr_col[k * STRIDE] = z[k] - (job ? s.x[3 + k] : s.x[k]);
    }
    const int wrank = __popc(wmask & ((1u << lane) - 1u));
    const int jidx = (int)__fdividef((float)wrank + 0.5f, (float)S), sub = wrank - jidx * S;
    const bool working = jidx < njobs;
    // lane of the jidx-th fixing env: position of the (jidx + 1)-th set bit of `busy`, by a 5-step binary search on popcounts
    int owner = lane;
    if (working) {
        unsigned m = busy;
        int n = jidx, pos = 0, t;
        t = __popc(m & 0xFFFFu); if (n >= t) { pos += 16; n -= t; m >>= 16; }
        t = __popc(m & 0xFFu);   if (n >= t) { pos += 8;  n -= t; m >>= 8; }
        t = __popc(m & 0xFu);    if (n >= t) { pos += 4;  n -= t; m >>= 4; }
        t = __popc(m & 0x3u);    if (n >= t) { pos += 2;  n -= t; m >>= 2; }
        t = (int)(m & 1u);       if (n >= t) { pos += 1; }
        owner = pos;
    }
    const int LO = __shfl_sync(wmask, job, owner);
    __syncwarp(wmask);                                       // innovations are published
    float* const Pc = s.P + (owner - lane);                  // the owner's column of the covariance tile
    float* const sc = scr_col + (owner - lane);
    float PH[3][9], Si[3][3], inn[3] = {0.f, 0.f, 0.f};
    if (working) {
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int j = 0; j < 9; ++j) PH[k][j] = Pc[((LO + k) * 9 + j) * STRIDE];
#pragma unroll
        for (int k = 0; k < 3; ++k) inn[k] = sc[k * STRIDE];
        float Sm[3][3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) Sm[i][j] = (LO ? PH[i][3 + j] : PH[i][j]) + (i == j ? (LO ? rvar_vel[i] : rvar_pos[i]) : 0.f);
        pv_inverse3(Sm, Si);
    }
    __syncwarp(wmask);                                       // every worker holds the old rows of H: rows may be overwritten now
    if (working) {
        for (int i = sub; i < 9; i += S) {
            float row[9];
#pragma unroll
            for (int j = 0; j < 9; ++j) row[j] = Pc[(i * 9 + j) * STRIDE];
            const float r0 = LO ? row[3] : row[0], r1 = LO ? row[4] : row[1], r2 = LO ? row[5] : row[2];
            float K[3];
#pragma unroll
            for (int j = 0; j < 3; ++j) K[j] = fmaf(r2, Si[2][j], fmaf(r1, Si[1][j], r0 * Si[0][j]));
            sc[(3 + i) * STRIDE] = fmaf(K[2], inn[2], fmaf(K[1], inn[1], K[0] * inn[0]));
            float w[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) w[k] = ((i == LO + k) ? 1.0f : 0.0f) - K[k];
            const bool inH = (i >= LO) && (i < LO + 3);
#pragma unroll
            for (int j = 0; j < 9; ++j) {
                const float acc3 = fmaf(w[2], PH[2][j], fmaf(w[1], PH[1][j], w[0] * PH[0][j]));
                Pc[(i * 9 + j) * STRIDE] = inH ? acc3 : (row[j] + acc3);
            }
        }
    }
    __syncwarp(wmask);                                       // increments are published
    if (job >= 0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) s.x[i] += scr_col[(3 + i) * STRIDE];
    }
}

// ------------------------------------------------------------------------------------------------ K2: attitude EKF
struct EKF4 {
    double q[4];        // wxyz
    double P[4][4];
};

// EKF.update(q/|q|, gyr, ang) -- ahrs_ekf.py:1301-1337, `ang` branch.  Dt = 1/frequency, g_noise = 0.3^2.
__device__ __forceinline__ void ekf_update(EKF4& s, const double g[3], const double ang[4], double Dt, double g_noise,
                                           double s_eps) {
    // caller-side normalisation (tasks/ekf_lee_landed.py:386: q=self.Q_state[idx]/np.linalg.norm(...))
    // (one reciprocal + four products instead of four float64 divisions: 1 ulp of float64 apart, parity bound 1e-9)
    const double inq = 1.0 / sqrt(fma(s.q[3], s.q[3], fma(s.q[2], s.q[2], fma(s.q[1], s.q[1], s.q[0] * s.q[0]))));
    double q[4] = {s.q[0] * inq, s.q[1] * inq, s.q[2] * inq, s.q[3] * inq};
    const double hd = 0.5 * Dt;
    // Omega(x) rows: [0,-x0,-x1,-x2],[x0,0,x2,-x1],[x1,-x2,0,x0],[x2,x1,-x0,0]          (:1100-1106); zero diagonal, so the
    // products with I + c Omega are written as "identity term + the three off-diagonal terms" (48 instead of 64 multiply-adds)
    const double x[3] = {hd * g[0], hd * g[1], hd * g[2]};                // F = I + Omega(0.5 Dt g)      (:1157-1158)
    const double Ox[4][4] = {{0.0, -x[0], -x[1], -x[2]}, {x[0], 0.0, x[2], -x[1]}, {x[1], -x[2], 0.0, x[0]}, {x[2], x[1], -x[0], 0.0}};
    double qt[4];                                                         // q_t = (I + 0.5 Dt Omega(g)) q    (:1132-1133)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double acc = q[i];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j != i) acc = fma(Ox[i][j], q[j], acc);
        qt[i] = acc;
    }
    // P_t = F P F^T + 0.5 Dt g_noise W W^T with W = 0.5 Dt [ -q_v ; q_w I + skew(q_v) ]                (:1320-1322);
    // W W^T = (0.5 Dt)^2 (|q|^2 I - q q^T) for this 4x3 quaternion-rate matrix
    double FP[4][4], Pt[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double a = s.P[i][j];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k != i) a = fma(Ox[i][k], s.P[k][j], a);
            FP[i][j] = a;
        }
    const double n2 = fma(q[3], q[3], fma(q[2], q[2], fma(q[1], q[1], q[0] * q[0])));
    const double qw = (hd * g_noise) * (hd * hd);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double a = FP[i][j];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k != j) a = fma(FP[i][k], Ox[j][k], a);
            Pt[i][j] = fma(qw, (i == j ? n2 : 0.0) - q[i] * q[j], a);
        }
    // S = P_t + eps I ; K = P_t S^-1  (Gauss-Jordan on the SPD 4x4, no pivoting)                       (:1332-1333)
    double S[4][4], Si[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { S[i][j] = Pt[i][j] + (i == j ? s_eps : 0.0); Si[i][j] = (i == j ? 1.0 : 0.0); }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const double ip = 1.0 / S[c][c];
#pragma unroll
        for (int j = 0; j < 4; ++j) { S[c][j] *= ip; Si[c][j] *= ip; }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if (r == c) continue;
            const double f = S[r][c];
#pragma unroll
            for (int j = 0; j < 4; ++j) { S[r][j] = fma(-f, S[c][j], S[r][j]); Si[r][j] = fma(-f, Si[c][j], Si[r][j]); }
        }
    }
    // K = P_t S^-1 ; P = (I - K) P_t ; q = normalize(q_t + K (ang - q_t)), evaluated as the reference writes them (:1333-1336).
    // (With H = I the update collapses algebraically to q = ang - eps S^-1 (ang - q_t), P = eps (I - eps S^-1), a third of the
    // work -- but `I - K` cancels to ~1e-9 relative in the literal form when P_t >> eps, so the two forms differ by up to 1e-9 in
    // later steps; parity with the reference's arithmetic is worth more here than ~100 float64 instructions.)
    double v[4], qn[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = ang[i] - qt[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) {               // one row of K at a time (row i of K feeds only q[i] and row i of P)
        double Ki[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double a = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) a = fma(Pt[i][k], Si[k][j], a);
            Ki[j] = a;
        }
        double a = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) a = fma(Ki[k], v[k], a);
        qn[i] = qt[i] + a;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            double b = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) b = fma((i == k ? 1.0 : 0.0) - Ki[k], Pt[k][j], b);
            s.P[i][j] = b;
        }
    }
    const double inn = 1.0 / sqrt(fma(qn[3], qn[3], fma(qn[2], qn[2], fma(qn[1], qn[1], qn[0] * qn[0]))));
#pragma unroll
    for (int i = 0; i < 4; ++i) s.q[i] = qn[i] * inn;
}

}  // namespace ozl
