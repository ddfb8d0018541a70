// Exact CPU twin of the batched estimators of ouzelum_b200/csrc/filters.cuh -- TEST INFRASTRUCTURE.
//
// Every function below restates its namesake in filters.cuh operation for operation: the same fused multiply-adds (fmaf / fma),
// the same products, sums, divisions and square roots, on the same operands, in the same order.  The device code uses only
// correctly rounded IEEE operations (+ - * /, sqrtf, fmaf, fma, sqrt, float <-> double conversions; every TU is built with
// -fmad=false), so this file, compiled with `gcc -ffp-contract=off -fno-fast-math` against a correctly rounded libm fma, must
// reproduce every output bit of the kernels that run these filters.
//
// Built twice (tests/filters_ref.py):
//   default                 PV scalar type float: the bit-exact twin of the kernels
//   -DFILTERS_REF_F64       PV scalar type double (fmaf -> fma, the rounding of the 3x3 inverse disappears): the same operation
//                           sequence in float64, the high-precision arbiter of the float32 arithmetic
// The attitude EKF is float64 on the device and identical in both builds.
//
// Covariance of one env: P[r * 9 + c] (the kernel's s.at(r, c)); batched drivers take the banks' plane layouts [9][N], [81][N],
// [4][N], [16][N] (SoA, element k of env i at [k * N + i]).
#include <math.h>
#include <stdint.h>

#ifdef FILTERS_REF_F64
typedef double real;
#define FMA(a, b, c) fma((a), (b), (c))
#define SQRT(a) sqrt(a)
#define ROUND_INV(a) (a)
#else
typedef float real;
#define FMA(a, b, c) fmaf((a), (b), (c))
#define SQRT(a) sqrtf(a)
#define ROUND_INV(a) ((float)(a))
#endif

int ozl_ref_real_size(void) { return (int)sizeof(real); }

// ------------------------------------------------------------------------------------------------ K3: PV filter
typedef struct {
    real x[9];
    real* P;                                  // 81 entries, row-major
} PVState;

#define AT(s, r, c) ((s)->P[(r) * 9 + (c)])

// pv_quat_to_R (filters.cuh): quaternion_to_matrix of PVFilter.py:113-142, wxyz in, normalises first
static void pv_quat_to_R(real r, real i, real j, real k, real R[3][3]) {
    const real n = SQRT(FMA(k, k, FMA(j, j, FMA(i, i, r * r))));
    r /= n; i /= n; j /= n; k /= n;
    const real two_s = (real)2.0 / FMA(k, k, FMA(j, j, FMA(i, i, r * r)));
    R[0][0] = FMA(-two_s, FMA(k, k, j * j), (real)1.0); R[0][1] = two_s * FMA(i, j, -(k * r)); R[0][2] = two_s * FMA(i, k, j * r);
    R[1][0] = two_s * FMA(i, j, k * r); R[1][1] = FMA(-two_s, FMA(k, k, i * i), (real)1.0); R[1][2] = two_s * FMA(j, k, -(i * r));
    R[2][0] = two_s * FMA(i, k, -(j * r)); R[2][1] = two_s * FMA(j, k, i * r); R[2][2] = FMA(-two_s, FMA(j, j, i * i), (real)1.0);
}

static real dot3(const real a0, const real a1, const real a2, const real b[3]) {
    return FMA(a2, b[2], FMA(a1, b[1], a0 * b[0]));
}

// pv_predict (filters.cuh): factored F P F^T, process noise added to each p/v entry right after its row of N is formed
static void pv_predict(PVState* s, const real acc[3], const real q_wxyz[4], real dt, real dt2, const real acc_var[3]) {
    real Rq[3][3], R[3][3];
    pv_quat_to_R(q_wxyz[0], q_wxyz[1], q_wxyz[2], q_wxyz[3], Rq);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) R[i][j] = Rq[j][i];                  // .T   (PVFilter.py:33-35)
    const real hdt2 = dt2 * (real)0.5;
    // ---- state
    {
        const real xv[3] = {s->x[3], s->x[4], s->x[5]};
        for (int i = 0; i < 3; ++i) {
            const real rv = dot3(R[i][0], R[i][1], R[i][2], xv), ra = dot3(R[i][0], R[i][1], R[i][2], acc);
            s->x[i] = FMA(hdt2, ra, FMA(dt, rv, s->x[i]));
            s->x[3 + i] = FMA(dt, ra, rv);
        }
    }
    // ---- M = F P, one column per iteration
    for (int c = 0; c < 9; ++c) {
        real pp[3], pv[3], pb[3];
        for (int j = 0; j < 3; ++j) { pp[j] = AT(s, j, c); pv[j] = AT(s, 3 + j, c); pb[j] = AT(s, 6 + j, c); }
        for (int i = 0; i < 3; ++i) {
            const real rv = dot3(R[i][0], R[i][1], R[i][2], pv), rb = dot3(R[i][0], R[i][1], R[i][2], pb);
            AT(s, i, c) = FMA(hdt2, rb, FMA(dt, rv, pp[i]));
            AT(s, 3 + i, c) = FMA(dt, rb, rv);
        }
    }
    // ---- C = R Q R^T
    real C[3][3];
    for (int i = 0; i < 3; ++i) {
        const real rq[3] = {R[i][0] * acc_var[0], R[i][1] * acc_var[1], R[i][2] * acc_var[2]};
        for (int j = 0; j < 3; ++j) C[i][j] = dot3(rq[0], rq[1], rq[2], R[j]);
    }
    const real k_pp = hdt2 * hdt2, k_pv = hdt2 * dt, k_vv = dt * dt;
    // ---- N = M F^T, one row per iteration, rows in three groups (p, v, b)
    for (int g = 0; g < 3; ++g) {
        const real kA = g == 0 ? k_pp : k_pv, kB = g == 0 ? k_pv : k_vv;
        for (int ri = 0; ri < 3; ++ri) {
            const int r = g * 3 + ri;
            real mp[3], mv[3], mb[3];
            for (int j = 0; j < 3; ++j) { mp[j] = AT(s, r, j); mv[j] = AT(s, r, 3 + j); mb[j] = AT(s, r, 6 + j); }
            for (int i = 0; i < 3; ++i) {
                const real rv = dot3(R[i][0], R[i][1], R[i][2], mv), rb = dot3(R[i][0], R[i][1], R[i][2], mb);
                real np = FMA(hdt2, rb, FMA(dt, rv, mp[i])), nv = FMA(dt, rb, rv);
                if (g < 2) { np = FMA(kA, C[ri][i], np); nv = FMA(kB, C[ri][i], nv); }
                AT(s, r, i) = np;
                AT(s, r, 3 + i) = nv;
            }
        }
    }
}

// pv_inverse3 (filters.cuh): adjugate in float64, rounded to the PV type once
static void pv_inverse3(const real S[3][3], real Si[3][3]) {
    const double s00 = S[0][0], s01 = S[0][1], s02 = S[0][2], s10 = S[1][0], s11 = S[1][1], s12 = S[1][2];
    const double s20 = S[2][0], s21 = S[2][1], s22 = S[2][2];
    const double c00 = fma(s11, s22, -(s12 * s21)), c01 = fma(s12, s20, -(s10 * s22)), c02 = fma(s10, s21, -(s11 * s20));
    const double id = 1.0 / fma(s02, c02, fma(s01, c01, s00 * c00));
    Si[0][0] = ROUND_INV(c00 * id); Si[1][0] = ROUND_INV(c01 * id); Si[2][0] = ROUND_INV(c02 * id);
    Si[0][1] = ROUND_INV(fma(s02, s21, -(s01 * s22)) * id);
    Si[1][1] = ROUND_INV(fma(s00, s22, -(s02 * s20)) * id);
    Si[2][1] = ROUND_INV(fma(s01, s20, -(s00 * s21)) * id);
    Si[0][2] = ROUND_INV(fma(s01, s12, -(s02 * s11)) * id);
    Si[1][2] = ROUND_INV(fma(s02, s10, -(s00 * s12)) * id);
    Si[2][2] = ROUND_INV(fma(s00, s11, -(s01 * s10)) * id);
}

// pv_correct<LO> (filters.cuh), per-thread form; LO = 0 position fix, 3 velocity fix.  pv_correct_coop has no twin here: it must
// give the bits of this form, and the GPU tests check exactly that.
static void pv_correct(PVState* s, const int LO, const real z[3], const real rvar[3]) {
    real PH[3][9];
    for (int k = 0; k < 3; ++k)
        for (int j = 0; j < 9; ++j) PH[k][j] = AT(s, LO + k, j);
    real S[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) S[i][j] = PH[i][LO + j] + (i == j ? rvar[i] : (real)0.0);
    real Si[3][3];
    pv_inverse3(S, Si);
    const real inn[3] = {z[0] - s->x[LO], z[1] - s->x[LO + 1], z[2] - s->x[LO + 2]};
    for (int g = 0; g < 3; ++g) {
        const int inH = (g * 3 == LO);
        real dxg[3];
        for (int ii = 0; ii < 3; ++ii) {
            const int i = g * 3 + ii;
            real row[9];
            for (int j = 0; j < 9; ++j) row[j] = AT(s, i, j);
            real K[3];
            for (int j = 0; j < 3; ++j) K[j] = FMA(row[LO + 2], Si[2][j], FMA(row[LO + 1], Si[1][j], row[LO] * Si[0][j]));
            dxg[ii] = FMA(K[2], inn[2], FMA(K[1], inn[1], K[0] * inn[0]));
            real w[3];
            for (int k = 0; k < 3; ++k) w[k] = ((inH && ii == k) ? (real)1.0 : (real)0.0) - K[k];
            if (inH) {
                for (int j = 0; j < 9; ++j) AT(s, i, j) = FMA(w[2], PH[2][j], FMA(w[1], PH[1][j], w[0] * PH[0][j]));
            } else {
                for (int j = 0; j < 9; ++j) AT(s, i, j) = row[j] + FMA(w[2], PH[2][j], FMA(w[1], PH[1][j], w[0] * PH[0][j]));
            }
        }
        s->x[g * 3 + 0] += dxg[0]; s->x[g * 3 + 1] += dxg[1]; s->x[g * 3 + 2] += dxg[2];
    }
}

// ------------------------------------------------------------------------------------------------ K2: attitude EKF (float64)
typedef struct {
    double q[4];        // wxyz
    double P[4][4];
} EKF4;

// ekf_update (filters.cuh): EKF.update(q/|q|, gyr, ang), `ang` branch, with the kernel's own normalisation
static void ekf_update(EKF4* s, const double g[3], const double ang[4], double Dt, double g_noise, double s_eps) {
    const double inq = 1.0 / sqrt(fma(s->q[3], s->q[3], fma(s->q[2], s->q[2], fma(s->q[1], s->q[1], s->q[0] * s->q[0]))));
    double q[4] = {s->q[0] * inq, s->q[1] * inq, s->q[2] * inq, s->q[3] * inq};
    const double hd = 0.5 * Dt;
    const double x[3] = {hd * g[0], hd * g[1], hd * g[2]};
    const double Ox[4][4] = {{0.0, -x[0], -x[1], -x[2]}, {x[0], 0.0, x[2], -x[1]}, {x[1], -x[2], 0.0, x[0]}, {x[2], x[1], -x[0], 0.0}};
    double qt[4];
    for (int i = 0; i < 4; ++i) {
        double acc = q[i];
        for (int j = 0; j < 4; ++j)
            if (j != i) acc = fma(Ox[i][j], q[j], acc);
        qt[i] = acc;
    }
    double FP[4][4], Pt[4][4];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            double a = s->P[i][j];
            for (int k = 0; k < 4; ++k)
                if (k != i) a = fma(Ox[i][k], s->P[k][j], a);
            FP[i][j] = a;
        }
    const double n2 = fma(q[3], q[3], fma(q[2], q[2], fma(q[1], q[1], q[0] * q[0])));
    const double qw = (hd * g_noise) * (hd * hd);
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            double a = FP[i][j];
            for (int k = 0; k < 4; ++k)
                if (k != j) a = fma(FP[i][k], Ox[j][k], a);
            Pt[i][j] = fma(qw, (i == j ? n2 : 0.0) - q[i] * q[j], a);
        }
    // S = P_t + eps I ; Gauss-Jordan on the SPD 4x4, no pivoting
    double S[4][4], Si[4][4];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) { S[i][j] = Pt[i][j] + (i == j ? s_eps : 0.0); Si[i][j] = (i == j ? 1.0 : 0.0); }
    for (int c = 0; c < 4; ++c) {
        const double ip = 1.0 / S[c][c];
        for (int j = 0; j < 4; ++j) { S[c][j] *= ip; Si[c][j] *= ip; }
        for (int r = 0; r < 4; ++r) {
            if (r == c) continue;
            const double f = S[r][c];
            for (int j = 0; j < 4; ++j) { S[r][j] = fma(-f, S[c][j], S[r][j]); Si[r][j] = fma(-f, Si[c][j], Si[r][j]); }
        }
    }
    double v[4], qn[4];
    for (int i = 0; i < 4; ++i) v[i] = ang[i] - qt[i];
    for (int i = 0; i < 4; ++i) {
        double Ki[4];
        for (int j = 0; j < 4; ++j) {
            double a = 0.0;
            for (int k = 0; k < 4; ++k) a = fma(Pt[i][k], Si[k][j], a);
            Ki[j] = a;
        }
        double a = 0.0;
        for (int k = 0; k < 4; ++k) a = fma(Ki[k], v[k], a);
        qn[i] = qt[i] + a;
        for (int j = 0; j < 4; ++j) {
            double b = 0.0;
            for (int k = 0; k < 4; ++k) b = fma((i == k ? 1.0 : 0.0) - Ki[k], Pt[k][j], b);
            s->P[i][j] = b;
        }
    }
    const double inn = 1.0 / sqrt(fma(qn[3], qn[3], fma(qn[2], qn[2], fma(qn[1], qn[1], qn[0] * qn[0]))));
    for (int i = 0; i < 4; ++i) s->q[i] = qn[i] * inn;
}

// ------------------------------------------------------------------------------------------------ batched drivers
// pv_step_kernel + ozl_pv_step (companions.cu): optional predict, then the position fix, then the velocity fix.  A fix fires where
// its mask is set or, without a mask, where (iter_base + i) % period == phase (period 0: never); no measurement pointer: no fix.
// pos_var / vel_var are used when *_given, else R = 0.  `dt` arrives as the host's double: the float build rounds it to float
// and forms dt2 = (float)((double)dt * dt) as ozl_pv_step does; the double build uses dt and dt * dt.
void ozl_ref_pv_step(int64_t n, real* x9, real* P81, const real* accel3, const real* quat4, const real* pos_meas3,
                     const real* vel_meas3, const uint8_t* pos_mask, const uint8_t* vel_mask, double dt_host, const real* acc_var,
                     const real* pos_var, const real* vel_var, int pos_var_given, int vel_var_given, int flip_qw, int do_predict,
                     uint32_t pos_period, uint32_t pos_phase, uint32_t vel_period, uint32_t vel_phase, uint64_t iter_base) {
#ifdef FILTERS_REF_F64
    const real dt = dt_host, dt2 = dt_host * dt_host;
#else
    const real dt = (float)dt_host, dt2 = (float)((double)dt * (double)dt);
#endif
    real av[3], pvar[3], vvar[3];
    for (int j = 0; j < 3; ++j) {
        av[j] = acc_var[j];
        pvar[j] = pos_var_given ? pos_var[j] : (real)0.0;
        vvar[j] = vel_var_given ? vel_var[j] : (real)0.0;
    }
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; ++i) {
        real P[81];
        PVState s;
        s.P = P;
        for (int k = 0; k < 9; ++k) s.x[k] = x9[k * n + i];
        for (int k = 0; k < 81; ++k) P[k] = P81[k * n + i];
        if (do_predict) {
            const real acc[3] = {accel3[i * 3], accel3[i * 3 + 1], accel3[i * 3 + 2]};
            const real* q4 = quat4 + i * 4;
            real q[4];
            if (flip_qw) { q[0] = q4[3]; q[1] = q4[0]; q[2] = q4[1]; q[3] = q4[2]; }
            else { q[0] = q4[0]; q[1] = q4[1]; q[2] = q4[2]; q[3] = q4[3]; }
            pv_predict(&s, acc, q, dt, dt2, av);
        }
        const uint64_t k = iter_base + (uint64_t)i;
        int pos_fix = 0, vel_fix = 0;
        if (pos_meas3) pos_fix = pos_mask ? (pos_mask[i] != 0) : (pos_period && (k % pos_period) == pos_phase);
        if (vel_meas3) vel_fix = vel_mask ? (vel_mask[i] != 0) : (vel_period && (k % vel_period) == vel_phase);
        if (pos_fix) pv_correct(&s, 0, pos_meas3 + i * 3, pvar);
        if (vel_fix) pv_correct(&s, 3, vel_meas3 + i * 3, vvar);
        for (int kk = 0; kk < 9; ++kk) x9[kk * n + i] = s.x[kk];
        for (int kk = 0; kk < 81; ++kk) P81[kk * n + i] = P[kk];
    }
}

// ekf_update_kernel (companions.cu): float32 sensors widened to double, `ang` reordered xyzw -> wxyz when asked, optional float32
// copy of the updated q (the PV filter's orientation input)
void ozl_ref_ekf_update(int64_t n, double* q4, double* P16, const float* gyr3, const float* ang4, int ang_xyzw, double Dt,
                        double g_noise, double s_eps, float* q_f32_out) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; ++i) {
        EKF4 s;
        for (int k = 0; k < 4; ++k) s.q[k] = q4[k * n + i];
        for (int k = 0; k < 16; ++k) s.P[k / 4][k % 4] = P16[k * n + i];
        const double g[3] = {(double)gyr3[i * 3], (double)gyr3[i * 3 + 1], (double)gyr3[i * 3 + 2]};
        const float* a4 = ang4 + i * 4;
        double a[4];
        if (ang_xyzw) { a[0] = a4[3]; a[1] = a4[0]; a[2] = a4[1]; a[3] = a4[2]; }
        else { a[0] = a4[0]; a[1] = a4[1]; a[2] = a4[2]; a[3] = a4[3]; }
        ekf_update(&s, g, a, Dt, g_noise, s_eps);
        for (int k = 0; k < 4; ++k) q4[k * n + i] = s.q[k];
        for (int k = 0; k < 16; ++k) P16[k * n + i] = s.P[k / 4][k % 4];
        if (q_f32_out)
            for (int k = 0; k < 4; ++k) q_f32_out[i * 4 + k] = (float)s.q[k];
    }
}
