// Philox4x32-10 counter RNG (device).  CPU twin: oracle/philox.py -- the two must agree bit for bit.
// counter = (global env id, step lo, step hi, purpose), key = 64-bit seed.
#pragma once
#include <stdint.h>

namespace ozl {

enum : uint32_t {
    P_TARGET = 0,    // r0,r1 -> target x,y ; r2 -> target z
    P_SPAWN = 1,     // r0,r1,r2 -> spawn offsets
    P_FAULT = 2,     // r0 -> rotor ; r1 -> onset ; r2 -> effectiveness  (fault_mode 2: r0 -> permutation ; r1 -> onset ; r2 -> count)
    P_DR0 = 3,       // mass, Ixx, Iyy, Izz
    P_DR1 = 4,       // arm, thrust-scale, yaw_km
    P_DR2 = 24,      // second uniforms of gaussian draws (mass, Ixx, Iyy, Izz)
    P_DR3 = 25,      //                                   (arm, thrust-scale, yaw_km)
    P_QDOF0 = 5,     // Quadcopter task: initial DOF positions 0..3
    P_QDOF1 = 6,     //                  initial DOF positions 4..7
    P_RFAULT = 7,    // fault_mode 2: w0..w3 -> effectiveness of rotors 0..3
    P_OBSNOISE = 8,  // +0..+3: 13 sensor-noise uniforms
    P_FLICKER = 12,  // global blackout draw (env word = GLOBAL_ENV)
    P_ACTION = 16,   // synthetic roll-out actions
    P_HUSKY = 20,    // waypoint-trajectory re-randomisation
};
constexpr uint32_t GLOBAL_ENV = 0xFFFFFFFFu;

// Inline everywhere, including the fused EKFLeeLanded kernel, where one out-of-line copy would save ~20 KB of code but was
// measured slower (ekf_lee_fused.cu).
static __device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += W0;
        k1 += W1;
    }
    return c;
}

__device__ __forceinline__ uint4 draw(uint64_t seed, uint32_t env, uint64_t step, uint32_t purpose) {
    return philox4x32_10(make_uint4(env, (uint32_t)step, (uint32_t)(step >> 32), purpose), (uint32_t)seed,
                         (uint32_t)(seed >> 32));
}

// Draws on rarely taken paths (episode reset: spawn, rotor fault, domain randomisation, target / trajectory re-draws).  A TU whose
// kernel is instruction-fetch bound defines OZL_COLD_DRAW_NOINLINE and these sites share ONE out-of-line copy of the ten rounds
// (~90 instructions each otherwise); the per-step draws stay inline everywhere.  Same function, same bits.
#ifdef OZL_COLD_DRAW_NOINLINE
static __device__ __noinline__ uint4 draw_cold(uint64_t seed, uint32_t env, uint64_t step, uint32_t purpose) {
    return draw(seed, env, step, purpose);
}
#else
__device__ __forceinline__ uint4 draw_cold(uint64_t seed, uint32_t env, uint64_t step, uint32_t purpose) {
    return draw(seed, env, step, purpose);
}
#endif

// uint32 -> [0,1): top 24 bits * 2^-24, exact in float32
__device__ __forceinline__ float u01(uint32_t r) { return (float)(r >> 8) * 5.9604644775390625e-08f; }

}  // namespace ozl
