// Internal (non-ABI) declarations shared by the translation units of libouzelum_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <cudaTypedefs.h>      // CUtensorMap and the encoder's type (no libcuda link: see tensor_map_encoder)
#include <stdint.h>
#include "../../include/ouzelum_b200.h"
#include "quad_env.cuh"

namespace ozl {

int set_error(const char* fmt, ...);   // stores a thread-local message, returns 1
int check_cuda(cudaError_t e, const char* what);
// cuTensorMapEncodeTiled, looked up once through cudaGetDriverEntryPoint; NULL if the driver does not provide it
PFN_cuTensorMapEncodeTiled tensor_map_encoder();

constexpr int kMetricSlots = 32;       // metric accumulators are striped over this many slots (256 B apart) to spread L2 atomics
constexpr int kMetricStride = 32;      // doubles per slot (16 used)

// Private state of one handle: float4-packed planes, so one env == one 16-byte lane per plane.
//   dynamic (read+written every step):  d0 {px,py,pz,qx} d1 {qy,qz,qw,vx} d2 {vy,vz,wx,wy} d3 {wz,T0,T1,T2} d4 {T3,ep_ret}
//   static  (read every step, written only on reset/resample):
//           s0 {tx,ty,tz,fault_eff} s1 {mass,ixx,iyy,izz} s2 {arm,thrust_scale,fault_word,yaw_km}
// Layout: tiles of kTile = 128 envs; inside a tile the planes are stored back to back
//   [d0 2 KiB][d1][d2][d3][d4 1 KiB][s0 2 KiB][s1][s2]  = 15360 bytes per tile
// so the CTA that owns a tile reads ONE contiguous 15 KiB region and writes ONE contiguous 9 KiB region (long DRAM bursts,
// 2 streams per CTA instead of 16), while a warp still touches 512 contiguous bytes per plane.
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * (7 * 16 + 8);
struct Planes {
    char* base;                 // arena
    unsigned long long* ctrl;   // [0..2] step-counter record {base, units, shift} (step_counter.cuh), [4] TMA-kernel tile scheduler (monotonic)
    double* metrics;            // kMetricSlots x kMetricStride
    unsigned long long* tile_seq;   // [tiles][2] {started, done}: per-tile step sequence of the tile-chained launches (tile_chain.cuh)
};
// k = 0..3: d0..d3, k = 4..6: s0..s2
__device__ __forceinline__ float4* plane4_ptr(const Planes& pl, int k, int64_t i) {
    const int64_t tile = i >> 7;
    const int lane = (int)(i & (kTile - 1));
    const int off = (k < 4 ? k * 2048 : 9216 + (k - 4) * 2048);
    return reinterpret_cast<float4*>(pl.base + tile * kTileBytes + off) + lane;
}
__device__ __forceinline__ float2* plane2_ptr(const Planes& pl, int64_t i) {
    return reinterpret_cast<float2*>(pl.base + (i >> 7) * kTileBytes + 8192) + (int)(i & (kTile - 1));
}

}  // namespace ozl

struct ozl_env {
    ozl_cfg cfg;
    ozl::DevCfg dev;
    ozl::Planes pl;
    int device;
    int sm_count;
    long long tma_min_tiles;    // >= this many whole tiles: use the persistent TMA-pipelined step kernel
    void* arena;                // single cudaMalloc backing all planes
    size_t arena_bytes;
    // host-consumer steps: completion word in pinned host memory, written by the last block of a step kernel after all its
    // zero-copy result stores (ozl_step_host_sync / ozl_step_host_wait poll it instead of synchronising the stream)
    volatile unsigned int* host_done;   // cudaHostAlloc'ed, one word; NULL if that failed (stream synchronise instead)
    unsigned int host_seq;              // sequence number of the last host step launched
    // tile-chained step launches (tile_chain.cuh): the graph node of the last chained launch captured on this handle
    // 2-D tensor map of the caller's [81][N] PV covariance planes with a [81][32] box (ekf_lee_fused.cu), cached per pointer
    alignas(64) unsigned char pv_tmap[128];
    const void* pv_tmap_ptr;
    int chain_mode;                     // OZL_EKF_CHAIN: 0 = never chain, 1 = chain launches that are provably adjacent in a stream capture
    unsigned long long chain_capture_id;
    void* chain_last_node;
    // privileged critic-state output (ozl_set_states_output): caller's [N, OZL_STATES_WIDTH] buffer or NULL, and the 2-D tensor
    // map over it (box [128 rows][32], 128-byte swizzle) through which the step kernels store one states tile per 128 envs
    float* states;
    alignas(64) unsigned char states_tmap[128];
    // scenario table (ozl_set_scenarios): device copy of the caller's [N, OZL_SCENARIO_WIDTH] rows, allocated on the first
    // registration and kept until ozl_destroy (re-registration overwrites it in place); `scn` is that buffer while a table is
    // registered and NULL otherwise -- the step launches pick the kernels that read it by this pointer
    float* scn_buf;
    float* scn;
};

// Step launches go through cudaLaunchKernelEx so that they can carry the programmatic-stream-serialization attribute (PDL):
// consecutive steps on a stream are strictly dependent, but the NEXT step's blocks can be made resident and parked in
// griddep_wait() while the current step drains, which takes the launch latency off the critical path of short steps.
template <typename... KArgs, typename... Args>
static inline int launch_pdl_smem(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                  Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...) != cudaSuccess;
}
template <typename... KArgs, typename... Args>
static inline int launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args... args) {
    return launch_pdl_smem(kernel, grid, block, 0, st, args...);
}

