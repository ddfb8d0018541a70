// TMA 1-D bulk copies (cp.async.bulk) and mbarrier helpers for sm_100a, shared by the step kernels (quad_step.cu) and the
// fused estimator kernel (ekf_lee_fused.cu).  SASS evidence: UBLKCP (bulk copy), SYNCS (mbarrier).
#pragma once
#include <stdint.h>

namespace ozl {

// TMA 1-D bulk copy shared -> global (SASS: UBLKCP).  Used to write the block's contiguous [BLOCK,13] observation
// tile with one instruction instead of a per-thread copy loop.
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// several copies in ONE bulk group: issue, ..., issue, commit
__device__ __forceinline__ void bulk_store_s2g_issue(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... and until the copies' global writes have been performed (before the thread signals a consumer outside the stream)
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sdst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// TMA 2-D tiled copies through a tensor map (cp.async.bulk.tensor.2d; SASS UTMALDG / UTMASTG): one instruction moves a whole
// [rows][cols] box between a row-strided global matrix and a dense shared-memory tile; columns beyond the matrix are zero-filled on
// loads and clipped on stores.  `tmap` is the generic address of a `const __grid_constant__ CUtensorMap` kernel parameter.
__device__ __forceinline__ void tma_load_2d(void* sdst, const void* tmap, int32_t x, int32_t y, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(sdst)),
                 "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void* tmap, int32_t x, int32_t y, const void* ssrc) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];" ::"l"(tmap), "r"(x), "r"(y), "r"(smem_u32(ssrc))
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

// Programmatic dependent launch (PDL).  A step kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may be
// made resident while its predecessor on the stream is still draining; griddep_wait() blocks until the predecessor has
// completed and its memory operations are visible (it returns at once when the launch carries no such dependency), and
// griddep_launch_dependents() lets the NEXT launch on the stream be staged the same way.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace ozl
