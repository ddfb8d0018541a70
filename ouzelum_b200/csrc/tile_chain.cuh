// Tile-chained step launches: consecutive launches of a step kernel whose CTA b touches only the envs of tile b may overlap
// TILE BY TILE instead of waiting for the whole previous grid.
//
// Why: a one-wave step kernel runs all its CTAs in lockstep -- every CTA reads at the start of the launch, computes in the
// middle and writes at the end -- so HBM idles during the arithmetic and the SMs idle during the two traffic bursts
// (EKFLeeLanded step at 65536 envs: 15.2 us with the arithmetic removed + ~12 us of arithmetic = 27 us; stage ablation in
// profiles/r02k_config3_ablation.jsonl).  With per-tile dependencies launch L+1's CTA b starts as soon as launch L's CTA b has
// finished and a CTA slot is free; the CTAs drift out of phase and the traffic of some overlaps the arithmetic of others.
//
// Protocol.  Two monotonic words per tile in the handle's arena, both ABSOLUTE step indices:
//     started[b]  the step index the NEXT launch's CTA b will execute          done[b]  steps completed by tile b
//   mode 0 (first launch of a chain / not provably adjacent to a chained launch): griddepcontrol.wait (everything before has
//     completed), S = the handle's global step record, started[b] <- S + 1 (store + fence), then the launch trigger.
//   mode 1 (chained, NO griddepcontrol.wait): S = atomicAdd(started[b], 1), then the launch trigger, then spin (ld.acquire.gpu)
//     until done[b] == S.
//   both: run step S on tile b; wait for the CTA's bulk stores to complete; block barrier; fence; st.release.gpu done[b] <- S + 1.
// The launches carry the programmatic-stream-serialization attribute, so a CTA of launch L+1 is scheduled only after EVERY CTA
// of launch L has passed its trigger, i.e. has read (mode 1: incremented) started[b]: the atomics on started[b] are executed in
// launch order, no CTA ever waits for a CTA that is not yet resident (no deadlock), and at most two launches share the SMs.
// The global step record is still retired by every launch (before the done-release), so it is exact whenever the stream has
// drained, which is the only time a mode-0 launch, any other kernel or the host reads it.
//
// The HOST decides the mode (ekf_lee_fused.cu): a launch is chained only when it is captured into a CUDA graph directly behind
// the previous chained launch of the same handle (cudaStreamGetCaptureInfo: same capture, the stream's only dependency is that
// launch's node) -- nothing can then sit between the two launches that writes what the step reads.  Everything else, eager
// launches included, runs in mode 0, which behaves exactly like a classic launch.
#pragma once
#include <stdint.h>
#include "bulk_copy.cuh"       // bulk_wait_all

namespace ozl {

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// thread 0 of the CTA, after the trigger: wait until the tile's previous step has been released
__device__ __forceinline__ void tile_chain_wait(const unsigned long long* seq, unsigned long long step) {
    while (ld_acquire_u64(seq + 1) != step) __nanosleep(64);
}

}  // namespace ozl
