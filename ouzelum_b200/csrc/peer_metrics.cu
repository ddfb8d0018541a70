// Multi-GPU metrics exchange over NVLink peer memory: the path's ONE collective -- the sum of the 16-double episode / reward
// metrics vector over all ranks every few steps (config 4; the reference's trainers scan `infos` on the host instead,
// RPO-LSTM/main.py:105-113) -- fused into the kernel that reads the metrics, with no NCCL kernel, no side stream and no fork / join
// in the step graph.
//
// Why not NCCL here: the payload is 128 bytes.  Captured into the step graph, an NCCL all-reduce needs a side stream (fork + join
// edges break the chain of programmatic launches) and a kernel of its own; measured on 8 B200s it costs 4.7 us per K = 20 step
// window (4.40 -> 4.74 us per 16384-env step, 0.93 weak-scaling efficiency) although the ranks share nothing else.
//
// Protocol (the LL idea of NCCL, over cudaIpc-mapped peer buffers):
//   * every rank owns a mailbox: ring of R entries x world senders x 16 lines; a line is 16 bytes {double value, u64 tag}
//     written with ONE 16-byte store, so a line is self-validating -- no fence, no separate flag, no ordering assumption
//     between different stores crossing NVLink;
//   * push (ozl_metrics_push, one launch, PDL-chained behind the step like ozl_metrics_read): 16 warps reduce the handle's
//     striped metric slots, then lane r of warp j stores {sum_j, seq + 1} into line [seq % R][my rank][j] of rank r's mailbox
//     (its own included) -- `world` 16-byte stores per metric, fire and forget; the device-side `seq` counter advances, so the
//     launch takes no host-changing argument and is CUDA-graph capturable;
//   * sum (ozl_metrics_sum, or folded into the NEXT push): thread (j, r) polls line [cons % R][r][j] of the LOCAL mailbox until
//     its tag is cons + 1, thread j adds the `world` values in rank order (deterministic, identical on every rank), `cons`
//     advances.  The poll is bounded (10 s, OZL_XCHG_TIMEOUT_MS): on expiry the result is NaN and the mailbox's error word is set -- a dead peer must
//     not hang the GPU.
//   A sender may run at most R - 1 exchanges ahead of the slowest receiver's sum (R = 8); the bench sums every push before the
//   next one.
#include <cstdlib>
#include <cstring>
#include <new>
#include "internal.h"
#include "bulk_copy.cuh"

namespace ozl {

constexpr int kXRing = 8;          // exchanges in flight
constexpr int kXMaxWorld = 16;

struct XLine { double v; unsigned long long tag; };

struct XDev {                       // device-side view passed by value
    XLine* peer[kXMaxWorld];        // every rank's mailbox as mapped into THIS process (peer[rank] = the local one)
    unsigned long long* ctl;        // local: [0] seq (pushes issued), [1] cons (sums done), [2] error
    long long timeout_cycles;       // bound of the receive poll
    int rank, world;
};

__device__ __forceinline__ XLine* xline(XLine* box, int world, unsigned long long seq, int sender, int j) {
    return box + ((seq % kXRing) * (unsigned long long)world + (unsigned long long)sender) * 16ull + (unsigned long long)j;
}
__device__ __forceinline__ void st_line(XLine* p, double v, unsigned long long tag) {
    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(__double_as_longlong(v)), "l"(tag) : "memory");
}
__device__ __forceinline__ void ld_line(const XLine* p, double& v, unsigned long long& tag) {
    long long b;
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(b), "=l"(tag) : "l"(p) : "memory");
    v = __longlong_as_double(b);
}

// Receive side, warp j = metric j, lane r = sender r.  Every ring entry of (sender, metric) is loaded up front -- the loads do not
// depend on the `cons` counter, so they fly together with the control-word and metrics loads (one L2 round trip for the whole kernel
// instead of three dependent ones: 2.2 -> ~1 us per exchange inside the step graph) -- and the entry `c % R` is picked afterwards;
// only if its tag is not there yet does the lane fall into the bounded poll.
struct XPre { double v[kXRing]; unsigned long long tag[kXRing]; };
__device__ __forceinline__ void xpreload(const XDev& x, int j, int lane, XPre& p) {
#pragma unroll
    for (int e = 0; e < kXRing; ++e) { p.v[e] = 0.0; p.tag[e] = 0ull; }
    if (lane < x.world) {
#pragma unroll
        for (int e = 0; e < kXRing; ++e) ld_line(xline(x.peer[x.rank], x.world, (unsigned long long)e, lane, j), p.v[e], p.tag[e]);
    }
}
__device__ __forceinline__ double xsum_metric(const XDev& x, unsigned long long c, int j, int lane, const XPre& p) {
    const int slot = (int)(c % kXRing);
    double v = 0.0;
    unsigned long long tag = 0ull;
#pragma unroll
    for (int e = 0; e < kXRing; ++e) { if (e == slot) { v = p.v[e]; tag = p.tag[e]; } }
    bool ok = true;
    if (lane < x.world && tag != c + 1ull) {
        const XLine* q = xline(x.peer[x.rank], x.world, c, lane, j);
        const long long t0 = clock64();
        ld_line(q, v, tag);
        while (tag != c + 1ull) {
            if (clock64() - t0 > x.timeout_cycles) { ok = false; break; }
            __nanosleep(100);
            ld_line(q, v, tag);
        }
    }
    if (lane >= x.world) v = 0.0;
    // rank-ordered sum (identical on every rank): sender 0, 1, 2, ...
    double s = 0.0;
    for (int r = 0; r < x.world; ++r) s += __shfl_sync(0xffffffffu, v, r);
    if (!__all_sync(0xffffffffu, ok)) {
        s = __longlong_as_double(0x7ff8000000000000ll);
        if (lane == 0) x.ctl[2] = 1ull;
    }
    return s;
}

// grid 1 x 512 threads: warp j handles metric j
__global__ void metrics_push_kernel(const Planes pl, const XDev x, double* local16, double* prev_sum16, const int clear) {
    griddep_wait();
    griddep_launch_dependents();
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // every load of the kernel is issued here, before the first use
    const unsigned long long seq = x.ctl[0], cons = x.ctl[1];
    XPre pre;
    if (prev_sum16) xpreload(x, j, lane, pre);
    double v = 0.0;
    for (int s = lane; s < kMetricSlots; s += 32) v += pl.metrics[s * kMetricStride + j];
    // (1) fold in the sum of the previous exchange if it is still outstanding and the caller wants it
    if (prev_sum16 && cons < seq) {
        const double s = xsum_metric(x, cons, j, lane, pre);
        if (lane == 0) prev_sum16[j] = s;
    }
    // (2) this rank's metrics
    if (clear) { for (int s = lane; s < kMetricSlots; s += 32) pl.metrics[s * kMetricStride + j] = 0.0; }
    v = warp_sum(v);
    if (lane == 0 && local16) local16[j] = v;
    // (3) one 16-byte store per (metric, receiver) over NVLink
    if (lane < x.world) st_line(xline(x.peer[lane], x.world, seq, x.rank, j), v, seq + 1ull);
    __syncthreads();
    if (threadIdx.x == 0) {
        x.ctl[0] = seq + 1ull;
        if (prev_sum16 && cons < seq) x.ctl[1] = cons + 1ull;
    }
}

__global__ void metrics_sum_kernel(const XDev x, double* sum16) {
    griddep_wait();
    griddep_launch_dependents();
    const int j = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned long long seq = x.ctl[0], cons = x.ctl[1];
    XPre pre;
    xpreload(x, j, lane, pre);
    if (cons >= seq) return;                       // nothing outstanding: sum16 keeps its value
    const double s = xsum_metric(x, cons, j, lane, pre);
    if (lane == 0) sum16[j] = s;
    __syncthreads();
    if (threadIdx.x == 0) x.ctl[1] = cons + 1ull;
}

}  // namespace ozl

using namespace ozl;

struct ozl_metrics_xchg {
    int rank, world, device;
    void* box;                      // local mailbox (cudaMalloc)
    size_t box_bytes;
    unsigned long long* ctl;
    void* peer[kXMaxWorld];
    bool opened[kXMaxWorld];        // mapped with cudaIpcOpenMemHandle (to be closed)
    bool connected;
    long long timeout_cycles;
};

static size_t xbox_bytes(int world) { return (size_t)kXRing * world * 16 * sizeof(XLine); }

extern "C" int ozl_metrics_xchg_create(int32_t rank, int32_t world, int32_t device, ozl_metrics_xchg** out) {
    if (!out) return set_error("ozl_metrics_xchg_create: NULL argument");
    if (world < 1 || world > kXMaxWorld || rank < 0 || rank >= world)
        return set_error("ozl_metrics_xchg_create: rank %d / world %d outside 1..%d", rank, world, kXMaxWorld);
    if (check_cuda(cudaSetDevice(device), "cudaSetDevice")) return 1;
    ozl_metrics_xchg* x = new (std::nothrow) ozl_metrics_xchg();
    if (!x) return set_error("out of host memory");
    x->rank = rank; x->world = world; x->device = device; x->connected = (world == 1);
    {
        const char* tv = getenv("OZL_XCHG_TIMEOUT_MS");
        const long long ms = tv ? atoll(tv) : 10000ll;
        x->timeout_cycles = (ms > 0 ? ms : 10000ll) * 1900000ll;          // ~1.9 GHz SM clock
    }
    x->box_bytes = xbox_bytes(world) + 256;
    if (check_cuda(cudaMalloc(&x->box, x->box_bytes), "cudaMalloc(metrics mailbox)")) { delete x; return 1; }
    if (check_cuda(cudaMemset(x->box, 0, x->box_bytes), "cudaMemset(metrics mailbox)")) { cudaFree(x->box); delete x; return 1; }
    x->ctl = (unsigned long long*)((char*)x->box + xbox_bytes(world));
    for (int r = 0; r < kXMaxWorld; ++r) { x->peer[r] = nullptr; x->opened[r] = false; }
    x->peer[rank] = x->box;
    if (check_cuda(cudaDeviceSynchronize(), "cudaDeviceSynchronize")) { cudaFree(x->box); delete x; return 1; }
    *out = x;
    return 0;
}

extern "C" int ozl_metrics_xchg_destroy(ozl_metrics_xchg* x) {
    if (!x) return 0;
    cudaSetDevice(x->device);
    for (int r = 0; r < x->world; ++r)
        if (x->opened[r]) cudaIpcCloseMemHandle(x->peer[r]);
    cudaFree(x->box);
    delete x;
    return 0;
}

extern "C" int ozl_metrics_xchg_ipc_handle(ozl_metrics_xchg* x, void* handle64) {
    if (!x || !handle64) return set_error("ozl_metrics_xchg_ipc_handle: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t h;
    if (check_cuda(cudaSetDevice(x->device), "cudaSetDevice")) return 1;
    if (check_cuda(cudaIpcGetMemHandle(&h, x->box), "cudaIpcGetMemHandle")) return 1;
    memcpy(handle64, &h, 64);
    return 0;
}

extern "C" int ozl_metrics_xchg_connect_ipc(ozl_metrics_xchg* x, const void* handles64xWorld) {
    if (!x || !handles64xWorld) return set_error("ozl_metrics_xchg_connect_ipc: NULL argument");
    if (getenv("OZL_XCHG_FAIL_IPC")) return set_error("ozl_metrics_xchg_connect_ipc: refused (OZL_XCHG_FAIL_IPC is set: fallback test)");
    if (check_cuda(cudaSetDevice(x->device), "cudaSetDevice")) return 1;
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank || x->peer[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles64xWorld + 64 * (size_t)r, 64);
        void* p = nullptr;
        if (check_cuda(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle(peer metrics mailbox)")) return 1;
        x->peer[r] = p; x->opened[r] = true;
    }
    x->connected = true;
    return 0;
}

extern "C" int ozl_metrics_xchg_connect_ptrs(ozl_metrics_xchg* x, void* const* boxes, const int32_t* devices) {
    if (!x || !boxes || !devices) return set_error("ozl_metrics_xchg_connect_ptrs: NULL argument");
    if (check_cuda(cudaSetDevice(x->device), "cudaSetDevice")) return 1;
    for (int r = 0; r < x->world; ++r) {
        if (r == x->rank) continue;
        if (!boxes[r]) return set_error("ozl_metrics_xchg_connect_ptrs: mailbox of rank %d is NULL", r);
        if (devices[r] != x->device) {
            int can = 0;
            if (check_cuda(cudaDeviceCanAccessPeer(&can, x->device, devices[r]), "cudaDeviceCanAccessPeer")) return 1;
            if (!can) return set_error("ozl_metrics_xchg_connect_ptrs: device %d cannot access device %d", x->device, devices[r]);
            const cudaError_t e = cudaDeviceEnablePeerAccess(devices[r], 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (check_cuda(e, "cudaDeviceEnablePeerAccess")) return 1;
        }
        x->peer[r] = boxes[r];
    }
    x->connected = true;
    return 0;
}

extern "C" int ozl_metrics_xchg_box(ozl_metrics_xchg* x, void** out) {
    if (!x || !out) return set_error("ozl_metrics_xchg_box: NULL argument");
    *out = x->box;
    return 0;
}

static int xdev_of(ozl_metrics_xchg* x, XDev& d, const char* who) {
    if (!x) return set_error("%s: NULL exchange", who);
    if (!x->connected) return set_error("%s: the exchange is not connected to its peers (ozl_metrics_xchg_connect_*)", who);
    for (int r = 0; r < kXMaxWorld; ++r) d.peer[r] = (XLine*)(r < x->world ? x->peer[r] : nullptr);
    d.ctl = x->ctl; d.rank = x->rank; d.world = x->world; d.timeout_cycles = x->timeout_cycles;
    return 0;
}

extern "C" int ozl_metrics_push(ozl_env* env, ozl_metrics_xchg* x, double* local16, double* prev_sum16, int32_t clear, void* stream) {
    if (!env) return set_error("ozl_metrics_push: NULL env");
    XDev d;
    if (xdev_of(x, d, "ozl_metrics_push")) return 1;
    if (x->device != env->device) return set_error("ozl_metrics_push: exchange on device %d, env on device %d", x->device, env->device);
    if (launch_pdl(metrics_push_kernel, dim3(1), dim3(512), (cudaStream_t)stream, env->pl, d, local16, prev_sum16, (int)clear))
        return check_cuda(cudaGetLastError(), "metrics_push_kernel");
    return 0;
}

extern "C" int ozl_metrics_sum(ozl_env* env, ozl_metrics_xchg* x, double* sum16, void* stream) {
    if (!env || !sum16) return set_error("ozl_metrics_sum: NULL argument");
    XDev d;
    if (xdev_of(x, d, "ozl_metrics_sum")) return 1;
    if (launch_pdl(metrics_sum_kernel, dim3(1), dim3(512), (cudaStream_t)stream, d, sum16))
        return check_cuda(cudaGetLastError(), "metrics_sum_kernel");
    return 0;
}

extern "C" int ozl_metrics_xchg_status(ozl_metrics_xchg* x, uint64_t* pushed, uint64_t* summed, uint64_t* error, void* stream) {
    if (!x) return set_error("ozl_metrics_xchg_status: NULL exchange");
    unsigned long long w[3];
    if (check_cuda(cudaMemcpyAsync(w, x->ctl, sizeof(w), cudaMemcpyDeviceToHost, (cudaStream_t)stream), "cudaMemcpyAsync")) return 1;
    if (check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "cudaStreamSynchronize")) return 1;
    if (pushed) *pushed = w[0];
    if (summed) *summed = w[1];
    if (error) *error = w[2];
    return 0;
}
