// Shared helpers for the octm kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/octm.h"

namespace octm {

// ---------------------------------------------------------------- host-side error plumbing
extern thread_local char g_last_error[512];
extern std::atomic<uint64_t> g_launches;

inline int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
    va_end(ap);
    return code;
}

inline int check_launch(const char* what) {
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(OCTM_ERR_LAUNCH, "%s: %s", what, cudaGetErrorString(e));
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return OCTM_OK;
}

// ---------------------------------------------------------------- per-kernel device timing (octm_profile_*)
// Off by default: a launch site costs one relaxed atomic load.  When enabled, every kernel launch of the
// library is bracketed by two CUDA events on ITS launch stream; octm_profile_report() turns them into
// per-kernel totals.  Used by bench.py on separate, untimed steps (never inside a timed region).
extern std::atomic<int> g_profile;
struct ProfScope {
    int slot;
    bool first;
    cudaStream_t stream;
    ProfScope(const char* name, cudaStream_t s) : slot(-1), first(true), stream(s) {
        if (g_profile.load(std::memory_order_relaxed)) begin(name);
    }
    ~ProfScope() {
        if (slot >= 0) end();
    }
    bool once() {
        const bool f = first;
        first = false;
        return f;
    }
    void begin(const char* name);
    void end();
};
#define OCTM_TIMED(name, stream) for (octm::ProfScope octm_ps_(name, stream); octm_ps_.once();)

int sm_count();            // SMs of the current device (cached per device)
// label_pass.cu: did the certificate reject more than a fifth of the maps of the last certified label pass on this device
// (or is that pinned by octm_label_pass_seed_policy)?  Speed heuristics only: results never depend on it.
bool stream_mostly_rejected();
int max_optin_smem();      // cudaDevAttrMaxSharedMemoryPerBlockOptin of the current device

// Persistent grid: min(want, the CTAs of `kern` resident at once on the current device); `fallback` CTAs per SM when the
// occupancy query fails.
template <class Kernel>
long long resident_grid(long long want, Kernel kern, int threads, size_t smem, int fallback) {
    int fit = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, kern, threads, smem) != cudaSuccess || fit < 1) {
        cudaGetLastError();
        fit = fallback;
    }
    const long long cap = static_cast<long long>(sm_count()) * fit;
    return want < cap ? want : cap;
}

// A zeroed, host-mapped uint32[2] per device and slot, allocated on first use: a one-thread kernel leaves a report in it
// and a later call reads it on the host without synchronisation.  nullptr when no cell can be had.
enum { kReportSeeds = 0, kReportWalks = 1 };      // label_pass.cu: rejected maps / maps; contour.cu: walks / contours
struct HostReport {
    uint32_t* host = nullptr;      // mapped, pinned
    uint32_t* dev = nullptr;       // the device's view of it
};
HostReport* host_report(int slot);

// contour.cu: the argument checks every contour entry point shares
int check_shape(int64_t n, int H, int W, int K, int max_pts);

// contour.cu: the contour workspace holds the vertices [n][K][2][max_pts] and the squared distances (same shape), each
// rounded up to 256 bytes, then a tail of words at tail_offset.  Without a workspace only tail_offset is set.
struct ContourWorkspace {
    size_t tail_offset;
    uint32_t* verts = nullptr;
    uint32_t* d2 = nullptr;
    uint32_t* tail = nullptr;
};
ContourWorkspace contour_workspace(int64_t n_items, int K, int max_pts, void* workspace = nullptr);

#ifdef __CUDACC__
// ---------------------------------------------------------------- device-side PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}

// Same wait for a thread that is expected to wait long (the producer, always a ring ahead): the
// suspend-time hint parks the thread in hardware instead of spinning on the issue port shared with
// the consumer warps of its scheduler.
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
            : "memory");
    } while (!done);
}

// L2 eviction policy for data that is read exactly once.
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}

// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
// dst, src 16-byte aligned; bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar,
                                         uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// TMA 2-D tiled copy global -> shared through a tensor map (SASS: UTMALDG), completion on an mbarrier.
// Out-of-range rows / columns of the box are filled with zeros and still count as transferred bytes.
__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const void* tmap, int x, int y, uint32_t bar_smem, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::
            "r"(dst_smem),
        "l"(tmap), "r"(x), "r"(y), "r"(bar_smem), "l"(policy)
        : "memory");
}

// mbarrier operations on raw shared-memory addresses (no generic -> shared conversion per call)
__device__ __forceinline__ void mbar_init_a(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_parked_a(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity), "r"(20000u)
            : "memory");
    } while (!done);
}

// orders prior generic-proxy accesses to shared memory before later async-proxy (TMA) accesses
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
// exclusive prefix SUM over the threads of a CTA (blockDim a multiple of 32, <= 1024) in thread order;
// s_warp: 33 elements of shared memory; `total` receives the sum over all threads.  Three CTA barriers.
template <class T>
__device__ __forceinline__ T block_excl_scan_sum(T v, T* s_warp, T& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        T w = s_warp[lane];
        T wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T n = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += n;
        }
        s_warp[lane] = wi - w;
        if (lane == 31) s_warp[32] = wi;
    }
    __syncthreads();
    const T res = s_warp[warp] + incl - v;
    total = s_warp[32];
    __syncthreads();
    return res;
}

#endif  // __CUDACC__

}  // namespace octm
