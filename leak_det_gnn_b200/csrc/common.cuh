// common.cuh -- shared host/device helpers for libltgnn (sm_100a only).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <utility>

#include "ltgnn.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libltgnn is written for sm_100a (Blackwell B200) only"
#endif

// ------------------------------------------------------------------------------------
// host side: error reporting + graph handle
// ------------------------------------------------------------------------------------
namespace ltgnn {

int fail(int code, const char* fmt, ...);  // records the thread-local message, returns code

#define LTGNN_CUDA_TRY(expr)                                                                         \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return ::ltgnn::fail(LTGNN_E_CUDA, "%s -> %s (%s:%d)", #expr, cudaGetErrorString(e__),   \
                                 __FILE__, __LINE__);                                                \
    } while (0)

#define LTGNN_REQUIRE(cond, code, ...)                      \
    do {                                                    \
        if (!(cond)) return ::ltgnn::fail(code, __VA_ARGS__); \
    } while (0)

// Every entry point runs on the device its tensors live on and leaves the caller's current device untouched
// (torch keeps its own notion of the current device; a stray cudaSetDevice would redirect later allocations).
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t enter(int device) {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) return e;
        if (prev != device) {
            e = cudaSetDevice(device);
            switched = (e == cudaSuccess);
        }
        return e;
    }
    ~DeviceGuard() {
        if (switched) cudaSetDevice(prev);
    }
};
#define LTGNN_USE_DEVICE(dev)           \
    ::ltgnn::DeviceGuard dev_guard__;   \
    LTGNN_CUDA_TRY(dev_guard__.enter(dev))

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// cuTensorMapEncodeTiled resolved through the runtime (no -lcuda link dependency)
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_tmapEncodeTiled tmap_encode_fn();

// per-device facts, queried once (cudaGetDeviceProperties costs ~1 ms per call)
struct DeviceInfo {
    bool ok = false;
    int cc_major = 0, cc_minor = 0;
    int sm_count = 0;
    int smem_optin = 0;   // max dynamic shared memory per block
    int smem_per_sm = 0;
};
// returns nullptr (and records the error) if the device cannot be queried
const DeviceInfo* device_info(int device);

// Launch `kernel` as clusters of `cluster_x` CTAs along x (grid.x must be a multiple of it).  A plain cudaLaunchKernelEx:
// capturable into a CUDA graph like a <<<>>> launch.
template <typename... Params, typename... Args>
cudaError_t launch_cluster(void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                           unsigned cluster_x, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster_x;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// out[i] (+)= sum_{c < n_parts} parts[c * stride + i], i < n, added in index order: the deterministic
// second stage of every cross-CTA reduction in this library (no float atomics anywhere)
int reduce_parts(const float* parts, int64_t stride, float* out, int n_parts, int n, int accumulate,
                 cudaStream_t stream);

// Device word the calling thread registered with ltgnn_seed_source (or nullptr): every dropout-bearing launch made from
// that thread hands it to its kernel, which adds the word -- read when the kernel RUNS -- to its drop_seed argument.
const uint64_t* seed_source();

}  // namespace ltgnn

struct ltgnn_graph {
    int device = 0;
    int sm_count = 0;
    int smem_optin = 0;  // max dynamic shared memory per block (opt-in), bytes
    int32_t n = 0;
    int32_t nnz = 0;
    // index 0: A_hat (row = target), index 1: A_hat^T (row = source)
    int32_t* rowptr[2] = {nullptr, nullptr};
    int2* colval[2] = {nullptr, nullptr};  // .x = column, .y = fp32 bits of the weight
    int32_t max_row_len[2] = {0, 0};
};

// ------------------------------------------------------------------------------------
// device side: PTX wrappers (mbarrier, TMA, tcgen05)
// ------------------------------------------------------------------------------------
namespace ltgnn {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// make mbarrier.init visible to the async (TMA / tcgen05) proxy
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// order generic-proxy smem writes before async-proxy reads (tcgen05.mma / TMA store)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Blocking wait with a watchdog: a lost arrival traps (launch fails with an error) instead of hanging
// the GPU.  try_wait itself suspends the warp in hardware for a bounded time, so the loop body is cold;
// 2^26 failed probes is seconds, real waits are microseconds.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
#ifdef LTGNN_DEBUG_WAIT
        if (++spins > (1u << 22)) {
            if ((threadIdx.x & 31) == 0) printf("mbar_wait timeout: block %d warp %d bar %x parity %u\n", blockIdx.x, threadIdx.x >> 5, smem_u32(bar), parity);
            __trap();
        }
#else
        if (++spins > (1u << 26)) __trap();
#endif
    }
}
// Same for waits that are NOT on the critical path (a producer running ahead of its consumer): the explicit
// suspend-time hint (ns) keeps the warp asleep longer per probe, so its polling does not take issue slots
// from the warps the SM is actually waiting for.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
            : "memory");
        if (ok) break;
#ifdef LTGNN_DEBUG_WAIT
        if (++spins > (1u << 16)) {
            if ((threadIdx.x & 31) == 0) printf("mbar_wait_relaxed timeout: block %d warp %d bar %x parity %u\n", blockIdx.x, threadIdx.x >> 5, smem_u32(bar), parity);
            __trap();
        }
#else
        if (++spins > (1u << 24)) __trap();
#endif
    }
}

// 3-D tiled TMA load global -> shared, completion on an mbarrier (coordinates innermost first)
__device__ __forceinline__ void tma_load_3d(void* dst_smem, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1,
                                            int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// 1-D bulk copy global -> shared (TMA without a tensor map): bytes a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// generic-proxy writes (global and shared) of this thread become visible to later async-proxy (TMA) accesses
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}

// streaming 128-bit global accesses (data touched once: keep it out of L1)
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void stg_stream(float4* p, const float4& v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// ---- counter-based RNG for dropout: Philox4x32 with 7 rounds (Salmon et al. 2011; 7 rounds pass
// BigCrush).  One call yields the four keep/drop decisions of one float4.  Statistically equivalent to,
// not bit-identical with, torch's dropout stream (SURVEY.md section 7 "Dropout RNG parity").
__device__ __forceinline__ uint4 philox4x32_7(uint32_t c0, uint32_t c1, uint32_t k0, uint32_t k1) {
    uint32_t c2 = 0x9E3779B9u, c3 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 7; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0;
        c1 = l1;
        c2 = h0 ^ c3 ^ k1;
        c3 = l0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
// seed of this launch: the drop_seed argument, plus the device-resident word of ltgnn_seed_source when one is set
__device__ __forceinline__ uint64_t launch_seed(uint64_t seed, const uint64_t* src) {
    return src ? seed + __ldg(reinterpret_cast<const unsigned long long*>(src)) : seed;
}
// inverted dropout on the float4 whose linear float4 index is `idx4`; thresh = p * 2^32
__device__ __forceinline__ void dropout4(float4& v, uint64_t idx4, uint64_t seed, uint32_t thresh, float keep_scale) {
    const uint4 r = philox4x32_7(static_cast<uint32_t>(idx4), static_cast<uint32_t>(idx4 >> 32),
                                 static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
    v.x = r.x >= thresh ? v.x * keep_scale : 0.f;
    v.y = r.y >= thresh ? v.y * keep_scale : 0.f;
    v.z = r.z >= thresh ? v.z * keep_scale : 0.f;
    v.w = r.w >= thresh ? v.w * keep_scale : 0.f;
}
// Same, 16 random bits per element: one Philox call decides 8 elements (v[0..7]); thresh16 = round(p * 2^16)
// and the caller scales by 1 / (1 - thresh16 / 2^16) so the estimator stays exactly unbiased.
__device__ __forceinline__ void dropout8(float* v, uint64_t idx8, uint64_t seed, uint32_t thresh16, float keep_scale) {
    const uint4 r = philox4x32_7(static_cast<uint32_t>(idx8), static_cast<uint32_t>(idx8 >> 32) ^ 0x5bd1e995u,
                                 static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = (w[i] & 0xffffu) >= thresh16 ? v[2 * i] * keep_scale : 0.f;
        v[2 * i + 1] = (w[i] >> 16) >= thresh16 ? v[2 * i + 1] * keep_scale : 0.f;
    }
}
// Same keep / drop decisions as dropout8 without the rescale (the caller folded 1 / (1 - p) into the producer of v).
// thresh_hi = thresh16 << 16: the high half of a word is compared in place, the low half after one shift.
__device__ __forceinline__ void dropout8_mask(float* v, uint64_t idx8, uint64_t seed, uint32_t thresh_hi) {
    const uint4 r = philox4x32_7(static_cast<uint32_t>(idx8), static_cast<uint32_t>(idx8 >> 32) ^ 0x5bd1e995u,
                                 static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = (w[i] << 16) >= thresh_hi ? v[2 * i] : 0.f;
        v[2 * i + 1] = w[i] >= thresh_hi ? v[2 * i + 1] : 0.f;
    }
}
// 16-bit-lane variant for a single float4 (same keep probability and scale as dropout8)
__device__ __forceinline__ void dropout4h(float4& v, uint64_t idx4, uint64_t seed, uint32_t thresh16, float keep_scale) {
    const uint4 r = philox4x32_7(static_cast<uint32_t>(idx4), static_cast<uint32_t>(idx4 >> 32) ^ 0x2545f491u,
                                 static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
    v.x = (r.x & 0xffffu) >= thresh16 ? v.x * keep_scale : 0.f;
    v.y = (r.x >> 16) >= thresh16 ? v.y * keep_scale : 0.f;
    v.z = (r.y & 0xffffu) >= thresh16 ? v.z * keep_scale : 0.f;
    v.w = (r.y >> 16) >= thresh16 ? v.w * keep_scale : 0.f;
}
// "Blocked-32" layout of row-per-thread tensors ([rows, W] logical): element (row, 4*f4 .. 4*f4+3) lives at float4
// index ((row / 32) * W/4 + f4) * 32 + row % 32.  A thread owns a row, so the 32 lanes of a warp read / write 512
// contiguous bytes per instruction instead of 32 segments a row apart (row-major costs 32 LSU wavefronts each).
__device__ __forceinline__ size_t b32(size_t row, int f4, int w4) { return ((row >> 5) * w4 + f4) * 32 + (row & 31); }

// exact floor(x / d) for any 32-bit x: magic = floor((2^64 - 1) / d) + 1 (host side, d >= 2)
__device__ __forceinline__ uint32_t fastdiv(uint32_t x, uint64_t magic) {
    return static_cast<uint32_t>(__umul64hi(static_cast<uint64_t>(x), magic));
}

// ---- thread-block clusters: distributed shared memory and the cluster-wide barrier ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// the shared::cluster address of the same shared::cta offset in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_v4(uint32_t addr, const float4& v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
// Every thread of every CTA of the cluster arrives (release: its shared::cluster writes are published) and later waits
// (acquire: the peers' writes before their arrive are visible).  Between the two a thread may do unrelated work.
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync() {
    cluster_arrive();
    cluster_wait();
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

}  // namespace ptx
}  // namespace ltgnn
