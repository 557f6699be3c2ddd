// gru_pred.cu -- one layer of the GRU normal-state predictor (reference models/predictor.py:84-111) at hidden 128,
// forward only: the frozen predictor's recurrence on the residual builder's windows.
//
// torch.nn.GRU equations and gate order (r, z, n), h_0 = 0:
//   r = sigma(gx_r + W_hr h),  z = sigma(gx_z + W_hz h),  n = tanh(gx_n + r * (W_hn h + b_hn)),  h' = (1 - z) n + z h
// where gx = x W_ih^T + b_ih (+ b_hr, b_hz folded into the r and z columns) is computed beforehand for every
// (sequence, step) row by ltgnn_linear: it is off the recurrence's critical path.
//
// The sensor-encoder kernel (gru.cu) keeps the whole recurrent weight resident in one SM; at H = 128 W_hh split hi/lo
// is 384 KiB and does not fit.  Here a CLUSTER of 4 CTAs owns a tile of 128 sequences for all L steps:
//   * CTA `rank` owns hidden units [32 rank, +32): its 96 x 128 slice of W_hh (r, z, hn rows of those units) is resident
//     in shared memory as TF32 hi/lo (96 KiB), ordered as two accumulator blocks of 48 rows (16 units x r | z | hn) so that
//     the gates of block 0 overlap the MMAs of block 1;
//   * every CTA holds the FULL h_{t-1} [128 x 128] as the A operand in tensor memory (hi | lo, 256 columns) next to a
//     96-column accumulator: each step is 16 K-steps x 3 tcgen05.mma (3xTF32, fp32-faithful) per block;
//   * 8 gate warps (thread = one sequence x 16 units) read the accumulator, add the gx row prefetched a step ahead, update
//     h in registers, store their slice into their own A columns and send it through distributed shared memory to the
//     3 peers (16 KiB per peer per step, double-buffered: 96 KiB of receive space);
//   * one cluster barrier per step publishes the slices; each CTA then moves what it received into its A columns.
// Shared memory 192 KiB + alignment; tensor memory 352 of 512 columns.  No atomics, fixed order: bitwise deterministic.
#include "umma.cuh"
#include "rowgemm_ts.cuh"

using namespace ltgnn;
using namespace ltgnn::ptx;
using namespace ltgnn::umma;
using ltgnn::rowgemm_ts::mma_tf32_ts;
using ltgnn::rowgemm_ts::tmem_wait_st;

namespace {

constexpr int H = 128;               // hidden size supported by this kernel
constexpr int kCluster = 4;          // CTAs per tile
constexpr int kUnits = H / kCluster; // 32 hidden units per CTA
constexpr int NB = 3 * kUnits;       // 96 rows of the resident W_hh slice
constexpr int kBlk = NB / 2;         // 48: one accumulator block = 16 units x (r | z | hn)
constexpr int kGateWarps = 8;
constexpr int kMmaWarp = kGateWarps;
constexpr int kThreads = (kGateWarps + 1) * 32;
constexpr uint32_t kAccCol = 0, kAhiCol = 128, kAloCol = 256;  // TMEM column map (352 of 512 used)
constexpr uint32_t kBBytes = NB * H * 4;                        // one of b_hi / b_lo: 48 KiB
constexpr uint32_t kSlotBytes = 128 * kUnits * 4;               // one peer's slice of h: 16 KiB
constexpr uint32_t kRecvBytes = 2 * (kCluster - 1) * kSlotBytes;  // double-buffered, 3 peers: 96 KiB
constexpr size_t kSmem = 1024 + 2ull * kBBytes + kRecvBytes;

struct GruLayerParams {
    const float* gx;    // [3][Q * L][H]: gate group g of row q * L + t
    const float* w_hh;  // [3H, H]
    const float* b_hn;  // [H]
    float* hseq;        // [Q, L, H] or nullptr
    float* h_last;      // [Q, H]
    uint32_t Q;
    int L;
    size_t plane;       // Q * L * H: floats per gate group of gx
};

// same fast forms as the sensor GRU (gru.cu)
__device__ __forceinline__ float rcp_approx(float v) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float sigmoidf_fast(float v) { return rcp_approx(1.f + __expf(-v)); }
__device__ __forceinline__ float tanhf_fast(float v) { return fmaf(2.f, rcp_approx(1.f + __expf(-2.f * v)), -1.f); }

__device__ __forceinline__ void load16(const float* src, float* v) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float4 a = ldg_stream(s4 + j);
        v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
    }
}
__device__ __forceinline__ void store16(float* dst, const float* v) {
    float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int j = 0; j < 4; ++j) stg_stream(d4 + j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
}
__device__ __forceinline__ void split16_store(uint32_t t_hi, uint32_t t_lo, const float* v) {
    float hi[16], lo[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) { hi[j] = tf32_hi(v[j]); lo[j] = v[j] - hi[j]; }
    tmem_st16(t_hi, hi);
    tmem_st16(t_lo, lo);
}

__global__ void __launch_bounds__(kThreads, 1)
gru_layer_fwd_kernel(const GruLayerParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_a, bar_d[2];
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;                 // B[n][k], n = 48 u + 16 g + jj <-> gate g of unit 32 rank + 16 u + jj
    uint8_t* b_lo = b_hi + kBBytes;
    uint8_t* recv = b_lo + kBBytes;       // [2 parity][3 slots][8 float4 columns][128 rows] float4

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const uint32_t tile = blockIdx.x / kCluster;
    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        mbar_init(&bar_a, kGateWarps);
        mbar_init(&bar_d[0], 1);
        mbar_init(&bar_d[1], 1);
        fence_mbar_init();
    }
    for (int i = tid; i < NB * (H / 4); i += kThreads) {
        const int n = i >> 5, c = i & 31;
        const int u = n / kBlk, g = (n % kBlk) >> 4, jj = n & 15;
        const int row = g * H + kUnits * static_cast<int>(rank) + 16 * u + jj;
        float4 hi, lo;
        split4(__ldg(reinterpret_cast<const float4*>(p.w_hh + static_cast<size_t>(row) * H) + c), hi, lo);
        const uint32_t off = sw128_offset(n, c, NB);
        *reinterpret_cast<float4*>(b_hi + off) = hi;
        *reinterpret_cast<float4*>(b_lo + off) = lo;
    }
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    cluster_sync();  // every peer is running (its receive buffer exists) before the first remote store
    const uint32_t tmem = tmem_base_s;
    const int L = p.L;

    if (warp < kGateWarps) {
        // warp (quad, half): TMEM lanes / sequences 32 quad .. +31, units u0 = 32 rank + 16 half .. +15 (accumulator block
        // `half`).  Half 0 finishes its gates while the tensor core still computes block 1.
        const int quad = warp & 3, half = warp >> 2;
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        const int r = quad * 32 + lane;
        const uint32_t q = tile * 128 + r;
        const bool valid = q < p.Q;
        const int u0 = kUnits * static_cast<int>(rank) + 16 * half;
        float bhn[16], h[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            bhn[j] = __ldg(p.b_hn + u0 + j);
            h[j] = 0.f;
        }
        const size_t row0 = static_cast<size_t>(valid ? q : 0) * L;  // gx / hseq row of step 0
        float gr[16], gz[16], gn[16];
        auto load_gx = [&](int t) {
            if (valid) {
                const float* src = p.gx + (row0 + t) * H + u0;
                load16(src, gr);
                load16(src + p.plane, gz);
                load16(src + 2 * p.plane, gn);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) gr[j] = gz[j] = gn[j] = 0.f;
            }
        };
        // A(0) = h_{-1} = 0: this warp zeroes 64 of the 128 columns of its lanes (hi and lo)
        {
            float z16[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) z16[j] = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                tmem_st16(tmem + lane_off + kAhiCol + 64 * half + 16 * c, z16);
                tmem_st16(tmem + lane_off + kAloCol + 64 * half + 16 * c, z16);
            }
        }
        tmem_wait_st();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_a);
        load_gx(0);

        // where this thread's 16 units land in a peer's receive buffer, and where the peers' slices land in ours
        const uint32_t recv_s = smem_u32(recv);
        uint32_t ph = 0;
        for (int t = 0; t < L; ++t) {
            mbar_wait(&bar_d[half], ph);
            fence_after_sync();
            float rr[16], zz[16], hn[16];
            tmem_ld16(tmem + lane_off + kAccCol + kBlk * half + 0, rr);
            tmem_ld16(tmem + lane_off + kAccCol + kBlk * half + 16, zz);
            tmem_ld16(tmem + lane_off + kAccCol + kBlk * half + 32, hn);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float rg = sigmoidf_fast(gr[j] + rr[j]);
                const float zg = sigmoidf_fast(gz[j] + zz[j]);
                const float n = tanhf_fast(fmaf(rg, hn[j] + bhn[j], gn[j]));
                h[j] = fmaf(zg, h[j] - n, n);  // (1 - z) n + z h
            }
            if (t + 1 < L) load_gx(t + 1);  // in flight through the exchange and the next step's MMAs
            if (valid && p.hseq) store16(p.hseq + (row0 + t) * H + u0, h);
            if (t + 1 < L) {
                // 1. publish this slice to the 3 peers (float4 column 4 half + j of slot "from rank" in their buffer)
                const uint32_t par_off = static_cast<uint32_t>(t & 1) * (kCluster - 1) * kSlotBytes;
#pragma unroll
                for (uint32_t k = 1; k < kCluster; ++k) {
                    const uint32_t dst = (rank + k) & (kCluster - 1);
                    // in CTA dst, a slice from rank sits in slot ((rank - dst) mod 4) - 1 = (4 - k) - 1
                    const uint32_t base = mapa_shared(recv_s + par_off + (kCluster - 1 - k) * kSlotBytes, dst);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        st_cluster_v4(base + ((4 * half + j) * 128 + r) * 16,
                                      make_float4(h[4 * j], h[4 * j + 1], h[4 * j + 2], h[4 * j + 3]));
                }
                __syncwarp();  // the cluster barrier and tcgen05.st are warp-collective (.aligned)
                cluster_arrive();
                // 2. own slice into A once every MMA of this step has read it (block 1 commits last)
                if (half == 0) mbar_wait(&bar_d[1], ph);
                fence_after_sync();
                split16_store(tmem + lane_off + kAhiCol + u0, tmem + lane_off + kAloCol + u0, h);
                // 3. the peers' slices: units 16 half .. +15 of each
                __syncwarp();
                cluster_wait();
#pragma unroll
                for (uint32_t s = 0; s < kCluster - 1; ++s) {
                    const uint32_t src = (rank + s + 1) & (kCluster - 1);  // slot s holds CTA (rank + s + 1)'s units
                    const float4* in = reinterpret_cast<const float4*>(recv + par_off + s * kSlotBytes);
                    float v[16];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 a = in[(4 * half + j) * 128 + r];
                        v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
                    }
                    const uint32_t col = kUnits * src + 16 * half;
                    split16_store(tmem + lane_off + kAhiCol + col, tmem + lane_off + kAloCol + col, v);
                }
                tmem_wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a);
            }
            ph ^= 1;
        }
        if (valid) store16(p.h_last + static_cast<size_t>(q) * H + u0, h);
    } else {
        // ------------------------------- MMA issuer -------------------------------
        const uint32_t idesc = idesc_tf32(128, kBlk);
        const uint32_t bh = desc_lo(smem_u32(b_hi)), bl = desc_lo(smem_u32(b_lo));
        constexpr uint32_t kg_units = NB * 128u >> 4;    // one 32-column k-atom block of B (96 rows x 128 B)
        constexpr uint32_t blk_units = kBlk * 128u >> 4;  // 48 rows of B inside a k-atom block
        uint32_t ph = 0;
        for (int t = 0; t < L; ++t) {
            mbar_wait(&bar_a, ph);
            ph ^= 1;
            fence_after_sync();
            if (elect_one()) {
#pragma unroll
                for (uint32_t u = 0; u < 2; ++u) {
                    const uint32_t d = tmem + kAccCol + kBlk * u;
#pragma unroll
                    for (uint32_t ks = 0; ks < H / 8; ++ks) {
                        const uint32_t boff = (ks >> 2) * kg_units + u * blk_units + 2 * (ks & 3);
                        mma_tf32_ts(d, tmem + kAloCol + 8 * ks, bh + boff, idesc, ks == 0 ? 0u : 1u);  // small terms first
                        mma_tf32_ts(d, tmem + kAhiCol + 8 * ks, bl + boff, idesc, 1u);
                        mma_tf32_ts(d, tmem + kAhiCol + 8 * ks, bh + boff, idesc, 1u);
                    }
                    commit(&bar_d[u]);
                }
            }
            __syncwarp();
            if (t + 1 < L) cluster_sync();  // the gate warps' per-step barrier counts every thread of the cluster
        }
    }
    fence_before_sync();
    __syncthreads();
    cluster_sync();  // no CTA leaves while a peer could still address its shared memory
    if (warp == kMmaWarp) {
        fence_after_sync();
        tmem_dealloc(tmem, 512);
    }
}

}  // namespace

extern "C" int ltgnn_gru_layer_fwd(int device, int64_t Q, int32_t L, int32_t Hdim, const float* gx, const float* w_hh,
                                   const float* b_hn, float* hseq, float* h_last, void* stream_) {
    LTGNN_REQUIRE(Q > 0 && L > 0, LTGNN_E_ARG, "gru_layer_fwd: Q=%lld L=%d", static_cast<long long>(Q), L);
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_layer_fwd: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(Q < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_layer_fwd: too many sequences");
    LTGNN_REQUIRE(gx && w_hh && b_hn && h_last, LTGNN_E_ARG, "gru_layer_fwd: null tensor");
    LTGNN_REQUIRE(aligned16(gx) && aligned16(w_hh) && aligned16(hseq) && aligned16(h_last), LTGNN_E_ALIGN,
                  "gru_layer_fwd: gx, w_hh, hseq and h_last must be 16-byte aligned");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "gru_layer_fwd: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_REQUIRE(kSmem <= static_cast<size_t>(di->smem_optin), LTGNN_E_SHAPE, "gru_layer_fwd: %zu B of shared memory", kSmem);
    LTGNN_USE_DEVICE(device);
    GruLayerParams p{gx, w_hh, b_hn, hseq, h_last, static_cast<uint32_t>(Q), L, static_cast<size_t>(Q) * L * H};
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gru_layer_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kSmem)));
    const int64_t tiles = (Q + 127) / 128;
    LTGNN_CUDA_TRY(launch_cluster(gru_layer_fwd_kernel, dim3(static_cast<unsigned>(tiles * kCluster)), dim3(kThreads), kSmem,
                                  static_cast<cudaStream_t>(stream_), kCluster, p));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}
