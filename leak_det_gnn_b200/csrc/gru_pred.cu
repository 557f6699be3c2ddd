// gru_pred.cu -- one layer of the GRU normal-state predictor (reference models/predictor.py:84-111) at hidden 128:
// the frozen predictor's recurrence on the residual builder's windows, and its training (saved-gates forward, backward
// through time, inter-layer dropout).
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
// The same kernel runs the shared sensor encoder at hidden 128 (kSensor): there the input term is formed in the gate
// threads from one residual and a time-feature projection shared by the window's sensors (ltgnn_gru_sensor_fwd).
// The windowed inference form (kWindows) runs overlapping windows of a series on one shared input projection: sequence q
// reads its step-t gx row at base[q] + t of a plane projected once per series row (ltgnn_gru_layer_fwd_windows).
#include "umma.cuh"
#include "rowgemm_ts.cuh"
#include "gru_dx.cuh"

using namespace ltgnn;
using namespace ltgnn::ptx;
using namespace ltgnn::umma;
using ltgnn::rowgemm_ts::mma_tf32_ts;
using ltgnn::rowgemm_ts::tmem_wait_st;
using ltgnn::ptx::launch_seed;
using ltgnn::ptx::philox4x32_7;

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
constexpr size_t kSensorSmem = kSmem + 3 * H * 4;                // + w_r for the sensor input form

struct GruLayerParams {
    const float* gx;    // [3][Q * L][H]: gate group g of row q * L + t
    const float* w_hh;  // [3H, H]
    const float* b_hn;  // [H]
    float* hseq;        // [Q, L, H] or nullptr
    float* h_last;      // [Q, H]
    uint32_t Q;
    int L;
    size_t plane;       // Q * L * H: floats per gate group of gx
    float* gates;       // training forward: [4][Q * L][H] = r | z | n | hn (hn = W_hn h_{t-1} + b_hn)
    // sensor input form: gx is T [3][B * L][H] (plane tplane) and sequence q = b S + s of the caller's B S sequences reads
    // gx_g = w_r[g] r[b, t, s] + T[g][b L + t]; local sequence q of this launch is sequence q0 + q of the B S
    const float* r_in;  // [B, L, S]
    const float* w_r;   // [3][H]: the residual column of W_ih
    uint32_t S;
    uint32_t q0;
    size_t tplane;      // B * L * H
    // windowed form: gx is [3][gx_rows][H] (plane gx_rows * H) and sequence q reads step t from row row_base[q] + t
    const int32_t* row_base;  // [Q]
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

// kTrain: also store every step's r, z, n and hn for the backward (hseq is then required).
// kSensor: the sensor encoder's input form (see GruLayerParams): one residual value and one T row per step instead of a
// gx row per sequence; every output is the planar form's, row (local q) L + t.
// kWindows (inference only): sequence q's gx rows start at row_base[q] instead of q L; hseq and h_last stay planar.
template <bool kTrain, bool kSensor = false, bool kWindows = false>
__global__ void __launch_bounds__(kThreads, 1)
gru_layer_fwd_kernel(const GruLayerParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_a, bar_d[2];
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;                 // B[n][k], n = 48 u + 16 g + jj <-> gate g of unit 32 rank + 16 u + jj
    uint8_t* b_lo = b_hi + kBBytes;
    uint8_t* recv = b_lo + kBBytes;       // [2 parity][3 slots][8 float4 columns][128 rows] float4
                                          // kSensor: then w_r [3][H] (kSensorSmem)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const uint32_t tile = blockIdx.x / kCluster;
    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if constexpr (kSensor) {
        for (int i = tid; i < 3 * H / 4; i += kThreads)
            reinterpret_cast<float4*>(recv + kRecvBytes)[i] = __ldg(reinterpret_cast<const float4*>(p.w_r) + i);
    }
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
        size_t xrow0 = row0;                                          // gx row of step 0
        if constexpr (kWindows) xrow0 = valid ? static_cast<size_t>(__ldg(p.row_base + q)) : 0;
        float gr[16], gz[16], gn[16];
        // sensor form: the T row of step 0 (b L) and the residual of step 0 (b L S + s)
        float xr = 0.f;
        size_t trow0 = 0;
        const float* rsrc = nullptr;
        if constexpr (kSensor) {
            const uint32_t qg = p.q0 + (valid ? q : 0), b = qg / p.S;
            trow0 = static_cast<size_t>(b) * L;
            rsrc = p.r_in + trow0 * p.S + (qg - b * p.S);
        }
        auto load_gx = [&](int t) {
            if (valid) {
                if constexpr (kSensor) {
                    const float* src = p.gx + (trow0 + t) * H + u0;
                    load16(src, gr);
                    load16(src + p.tplane, gz);
                    load16(src + 2 * p.tplane, gn);
                    xr = __ldg(rsrc + static_cast<size_t>(t) * p.S);
                } else {
                    const float* src = p.gx + (xrow0 + t) * H + u0;
                    load16(src, gr);
                    load16(src + p.plane, gz);
                    load16(src + 2 * p.plane, gn);
                }
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
                if constexpr (kSensor) {  // the input term, formed here so that its loads stay off the critical path
                    const float* wr = reinterpret_cast<const float*>(recv + kRecvBytes) + u0 + j;  // warp-uniform
                    gr[j] = fmaf(wr[0], xr, gr[j]);
                    gz[j] = fmaf(wr[H], xr, gz[j]);
                    gn[j] = fmaf(wr[2 * H], xr, gn[j]);
                }
                const float rg = sigmoidf_fast(gr[j] + rr[j]);
                const float zg = sigmoidf_fast(gz[j] + zz[j]);
                const float n = tanhf_fast(fmaf(rg, hn[j] + bhn[j], gn[j]));
                h[j] = fmaf(zg, h[j] - n, n);  // (1 - z) n + z h
                if constexpr (kTrain) {
                    rr[j] = rg;
                    zz[j] = zg;
                    gn[j] = n;
                    hn[j] += bhn[j];
                }
            }
            if constexpr (kTrain) {
                if (valid) {
                    float* g = p.gates + (row0 + t) * H + u0;
                    store16(g, rr);
                    store16(g + p.plane, zz);
                    store16(g + 2 * p.plane, gn);
                    store16(g + 3 * p.plane, hn);
                }
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


// =====================================================================================================
// backward through time of one layer, from the gates r | z | n | hn and the states the training forward saved.  Per step
// t = L-1 .. 0, with dh = d loss / d h_t (the carried gradient plus dh_seq[t], the gradient from the layer above):
//   dn_pre = dh (1 - z)(1 - n^2);  dz_pre = dh (h_{t-1} - n) z (1 - z);  dr_pre = dn_pre hn r (1 - r);  dhn = dn_pre r
//   dG(t) = [dr_pre | dz_pre | dn_pre | dhn]  -> HBM, planar, for the weight gradients (ltgnn_wgrad_tc)
//   dh_{t-1} = dh z + [dr_pre | dz_pre | dhn] [W_hr; W_hz; W_hn]
// The cluster shape is the forward's: CTA `rank` owns hidden units [32 rank, +32) and holds the 96 x 128 slice of W_hh
// of their r, z and hn rows, transposed to K-major (B[n = h column][k = 32 g + unit]), hi / lo in 96 KiB of shared memory.
// Its 96 gate columns (hi | lo, 192 tensor-memory columns) times that slice give a 128 x 128 PARTIAL of the contraction
// over the 3H gate rows (12 K-steps x 3 tcgen05.mma).  Each CTA sends the three 32-column blocks that belong to its peers
// into their double-buffered receive space (3 x 16 KiB per step, the forward's scheme); after one cluster barrier the
// owner adds the four partials in rank order.  Shared memory 192 KiB + alignment; tensor memory 320 of 512 columns.
// No atomics, fixed order: bitwise deterministic.
// =====================================================================================================
constexpr uint32_t kBwAccCol = 0, kBwAhiCol = H, kBwAloCol = H + NB;  // 128 | 96 | 96

struct GruLayerBwdParams {
    const float* w_hh;     // [3H, H]
    const float* gates;    // [4][Q * L][H]: r | z | n | hn
    const float* hseq;     // [Q * L][H]
    const float* dh_last;  // [Q, H] or nullptr
    const float* dh_seq;   // [Q * L][H] or nullptr
    float* dG;             // [4][Q * L][H]: dr_pre | dz_pre | dn_pre | dhn
    uint32_t Q;
    int L;
    size_t plane;          // Q * L * H
};

__global__ void __launch_bounds__(kThreads, 1)
gru_layer_bwd_kernel(const GruLayerBwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_a, bar_d;
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;                 // B[n][k] = w_hh[g H + 32 rank + u][n], k = 32 g + u: three k-atoms, one per gate
    uint8_t* b_lo = b_hi + kBBytes;
    uint8_t* recv = b_lo + kBBytes;       // [2 parity][3 slots][8 float4 columns][128 rows] float4

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const uint32_t tile = blockIdx.x / kCluster;
    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        mbar_init(&bar_a, kGateWarps);
        mbar_init(&bar_d, 1);
        fence_mbar_init();
    }
    for (int i = tid; i < NB * H; i += kThreads) {
        const int k = i / H, n = i - k * H;  // consecutive threads read consecutive columns of one W_hh row
        const int row = (k / kUnits) * H + kUnits * static_cast<int>(rank) + (k % kUnits);
        const float w = __ldg(p.w_hh + static_cast<size_t>(row) * H + n);
        const float hi = tf32_hi(w), lo = w - hi;
        const uint32_t off = sw128_offset(n, k >> 2, H) + (k & 3) * 4;
        *reinterpret_cast<float*>(b_hi + off) = hi;
        *reinterpret_cast<float*>(b_lo + off) = lo;
    }
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    cluster_sync();  // every peer is running (its receive buffer exists) before the first remote store
    const uint32_t tmem = tmem_base_s;
    const int L = p.L;

    if (warp < kGateWarps) {
        // warp (quad, half): TMEM lanes / sequences 32 quad .. +31, units u0 = 32 rank + 16 half .. +15
        const int quad = warp & 3, half = warp >> 2;
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        const int r = quad * 32 + lane;
        const uint32_t q = tile * 128 + r;
        const bool valid = q < p.Q;
        const int u0 = kUnits * static_cast<int>(rank) + 16 * half;
        const size_t row0 = static_cast<size_t>(valid ? q : 0) * L;
        float dh[16], gr[16], gz[16], gn[16], ghn[16], hm[16];
        auto zero16 = [](float* v) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = 0.f;
        };
        if (valid && p.dh_last) load16(p.dh_last + static_cast<size_t>(q) * H + u0, dh);
        else zero16(dh);
        auto load_step = [&](int t) {  // saved gates and h_{t-1} (zero at t = 0); zeros for pad rows
            if (valid) {
                const float* g = p.gates + (row0 + t) * H + u0;
                load16(g, gr);
                load16(g + p.plane, gz);
                load16(g + 2 * p.plane, gn);
                load16(g + 3 * p.plane, ghn);
                if (t > 0) load16(p.hseq + (row0 + t - 1) * H + u0, hm);
                else zero16(hm);
            } else {
                zero16(gr); zero16(gz); zero16(gn); zero16(ghn); zero16(hm);
            }
        };
        // the gradient from the layer above, dh_seq[t], joins the carried gradient before step t (its load is issued
        // while the previous step's MMAs run)
        const bool seq = valid && p.dh_seq;
        auto add_seq = [&](const float* ds) {
#pragma unroll
            for (int j = 0; j < 16; ++j) dh[j] += ds[j];
        };
        if (seq) {
            float ds[16];
            load16(p.dh_seq + (row0 + L - 1) * H + u0, ds);
            add_seq(ds);
        }
        load_step(L - 1);
        const uint32_t recv_s = smem_u32(recv);
        uint32_t ph = 0;
        for (int t = L - 1; t >= 0; --t) {
            // in place: gr <- dr_pre, gz <- dz_pre, gn <- dn_pre, ghn <- dhn, dh <- dh z
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float g = dh[j];
                const float rg = gr[j], zg = gz[j], n = gn[j];
                const float dnp = g * (1.f - zg) * (1.f - n * n);
                gz[j] = g * (hm[j] - n) * zg * (1.f - zg);
                gr[j] = dnp * ghn[j] * rg * (1.f - rg);
                ghn[j] = dnp * rg;
                gn[j] = dnp;
                dh[j] = g * zg;
            }
            if (valid) {
                float* d = p.dG + (row0 + t) * H + u0;
                store16(d, gr);
                store16(d + p.plane, gz);
                store16(d + 2 * p.plane, gn);
                store16(d + 3 * p.plane, ghn);
            }
            if (t == 0) break;  // dh_{-1} is not needed
            // A = this CTA's 96 gate columns [dr | dz | dhn] of its 32 units; the previous step's MMAs have completed
            // (their commit was waited for below), so the columns are free
            split16_store(tmem + lane_off + kBwAhiCol + 16 * half, tmem + lane_off + kBwAloCol + 16 * half, gr);
            split16_store(tmem + lane_off + kBwAhiCol + kUnits + 16 * half, tmem + lane_off + kBwAloCol + kUnits + 16 * half, gz);
            split16_store(tmem + lane_off + kBwAhiCol + 2 * kUnits + 16 * half,
                          tmem + lane_off + kBwAloCol + 2 * kUnits + 16 * half, ghn);
            tmem_wait_st();
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_a);
            float ds[16];
            if (seq) load16(p.dh_seq + (row0 + t - 1) * H + u0, ds);
            mbar_wait(&bar_d, ph);
            fence_after_sync();
            // 1. the peers' 32-column blocks of the partial into their receive space (slot of "from rank", as the forward)
            const uint32_t par_off = static_cast<uint32_t>(t & 1) * (kCluster - 1) * kSlotBytes;
#pragma unroll
            for (uint32_t k = 1; k < kCluster; ++k) {
                const uint32_t dst = (rank + k) & (kCluster - 1);
                float v[16];
                tmem_ld16(tmem + lane_off + kBwAccCol + kUnits * dst + 16 * half, v);
                const uint32_t base = mapa_shared(recv_s + par_off + (kCluster - 1 - k) * kSlotBytes, dst);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    st_cluster_v4(base + ((4 * half + j) * 128 + r) * 16,
                                  make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
            }
            if (seq) add_seq(ds);  // dh_{t-1} = (dh_t z + dh_seq[t-1]) + partial 0 + 1 + 2 + 3, in this order
            load_step(t - 1);      // in flight through the cluster barrier
            __syncwarp();      // the cluster barrier is warp-collective (.aligned)
            cluster_arrive();
            cluster_wait();
            // 2. the four partials of this thread's units, added to dh in rank order; the own one is still in the accumulator
            // (the next MMA waits for this step's bar_a arrival), so it is not held in registers across the barrier
#pragma unroll
            for (uint32_t c = 0; c < kCluster; ++c) {
                float v[16];
                if (c == rank) {
                    tmem_ld16(tmem + lane_off + kBwAccCol + kUnits * rank + 16 * half, v);
                } else {
                    const uint32_t s = (c - rank - 1) & (kCluster - 1);  // slot s holds CTA (rank + s + 1)'s partial
                    const float4* in = reinterpret_cast<const float4*>(recv + par_off + s * kSlotBytes);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 a = in[(4 * half + j) * 128 + r];
                        v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
                    }
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) dh[j] += v[j];
            }
            ph ^= 1;
        }
    } else {
        // ------------------------------- MMA issuer -------------------------------
        const uint32_t idesc = idesc_tf32(128, H);
        const uint32_t bh = desc_lo(smem_u32(b_hi)), bl = desc_lo(smem_u32(b_lo));
        constexpr uint32_t kg_units = H * 128u >> 4;  // one 32-column k-atom block of B (128 rows x 128 B)
        uint32_t ph = 0;
        for (int t = L - 1; t > 0; --t) {
            mbar_wait(&bar_a, ph);
            ph ^= 1;
            fence_after_sync();
            if (elect_one()) {
#pragma unroll
                for (uint32_t ks = 0; ks < NB / 8; ++ks) {
                    const uint32_t boff = (ks >> 2) * kg_units + 2 * (ks & 3);
                    mma_tf32_ts(tmem + kBwAccCol, tmem + kBwAloCol + 8 * ks, bh + boff, idesc, ks == 0 ? 0u : 1u);
                    mma_tf32_ts(tmem + kBwAccCol, tmem + kBwAhiCol + 8 * ks, bl + boff, idesc, 1u);
                    mma_tf32_ts(tmem + kBwAccCol, tmem + kBwAhiCol + 8 * ks, bh + boff, idesc, 1u);
                }
                commit(&bar_d);
            }
            __syncwarp();
            cluster_sync();  // the gate warps' per-step barrier counts every thread of the cluster
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

// ---- inter-layer dropout (nn.GRU applies it to every layer's output but the last, in train mode), off the recurrence.
// Thread = one 32-unit word of a row: y = x * keep / (1 - p) with Philox (launch seed + ltgnn_seed_source word), bit b
// of live[word] = unit 32 (word % 4) + b kept.  p = 0 copies x bit for bit.
__global__ void __launch_bounds__(256)
gru_dropout_kernel(const float4* __restrict__ x, uint32_t thresh, float keep_scale, uint64_t drop_seed,
                   const uint64_t* seed_src, float4* __restrict__ y, uint32_t* __restrict__ live, uint32_t n_words) {
    const uint32_t w = blockIdx.x * 256 + threadIdx.x;
    if (w >= n_words) return;
    const uint64_t seed = thresh ? launch_seed(drop_seed, seed_src) : 0;
    uint32_t bits = thresh ? 0u : ~0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint64_t idx4 = static_cast<uint64_t>(w) * 8 + j;
        float4 v = ldg_stream(x + idx4);
        if (thresh) {
            const uint4 rv = philox4x32_7(static_cast<uint32_t>(idx4), static_cast<uint32_t>(idx4 >> 32),
                                          static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
            const bool k0 = rv.x >= thresh, k1 = rv.y >= thresh, k2 = rv.z >= thresh, k3 = rv.w >= thresh;
            v.x = k0 ? v.x * keep_scale : 0.f;
            v.y = k1 ? v.y * keep_scale : 0.f;
            v.z = k2 ? v.z * keep_scale : 0.f;
            v.w = k3 ? v.w * keep_scale : 0.f;
            bits |= (static_cast<uint32_t>(k0) | static_cast<uint32_t>(k1) << 1 | static_cast<uint32_t>(k2) << 2 |
                     static_cast<uint32_t>(k3) << 3) << (4 * j);
        }
        stg_stream(y + idx4, v);
    }
    live[w] = bits;
}

// dx = (dy[0] + dy[1] + ...) * (live ? keep / (1 - p) : 1), the parts added in index order
__global__ void __launch_bounds__(256)
gru_dropout_bwd_kernel(const float4* __restrict__ dy, int n_parts, size_t plane4, const uint32_t* __restrict__ live,
                       float keep_scale, float4* __restrict__ dx, uint32_t n_words) {
    const uint32_t w = blockIdx.x * 256 + threadIdx.x;
    if (w >= n_words) return;
    const uint32_t bits = live ? __ldg(live + w) : ~0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const size_t idx4 = static_cast<size_t>(w) * 8 + j;
        float4 s = ldg_stream(dy + idx4);
        for (int k = 1; k < n_parts; ++k) {
            const float4 a = ldg_stream(dy + k * plane4 + idx4);
            s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
        }
        if (live) {
            const uint32_t nib = bits >> (4 * j);
            s.x = nib & 1u ? s.x * keep_scale : 0.f;
            s.y = nib & 2u ? s.y * keep_scale : 0.f;
            s.z = nib & 4u ? s.z * keep_scale : 0.f;
            s.w = nib & 8u ? s.w * keep_scale : 0.f;
        }
        stg_stream(dx + idx4, s);
    }
}

// the device and shape checks every entry point of this file makes
int check_device(int device, const char* fn, size_t smem = kSmem) {
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "%s: device is sm_%d%d, need sm_100", fn, di->cc_major,
                  di->cc_minor);
    LTGNN_REQUIRE(smem <= static_cast<size_t>(di->smem_optin), LTGNN_E_SHAPE, "%s: %zu B of shared memory", fn, smem);
    return LTGNN_OK;
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
    GruLayerParams p{gx, w_hh, b_hn, hseq, h_last, static_cast<uint32_t>(Q), L, static_cast<size_t>(Q) * L * H, nullptr};
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gru_layer_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kSmem)));
    const int64_t tiles = (Q + 127) / 128;
    LTGNN_CUDA_TRY(launch_cluster(gru_layer_fwd_kernel<false>, dim3(static_cast<unsigned>(tiles * kCluster)), dim3(kThreads), kSmem,
                                  static_cast<cudaStream_t>(stream_), kCluster, p));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_layer_fwd_train(int device, int64_t Q, int32_t L, int32_t Hdim, const float* gx, const float* w_hh,
                                         const float* b_hn, float* hseq, float* h_last, float* gates, void* stream_) {
    LTGNN_REQUIRE(Q > 0 && L > 0, LTGNN_E_ARG, "gru_layer_fwd_train: Q=%lld L=%d", static_cast<long long>(Q), L);
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_layer_fwd_train: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(Q < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_layer_fwd_train: too many sequences");
    LTGNN_REQUIRE(gx && w_hh && b_hn && hseq && h_last && gates, LTGNN_E_ARG, "gru_layer_fwd_train: null tensor");
    LTGNN_REQUIRE(aligned16(gx) && aligned16(w_hh) && aligned16(hseq) && aligned16(h_last) && aligned16(gates), LTGNN_E_ALIGN,
                  "gru_layer_fwd_train: gx, w_hh, hseq, h_last and gates must be 16-byte aligned");
    if (int rc = check_device(device, "gru_layer_fwd_train")) return rc;
    LTGNN_USE_DEVICE(device);
    GruLayerParams p{gx, w_hh, b_hn, hseq, h_last, static_cast<uint32_t>(Q), L, static_cast<size_t>(Q) * L * H, gates};
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gru_layer_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kSmem)));
    const int64_t tiles = (Q + 127) / 128;
    LTGNN_CUDA_TRY(launch_cluster(gru_layer_fwd_kernel<true>, dim3(static_cast<unsigned>(tiles * kCluster)), dim3(kThreads), kSmem,
                                  static_cast<cudaStream_t>(stream_), kCluster, p));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_sensor_fwd(int device, int64_t B, int32_t L, int32_t S, int64_t q0, int64_t Q, int32_t Hdim,
                                    const float* r, const float* tproj, const float* w_r, const float* w_hh,
                                    const float* b_hn, float* hseq, float* h_last, float* gates, void* stream_) {
    LTGNN_REQUIRE(B > 0 && L > 0 && S > 0 && q0 >= 0 && Q > 0 && q0 + Q <= B * S, LTGNN_E_ARG,
                  "gru_sensor_fwd: B=%lld L=%d S=%d q0=%lld Q=%lld", static_cast<long long>(B), L, S,
                  static_cast<long long>(q0), static_cast<long long>(Q));
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_sensor_fwd: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(B * S < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_sensor_fwd: too many sequences");
    LTGNN_REQUIRE(r && tproj && w_r && w_hh && b_hn && h_last && (hseq || !gates), LTGNN_E_ARG,
                  "gru_sensor_fwd: null tensor (gates needs hseq)");
    LTGNN_REQUIRE(aligned16(tproj) && aligned16(w_r) && aligned16(w_hh) && aligned16(hseq) && aligned16(h_last) &&
                  aligned16(gates), LTGNN_E_ALIGN, "gru_sensor_fwd: tproj, w_r, w_hh, hseq, h_last and gates must be 16-byte aligned");
    if (int rc = check_device(device, "gru_sensor_fwd", kSensorSmem)) return rc;
    LTGNN_USE_DEVICE(device);
    GruLayerParams p{tproj, w_hh, b_hn, hseq, h_last, static_cast<uint32_t>(Q), L, static_cast<size_t>(Q) * L * H, gates,
                     r, w_r, static_cast<uint32_t>(S), static_cast<uint32_t>(q0), static_cast<size_t>(B) * L * H};
    auto kernel = gates ? gru_layer_fwd_kernel<true, true> : gru_layer_fwd_kernel<false, true>;
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kSensorSmem)));
    const int64_t tiles = (Q + 127) / 128;
    LTGNN_CUDA_TRY(launch_cluster(kernel, dim3(static_cast<unsigned>(tiles * kCluster)), dim3(kThreads), kSensorSmem,
                                  static_cast<cudaStream_t>(stream_), kCluster, p));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_layer_fwd_windows(int device, int64_t Q, int32_t L, int32_t Hdim, const float* gx, int64_t gx_rows,
                                           const int32_t* row_base, const float* w_hh, const float* b_hn, float* hseq,
                                           float* h_last, void* stream_) {
    LTGNN_REQUIRE(Q > 0 && L > 0 && gx_rows >= L, LTGNN_E_ARG, "gru_layer_fwd_windows: Q=%lld L=%d gx_rows=%lld",
                  static_cast<long long>(Q), L, static_cast<long long>(gx_rows));
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_layer_fwd_windows: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(Q < (1ll << 31) - 128 && gx_rows < (1ll << 31), LTGNN_E_SHAPE,
                  "gru_layer_fwd_windows: too many sequences or gx rows");
    LTGNN_REQUIRE(gx && row_base && w_hh && b_hn && h_last, LTGNN_E_ARG, "gru_layer_fwd_windows: null tensor");
    LTGNN_REQUIRE(aligned16(gx) && aligned16(w_hh) && aligned16(hseq) && aligned16(h_last) &&
                  reinterpret_cast<uintptr_t>(row_base) % 4 == 0, LTGNN_E_ALIGN,
                  "gru_layer_fwd_windows: gx, w_hh, hseq and h_last must be 16-byte aligned, row_base 4-byte aligned");
    if (int rc = check_device(device, "gru_layer_fwd_windows")) return rc;
    LTGNN_USE_DEVICE(device);
    GruLayerParams p{gx, w_hh, b_hn, hseq, h_last, static_cast<uint32_t>(Q), L, static_cast<size_t>(gx_rows) * H, nullptr,
                     nullptr, nullptr, 0u, 0u, 0, row_base};
    auto kernel = gru_layer_fwd_kernel<false, false, true>;
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kSmem)));
    const int64_t tiles = (Q + 127) / 128;
    LTGNN_CUDA_TRY(launch_cluster(kernel, dim3(static_cast<unsigned>(tiles * kCluster)), dim3(kThreads), kSmem,
                                  static_cast<cudaStream_t>(stream_), kCluster, p));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_resident_tiles(int device, int32_t* tiles) {
    LTGNN_REQUIRE(tiles, LTGNN_E_ARG, "gru_resident_tiles: null output");
    if (int rc = check_device(device, "gru_resident_tiles", kSensorSmem)) return rc;
    LTGNN_USE_DEVICE(device);
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gru_layer_fwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(kSensorSmem)));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kCluster);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kSensorSmem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kCluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    LTGNN_CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, gru_layer_fwd_kernel<true, true>, &cfg));
    *tiles = n;
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_layer_bwd(int device, int64_t Q, int32_t L, int32_t Hdim, const float* w_hh, const float* gates,
                                   const float* hseq, const float* dh_last, const float* dh_seq, float* dG, void* stream_) {
    LTGNN_REQUIRE(Q > 0 && L > 0, LTGNN_E_ARG, "gru_layer_bwd: Q=%lld L=%d", static_cast<long long>(Q), L);
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_layer_bwd: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(Q < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_layer_bwd: too many sequences");
    LTGNN_REQUIRE(w_hh && gates && hseq && dG && (dh_last || dh_seq), LTGNN_E_ARG,
                  "gru_layer_bwd: null tensor (dh_last and dh_seq may not both be NULL)");
    LTGNN_REQUIRE(aligned16(w_hh) && aligned16(gates) && aligned16(hseq) && aligned16(dh_last) && aligned16(dh_seq) &&
                  aligned16(dG), LTGNN_E_ALIGN, "gru_layer_bwd: every tensor must be 16-byte aligned");
    if (int rc = check_device(device, "gru_layer_bwd")) return rc;
    LTGNN_USE_DEVICE(device);
    GruLayerBwdParams p{w_hh, gates, hseq, dh_last, dh_seq, dG, static_cast<uint32_t>(Q), L, static_cast<size_t>(Q) * L * H};
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gru_layer_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kSmem)));
    const int64_t tiles = (Q + 127) / 128;
    LTGNN_CUDA_TRY(launch_cluster(gru_layer_bwd_kernel, dim3(static_cast<unsigned>(tiles * kCluster)), dim3(kThreads), kSmem,
                                  static_cast<cudaStream_t>(stream_), kCluster, p));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_dropout(int device, int64_t M, int32_t Hdim, const float* x, float drop_p, uint64_t drop_seed,
                                 float* y, uint32_t* live, void* stream_) {
    LTGNN_REQUIRE(M > 0 && M < (1ll << 31), LTGNN_E_ARG, "gru_dropout: M=%lld", static_cast<long long>(M));
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_dropout: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, LTGNN_E_ARG, "gru_dropout: drop_p=%g", static_cast<double>(drop_p));
    LTGNN_REQUIRE(x && y && live, LTGNN_E_ARG, "gru_dropout: null tensor");
    LTGNN_REQUIRE(aligned16(x) && aligned16(y) && aligned16(live), LTGNN_E_ALIGN, "gru_dropout: 16-byte alignment");
    if (int rc = check_device(device, "gru_dropout")) return rc;
    LTGNN_USE_DEVICE(device);
    const double t = static_cast<double>(drop_p) * 4294967296.0;
    const uint32_t thresh = drop_p > 0.f ? static_cast<uint32_t>(t < 4294967295.0 ? t : 4294967295.0) : 0u;
    const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    const uint32_t n_words = static_cast<uint32_t>(M * (H / 32));
    gru_dropout_kernel<<<(n_words + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream_)>>>(
        reinterpret_cast<const float4*>(x), thresh, keep_scale, drop_seed, seed_source(), reinterpret_cast<float4*>(y), live,
        n_words);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_dropout_bwd(int device, int64_t M, int32_t Hdim, const float* dy, int32_t n_parts,
                                     const uint32_t* live, float drop_p, float* dx, void* stream_) {
    LTGNN_REQUIRE(M > 0 && M < (1ll << 31), LTGNN_E_ARG, "gru_dropout_bwd: M=%lld", static_cast<long long>(M));
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_dropout_bwd: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(n_parts >= 1 && n_parts <= 4, LTGNN_E_ARG, "gru_dropout_bwd: n_parts=%d", n_parts);
    LTGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, LTGNN_E_ARG, "gru_dropout_bwd: drop_p=%g", static_cast<double>(drop_p));
    LTGNN_REQUIRE(dy && dx, LTGNN_E_ARG, "gru_dropout_bwd: null tensor");
    LTGNN_REQUIRE(aligned16(dy) && aligned16(dx) && aligned16(live), LTGNN_E_ALIGN, "gru_dropout_bwd: 16-byte alignment");
    if (int rc = check_device(device, "gru_dropout_bwd")) return rc;
    LTGNN_USE_DEVICE(device);
    const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    const uint32_t n_words = static_cast<uint32_t>(M * (H / 32));
    gru_dropout_bwd_kernel<<<(n_words + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream_)>>>(
        reinterpret_cast<const float4*>(dy), n_parts, static_cast<size_t>(M) * (H / 4), live, keep_scale,
        reinterpret_cast<float4*>(dx), n_words);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

// ---- input gradient of the sensor encoder (gru_dx.cuh) from one slab's dG: input planes r, z, n = 0, 1, 2 of 4
namespace {
struct DgPlanarSlab {
    const float* dg;  // [4][Q * L][H], row (q - q0) L + t
    int64_t rows;     // Q * L
    size_t plane;     // Q * L * H
    uint32_t q0;
    int L;
    __device__ __forceinline__ bool decode(int64_t row, uint32_t& q, uint32_t& t) const {
        const uint32_t ql = static_cast<uint32_t>(row / L);
        t = static_cast<uint32_t>(row - static_cast<int64_t>(ql) * L);
        q = q0 + ql;
        return true;
    }
    // a thread reads its row's 512 contiguous bytes per plane: L1-allocating loads, so that the second float4 of each
    // 32-byte sector the warp fetched is served from L1
    __device__ __forceinline__ float4 load(int64_t row, int g, int j4) const {
        return __ldg(reinterpret_cast<const float4*>(dg + g * plane + static_cast<size_t>(row) * H) + j4);
    }
};
}  // namespace

extern "C" int ltgnn_gru_sensor_bwd_dx(int device, int64_t B, int32_t L, int32_t S, int32_t F, int64_t q0, int64_t Q,
                                       int32_t Hdim, const float* w_ih, const float* dG, float* dr, float* dxt,
                                       void* stream_) {
    LTGNN_REQUIRE(B > 0 && L > 0 && S > 0 && F >= 0 && q0 >= 0 && Q > 0 && q0 + Q <= B * S, LTGNN_E_ARG,
                  "gru_sensor_bwd_dx: B=%lld L=%d S=%d F=%d q0=%lld Q=%lld", static_cast<long long>(B), L, S, F,
                  static_cast<long long>(q0), static_cast<long long>(Q));
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_sensor_bwd_dx: hidden size %d not supported (128 only)", Hdim);
    LTGNN_REQUIRE(1 + F < gru_dx::kCols, LTGNN_E_SHAPE, "gru_sensor_bwd_dx: %d time features, at most %d", F,
                  gru_dx::kCols - 2);
    LTGNN_REQUIRE(B * S < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_sensor_bwd_dx: too many sequences");
    LTGNN_REQUIRE(w_ih && dG && (dr || dxt) && (F > 0 || !dxt), LTGNN_E_ARG,
                  "gru_sensor_bwd_dx: null tensor (dr or dxt required; dxt needs F > 0)");
    LTGNN_REQUIRE(aligned16(dG) && reinterpret_cast<uintptr_t>(w_ih) % 4 == 0 && reinterpret_cast<uintptr_t>(dr) % 4 == 0 &&
                  reinterpret_cast<uintptr_t>(dxt) % 4 == 0, LTGNN_E_ALIGN,
                  "gru_sensor_bwd_dx: dG must be 16-byte aligned, w_ih, dr and dxt 4-byte aligned");
    const size_t smem = gru_dx::smem_bytes(H);
    if (int rc = check_device(device, "gru_sensor_bwd_dx", smem)) return rc;
    LTGNN_USE_DEVICE(device);
    DgPlanarSlab lay{dG, Q * L, static_cast<size_t>(Q) * L * H, static_cast<uint32_t>(q0), L};
    auto kernel = gru_dx::gru_bwd_dx_kernel<H, DgPlanarSlab>;
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kernel<<<gru_dx::grid_for(lay.rows, device_info(device)->sm_count), gru_dx::kThreads, smem,
             static_cast<cudaStream_t>(stream_)>>>(lay, w_ih, dr, dxt, static_cast<uint32_t>(S), L, F,
                                                   S >= 2 ? (~0ull / static_cast<uint64_t>(S)) + 1 : 0ull);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}
