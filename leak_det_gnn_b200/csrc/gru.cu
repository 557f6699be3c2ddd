// gru.cu -- the shared per-sensor GRU encoder that feeds the message-passing path (SURVEY.md 8f, rank 2).
//
// Reference: models/detector.py:28-73 -- `nn.GRU(input_size=1+9, hidden_size=64, batch_first=True)` over
// B*S sequences of L steps (input = [residual_s(t), 9 time features of the window]); only the last hidden
// state is used.  The reference (and round-1's drop-in) call cuDNN, which at B*S = 118 784, L = 288 spends
// ~225 ms forward / ~450 ms backward on 1 TFLOP of recurrent GEMM (per-timestep launches, 4 TFLOP/s).
//
// Here: one persistent CTA per SM owns a tile of 128 sequences for all L steps.
//   * the recurrent weights AND the input weights AND the biases form ONE resident tensor-core operand
//     B[4H x 96] (rows: r | z | W_hn h + b_hn | W_in x + b_in; columns: h(64) | x(1) | tf(9) | 1 | 0-pad),
//     split TF32 hi/lo in shared memory (192 KB);
//   * the state lives in TENSOR MEMORY: A[128 x 96] = [h_{t-1} | x_t | tf_t | 1] as hi/lo columns, written
//     by the gate warps with tcgen05.st, consumed by tcgen05.mma (A from TMEM, 3xTF32) into a 256-column
//     accumulator -- the hidden state never touches shared or global memory between steps;
//   * 8 gate warps (thread = one sequence x 32 hidden units) read the four pre-activation groups with
//     tcgen05.ld, apply sigmoid/tanh, update h in registers and store the next A.
// PyTorch gate order and equations (torch.nn.GRU): r, z, n;  n = tanh(W_in x + b_in + r * (W_hn h + b_hn));
// h' = (1 - z) * n + z * h.
#include "umma.cuh"
#include "rowgemm_ts.cuh"
#include "tgrad.cuh"
#include "gru_dx.cuh"

using namespace ltgnn;
using namespace ltgnn::ptx;
using namespace ltgnn::umma;
using ltgnn::rowgemm_ts::mma_tf32_ts;
using ltgnn::rowgemm_ts::tmem_wait_st;

namespace {

constexpr int H = 64;            // hidden size supported by this kernel
constexpr int KA = 96;           // augmented K: h(64) | x | tf(F <= 29) | 1 | pad
constexpr int NG = 4 * H;        // 256 accumulator columns
constexpr int kGateWarps = 8;
constexpr int kAuxIn = 31;       // x + up to 30 time features, held in registers one step ahead
constexpr int kMmaWarp = kGateWarps;
constexpr int kThreads = (kGateWarps + 1) * 32;
constexpr uint32_t kAccCol = 0, kAhiCol = NG, kAloCol = NG + KA;  // TMEM column map (448 of 512 used)
constexpr int kDg3W4 = 3 * H / 4;  // float4 per row of the saved r | z | n

struct GruParams {
    const float* r;      // [B, L, S]
    const float* tf;     // [B, L, F] or nullptr (F = 0)
    const float* w_ih;   // [3H, 1 + F]
    const float* w_hh;   // [3H, H]
    const float* b_ih;   // [3H]
    const float* b_hh;   // [3H]
    float* h_last;       // [Q, H]
    float* hseq;         // blocked-32 [L * Qp, H] or nullptr
    float* gates;        // blocked-32 [L * Qp, 3H] (r | z | n: the backward rebuilds W_hn h + b_hn) or nullptr
    uint32_t Q;          // B * S sequences
    uint32_t Qp;         // Q rounded up to a multiple of 128
    int L, S, F;
    uint64_t magic_s;    // fastdiv constant of S (S >= 2), 0 when S == 1
};

__device__ __forceinline__ float rcp_approx(float v) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float sigmoidf_fast(float v) { return rcp_approx(1.f + __expf(-v)); }
__device__ __forceinline__ float tanhf_fast(float v) { return fmaf(2.f, rcp_approx(1.f + __expf(-2.f * v)), -1.f); }

// saved tensors use the blocked-32 layout (common.cuh): rows = t * Qp + q with Qp = Q rounded up to 128

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]),
          "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
        : "memory");
}

// element (n, k) of the fused operand described in the file header.  Rows are ordered in 4 blocks of 64 so that
// the step GEMM can be issued as 4 independent N = 64 accumulator blocks, block u holding all four gate
// pre-activations of hidden units [16u, 16u + 16):  n = 64 u + 16 g + jj  <->  gate g, unit 16 u + jj.
__device__ __forceinline__ float fused_weight(const GruParams& p, int n, int k) {
    const int g = (n >> 4) & 3, j = ((n >> 6) << 4) | (n & 15);
    const int fi = 1 + p.F;  // row length of w_ih
    const int kx = H, kb = H + 1 + p.F;  // column of x, column of the constant 1
    if (g < 2) {
        const int row = g * H + j;
        if (k < H) return __ldg(p.w_hh + row * H + k);
        if (k >= kx && k < kb) return __ldg(p.w_ih + row * fi + (k - kx));
        if (k == kb) return __ldg(p.b_ih + row) + __ldg(p.b_hh + row);
        return 0.f;
    }
    const int row = 2 * H + j;
    if (g == 2) {
        if (k < H) return __ldg(p.w_hh + row * H + k);
        if (k == kb) return __ldg(p.b_hh + row);
        return 0.f;
    }
    if (k >= kx && k < kb) return __ldg(p.w_ih + row * fi + (k - kx));
    if (k == kb) return __ldg(p.b_ih + row);
    return 0.f;
}

__global__ void __launch_bounds__(kThreads, 1)
gru_fwd_kernel(const GruParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_a, bar_d[4];
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;
    uint8_t* b_lo = b_hi + NG * KA * 4;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        mbar_init(&bar_a, kGateWarps);
        for (int u = 0; u < 4; ++u) mbar_init(&bar_d[u], 1);
        fence_mbar_init();
    }
    for (int i = tid; i < NG * KA; i += kThreads) {
        const int n = i / KA, k = i - n * KA;
        const float w = fused_weight(p, n, k);
        const float hi = tf32_hi(w);
        const uint32_t off = sw128_offset(n, k >> 2, NG) + (k & 3) * 4;
        *reinterpret_cast<float*>(b_hi + off) = hi;
        *reinterpret_cast<float*>(b_lo + off) = w - hi;
    }
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = tmem_base_s;
    const uint32_t n_tiles = (p.Q + 127) / 128;
    uint32_t ph_a = 0, ph_d = 0;  // phases of the two barriers, advanced identically by every role

    if (warp < kGateWarps) {
        // warp (quad, half): TMEM lanes 32 quad .. +31; accumulator blocks u = half and half + 2, i.e. hidden
        // units [16 half, +16) and [32 + 16 half, +16).  The tensor core produces the 4 blocks one after the
        // other, so the sigmoid / tanh work of block u overlaps the MMAs of blocks u+1...
        const int quad = warp & 3, half = warp >> 2;
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const uint32_t q = tile * 128 + quad * 32 + lane;  // sequence index = b * S + s
            const bool valid = q < p.Q;
            const uint32_t b = p.magic_s ? fastdiv(valid ? q : 0, p.magic_s) : (valid ? q : 0);
            const uint32_t s = (valid ? q : 0) - b * p.S;
            const float* rp = p.r + static_cast<size_t>(b) * p.L * p.S + s;      // + t * S
            const float* tp = p.tf ? p.tf + static_cast<size_t>(b) * p.L * p.F : nullptr;  // + t * F
            float h[32];  // h[16 pass + jj] = unit 16 (half + 2 pass) + jj
#pragma unroll
            for (int j = 0; j < 32; ++j) h[j] = 0.f;

            // ---- A(0) = [0 | x_0 | tf_0 | 1]
            {
                float z16[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) z16[j] = 0.f;
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    tmem_st16(tmem + lane_off + kAhiCol + 16 * (half + 2 * pass), z16);
                    tmem_st16(tmem + lane_off + kAloCol + 16 * (half + 2 * pass), z16);
                }
            }
            // columns 64..95 of A for step t (half 0 warps only).  The inputs do not depend on the recurrence: they
            // are fetched one step ahead (load_aux at the top of step t - 1) so that their L2 / HBM latency is not
            // paid between the last gate and the next MMA.
            float xin[kAuxIn];
            auto load_aux = [&](int t) {
#pragma unroll
                for (int j = 0; j < kAuxIn; ++j) xin[j] = 0.f;
                if (valid && t < p.L) {
                    xin[0] = __ldg(rp + static_cast<size_t>(t) * p.S);
#pragma unroll
                    for (int j = 1; j < kAuxIn; ++j)  // compile-time register indices
                        if (j <= p.F) xin[j] = __ldg(tp + static_cast<size_t>(t) * p.F + (j - 1));
                }
            };
            auto store_aux = [&]() {
                float a[32], lo[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) a[j] = j < kAuxIn ? xin[j] : 0.f;
                // the constant-one column sits right after the time features
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (j == 1 + p.F) a[j] = 1.f;
                    const float hi = tf32_hi(a[j]);
                    lo[j] = a[j] - hi;
                    a[j] = hi;
                }
                rowgemm_ts::tmem_st32(tmem + lane_off + kAhiCol + H, a);
                rowgemm_ts::tmem_st32(tmem + lane_off + kAloCol + H, lo);
            };
            if (half == 0) {
                load_aux(0);
                store_aux();
            }
            tmem_wait_st();
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_a);

            for (int t = 0; t < p.L; ++t) {
                const size_t row = static_cast<size_t>(t) * p.Qp + q;
                if (half == 0) load_aux(t + 1);  // in flight while this step's MMAs and gates run
                float hhi[32], hlo[32];
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    const int u = half + 2 * pass;
                    mbar_wait(&bar_d[u], ph_d);
                    fence_after_sync();
                    float rr[16], zz[16], hn[16], in[16];
                    tmem_ld16(tmem + lane_off + kAccCol + 64 * u + 0, rr);
                    tmem_ld16(tmem + lane_off + kAccCol + 64 * u + 16, zz);
                    tmem_ld16(tmem + lane_off + kAccCol + 64 * u + 32, hn);
                    tmem_ld16(tmem + lane_off + kAccCol + 64 * u + 48, in);
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float r = sigmoidf_fast(rr[j]);
                        const float z = sigmoidf_fast(zz[j]);
                        const float n = tanhf_fast(fmaf(r, hn[j], in[j]));
                        const float hv = fmaf(z, h[16 * pass + j] - n, n);  // (1 - z) n + z h
                        h[16 * pass + j] = hv;
                        hhi[16 * pass + j] = tf32_hi(hv);
                        hlo[16 * pass + j] = hv - hhi[16 * pass + j];
                        rr[j] = r;
                        zz[j] = z;
                        in[j] = n;
                    }
                    const int f0 = 4 * u;  // float4 index of unit 16 u within a 64-wide group
                    if (p.gates) {
                        float4* g4 = reinterpret_cast<float4*>(p.gates);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            stg_stream(g4 + b32(row, 0 * (H / 4) + f0 + j, kDg3W4), make_float4(rr[4 * j], rr[4 * j + 1], rr[4 * j + 2], rr[4 * j + 3]));
                            stg_stream(g4 + b32(row, 1 * (H / 4) + f0 + j, kDg3W4), make_float4(zz[4 * j], zz[4 * j + 1], zz[4 * j + 2], zz[4 * j + 3]));
                            stg_stream(g4 + b32(row, 2 * (H / 4) + f0 + j, kDg3W4), make_float4(in[4 * j], in[4 * j + 1], in[4 * j + 2], in[4 * j + 3]));
                        }
                    }
                    if (p.hseq) {
                        float4* h4 = reinterpret_cast<float4*>(p.hseq);
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            stg_stream(h4 + b32(row, f0 + j, H / 4),
                                       make_float4(h[16 * pass + 4 * j], h[16 * pass + 4 * j + 1], h[16 * pass + 4 * j + 2],
                                                   h[16 * pass + 4 * j + 3]));
                    }
                }
                if (t + 1 < p.L) {
                    // A may only be overwritten once every MMA of this step has read it: block 3 commits last
                    if (half == 0) mbar_wait(&bar_d[3], ph_d);
                    fence_after_sync();
#pragma unroll
                    for (int pass = 0; pass < 2; ++pass) {
                        tmem_st16(tmem + lane_off + kAhiCol + 16 * (half + 2 * pass), hhi + 16 * pass);
                        tmem_st16(tmem + lane_off + kAloCol + 16 * (half + 2 * pass), hlo + 16 * pass);
                    }
                    if (half == 0) store_aux();
                    tmem_wait_st();
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bar_a);
                }
                ph_d ^= 1;
            }
            if (valid) {
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    float4* dst = reinterpret_cast<float4*>(p.h_last + static_cast<size_t>(q) * H + 16 * (half + 2 * pass));
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        dst[j] = make_float4(h[16 * pass + 4 * j], h[16 * pass + 4 * j + 1], h[16 * pass + 4 * j + 2],
                                             h[16 * pass + 4 * j + 3]);
                }
            }
            // the next tile's A(0) store must not overtake the last MMAs of this tile
            if (half == 0) mbar_wait(&bar_d[3], ph_d ^ 1);
            fence_before_sync();
        }
    } else {
        // ------------------------------- MMA issuer -------------------------------
        const uint32_t idesc = idesc_tf32(128, 64);
        const uint32_t bh = desc_lo(smem_u32(b_hi)), bl = desc_lo(smem_u32(b_lo));
        constexpr uint32_t kg_units = NG * 128u >> 4;   // one 32-column k-atom block of B (256 rows x 128 B)
        constexpr uint32_t blk_units = 64 * 128u >> 4;  // 64 rows of B inside a k-atom block
        const uint32_t n_ks = static_cast<uint32_t>(H + p.F + 2 + 7) / 8;  // K-steps that hold data: 10 for F = 9
        for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int t = 0; t < p.L; ++t) {
                mbar_wait(&bar_a, ph_a);
                ph_a ^= 1;
                fence_after_sync();
                if (elect_one()) {
#pragma unroll
                    for (uint32_t u = 0; u < 4; ++u) {
                        const uint32_t d = tmem + kAccCol + 64 * u;
                        for (uint32_t ks = 0; ks < n_ks; ++ks) {
                            const uint32_t boff = (ks >> 2) * kg_units + u * blk_units + 2 * (ks & 3);
                            mma_tf32_ts(d, tmem + kAloCol + 8 * ks, bh + boff, idesc, ks == 0 ? 0u : 1u);
                            mma_tf32_ts(d, tmem + kAhiCol + 8 * ks, bl + boff, idesc, 1u);
                            mma_tf32_ts(d, tmem + kAhiCol + 8 * ks, bh + boff, idesc, 1u);
                        }
                        commit(&bar_d[u]);
                    }
                }
                __syncwarp();
            }
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == kMmaWarp) {
        fence_after_sync();
        tmem_dealloc(tmem, 512);
    }
}


// =====================================================================================================
// backward through time, from the gates r, z, n and the states the forward saved.  Per step t = L-1 .. 0 and tile of 128
// sequences, with dh = d loss / d h_t:
//   hn = W_hn h_{t-1} + b_hn                       rebuilt by one 64-column tcgen05 GEMM (A = h_{t-1} hi / lo in TMEM)
//   dn = dh (1 - z);  dn_pre = dn (1 - n^2);  dz_pre = dh (h_{t-1} - n) z (1 - z);
//   dr_pre = dn_pre * hn * r (1 - r);  dhn = dn_pre * r;  din = dn_pre
//   dG(t) = [dr_pre | dz_pre | dhn | din]  -> written to HBM for the weight-gradient GEMM (tgrad.cuh)
//   dh_{t-1} = dh z + [dr_pre | dz_pre | dhn] [W_hr; W_hz; W_hn]      (second tcgen05 GEMM, A = dG hi / lo in TMEM)
// No transcendental is recomputed.  Rebuilding hn instead of saving it spares the forward's writes and the BPTT's reads
// of one gate group (8.75 GB at B*S = 118 784, L = 288); the second MMA round trip stays under the HBM time of the step.
// Tensor memory (448 of 512 columns): dh accumulator 64 | 192 columns that hold the hn accumulator (the first 64), then
// dG lo | 192 columns that hold h_{t-1} hi + lo (the first 128), then dG hi.  Every reuse is by the thread that owned the
// columns, after the MMA that read them has committed.
// =====================================================================================================
constexpr int KB = 3 * H;  // 192: K of the dh_{t-1} GEMM
constexpr uint32_t kR_accDh = 0, kR_accR = H, kR_a = H + KB;  // 64 | 192 | 192
constexpr int kGateWarpsHn = 16, kThreadsHn = kGateWarpsHn * 32;  // 4 gate warps per scheduler hide the loads

__device__ __forceinline__ void tmem_st4(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]),
                 "f"(v[3])
                 : "memory");
}

struct GruBwdHnParams {
    const float* w_hh;     // [3H, H]
    const float* b_hh;     // [3H]
    const float* gates;    // blocked-32 [L * Qp, 3H]: r | z | n
    const float* hseq;     // blocked-32 [L * Qp, H]
    const float* dh_last;  // [Q, H]
    float* dG;             // blocked-32 [L * Qp, 4H]
    uint32_t Q, Qp;
    int L;
};

__global__ void __launch_bounds__(kThreadsHn, 1)
gru_bwd_hn_kernel(const GruBwdHnParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_a1, bar_a2, bar_r, bar_d;
    __shared__ uint32_t tmem_base_s;
    __shared__ float4 bhn_s[H / 4];  // b_hh of the n rows
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b1_hi = smem;                  // B1[n = unit (64)][k = h column (64)] = w_hh[2H + n][k], K-major SW128
    uint8_t* b1_lo = b1_hi + H * H * 4;
    uint8_t* b2_hi = b1_lo + H * H * 4;     // B2[n = h column (64)][k = gate row (192)] = w_hh[k][n], K-major SW128
    uint8_t* b2_lo = b2_hi + H * KB * 4;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        mbar_init(&bar_a1, kGateWarpsHn);
        mbar_init(&bar_a2, kGateWarpsHn);
        mbar_init(&bar_r, 1);
        mbar_init(&bar_d, 1);
        fence_mbar_init();
    }
    for (int i = tid; i < KB * H; i += kThreadsHn) {
        const int k = i / H, n = i - k * H;  // w_hh[k][n]: k = gate row, n = h column
        const float w = __ldg(p.w_hh + i);
        const float hi = tf32_hi(w), lo = w - hi;
        const uint32_t o2 = sw128_offset(n, k >> 2, H) + (k & 3) * 4;
        *reinterpret_cast<float*>(b2_hi + o2) = hi;
        *reinterpret_cast<float*>(b2_lo + o2) = lo;
        if (k >= 2 * H) {
            const uint32_t o1 = sw128_offset(k - 2 * H, n >> 2, H) + (n & 3) * 4;
            *reinterpret_cast<float*>(b1_hi + o1) = hi;
            *reinterpret_cast<float*>(b1_lo + o1) = lo;
        }
    }
    if (tid < H) reinterpret_cast<float*>(bhn_s)[tid] = __ldg(p.b_hh + 2 * H + tid);
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = tmem_base_s;
    const uint32_t n_tiles = (p.Q + 127) / 128;
    uint32_t ph = 0;  // one phase bit serves all four barriers: each completes exactly once per step

    {
        // 16 gate warps: thread = one sequence (TMEM lane) x 16 hidden units [16 part, +16).  Warp 0 also issues the
        // two GEMMs of a step (it would only wait for them otherwise): 16 warps = 4 per scheduler, 128 registers each.
        const uint32_t idesc1 = idesc_tf32(128, H), idesc2 = idesc_tf32(128, H);
        const uint32_t b1h = desc_lo(smem_u32(b1_hi)), b1l = desc_lo(smem_u32(b1_lo));
        const uint32_t b2h = desc_lo(smem_u32(b2_hi)), b2l = desc_lo(smem_u32(b2_lo));
        constexpr uint32_t kg1 = H * 128u >> 4, kg2 = H * 128u >> 4;  // one 32-column k-atom block of B1 / B2
        const int quad = warp & 3, part = warp >> 2;
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        const int j0 = part * 16;
        const float4* h4 = reinterpret_cast<const float4*>(p.hseq);
        float4* dg4 = reinterpret_cast<float4*>(p.dG);
        for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const uint32_t q = tile * 128 + quad * 32 + lane;
            const bool valid = q < p.Q;
            const float4* g4 = reinterpret_cast<const float4*>(p.gates);
            float dh[16], hm[16];
            {
                const float4* src = reinterpret_cast<const float4*>(p.dh_last + static_cast<size_t>(valid ? q : 0) * H + j0);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 v = valid ? __ldg(src + j) : make_float4(0.f, 0.f, 0.f, 0.f);
                    dh[4 * j] = v.x; dh[4 * j + 1] = v.y; dh[4 * j + 2] = v.z; dh[4 * j + 3] = v.w;
                }
            }
            auto load_h = [&](int t) {  // h_{t-1}[j0 .. j0 + 16): zero for t = 0 and for pad rows
                const size_t prow = static_cast<size_t>(t > 0 ? t - 1 : 0) * p.Qp + q;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 v = (valid && t > 0) ? ldg_stream(h4 + b32(prow, (j0 >> 2) + j, H / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    hm[4 * j] = v.x; hm[4 * j + 1] = v.y; hm[4 * j + 2] = v.z; hm[4 * j + 3] = v.w;
                }
            };
            load_h(p.L - 1);
            for (int t = p.L - 1; t >= 0; --t) {
                const size_t row = static_cast<size_t>(t) * p.Qp + q;
                // ---- A = h_{t-1} (hi | lo), this thread's 16 of the 64 columns
#pragma unroll
                for (int c = 0; c < 16; c += 16) {
                    float hi[16], lo[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) { hi[j] = tf32_hi(hm[c + j]); lo[j] = hm[c + j] - hi[j]; }
                    tmem_st16(tmem + lane_off + kR_a + j0 + c, hi);
                    tmem_st16(tmem + lane_off + kR_a + H + j0 + c, lo);
                }
                tmem_wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a1);
                {
                    const int f0 = j0 >> 2;  // float4 index of this thread's units inside a 64-wide group
                    // saved r | z | n: requested before the first GEMM is waited for
                    float4 r4[4], z4[4], n4[4];
                    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        r4[j] = valid ? ldg_stream(g4 + b32(row, 0 * (H / 4) + f0 + j, kDg3W4)) : zero;
                        z4[j] = valid ? ldg_stream(g4 + b32(row, 1 * (H / 4) + f0 + j, kDg3W4)) : zero;
                        n4[j] = valid ? ldg_stream(g4 + b32(row, 2 * (H / 4) + f0 + j, kDg3W4)) : zero;
                    }
                    if (warp == 0) {  // hn pre-activations = h_{t-1} W_hn^T
                        mbar_wait(&bar_a1, ph);
                        fence_after_sync();
                        if (elect_one()) {
#pragma unroll
                            for (uint32_t ks = 0; ks < H / 8; ++ks) {
                                const uint32_t boff = (ks >> 2) * kg1 + 2 * (ks & 3);
                                mma_tf32_ts(tmem + kR_accR, tmem + kR_a + H + 8 * ks, b1h + boff, idesc1, ks == 0 ? 0u : 1u);
                                mma_tf32_ts(tmem + kR_accR, tmem + kR_a + 8 * ks, b1l + boff, idesc1, 1u);
                                mma_tf32_ts(tmem + kR_accR, tmem + kR_a + 8 * ks, b1h + boff, idesc1, 1u);
                            }
                            commit(&bar_r);
                        }
                        __syncwarp();
                    }
                    mbar_wait(&bar_r, ph);
                    fence_after_sync();
                    float hn[16];
                    tmem_ld16(tmem + lane_off + kR_accR + j0, hn);
                    // four units at a time: dG to HBM, its hi / lo to tensor memory (hi over the consumed h_{t-1}
                    // columns, lo over the consumed hn columns), so that no 16-wide temporaries stay live
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float4 bb = bhn_s[f0 + j];
                        const float rr[4] = {r4[j].x, r4[j].y, r4[j].z, r4[j].w}, zz[4] = {z4[j].x, z4[j].y, z4[j].z, z4[j].w};
                        const float nn[4] = {n4[j].x, n4[j].y, n4[j].z, n4[j].w}, bh[4] = {bb.x, bb.y, bb.z, bb.w};
                        float dr[4], dz[4], dhn[4], din[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float g = dh[4 * j + e], hv = hn[4 * j + e] + bh[e];
                            const float dnp = g * (1.f - zz[e]) * (1.f - nn[e] * nn[e]);
                            dz[e] = g * (hm[4 * j + e] - nn[e]) * zz[e] * (1.f - zz[e]);
                            dr[e] = dnp * hv * rr[e] * (1.f - rr[e]);
                            dhn[e] = dnp * rr[e];
                            din[e] = dnp;
                            dh[4 * j + e] = g * zz[e];  // the accumulator of the second GEMM is added after the wait below
                        }
                        // pad rows carry zeros (their dh is zero)
                        stg_stream(dg4 + b32(row, 0 * (H / 4) + f0 + j, H), make_float4(dr[0], dr[1], dr[2], dr[3]));
                        stg_stream(dg4 + b32(row, 1 * (H / 4) + f0 + j, H), make_float4(dz[0], dz[1], dz[2], dz[3]));
                        stg_stream(dg4 + b32(row, 2 * (H / 4) + f0 + j, H), make_float4(dhn[0], dhn[1], dhn[2], dhn[3]));
                        stg_stream(dg4 + b32(row, 3 * (H / 4) + f0 + j, H), make_float4(din[0], din[1], din[2], din[3]));
                        float hi[4], lo[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) { hi[e] = tf32_hi(dr[e]); lo[e] = dr[e] - hi[e]; }
                        tmem_st4(tmem + lane_off + kR_a + 0 * H + j0 + 4 * j, hi);
                        tmem_st4(tmem + lane_off + kR_accR + 0 * H + j0 + 4 * j, lo);
#pragma unroll
                        for (int e = 0; e < 4; ++e) { hi[e] = tf32_hi(dz[e]); lo[e] = dz[e] - hi[e]; }
                        tmem_st4(tmem + lane_off + kR_a + 1 * H + j0 + 4 * j, hi);
                        tmem_st4(tmem + lane_off + kR_accR + 1 * H + j0 + 4 * j, lo);
#pragma unroll
                        for (int e = 0; e < 4; ++e) { hi[e] = tf32_hi(dhn[e]); lo[e] = dhn[e] - hi[e]; }
                        tmem_st4(tmem + lane_off + kR_a + 2 * H + j0 + 4 * j, hi);
                        tmem_st4(tmem + lane_off + kR_accR + 2 * H + j0 + 4 * j, lo);
                    }
                }
                tmem_wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a2);
                if (t > 0) load_h(t - 1);  // h_{t-2}: in flight while the second GEMM runs
                if (warp == 0) {  // dh_{t-1} += [dr | dz | dhn] W_hh
                    mbar_wait(&bar_a2, ph);
                    fence_after_sync();
                    if (elect_one()) {
#pragma unroll
                        for (uint32_t ks = 0; ks < KB / 8; ++ks) {
                            const uint32_t boff = (ks >> 2) * kg2 + 2 * (ks & 3);
                            mma_tf32_ts(tmem + kR_accDh, tmem + kR_accR + 8 * ks, b2h + boff, idesc2, ks == 0 ? 0u : 1u);
                            mma_tf32_ts(tmem + kR_accDh, tmem + kR_a + 8 * ks, b2l + boff, idesc2, 1u);
                            mma_tf32_ts(tmem + kR_accDh, tmem + kR_a + 8 * ks, b2h + boff, idesc2, 1u);
                        }
                        commit(&bar_d);
                    }
                    __syncwarp();
                }
                mbar_wait(&bar_d, ph);
                fence_after_sync();
#pragma unroll
                for (int c = 0; c < 16; c += 16) {
                    float acc[16];
                    tmem_ld16(tmem + lane_off + kR_accDh + j0 + c, acc);
#pragma unroll
                    for (int j = 0; j < 16; ++j) dh[c + j] += acc[j];
                }
                fence_before_sync();
                ph ^= 1;
            }
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        fence_after_sync();
        tmem_dealloc(tmem, 512);
    }
}

}  // namespace

extern "C" int ltgnn_gru_fwd(int device, int64_t B, int32_t L, int32_t S, int32_t F, int32_t Hdim, const float* r,
                             const float* tf, const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                             float* h_last, float* hseq, float* gates, void* stream_) {
    LTGNN_REQUIRE(B >= 0 && L > 0 && S > 0 && F >= 0, LTGNN_E_ARG, "gru_fwd: B=%lld L=%d S=%d F=%d",
                  static_cast<long long>(B), L, S, F);
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_fwd: hidden size %d not supported (64 only)", Hdim);
    LTGNN_REQUIRE(H + 1 + F + 1 <= KA && 1 + F <= kAuxIn, LTGNN_E_SHAPE, "gru_fwd: %d time features do not fit the fused operand", F);
    LTGNN_REQUIRE(B * S < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_fwd: too many sequences");
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(r && w_ih && w_hh && b_ih && b_hh && h_last && (tf || F == 0), LTGNN_E_ARG, "gru_fwd: null tensor");
    LTGNN_REQUIRE(aligned16(h_last) && aligned16(hseq) && aligned16(gates), LTGNN_E_ALIGN, "gru_fwd: outputs must be 16-byte aligned");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "gru_fwd: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_USE_DEVICE(device);
    GruParams p{r, F ? tf : nullptr, w_ih, w_hh, b_ih, b_hh, h_last, hseq, gates, static_cast<uint32_t>(B * S),
                static_cast<uint32_t>((B * S + 127) / 128 * 128), L, S, F,
                S >= 2 ? (~0ull / static_cast<uint64_t>(S)) + 1 : 0ull};
    const size_t smem = 1024 + 2ull * NG * KA * 4;
    LTGNN_REQUIRE(smem <= static_cast<size_t>(di->smem_optin), LTGNN_E_SHAPE, "gru_fwd: %zu B of shared memory", smem);
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gru_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    const int64_t tiles = (B * S + 127) / 128;
    const int grid = static_cast<int>(tiles < di->sm_count ? tiles : di->sm_count);
    gru_fwd_kernel<<<grid, kThreads, smem, static_cast<cudaStream_t>(stream_)>>>(p);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gru_bwd_dg_hn(int device, int64_t Q, int32_t L, int32_t Hdim, const float* w_hh, const float* b_hh,
                                   const float* gates3, const float* hseq, const float* dh_last, float* dG,
                                   void* stream_) {
    LTGNN_REQUIRE(Q >= 0 && L > 0, LTGNN_E_ARG, "gru_bwd_dg_hn: Q=%lld L=%d", static_cast<long long>(Q), L);
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_bwd_dg_hn: hidden size %d not supported (64 only)", Hdim);
    LTGNN_REQUIRE(Q < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_bwd_dg_hn: too many sequences");
    if (Q == 0) return LTGNN_OK;
    LTGNN_REQUIRE(w_hh && b_hh && gates3 && hseq && dh_last && dG, LTGNN_E_ARG, "gru_bwd_dg_hn: null tensor");
    LTGNN_REQUIRE(aligned16(gates3) && aligned16(hseq) && aligned16(dh_last) && aligned16(dG), LTGNN_E_ALIGN,
                  "gru_bwd_dg_hn: 16-byte alignment required");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "gru_bwd_dg_hn: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_USE_DEVICE(device);
    GruBwdHnParams p{w_hh, b_hh, gates3, hseq, dh_last, dG, static_cast<uint32_t>(Q),
                     static_cast<uint32_t>((Q + 127) / 128 * 128), L};
    const size_t smem = 1024 + 2ull * H * H * 4 + 2ull * H * KB * 4;
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gru_bwd_hn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    const int64_t tiles = (Q + 127) / 128;
    const int grid = static_cast<int>(tiles < di->sm_count ? tiles : di->sm_count);
    gru_bwd_hn_kernel<<<grid, kThreadsHn, smem, static_cast<cudaStream_t>(stream_)>>>(p);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

// ---- weight gradients: dBfused[4H, 96] = sum over (t, q) of dG(t, q)^T [h_{t-1}(q) | x | tf | 1 | 0]  (tgrad.cuh)
namespace {
struct DgRows {  // the 256 dG columns of row rho = t * Qp + q (blocked-32 storage)
    static constexpr bool kRowFast = true;
    const float4* dg;
    __device__ __forceinline__ float4 operator()(uint32_t row, int c) const { return ptx::ldg_stream(dg + b32(row, c, H)); }
};
struct GruInputRows {  // the forward's A operand, rebuilt on the fly
    static constexpr bool kRowFast = true;
    const float4* hseq;  // blocked-32 [L * Qp, H]
    const float* r;      // [B, L, S]
    const float* tf;     // [B, L, F]
    uint32_t Q, Qp, S;
    int L, F;
    uint64_t magic_qp, magic_s;
    __device__ __forceinline__ float4 operator()(uint32_t row, int c) const {
        if (c < 16) {
            if (row < Qp) return make_float4(0.f, 0.f, 0.f, 0.f);  // t = 0: h_{-1} = 0
            return ptx::ldg_stream(hseq + b32(row - Qp, c, H / 4));
        }
        const uint32_t t = ptx::fastdiv(row, magic_qp);
        const uint32_t q = row - t * Qp;
        if (q >= Q) return make_float4(0.f, 0.f, 0.f, 0.f);     // pad row
        const uint32_t b = magic_s ? ptx::fastdiv(q, magic_s) : q;
        const uint32_t s = q - b * S;
        float v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = 4 * (c - 16) + i;
            float x = 0.f;
            if (e == 0) x = __ldg(r + (static_cast<size_t>(b) * L + t) * S + s);
            else if (e <= F) x = __ldg(tf + (static_cast<size_t>(b) * L + t) * F + (e - 1));
            else if (e == F + 1) x = 1.f;
            v[i] = x;
        }
        return make_float4(v[0], v[1], v[2], v[3]);
    }
};
}  // namespace

extern "C" int64_t ltgnn_gru_ws_floats(int device) {
    const DeviceInfo* di = device_info(device);
    return di ? static_cast<int64_t>(di->sm_count) * NG * KA : -1;
}

extern "C" int ltgnn_gru_bwd_w(int device, int64_t B, int32_t L, int32_t S, int32_t F, int32_t Hdim, const float* r,
                               const float* tf, const float* hseq, const float* dG, float* dBfused, float* ws,
                               void* stream_) {
    LTGNN_REQUIRE(B >= 0 && L > 0 && S > 0 && F >= 0, LTGNN_E_ARG, "gru_bwd_w: B=%lld L=%d S=%d F=%d",
                  static_cast<long long>(B), L, S, F);
    LTGNN_REQUIRE(Hdim == H && H + 1 + F + 1 <= KA, LTGNN_E_SHAPE, "gru_bwd_w: H=%d F=%d not supported", Hdim, F);
    LTGNN_REQUIRE(r && hseq && dG && dBfused && ws && (tf || F == 0), LTGNN_E_ARG, "gru_bwd_w: null tensor");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (B == 0) {
        LTGNN_CUDA_TRY(cudaMemsetAsync(dBfused, 0, sizeof(float) * NG * KA, stream));
        return LTGNN_OK;
    }
    const int64_t Q = B * S, Qp = (Q + 127) / 128 * 128, M = Qp * L;
    LTGNN_REQUIRE(M < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_bwd_w: L*B*S=%lld rows exceed the 32-bit row index",
                  static_cast<long long>(M));
    GruInputRows x{reinterpret_cast<const float4*>(hseq), r, tf, static_cast<uint32_t>(Q), static_cast<uint32_t>(Qp),
                   static_cast<uint32_t>(S), L, F, (~0ull / static_cast<uint64_t>(Qp)) + 1,
                   S >= 2 ? (~0ull / static_cast<uint64_t>(S)) + 1 : 0ull};
    DgRows g{reinterpret_cast<const float4*>(dG)};
    int grid = 0;
    int rc = tgrad::launch<2, 8, 4, 16>(device, g, x, ws, M, KA, &grid, stream, "gru_bwd_w");  // all 256 rows in one pass over X
    if (rc) return rc;
    return tgrad::gather(ws, grid, KA, 0, NG, 0, KA, dBfused, KA, 0, stream, NG);
}

// ---- input gradient (gru_dx.cuh) from the BPTT's dG: input groups r, z and in = columns 0, 1 and 3 of 4
namespace {
struct DgBlocked {
    const float4* dg;  // blocked-32 [L * Qp, 4H]
    int64_t rows;      // L * Qp
    uint32_t Q, Qp;
    uint64_t magic_qp;
    __device__ __forceinline__ bool decode(int64_t row, uint32_t& q, uint32_t& t) const {
        t = ptx::fastdiv(static_cast<uint32_t>(row), magic_qp);
        q = static_cast<uint32_t>(row) - t * Qp;
        return q < Q;
    }
    __device__ __forceinline__ float4 load(int64_t row, int g, int j4) const {
        return ptx::ldg_stream(dg + b32(static_cast<size_t>(row), (g == 2 ? 3 : g) * (H / 4) + j4, H));
    }
};
}  // namespace

extern "C" int ltgnn_gru_bwd_dx(int device, int64_t B, int32_t L, int32_t S, int32_t F, int32_t Hdim, const float* w_ih,
                                const float* dG, float* dr, float* dxt, void* stream_) {
    LTGNN_REQUIRE(B >= 0 && L > 0 && S > 0 && F >= 0, LTGNN_E_ARG, "gru_bwd_dx: B=%lld L=%d S=%d F=%d",
                  static_cast<long long>(B), L, S, F);
    LTGNN_REQUIRE(Hdim == H, LTGNN_E_SHAPE, "gru_bwd_dx: hidden size %d not supported (64 only)", Hdim);
    LTGNN_REQUIRE(1 + F < gru_dx::kCols, LTGNN_E_SHAPE, "gru_bwd_dx: %d time features, at most %d", F, gru_dx::kCols - 2);
    LTGNN_REQUIRE(B * S < (1ll << 31) - 128, LTGNN_E_SHAPE, "gru_bwd_dx: too many sequences");
    const int64_t Q = B * S, Qp = (Q + 127) / 128 * 128;
    LTGNN_REQUIRE(Qp * L < (1ll << 31), LTGNN_E_SHAPE, "gru_bwd_dx: L*B*S=%lld rows exceed the 32-bit row index",
                  static_cast<long long>(Qp * L));
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(w_ih && dG && (dr || dxt) && (F > 0 || !dxt), LTGNN_E_ARG,
                  "gru_bwd_dx: null tensor (dr or dxt required; dxt needs F > 0)");
    LTGNN_REQUIRE(aligned16(dG) && reinterpret_cast<uintptr_t>(w_ih) % 4 == 0 && reinterpret_cast<uintptr_t>(dr) % 4 == 0 &&
                  reinterpret_cast<uintptr_t>(dxt) % 4 == 0, LTGNN_E_ALIGN,
                  "gru_bwd_dx: dG must be 16-byte aligned, w_ih, dr and dxt 4-byte aligned");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "gru_bwd_dx: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_USE_DEVICE(device);
    DgBlocked lay{reinterpret_cast<const float4*>(dG), Qp * L, static_cast<uint32_t>(Q), static_cast<uint32_t>(Qp),
                  (~0ull / static_cast<uint64_t>(Qp)) + 1};
    auto kernel = gru_dx::gru_bwd_dx_kernel<H, DgBlocked>;
    const size_t smem = gru_dx::smem_bytes(H);
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    kernel<<<gru_dx::grid_for(lay.rows, di->sm_count), gru_dx::kThreads, smem, static_cast<cudaStream_t>(stream_)>>>(
        lay, w_ih, dr, dxt, static_cast<uint32_t>(S), L, F, S >= 2 ? (~0ull / static_cast<uint64_t>(S)) + 1 : 0ull);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}
