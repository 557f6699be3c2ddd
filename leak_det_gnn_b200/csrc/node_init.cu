// node_init.cu -- node-feature initialisation of the detector and its backward.
//
// Reference (models/detector.py:178-190): h0 = zeros(B, N, d_s); h0[:, sensor_idx] = h_s; mask = sensor
// indicator; x0 = dropout(relu(Linear_{d_s+1 -> D}(cat[h0, mask]))).  That materialises three full
// (B, N, .) tensors and runs a (B*N) x 65 x 64 GEMM in which 632 of 661 rows are all-zero inputs.
// Here: a non-sensor row is the batch-independent constant relu(bias); a sensor row is
// relu(W[:, :d_s] h_s + W[:, d_s] + bias).  HBM traffic = one write of x0 (forward), one read of
// dx0 and x0 (backward); the 29-row GEMMs run on CUDA cores out of shared memory (0.1 % of the bytes).
#include "functors.cuh"
#include "rowgemm.cuh"
#include "tgrad.cuh"

using namespace ltgnn;

namespace {

constexpr int kThreads = 256;

struct InitParams {
    const float* hs;        // [B, S, ds]
    const float* W;         // [D, ds + 1]  (torch Linear layout)
    const float* bias;      // [D]
    const int32_t* slot;    // [N]: sensor slot of node i, or -1
    int64_t B;
    int32_t N, S, ds, D;
    uint32_t drop_thresh;
    float keep_scale;
    uint64_t drop_seed;
    const uint64_t* seed_src;  // ltgnn_seed_source word or nullptr
};

// ---------------------------------------- forward ----------------------------------------
__global__ void __launch_bounds__(kThreads)
node_init_fwd_kernel(const InitParams p, float* __restrict__ X0, uint32_t* __restrict__ live_out) {
    extern __shared__ __align__(16) float sm[];
    const int ds1 = p.ds + 1, D = p.D, d4 = D >> 2;
    float* Wt = sm;                   // [ds+1][D]  transposed weight
    float* base = Wt + ds1 * D;       // [D] relu(bias)
    float* cst = base + D;            // [D] W[:, ds] + bias
    float* hs = cst + D;              // [S][ds]
    float* sens = hs + p.S * p.ds;    // [S][D]
    const int tid = threadIdx.x;

    for (int i = tid; i < D * ds1; i += kThreads) {
        const int j = i / ds1, k = i - j * ds1;
        Wt[k * D + j] = __ldg(p.W + i);
    }
    __syncthreads();
    for (int j = tid; j < D; j += kThreads) {
        const float b = __ldg(p.bias + j);
        base[j] = fmaxf(b, 0.f);
        cst[j] = Wt[p.ds * D + j] + b;
    }

    for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
        __syncthreads();  // previous window's sens/hs fully consumed
        const float* hsb = p.hs + b * p.S * p.ds;
        for (int i = tid; i < p.S * p.ds; i += kThreads) hs[i] = __ldg(hsb + i);
        __syncthreads();
        for (int i = tid; i < p.S * d4; i += kThreads) {  // thread = (sensor row, 4 output columns)
            const int s = i / d4, j = (i - s * d4) * 4;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            const float* h = hs + s * p.ds;
#pragma unroll 8
            for (int k = 0; k < p.ds; ++k) {
                const float4 w = *reinterpret_cast<const float4*>(Wt + k * D + j);
                const float hk = h[k];
                acc.x = fmaf(hk, w.x, acc.x); acc.y = fmaf(hk, w.y, acc.y);
                acc.z = fmaf(hk, w.z, acc.z); acc.w = fmaf(hk, w.w, acc.w);
            }
            const float4 cj = *reinterpret_cast<const float4*>(cst + j);
            *reinterpret_cast<float4*>(sens + s * D + j) = make_float4(fmaxf(acc.x + cj.x, 0.f), fmaxf(acc.y + cj.y, 0.f),
                                                                       fmaxf(acc.z + cj.z, 0.f), fmaxf(acc.w + cj.w, 0.f));
        }
        __syncthreads();
        float4* out = reinterpret_cast<float4*>(X0) + b * p.N * d4;
        const int d8 = d4 >> 1;  // a thread writes 8 consecutive features: one Philox call decides all of them
        const int c = (tid % d8) * 2, rstep = kThreads / d8;  // kThreads % d8 == 0: a thread keeps its column group
        for (int r = tid / d8; r < p.N; r += rstep) {
            const int i = r * d8 + (c >> 1);
            const int sl = __ldg(p.slot + r);
            const float4* src = reinterpret_cast<const float4*>(sl < 0 ? base + c * 4 : sens + sl * D + c * 4);
            float v[8];
            *reinterpret_cast<float4*>(v) = src[0];
            *reinterpret_cast<float4*>(v + 4) = src[1];
            if (p.drop_thresh)
                ptx::dropout8(v, static_cast<uint64_t>(b * p.N * d8 + i), ptx::launch_seed(p.drop_seed, p.seed_src), p.drop_thresh,
                              p.keep_scale);
            ptx::stg_stream(out + 2 * i, *reinterpret_cast<const float4*>(v));
            ptx::stg_stream(out + 2 * i + 1, *reinterpret_cast<const float4*>(v + 4));
            if (live_out) {
                // 1-bit form of x0 > 0 for the backward: the 4 threads of a 32-feature slice (same row, so they run
                // this loop together) assemble one word, layout [b][D/32][N]
                // bit 8 c + q <-> element 4 q + c of the slice (see ltgnn_spmm_fused); this thread holds q = 2 t, 2 t + 1
                uint32_t w = 0;
#pragma unroll
                for (int cc = 0; cc < 4; ++cc)
                    w |= ((v[cc] > 0.f ? 1u : 0u) << (8 * cc)) | ((v[4 + cc] > 0.f ? 1u : 0u) << (8 * cc + 1));
                w <<= 2 * (tid & 3);
                const uint32_t grp = 0xfu << (tid & 28);
                w |= __shfl_xor_sync(grp, w, 1);
                w |= __shfl_xor_sync(grp, w, 2);
                if ((tid & 3) == 0) live_out[(b * (D >> 5) + (c >> 3)) * p.N + r] = w;
            }
        }
    }
}

// Same result for sensor sets too large to stage (the 100k-node network has 1 000 sensors: 768 KB of embeddings per
// window): only the transposed weight lives in shared memory, and the thread that owns (row, 8 features) of a sensor row
// forms its 8 dot products straight from the embeddings in global memory.  Sensor rows are ~1 % of the rows there.
__global__ void __launch_bounds__(kThreads)
node_init_fwd_direct_kernel(const InitParams p, float* __restrict__ X0, uint32_t* __restrict__ live_out) {
    extern __shared__ __align__(16) float sm[];
    const int ds1 = p.ds + 1, D = p.D, d4 = D >> 2;
    float* Wt = sm;                   // [ds+1][D]  transposed weight
    float* base = Wt + ds1 * D;       // [D] relu(bias)
    float* cst = base + D;            // [D] W[:, ds] + bias
    const int tid = threadIdx.x;
    for (int i = tid; i < D * ds1; i += kThreads) {
        const int j = i / ds1, k = i - j * ds1;
        Wt[k * D + j] = __ldg(p.W + i);
    }
    __syncthreads();
    for (int j = tid; j < D; j += kThreads) {
        const float b = __ldg(p.bias + j);
        base[j] = fmaxf(b, 0.f);
        cst[j] = Wt[p.ds * D + j] + b;
    }
    __syncthreads();
    const int d8 = d4 >> 1;
    const int c = (tid % d8) * 2, rstep = kThreads / d8;
    // work unit = (window, block of rows): the large graphs come with few windows
    const int rows_per_unit = rstep * 64;
    const int units_per_b = (p.N + rows_per_unit - 1) / rows_per_unit;
    for (int64_t u = blockIdx.x; u < p.B * units_per_b; u += gridDim.x) {
        const int64_t b = u / units_per_b;
        const int r_lo = static_cast<int>(u - b * units_per_b) * rows_per_unit;
        const int r_hi = r_lo + rows_per_unit < p.N ? r_lo + rows_per_unit : p.N;
        float4* out = reinterpret_cast<float4*>(X0) + b * p.N * d4;
        for (int r = r_lo + tid / d8; r < r_hi; r += rstep) {
            const int i = r * d8 + (c >> 1);
            const int sl = __ldg(p.slot + r);
            float v[8];
            if (sl < 0) {
                *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(base + c * 4);
                *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(base + c * 4 + 4);
            } else {
                const float* h = p.hs + (b * p.S + sl) * p.ds;
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = 0.f;
                for (int k = 0; k < p.ds; ++k) {
                    const float hk = __ldg(h + k);
                    const float4 w0 = *reinterpret_cast<const float4*>(Wt + k * D + c * 4);
                    const float4 w1 = *reinterpret_cast<const float4*>(Wt + k * D + c * 4 + 4);
                    v[0] = fmaf(hk, w0.x, v[0]); v[1] = fmaf(hk, w0.y, v[1]); v[2] = fmaf(hk, w0.z, v[2]); v[3] = fmaf(hk, w0.w, v[3]);
                    v[4] = fmaf(hk, w1.x, v[4]); v[5] = fmaf(hk, w1.y, v[5]); v[6] = fmaf(hk, w1.z, v[6]); v[7] = fmaf(hk, w1.w, v[7]);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j] + cst[c * 4 + j], 0.f);
            }
            if (p.drop_thresh)
                ptx::dropout8(v, static_cast<uint64_t>(b * p.N * d8 + i), ptx::launch_seed(p.drop_seed, p.seed_src), p.drop_thresh,
                              p.keep_scale);
            ptx::stg_stream(out + 2 * i, *reinterpret_cast<const float4*>(v));
            ptx::stg_stream(out + 2 * i + 1, *reinterpret_cast<const float4*>(v + 4));
            if (live_out) {  // same word layout as node_init_fwd_kernel
                uint32_t w = 0;
#pragma unroll
                for (int cc = 0; cc < 4; ++cc)
                    w |= ((v[cc] > 0.f ? 1u : 0u) << (8 * cc)) | ((v[4 + cc] > 0.f ? 1u : 0u) << (8 * cc + 1));
                w <<= 2 * (tid & 3);
                const uint32_t grp = 0xfu << (tid & 28);
                w |= __shfl_xor_sync(grp, w, 1);
                w |= __shfl_xor_sync(grp, w, 2);
                if ((tid & 3) == 0) live_out[(b * (D >> 5) + (c >> 3)) * p.N + r] = w;
            }
        }
    }
}

// ---------------------------------------- backward ----------------------------------------
// (1) one pure streaming kernel over dx0 / x0: gate, per-column sums (-> d bias) and the gated gradient of the S
//     sensor rows of every window, written compactly to dz [B, S, D] (4 % of the bytes);
// (2) d h_s = dz W[:, :ds] on the row-GEMM skeleton and dW = dz^T [h_s | 1] on the tensor-core weight-gradient
//     skeleton, both over the B*S sensor rows only.
// ltgnn_node_init_bwd_from_layer replaces (1) when dx0 is the first GCN layer's input gradient G1 W1: the tensor-core GEMM
// that would form it does the gate, the column sums and the sensor-row extraction in its epilogue (GateSumEpilogue,
// functors.cuh) and never stores dx0 -- one read of G1 instead of a write and a read of dx0.

// colsum partial layout: part[cta][D]
// kBits: the gate comes as 1 bit per element (`live`, layout [b][D/32][N]) instead of the float tensor X0
template <bool kBits>
__global__ void __launch_bounds__(kThreads)
gate_extract_kernel(const float4* __restrict__ dX0, const float4* __restrict__ X0, const uint32_t* __restrict__ live,
                    const int32_t* __restrict__ slot, float gate_scale, float4* __restrict__ dz,
                    float* __restrict__ part, int64_t B, int N, int S, int d4, int units_per_b, int rows_per_unit) {
    __shared__ float4 red[kThreads];
    const int tid = threadIdx.x;
    float4 csum = make_float4(0.f, 0.f, 0.f, 0.f);  // kThreads % d4 == 0: a thread keeps its column group
    const int n4 = N * d4;
    const int c = tid % d4, rstep = kThreads / d4;  // a thread keeps its float4 column: no division in the loop
    // work unit = (window, block of rows): a large graph comes with few windows, and one CTA per window would leave
    // most of the machine idle (the 100k-node network: 16 windows)
    for (int64_t u = blockIdx.x; u < B * units_per_b; u += gridDim.x) {
        const int64_t b = u / units_per_b;
        const int r_lo = static_cast<int>(u - b * units_per_b) * rows_per_unit;
        const int r_hi = r_lo + rows_per_unit < N ? r_lo + rows_per_unit : N;
        const float4* gb = dX0 + b * n4 + c;
        const float4* xb = kBits ? nullptr : X0 + b * n4 + c;
        const uint32_t* lw = kBits ? live + (b * (d4 >> 3) + (c >> 3)) * N : nullptr;
        float4* dzb = dz + b * S * d4 + c;
        for (int r0 = r_lo + tid / d4; r0 < r_hi; r0 += 4 * rstep) {
            float4 g[4], x[4];
            uint32_t m[4];
            int sl[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int r = r0 + u * rstep;
                if (r < r_hi) {
                    g[u] = ptx::ldg_stream(gb + r * d4);
                    if (kBits) m[u] = __ldg(lw + r) >> (c & 7);
                    else x[u] = ptx::ldg_stream(xb + r * d4);
                    sl[u] = __ldg(slot + r);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (r0 + u * rstep < r_hi) {
                    if (kBits) {
                        g[u].x = (m[u] & 0x1u) ? g[u].x * gate_scale : 0.f;
                        g[u].y = (m[u] & 0x100u) ? g[u].y * gate_scale : 0.f;
                        g[u].z = (m[u] & 0x10000u) ? g[u].z * gate_scale : 0.f;
                        g[u].w = (m[u] & 0x1000000u) ? g[u].w * gate_scale : 0.f;
                    } else {
                        g[u].x = x[u].x > 0.f ? g[u].x * gate_scale : 0.f;
                        g[u].y = x[u].y > 0.f ? g[u].y * gate_scale : 0.f;
                        g[u].z = x[u].z > 0.f ? g[u].z * gate_scale : 0.f;
                        g[u].w = x[u].w > 0.f ? g[u].w * gate_scale : 0.f;
                    }
                    csum.x += g[u].x; csum.y += g[u].y; csum.z += g[u].z; csum.w += g[u].w;
                    if (sl[u] >= 0) dzb[sl[u] * d4] = g[u];
                }
            }
        }
    }
    red[tid] = csum;
    __syncthreads();
    if (tid < d4) {
        float4 t = red[tid];
        for (int k = tid + d4; k < kThreads; k += d4) {
            const float4 o = red[k];
            t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
        }
        reinterpret_cast<float4*>(part)[static_cast<size_t>(blockIdx.x) * d4 + tid] = t;
    }
}

int check_common(int device, int64_t B, int32_t N, int32_t S, int32_t ds, int32_t D, const DeviceInfo** di,
                 const char* who) {
    LTGNN_REQUIRE(B >= 0 && N > 0 && S >= 0 && ds > 0 && D > 0, LTGNN_E_ARG, "%s: B=%lld N=%d S=%d ds=%d D=%d", who,
                  static_cast<long long>(B), N, S, ds, D);
    LTGNN_REQUIRE(D % 4 == 0 && kThreads % (D / 4) == 0, LTGNN_E_SHAPE, "%s: D=%d must be 4 * a divisor of %d", who, D,
                  kThreads);
    *di = device_info(device);
    if (!*di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE((*di)->cc_major == 10, LTGNN_E_UNSUPPORTED, "%s: device is sm_%d%d, need sm_100", who,
                  (*di)->cc_major, (*di)->cc_minor);
    return LTGNN_OK;
}

// 16 random bits per element everywhere: keep probability 1 - round(p * 2^16) / 2^16, scale its exact inverse
uint32_t thresh_of(float p) { return p > 0.f ? static_cast<uint32_t>(static_cast<double>(p) * 65536.0 + 0.5) : 0u; }
float scale_of(float p) { return 1.f / (1.f - static_cast<float>(thresh_of(p)) / 65536.f); }

}  // namespace

extern "C" int ltgnn_node_init_fwd(int device, int64_t B, int32_t N, int32_t S, int32_t ds, int32_t D, const float* hs,
                                   const int32_t* slot, const float* W, const float* bias, float drop_p,
                                   uint64_t drop_seed, float* X0, uint32_t* live_out, void* stream_) {
    const DeviceInfo* di;
    int rc = check_common(device, B, N, S, ds, D, &di, "node_init_fwd");
    if (rc) return rc;
    LTGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, LTGNN_E_ARG, "node_init_fwd: dropout p=%f", drop_p);
    LTGNN_REQUIRE(D % 8 == 0, LTGNN_E_SHAPE, "node_init_fwd: D=%d must be a multiple of 8", D);
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(hs && slot && W && bias && X0, LTGNN_E_ARG, "node_init_fwd: null tensor");
    LTGNN_REQUIRE(aligned16(X0), LTGNN_E_ALIGN, "node_init_fwd: X0 must be 16-byte aligned");
    LTGNN_USE_DEVICE(device);
    InitParams p{hs, W, bias, slot, B, N, S, ds, D, thresh_of(drop_p), scale_of(drop_p), drop_seed, seed_source()};
    const size_t smem = sizeof(float) * (static_cast<size_t>(ds + 1) * D + 2 * D + static_cast<size_t>(S) * ds +
                                         static_cast<size_t>(S) * D);
    LTGNN_REQUIRE(!live_out || D % 32 == 0, LTGNN_E_SHAPE, "node_init_fwd: live_out needs D %% 32 == 0 (D=%d)", D);
    if (smem > static_cast<size_t>(di->smem_optin)) {  // sensor set too large to stage: rows formed straight from global
        const size_t smem_d = sizeof(float) * (static_cast<size_t>(ds + 1) * D + 2 * D);
        LTGNN_REQUIRE(smem_d <= static_cast<size_t>(di->smem_optin), LTGNN_E_SHAPE, "node_init_fwd: %zu B of shared memory",
                      smem_d);
        LTGNN_CUDA_TRY(cudaFuncSetAttribute(node_init_fwd_direct_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            static_cast<int>(smem_d)));
        node_init_fwd_direct_kernel<<<di->sm_count * 4, kThreads, smem_d, static_cast<cudaStream_t>(stream_)>>>(p, X0, live_out);
        LTGNN_CUDA_TRY(cudaGetLastError());
        return LTGNN_OK;
    }
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(node_init_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    const int64_t cap = static_cast<int64_t>(di->sm_count) * 6;
    const int grid = static_cast<int>(B < cap ? B : cap);
    node_init_fwd_kernel<<<grid, kThreads, smem, static_cast<cudaStream_t>(stream_)>>>(p, X0, live_out);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

// workspace (ltgnn_node_init_bwd and ltgnn_node_init_bwd_from_layer):
//   dz [B,S,D] | colsum partials [n_stream_ctas][D] | weight-gradient partials
static int stream_ctas(const DeviceInfo* di) { return di->sm_count * 8; }
static int dw_cols(int ds) { return (ds + 1 + 31) / 32 * 32; }  // [h_s | 1] padded to whole 32-column blocks

extern "C" int64_t ltgnn_node_init_ws_floats(int device, int64_t B, int32_t S, int32_t ds, int32_t D) {
    const DeviceInfo* di = device_info(device);
    if (!di) return -1;
    return B * S * D + static_cast<int64_t>(stream_ctas(di)) * D +
           static_cast<int64_t>(di->sm_count) * tgrad::kMo * dw_cols(ds);
}

// (2a) d h_s [M, ds] = dz [M, D] * W[:, :ds]   (W is [D, ds+1] row-major: a [K, N] operand with ld = ds+1)
// (2b) dW [D, ds+1] = dz^T [h_s | 1]
static int sensor_row_grads(int device, int64_t M, int32_t ds, int32_t D, const float* hs, const float* W, const float* dz,
                            float* wpart, float* dhs, float* dW, cudaStream_t stream) {
    functors::RowLoader ld{reinterpret_cast<const float4*>(dz), D / 4};
    functors::StoreEpilogue ep{dhs, nullptr, nullptr, 1.f, ds, 0};
    rowgemm::BSpec bs{W, ds + 1, 1, 1};
    int rc = rowgemm::launch(device, ld, ep, bs, M, D, ds, stream, "node_init_bwd(dhs)");
    if (rc) return rc;
    functors::StackedRows g{reinterpret_cast<const float4*>(dz), nullptr, D / 4, 0};
    functors::RowsThenOne x{reinterpret_cast<const float4*>(hs), ds / 4};
    int grid = 0;
    rc = tgrad::launch(device, g, x, wpart, M, dw_cols(ds), &grid, stream, "node_init_bwd(dW)");
    if (rc) return rc;
    return tgrad::gather(wpart, grid, dw_cols(ds), 0, D, 0, ds + 1, dW, ds + 1, 0, stream);
}

extern "C" int ltgnn_node_init_bwd(int device, int64_t B, int32_t N, int32_t S, int32_t ds, int32_t D, const float* hs,
                                   const int32_t* slot, const float* W, const float* dX0, const float* X0,
                                   const uint32_t* live_in, float gate_scale, float* dhs, float* dW, float* dbias,
                                   float* ws, void* stream_) {
    const DeviceInfo* di;
    int rc = check_common(device, B, N, S, ds, D, &di, "node_init_bwd");
    if (rc) return rc;
    LTGNN_REQUIRE(D == 64 || D == 128, LTGNN_E_SHAPE, "node_init_bwd: D=%d must be 64 or 128", D);
    LTGNN_REQUIRE(ds % 32 == 0 && ds <= 224, LTGNN_E_SHAPE, "node_init_bwd: ds=%d must be a multiple of 32", ds);
    LTGNN_REQUIRE(hs && slot && W && dX0 && (X0 || live_in) && dhs && dW && dbias && ws, LTGNN_E_ARG,
                  "node_init_bwd: null tensor");
    LTGNN_REQUIRE(aligned16(dX0) && aligned16(X0) && aligned16(ws) && aligned16(hs) && aligned16(dhs), LTGNN_E_ALIGN,
                  "node_init_bwd: 16-byte alignment required");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    LTGNN_USE_DEVICE(device);
    const int n_w = D * (ds + 1), d4 = D / 4;
    if (B == 0) {
        LTGNN_CUDA_TRY(cudaMemsetAsync(dW, 0, sizeof(float) * n_w, stream));
        LTGNN_CUDA_TRY(cudaMemsetAsync(dbias, 0, sizeof(float) * D, stream));
        return LTGNN_OK;
    }
    float* dz = ws;
    float* cpart = dz + B * S * D;
    float* wpart = cpart + static_cast<int64_t>(stream_ctas(di)) * D;

    // (1) streaming pass
    int units_per_b = static_cast<int>((stream_ctas(di) + B - 1) / B);
    const int max_units = (N + 1023) / 1024;  // at least 1024 rows per unit
    if (units_per_b > max_units) units_per_b = max_units;
    const int rows_per_unit = (N + units_per_b - 1) / units_per_b;
    const int64_t n_units = B * units_per_b;
    const int64_t g1 = n_units < stream_ctas(di) ? n_units : stream_ctas(di);
    if (live_in)  // 1 bit per element instead of the float activations: half the bytes of this pass
        gate_extract_kernel<true><<<static_cast<int>(g1), kThreads, 0, stream>>>(
            reinterpret_cast<const float4*>(dX0), nullptr, live_in, slot, gate_scale, reinterpret_cast<float4*>(dz),
            cpart, B, N, S, d4, units_per_b, rows_per_unit);
    else
        gate_extract_kernel<false><<<static_cast<int>(g1), kThreads, 0, stream>>>(
            reinterpret_cast<const float4*>(dX0), reinterpret_cast<const float4*>(X0), nullptr, slot, gate_scale,
            reinterpret_cast<float4*>(dz), cpart, B, N, S, d4, units_per_b, rows_per_unit);
    LTGNN_CUDA_TRY(cudaGetLastError());
    rc = reduce_parts(cpart, D, dbias, static_cast<int>(g1), D, 0, stream);
    if (rc) return rc;
    return sensor_row_grads(device, B * S, ds, D, hs, W, dz, wpart, dhs, dW, stream);
}

extern "C" int ltgnn_node_init_bwd_from_layer(int device, int64_t B, int32_t N, int32_t S, int32_t ds, int32_t D,
                                              int32_t K, const float* hs, const int32_t* slot, const float* W,
                                              const float* G1, const float* W1, const uint32_t* live_in,
                                              float gate_scale, float* dhs, float* dW, float* dbias, float* ws,
                                              void* stream_) {
    const DeviceInfo* di;
    int rc = check_common(device, B, N, S, ds, D, &di, "node_init_bwd_from_layer");
    if (rc) return rc;
    LTGNN_REQUIRE(D == 64 || D == 128, LTGNN_E_SHAPE, "node_init_bwd_from_layer: D=%d must be 64 or 128", D);
    LTGNN_REQUIRE(ds % 32 == 0 && ds <= 224, LTGNN_E_SHAPE, "node_init_bwd_from_layer: ds=%d must be a multiple of 32",
                  ds);
    LTGNN_REQUIRE(K > 0 && K % 32 == 0 && K <= 128, LTGNN_E_SHAPE,
                  "node_init_bwd_from_layer: K=%d must be a multiple of 32 up to 128", K);
    LTGNN_REQUIRE(B * N < (1ll << 31) - 128, LTGNN_E_SHAPE, "node_init_bwd_from_layer: B*N=%lld rows",
                  static_cast<long long>(B * N));
    LTGNN_REQUIRE(hs && slot && W && G1 && W1 && live_in && dhs && dW && dbias && ws, LTGNN_E_ARG,
                  "node_init_bwd_from_layer: null tensor");
    LTGNN_REQUIRE(aligned16(G1) && aligned16(W1) && aligned16(ws) && aligned16(hs) && aligned16(dhs), LTGNN_E_ALIGN,
                  "node_init_bwd_from_layer: 16-byte alignment required");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    LTGNN_USE_DEVICE(device);
    if (B == 0) {
        LTGNN_CUDA_TRY(cudaMemsetAsync(dW, 0, sizeof(float) * D * (ds + 1), stream));
        LTGNN_CUDA_TRY(cudaMemsetAsync(dbias, 0, sizeof(float) * D, stream));
        return LTGNN_OK;
    }
    float* dz = ws;
    float* cpart = dz + B * S * D;  // one row per GEMM CTA: at most sm_count <= stream_ctas rows
    float* wpart = cpart + static_cast<int64_t>(stream_ctas(di)) * D;

    // (1) dX0 = G1 W1 on the tensor cores; the epilogue keeps only the gated column sums and sensor rows of it
    functors::GateSumEpilogue ep{dz, cpart, live_in, slot, gate_scale, D, static_cast<uint32_t>(N),
                                 static_cast<uint32_t>(S)};
    int parts = 0;
    rc = functors::linear_gate_sums(device, B * N, K, G1, W1, ep, &parts, stream);
    if (rc) return rc;
    rc = reduce_parts(cpart, D, dbias, parts, D, 0, stream);
    if (rc) return rc;
    return sensor_row_grads(device, B * S, ds, D, hs, W, dz, wpart, dhs, dW, stream);
}
