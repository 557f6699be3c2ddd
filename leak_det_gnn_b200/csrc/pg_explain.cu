// pg_explain.cu -- PyG's PGExplainer edge network on the node embeddings of the leak detector's last GCN layer.
//
//   The edge MLP is Linear(2D, 64) -> ReLU -> Linear(64, 1) on [z[src] | z[dst]].  Its first layer is linear in the
//   concatenation, so it factors per node: [P | Q] = z [W1a; W1b]^T is ONE node-level GEMM (ltgnn_linear, B*N rows,
//   K = D, N = 128) and per edge e = (src, dst) of window b
//       pre = (P[b, src] + Q[b, dst]) + b1,   h = relu(pre),   logit = w2 . h + b2.
//   forward     one warp per 32 (window, edge) rows: for each, lane l holds units 2l, 2l+1 (float2 reads of the [P | Q]
//               rows through L2) and the dot product is a fixed xor-shuffle tree; then lane j finishes edge j.  Training: the concrete sample s = (log eps - log(1 - eps)
//               + logit) / T with eps = (1 - 2 bias) U + bias, U from Philox keyed by seed + the ltgnn_seed_source word,
//               1 / T read from a device scalar; writes s, mask = sigmoid(s) and the 64-bit ReLU gate.  Explaining:
//               mask = sigmoid(logit) only.
//   backward    one warp per (window, node), from d mask: d logit = d mask s'(1 - s') / T on every edge, the gated
//               hidden gradient gh = d logit w2 [pre > 0], summed into R[b, n, :64] over the edges leaving n and into
//               R[b, n, 64:] over the edges entering n, each in ascending edge order (host-built CSRs by source and by
//               target) -- d[P | Q], whose weight gradient is ltgnn_wgrad_tc's R^T z.  d b1, d w2 (h recomputed in the
//               forward's order) and d b2 are per-CTA partials finished by reduce_parts.
//   No atomics, no allocation, no host synchronisation; the gathers go through L2, so any graph size runs.
#include "common.cuh"

using namespace ltgnn;

namespace {

constexpr int kHid = 64;            // PGExplainer's hidden width
constexpr int kPQ = 2 * kHid;       // [P | Q] row
constexpr int kWarps = 8;           // 256 threads
constexpr int kParts = 2 * kHid + 1;   // d b1 [64] | d w2 [64] | d b2
constexpr int kPartStride = 132;

__device__ __forceinline__ float sigmoidf(float x) { return 1.f / (1.f + expf(-x)); }

__global__ void __launch_bounds__(256)
pg_edge_fwd_kernel(int64_t rows, int32_t n, int32_t n_edges, const int32_t* __restrict__ src,
                   const int32_t* __restrict__ dst, const float* __restrict__ pq, const float* __restrict__ b1,
                   const float* __restrict__ w2, const float* __restrict__ b2, const float* __restrict__ inv_t,
                   float eps_scale, float eps_bias, uint64_t seed, const uint64_t* __restrict__ seed_src,
                   float* __restrict__ mask, float* __restrict__ s_out, uint2* __restrict__ gate,
                   float* __restrict__ uniform) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    const float2 bb = __ldg(reinterpret_cast<const float2*>(b1) + lane);
    const float2 ww = __ldg(reinterpret_cast<const float2*>(w2) + lane);
    const float c2 = __ldg(b2);
    const bool train = inv_t != nullptr;
    const float it = train ? __ldg(inv_t) : 1.f;
    const uint64_t key = train ? ptx::launch_seed(seed, seed_src) : 0;
    // a warp takes 32 consecutive edges: their logits one after the other (all lanes), then one edge per lane for the
    // sample, the sigmoid and the stores
    for (int64_t r0 = ((static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5) * 32; r0 < rows;
         r0 += nwarps * 32) {
        const int cnt = rows - r0 < 32 ? static_cast<int>(rows - r0) : 32;
        float my_logit = 0.f;
        uint32_t my_g0 = 0, my_g1 = 0;
#pragma unroll 1  // unrolled, the loop spills
        for (int j = 0; j < cnt; ++j) {
            const int64_t r = r0 + j;
            const int64_t b = r / n_edges;
            const int e = static_cast<int>(r - b * n_edges);
            const int64_t ps = (b * n + __ldg(src + e)) * kPQ, qd = (b * n + __ldg(dst + e)) * kPQ + kHid;
            const float2 p = __ldg(reinterpret_cast<const float2*>(pq + ps) + lane);
            const float2 q = __ldg(reinterpret_cast<const float2*>(pq + qd) + lane);
            const float pre0 = __fadd_rn(__fadd_rn(p.x, q.x), bb.x), pre1 = __fadd_rn(__fadd_rn(p.y, q.y), bb.y);
            const float h0 = pre0 > 0.f ? pre0 : 0.f, h1 = pre1 > 0.f ? pre1 : 0.f;
            float acc = __fmaf_rn(ww.y, h1, __fmul_rn(ww.x, h0));
#pragma unroll
            for (int o = 16; o; o >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, o));  // same bits in every lane
            const uint32_t g0 = __ballot_sync(0xffffffffu, pre0 > 0.f), g1 = __ballot_sync(0xffffffffu, pre1 > 0.f);
            if (lane == j) {
                my_logit = __fadd_rn(acc, c2);
                my_g0 = g0;
                my_g1 = g1;
            }
        }
        if (lane >= cnt) continue;
        const int64_t r = r0 + lane;
        if (!train) {
            mask[r] = sigmoidf(my_logit);
            continue;
        }
        const uint4 rnd = ptx::philox4x32_7(static_cast<uint32_t>(r), static_cast<uint32_t>(r >> 32) ^ 0x3c6ef372u,
                                            static_cast<uint32_t>(key), static_cast<uint32_t>(key >> 32));
        const float u = static_cast<float>(rnd.x >> 8) * 0x1p-24f;                  // U[0, 1), 24 bits
        const float eps = __fadd_rn(__fmul_rn(eps_scale, u), eps_bias);
        const float sv = __fmul_rn(__fadd_rn(__fsub_rn(logf(eps), logf(__fsub_rn(1.f, eps))), my_logit), it);
        s_out[r] = sv;
        mask[r] = sigmoidf(sv);
        gate[r] = make_uint2(my_g0, my_g1);  // bit l of word j <-> unit 2l + j
        if (uniform) uniform[r] = u;
    }
}

__global__ void __launch_bounds__(256)
pg_edge_bwd_kernel(int64_t rows, int32_t n, int32_t n_edges, const int32_t* __restrict__ out_ptr,
                   const int32_t* __restrict__ out_edge, const int32_t* __restrict__ in_ptr,
                   const int32_t* __restrict__ in_edge, const int32_t* __restrict__ dst, const float* __restrict__ pq,
                   const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ inv_t,
                   const float* __restrict__ mask, const float* __restrict__ dmask, const uint2* __restrict__ gate,
                   float* __restrict__ R, float* __restrict__ parts) {
    __shared__ float red[kWarps][kPartStride];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    const float2 bb = __ldg(reinterpret_cast<const float2*>(b1) + lane);
    const float2 ww = __ldg(reinterpret_cast<const float2*>(w2) + lane);
    const float it = __ldg(inv_t);
    float2 db1 = make_float2(0.f, 0.f), dw2 = make_float2(0.f, 0.f);
    float db2 = 0.f;
    for (int64_t r = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; r < rows; r += nwarps) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        const float2 p = __ldg(reinterpret_cast<const float2*>(pq + r * kPQ) + lane);
        const float* mb = mask + b * n_edges;
        const float* db = dmask + b * n_edges;
        const uint2* gb = gate + b * n_edges;
        float2 rs = make_float2(0.f, 0.f), rd = make_float2(0.f, 0.f);
        for (int k = __ldg(out_ptr + i), end = __ldg(out_ptr + i + 1); k < end; ++k) {  // edges with src = i
            const int e = __ldg(out_edge + k);
            const float m = __ldg(mb + e);
            const float dl = __fmul_rn(__fmul_rn(__ldg(db + e), __fmul_rn(m, __fsub_rn(1.f, m))), it);
            const uint2 g = __ldg(gb + e);
            const float2 q = __ldg(reinterpret_cast<const float2*>(pq + (b * n + __ldg(dst + e)) * kPQ + kHid) + lane);
            const float pre0 = __fadd_rn(__fadd_rn(p.x, q.x), bb.x), pre1 = __fadd_rn(__fadd_rn(p.y, q.y), bb.y);
            const float gh0 = (g.x >> lane) & 1u ? __fmul_rn(dl, ww.x) : 0.f;
            const float gh1 = (g.y >> lane) & 1u ? __fmul_rn(dl, ww.y) : 0.f;
            rs.x = __fadd_rn(rs.x, gh0);
            rs.y = __fadd_rn(rs.y, gh1);
            db1.x = __fadd_rn(db1.x, gh0);
            db1.y = __fadd_rn(db1.y, gh1);
            dw2.x = __fmaf_rn(dl, pre0 > 0.f ? pre0 : 0.f, dw2.x);
            dw2.y = __fmaf_rn(dl, pre1 > 0.f ? pre1 : 0.f, dw2.y);
            db2 = __fadd_rn(db2, dl);
        }
        for (int k = __ldg(in_ptr + i), end = __ldg(in_ptr + i + 1); k < end; ++k) {  // edges with dst = i
            const int e = __ldg(in_edge + k);
            const float m = __ldg(mb + e);
            const float dl = __fmul_rn(__fmul_rn(__ldg(db + e), __fmul_rn(m, __fsub_rn(1.f, m))), it);
            const uint2 g = __ldg(gb + e);
            rd.x = __fadd_rn(rd.x, (g.x >> lane) & 1u ? __fmul_rn(dl, ww.x) : 0.f);
            rd.y = __fadd_rn(rd.y, (g.y >> lane) & 1u ? __fmul_rn(dl, ww.y) : 0.f);
        }
        reinterpret_cast<float2*>(R + r * kPQ)[lane] = rs;
        reinterpret_cast<float2*>(R + r * kPQ + kHid)[lane] = rd;
    }
    // this CTA's partials: warps added in index order
    red[wid][2 * lane] = db1.x;
    red[wid][2 * lane + 1] = db1.y;
    red[wid][kHid + 2 * lane] = dw2.x;
    red[wid][kHid + 2 * lane + 1] = dw2.y;
    if (lane == 0) red[wid][2 * kHid] = db2;
    __syncthreads();
    for (int j = threadIdx.x; j < kParts; j += blockDim.x) {
        float a = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) a = __fadd_rn(a, red[w][j]);
        parts[static_cast<int64_t>(blockIdx.x) * kPartStride + j] = a;
    }
}

int bwd_grid(const DeviceInfo* di) { return di->sm_count * 4; }

bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

}  // namespace

extern "C" int ltgnn_pg_edge_fwd(int device, int64_t B, int32_t N, int32_t E, const int32_t* src, const int32_t* dst,
                                 const float* pq, const float* b1, const float* w2, const float* b2, const float* inv_t,
                                 float bias, uint64_t seed, float* mask, float* s, uint32_t* gate, float* uniform,
                                 void* stream_) {
    LTGNN_REQUIRE(B >= 0 && N > 0 && E >= 0, LTGNN_E_ARG, "pg_edge_fwd: B=%lld N=%d E=%d", static_cast<long long>(B), N,
                  E);
    LTGNN_REQUIRE(bias >= 0.f && bias <= 0.5f, LTGNN_E_ARG, "pg_edge_fwd: bias %g outside [0, 0.5]", bias);
    if (B == 0 || E == 0) return LTGNN_OK;
    LTGNN_REQUIRE(src && dst && pq && b1 && w2 && b2 && mask, LTGNN_E_ARG, "pg_edge_fwd: null pointer");
    LTGNN_REQUIRE(inv_t ? (s && gate) : (!s && !gate && !uniform), LTGNN_E_ARG,
                  "pg_edge_fwd: training (inv_t) writes s and gate; explaining writes the mask only");
    LTGNN_REQUIRE(aligned8(pq) && aligned8(b1) && aligned8(w2) && aligned8(gate), LTGNN_E_ALIGN,
                  "pg_edge_fwd: pq, b1, w2 and gate must be 8-byte aligned");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "pg_edge_fwd: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_USE_DEVICE(device);
    const int64_t rows = B * E;
    const int64_t blocks = (rows + 32 * kWarps - 1) / (32 * kWarps), cap = static_cast<int64_t>(di->sm_count) * 16;
    pg_edge_fwd_kernel<<<static_cast<unsigned>(blocks < cap ? blocks : cap), 256, 0,
                         static_cast<cudaStream_t>(stream_)>>>(
        rows, N, E, src, dst, pq, b1, w2, b2, inv_t, static_cast<float>(1.0 - 2.0 * bias), bias, seed,
        inv_t ? seed_source() : nullptr, mask, s, reinterpret_cast<uint2*>(gate), uniform);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int64_t ltgnn_pg_edge_bwd_ws_floats(int device) {
    const DeviceInfo* di = device_info(device);
    return di ? static_cast<int64_t>(bwd_grid(di)) * kPartStride : -1;
}

extern "C" int ltgnn_pg_edge_bwd(int device, int64_t B, int32_t N, int32_t E, const int32_t* out_ptr,
                                 const int32_t* out_edge, const int32_t* in_ptr, const int32_t* in_edge,
                                 const int32_t* dst, const float* pq, const float* b1, const float* w2,
                                 const float* inv_t, const float* mask, const float* dmask, const uint32_t* gate,
                                 float* R, float* dparams, float* ws, void* stream_) {
    LTGNN_REQUIRE(B >= 0 && N > 0 && E >= 0, LTGNN_E_ARG, "pg_edge_bwd: B=%lld N=%d E=%d", static_cast<long long>(B), N,
                  E);
    LTGNN_REQUIRE(out_ptr && out_edge && in_ptr && in_edge && dst && pq && b1 && w2 && inv_t && mask && dmask && gate &&
                  R && dparams && ws, LTGNN_E_ARG, "pg_edge_bwd: null pointer");
    LTGNN_REQUIRE(aligned8(pq) && aligned8(b1) && aligned8(w2) && aligned8(gate) && aligned8(R), LTGNN_E_ALIGN,
                  "pg_edge_bwd: pq, b1, w2, gate and R must be 8-byte aligned");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "pg_edge_bwd: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_USE_DEVICE(device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int grid = bwd_grid(di);
    pg_edge_bwd_kernel<<<grid, 256, 0, stream>>>(B * N, N, E, out_ptr, out_edge, in_ptr, in_edge, dst, pq, b1, w2, inv_t,
                                                 mask, dmask, reinterpret_cast<const uint2*>(gate), R, ws);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return reduce_parts(ws, kPartStride, dparams, grid, kParts, 0, stream);
}
