// edge_weight.cu -- weighted adjacency on the device: PyG's gcn_norm of per-call edge weights and the gradient with
// respect to the adjacency values.
//
//   normalisation  norm_k = dis[src_k] * w_k * dis[dst_k],  dis = deg^-1/2 (inf -> 0),  deg[i] = sum of w over row i of
//                  A_hat (entries with dst = i) in row order: edge order, self loop last -- the order of PyG's sequential
//                  scatter_add on CPU, so at w = 1 the values equal the handle's host-built ones.  One thread per
//                  (window, node) walks its rows: no atomics, no allocation, no host synchronisation.
//   its backward   d w_e = d norm_k dis[src] dis[dst] + d deg[dst],  d deg = -1/2 dis^3 d dis,
//                  d dis[i] = sum over row i of A_hat (i = dst) and of A_hat^T (i = src), fixed order.
//   adjacency grad dA[b, k] = sum_d Gg[b, i_k, d] XW[b, j_k, d] over the CSR pattern of A_hat (an SDDMM): Gg is the
//                  upstream gradient gated as the layer's backward gates it (live bits or float gate, times gate_scale).
//                  One warp per (window, row): the row of Gg stays in registers, every neighbour row of XW is read
//                  through L2 (a window's XW is a few hundred KB), dot products reduced by a fixed shuffle tree.  For
//                  weights shared by every window the (B, nnz) result is summed over windows by reduce_parts.
#include "common.cuh"

using namespace ltgnn;

namespace {

__device__ __forceinline__ float edge_w(const float* wb, const int32_t e) { return e >= 0 ? __ldg(wb + e) : 1.f; }

// dis[b, i] = deg^-1/2 (inf -> 0) as ATen's pow(-0.5): one correctly rounded sqrt, one correctly rounded division
__global__ void __launch_bounds__(256)
edge_norm_dis_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ ent_edge, const float* __restrict__ w,
                     int64_t w_stride, int32_t n, int64_t rows, float* __restrict__ dis) {
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
         r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        const float* wb = w + b * w_stride;
        float deg = 0.f;
        for (int k = __ldg(rowptr + i), e = __ldg(rowptr + i + 1); k < e; ++k) deg += edge_w(wb, __ldg(ent_edge + k));
        float d = __fdiv_rn(1.f, __fsqrt_rn(deg));
        dis[r] = isinf(d) ? 0.f : d;
    }
}

// vals[b, k] over the rows of A_hat, t_vals[b, k'] over the rows of A_hat^T; both (dis[src] * w) * dis[dst]
__global__ void __launch_bounds__(256)
edge_norm_vals_kernel(const int32_t* __restrict__ rowptr, const int2* __restrict__ colval, const int32_t* __restrict__ t_rowptr,
                      const int2* __restrict__ t_colval, const int32_t* __restrict__ ent_edge,
                      const int32_t* __restrict__ t_ent_edge, const float* __restrict__ w, int64_t w_stride, int32_t n,
                      int32_t nnz, int64_t rows, const float* __restrict__ dis, float* __restrict__ vals,
                      float* __restrict__ t_vals) {
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
         r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        const float* wb = w + b * w_stride;
        const float* db = dis + b * n;
        const float di = db[i];
        for (int k = __ldg(rowptr + i), e = __ldg(rowptr + i + 1); k < e; ++k)  // i = dst
            vals[b * nnz + k] = __fmul_rn(__fmul_rn(db[__ldg(colval + k).x], edge_w(wb, __ldg(ent_edge + k))), di);
        for (int k = __ldg(t_rowptr + i), e = __ldg(t_rowptr + i + 1); k < e; ++k)  // i = src
            t_vals[b * nnz + k] = __fmul_rn(__fmul_rn(di, edge_w(wb, __ldg(t_ent_edge + k))), db[__ldg(t_colval + k).x]);
    }
}

// ddeg[b, i] = -1/2 dis^3 (sum over entries with dst = i of dval dis[src] w  +  over entries with src = i of dval w dis[dst])
__global__ void __launch_bounds__(256)
edge_norm_ddeg_kernel(const int32_t* __restrict__ rowptr, const int2* __restrict__ colval, const int32_t* __restrict__ t_rowptr,
                      const int2* __restrict__ t_colval, const int32_t* __restrict__ ent_edge,
                      const int32_t* __restrict__ t_ent_edge, const int32_t* __restrict__ t_perm, const float* __restrict__ w,
                      int64_t w_stride, int32_t n, int32_t nnz, int64_t rows, const float* __restrict__ dis,
                      const float* __restrict__ dvals, float* __restrict__ ddeg) {
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
         r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        const float* wb = w + b * w_stride;
        const float* db = dis + b * n;
        const float* gb = dvals + b * nnz;
        float s = 0.f;
        for (int k = __ldg(rowptr + i), e = __ldg(rowptr + i + 1); k < e; ++k)
            s += gb[k] * (db[__ldg(colval + k).x] * edge_w(wb, __ldg(ent_edge + k)));
        for (int k = __ldg(t_rowptr + i), e = __ldg(t_rowptr + i + 1); k < e; ++k)
            s += gb[__ldg(t_perm + k)] * (edge_w(wb, __ldg(t_ent_edge + k)) * db[__ldg(t_colval + k).x]);
        const float di = db[i];
        ddeg[r] = di == 0.f ? 0.f : -0.5f * di * di * di * s;
    }
}

// dw[b, e] = dval_k dis[src] dis[dst] + ddeg[dst] for the entry k of edge e (each kept edge owns exactly one entry)
__global__ void __launch_bounds__(256)
edge_norm_dw_kernel(const int32_t* __restrict__ rowptr, const int2* __restrict__ colval, const int32_t* __restrict__ ent_edge,
                    int32_t n, int32_t nnz, int32_t n_edges, int64_t rows, const float* __restrict__ dis,
                    const float* __restrict__ dvals, const float* __restrict__ ddeg, float* __restrict__ dw) {
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
         r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        const float* db = dis + b * n;
        const float di = db[i], dd = ddeg[r];
        for (int k = __ldg(rowptr + i), e = __ldg(rowptr + i + 1); k < e; ++k) {
            const int32_t ed = __ldg(ent_edge + k);
            if (ed >= 0) dw[b * n_edges + ed] = dvals[b * nnz + k] * (db[__ldg(colval + k).x] * di) + dd;
        }
    }
}

// dA[b, k] (+)= <Gg[b, i], XW[b, col_k]> for the entries k of row i; one warp per (b, i), D % 4 == 0
__global__ void __launch_bounds__(256)
adj_grad_kernel(const int32_t* __restrict__ rowptr, const int2* __restrict__ colval, const float4* __restrict__ G,
                const float4* __restrict__ gate, const uint32_t* __restrict__ live, float gate_scale,
                const float4* __restrict__ XW, int32_t n, int32_t nnz, int32_t d4, int64_t rows, int accumulate,
                float* __restrict__ dA) {
    constexpr int kMaxD4 = 64;  // D <= 256
    const int lane = threadIdx.x & 31;
    const int64_t warps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        float4 gg[kMaxD4 / 32];
#pragma unroll
        for (int u = 0; u < kMaxD4 / 32; ++u) {
            const int c4 = lane + 32 * u;
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c4 < d4) {
                x = __ldg(G + r * d4 + c4);
                if (live) {
                    const uint32_t m = __ldg(live + (b * (d4 >> 3) + (c4 >> 3)) * n + i) >> (c4 & 7);
                    x.x = (m & 1u) ? x.x * gate_scale : 0.f; x.y = (m & 0x100u) ? x.y * gate_scale : 0.f;
                    x.z = (m & 0x10000u) ? x.z * gate_scale : 0.f; x.w = (m & 0x1000000u) ? x.w * gate_scale : 0.f;
                } else if (gate) {
                    const float4 m = __ldg(gate + r * d4 + c4);
                    x.x = m.x > 0.f ? x.x * gate_scale : 0.f; x.y = m.y > 0.f ? x.y * gate_scale : 0.f;
                    x.z = m.z > 0.f ? x.z * gate_scale : 0.f; x.w = m.w > 0.f ? x.w * gate_scale : 0.f;
                }
            }
            gg[u] = x;
        }
        const float4* xb = XW + b * static_cast<int64_t>(n) * d4;
        for (int k = __ldg(rowptr + i), e = __ldg(rowptr + i + 1); k < e; ++k) {
            const int j = __ldg(colval + k).x;
            float s = 0.f;
#pragma unroll
            for (int u = 0; u < kMaxD4 / 32; ++u) {
                const int c4 = lane + 32 * u;
                if (c4 < d4) {
                    const float4 x = __ldg(xb + static_cast<int64_t>(j) * d4 + c4);
                    s += gg[u].x * x.x + gg[u].y * x.y + gg[u].z * x.z + gg[u].w * x.w;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) {
                float* out = dA + b * nnz + k;
                *out = accumulate ? *out + s : s;
            }
        }
    }
}

int grid_for(const ltgnn_graph* g, int64_t threads) {
    int64_t blocks = (threads + 255) / 256;
    const int64_t cap = static_cast<int64_t>(g->sm_count) * 16;
    return static_cast<int>(blocks < cap ? blocks : cap);
}

}  // namespace

extern "C" int ltgnn_edge_norm_fwd(ltgnn_graph_t g, int64_t Bw, int32_t n_edges, const float* w, int64_t w_stride,
                                   const int32_t* ent_edge, const int32_t* t_ent_edge, float* dis, float* vals,
                                   float* t_vals, void* stream_) {
    LTGNN_REQUIRE(g != nullptr, LTGNN_E_ARG, "edge_norm_fwd: null graph handle");
    LTGNN_REQUIRE(Bw >= 0 && n_edges >= 0, LTGNN_E_ARG, "edge_norm_fwd: Bw=%lld E=%d", static_cast<long long>(Bw), n_edges);
    LTGNN_REQUIRE(w_stride == 0 || w_stride == n_edges, LTGNN_E_ARG, "edge_norm_fwd: w_stride must be 0 or E");
    if (Bw == 0) return LTGNN_OK;
    LTGNN_REQUIRE((w || n_edges == 0) && ent_edge && t_ent_edge && dis && vals && t_vals, LTGNN_E_ARG,
                  "edge_norm_fwd: null pointer");
    LTGNN_USE_DEVICE(g->device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int64_t rows = Bw * g->n;
    edge_norm_dis_kernel<<<grid_for(g, rows), 256, 0, stream>>>(g->rowptr[0], ent_edge, w, w_stride, g->n, rows, dis);
    LTGNN_CUDA_TRY(cudaGetLastError());
    edge_norm_vals_kernel<<<grid_for(g, rows), 256, 0, stream>>>(g->rowptr[0], g->colval[0], g->rowptr[1], g->colval[1],
                                                                 ent_edge, t_ent_edge, w, w_stride, g->n, g->nnz, rows,
                                                                 dis, vals, t_vals);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_edge_norm_bwd(ltgnn_graph_t g, int64_t Bw, int32_t n_edges, const float* w, int64_t w_stride,
                                   const int32_t* ent_edge, const int32_t* t_ent_edge, const int32_t* t_perm,
                                   const float* dis, const float* dvals, float* ddeg, float* dw, void* stream_) {
    LTGNN_REQUIRE(g != nullptr, LTGNN_E_ARG, "edge_norm_bwd: null graph handle");
    LTGNN_REQUIRE(Bw >= 0 && n_edges >= 0, LTGNN_E_ARG, "edge_norm_bwd: Bw=%lld E=%d", static_cast<long long>(Bw), n_edges);
    LTGNN_REQUIRE(w_stride == 0 || w_stride == n_edges, LTGNN_E_ARG, "edge_norm_bwd: w_stride must be 0 or E");
    if (Bw == 0 || n_edges == 0) return LTGNN_OK;
    LTGNN_REQUIRE(w && ent_edge && t_ent_edge && t_perm && dis && dvals && ddeg && dw, LTGNN_E_ARG,
                  "edge_norm_bwd: null pointer");
    LTGNN_USE_DEVICE(g->device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int64_t rows = Bw * g->n;
    LTGNN_CUDA_TRY(cudaMemsetAsync(dw, 0, sizeof(float) * Bw * n_edges, stream));  // edges of dropped duplicate loops
    edge_norm_ddeg_kernel<<<grid_for(g, rows), 256, 0, stream>>>(g->rowptr[0], g->colval[0], g->rowptr[1], g->colval[1],
                                                                 ent_edge, t_ent_edge, t_perm, w, w_stride, g->n, g->nnz,
                                                                 rows, dis, dvals, ddeg);
    LTGNN_CUDA_TRY(cudaGetLastError());
    edge_norm_dw_kernel<<<grid_for(g, rows), 256, 0, stream>>>(g->rowptr[0], g->colval[0], ent_edge, g->n, g->nnz,
                                                               n_edges, rows, dis, dvals, ddeg, dw);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_gcn_adj_grad(ltgnn_graph_t g, int64_t B, int32_t D, const float* G, const float* gate,
                                  const uint32_t* live_in, float gate_scale, const float* XW, float* dA, int accumulate,
                                  float* dA_sum, void* stream_) {
    LTGNN_REQUIRE(g != nullptr, LTGNN_E_ARG, "gcn_adj_grad: null graph handle");
    LTGNN_REQUIRE(B >= 0 && D > 0, LTGNN_E_ARG, "gcn_adj_grad: B=%lld D=%d", static_cast<long long>(B), D);
    LTGNN_REQUIRE(D % 4 == 0 && D <= 256, LTGNN_E_SHAPE, "gcn_adj_grad: D=%d must be a multiple of 4, <= 256", D);
    LTGNN_REQUIRE(!(gate && live_in), LTGNN_E_ARG, "gcn_adj_grad: pass the gate as floats or as bits, not both");
    LTGNN_REQUIRE(!live_in || D % 32 == 0, LTGNN_E_SHAPE, "gcn_adj_grad: 1-bit gates need D %% 32 == 0");
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(G && XW && dA, LTGNN_E_ARG, "gcn_adj_grad: null tensor");
    LTGNN_REQUIRE(aligned16(G) && aligned16(XW) && aligned16(gate), LTGNN_E_ALIGN,
                  "gcn_adj_grad: G, XW and gate must be 16-byte aligned");
    LTGNN_USE_DEVICE(g->device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int64_t rows = B * g->n;
    int64_t blocks = (rows + 7) / 8;  // 8 warps per block, one row each
    const int64_t cap = static_cast<int64_t>(g->sm_count) * 32;
    if (blocks > cap) blocks = cap;
    adj_grad_kernel<<<static_cast<int>(blocks), 256, 0, stream>>>(
        g->rowptr[0], g->colval[0], reinterpret_cast<const float4*>(G), reinterpret_cast<const float4*>(gate), live_in,
        gate_scale, reinterpret_cast<const float4*>(XW), g->n, g->nnz, D / 4, rows, dA_sum ? 0 : accumulate, dA);
    LTGNN_CUDA_TRY(cudaGetLastError());
    if (dA_sum) {  // one set of weights shared by every window: sum the windows, fixed two-stage order
        LTGNN_REQUIRE(B < (1ll << 31), LTGNN_E_SHAPE, "gcn_adj_grad: B too large");
        return reduce_parts(dA, g->nnz, dA_sum, static_cast<int>(B), g->nnz, accumulate, stream);
    }
    return LTGNN_OK;
}
