// edge_mask.cu -- PyG's explainer edge mask on the weighted adjacency, and one GNNExplainer epoch's mask update.
//
//   message mask   vals[b, k] = base[k] * f,  f = mask[b, edge(k)] for an entry k off the diagonal, 1 for the self loop
//                  gcn_norm appended (PyG's explain_message: edge_mask[loop_mask] then cat(ones(N)); an input self loop
//                  is dropped by add_remaining_self_loops, so its mask value is never read and its gradient is 0).  base is
//                  the per-call normalisation (ltgnn_edge_norm_fwd) or the handle's own values; both orders are written,
//                  t_vals[b, k'] = t_base[k'] * f -- the same products, since t_base = base[t_perm] bit for bit.  The
//                  mask multiplies the normalised value: degrees do not see it.  One thread per (window, node) walks
//                  that node's rows of A_hat and A_hat^T: no atomics, no allocation, no host synchronisation.
//   its backward   d mask[b, edge(k)] = dvals[b, k] * base[k],  d base[b, k] = dvals[b, k] * f;  a mask (or base) shared
//                  by every window gets the sum of its B rows through reduce_parts (fixed two-stage order).
//   explain step   GNNExplainer (PyG 2.x, edge_mask_type='object', edge_reduction='sum') on the logits m of a (B, E) mask
//                  s = sigmoid(m): d m from d loss / d s, the size and entropy regularisers on the hard mask, Adam, and the
//                  new m and s -- one block per window, one pass over its E logits.
#include "common.cuh"

using namespace ltgnn;

namespace {

__device__ __forceinline__ float base_val(const float* bb, const int2 cv, const int k) {
    return bb ? __ldg(bb + k) : __int_as_float(cv.y);
}

template <bool kBase>
__global__ void __launch_bounds__(256)
edge_mask_fwd_kernel(const int32_t* __restrict__ rowptr, const int2* __restrict__ colval,
                     const int32_t* __restrict__ t_rowptr, const int2* __restrict__ t_colval,
                     const int32_t* __restrict__ ent_edge, const int32_t* __restrict__ t_ent_edge,
                     const float* __restrict__ mask, int64_t mask_stride, const float* __restrict__ base,
                     const float* __restrict__ t_base, int64_t base_stride, int32_t n, int32_t nnz, int64_t rows,
                     float* __restrict__ vals, float* __restrict__ t_vals) {
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
         r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        const float* mb = mask + b * mask_stride;
        const float* bb = base + b * base_stride;
        const float* tb = t_base + b * base_stride;
        for (int k = __ldg(rowptr + i), e = __ldg(rowptr + i + 1); k < e; ++k) {  // i = dst
            const int2 cv = __ldg(colval + k);
            const float v = kBase ? __ldg(bb + k) : __int_as_float(cv.y);
            vals[b * nnz + k] = cv.x == i ? v : __fmul_rn(v, __ldg(mb + __ldg(ent_edge + k)));
        }
        for (int k = __ldg(t_rowptr + i), e = __ldg(t_rowptr + i + 1); k < e; ++k) {  // i = src
            const int2 cv = __ldg(t_colval + k);
            const float v = kBase ? __ldg(tb + k) : __int_as_float(cv.y);
            t_vals[b * nnz + k] = cv.x == i ? v : __fmul_rn(v, __ldg(mb + __ldg(t_ent_edge + k)));
        }
    }
}

__global__ void __launch_bounds__(256)
edge_mask_bwd_kernel(const int32_t* __restrict__ rowptr, const int2* __restrict__ colval,
                     const int32_t* __restrict__ ent_edge, const float* __restrict__ mask, int64_t mask_stride,
                     const float* __restrict__ base, int64_t base_stride, int32_t n, int32_t nnz, int32_t n_edges,
                     int64_t rows, const float* __restrict__ dvals, float* __restrict__ dmask, float* __restrict__ dbase) {
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
         r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t b = r / n;
        const int i = static_cast<int>(r - b * n);
        const float* mb = mask + b * mask_stride;
        const float* bb = base ? base + b * base_stride : nullptr;
        for (int k = __ldg(rowptr + i), e = __ldg(rowptr + i + 1); k < e; ++k) {
            const int2 cv = __ldg(colval + k);
            const float g = __ldg(dvals + b * nnz + k);
            if (cv.x == i) {  // gcn_norm's self loop: factor 1, no mask value
                if (dbase) dbase[b * nnz + k] = g;
                continue;
            }
            const int32_t ed = __ldg(ent_edge + k);
            dmask[b * n_edges + ed] = __fmul_rn(g, base_val(bb, cv, k));
            if (dbase) dbase[b * nnz + k] = __fmul_rn(g, __ldg(mb + ed));
        }
    }
}

constexpr float kEntEps = 1e-15f;  // PyG's EPS in GNNExplainer's entropy

// One block per window row: dm = dL/ds * s(1-s) (+ the regularisers on the hard mask), Adam, m and s = sigmoid(m).
// record: epoch 0 -- no regulariser; hard = (dm != 0) and its per-window count (integer: exact in any order).
__global__ void __launch_bounds__(256)
explain_step_kernel(int64_t B, int32_t E, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ s,
                    float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq, uint8_t* __restrict__ hard,
                    int32_t* __restrict__ n_hard, const int32_t* __restrict__ step, double lr, double beta1, double beta2,
                    double eps, float edge_size, float edge_ent, int record) {
    __shared__ int32_t red[256];
    // torch.optim.Adam's bias corrections (computed in double there, from a host-side step count)
    const int t = __ldg(step) + 1;
    const float step_size = static_cast<float>(lr / (1.0 - pow(beta1, t)));
    const float bc2_sqrt = static_cast<float>(sqrt(1.0 - pow(beta2, t)));
    const float b1c = static_cast<float>(1.0 - beta1), b2 = static_cast<float>(beta2), b2c = static_cast<float>(1.0 - beta2);
    const float epsf = static_cast<float>(eps);
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
        const int64_t row = b * E;
        float ent_coef = 0.f;
        if (!record) {
            const int32_t nh = __ldg(n_hard + b);
            ent_coef = nh > 0 ? edge_ent / static_cast<float>(nh) : 0.f;  // no hard entry: PyG's mean is NaN, its mask 0
        }
        int32_t cnt = 0;
        for (int e = threadIdx.x; e < E; e += blockDim.x) {
            const int64_t idx = row + e;
            const float sv = s[idx];
            const float sp = sv * (1.f - sv);
            float dm = __ldg(g + idx) * sp;
            if (record) {
                const bool h = dm != 0.f;
                hard[idx] = h;
                cnt += h;
            } else if (hard[idx]) {
                // d/ds [edge_size s + coef * H(s)],  H(s) = -s log(s + EPS) - (1 - s) log(1 - s + EPS)
                const float q = 1.f - sv;
                const float dh = -logf(sv + kEntEps) - sv / (sv + kEntEps) + logf(q + kEntEps) + q / (q + kEntEps);
                dm += (edge_size + ent_coef * dh) * sp;
            }
            float a = exp_avg[idx], v = exp_avg_sq[idx];
            a += b1c * (dm - a);                      // lerp(grad, 1 - beta1)
            v = v * b2 + b2c * dm * dm;
            exp_avg[idx] = a;
            exp_avg_sq[idx] = v;
            const float mv = m[idx] - step_size * (a / (sqrtf(v) / bc2_sqrt + epsf));
            m[idx] = mv;
            s[idx] = 1.f / (1.f + expf(-mv));
        }
        if (record) {
            red[threadIdx.x] = cnt;
            __syncthreads();
            for (int w = blockDim.x >> 1; w > 0; w >>= 1) {
                if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
                __syncthreads();
            }
            if (threadIdx.x == 0) n_hard[b] = red[0];
            __syncthreads();
        }
    }
}

__global__ void explain_step_count_kernel(int32_t* step) { *step += 1; }

int grid_for(const ltgnn_graph* g, int64_t threads) {
    int64_t blocks = (threads + 255) / 256;
    const int64_t cap = static_cast<int64_t>(g->sm_count) * 16;
    return static_cast<int>(blocks < cap ? blocks : cap);
}

}  // namespace

extern "C" int ltgnn_edge_mask_fwd(ltgnn_graph_t g, int64_t B, int32_t n_edges, const float* mask, int64_t mask_stride,
                                   const float* base, const float* t_base, int64_t base_stride, const int32_t* ent_edge,
                                   const int32_t* t_ent_edge, float* vals, float* t_vals, void* stream_) {
    LTGNN_REQUIRE(g != nullptr, LTGNN_E_ARG, "edge_mask_fwd: null graph handle");
    LTGNN_REQUIRE(B >= 0 && n_edges >= 0, LTGNN_E_ARG, "edge_mask_fwd: B=%lld E=%d", static_cast<long long>(B), n_edges);
    LTGNN_REQUIRE(mask_stride == 0 || mask_stride == n_edges, LTGNN_E_ARG, "edge_mask_fwd: mask_stride must be 0 or E");
    LTGNN_REQUIRE(base_stride == 0 || base_stride == g->nnz, LTGNN_E_ARG, "edge_mask_fwd: base_stride must be 0 or nnz");
    LTGNN_REQUIRE(!base == !t_base, LTGNN_E_ARG, "edge_mask_fwd: pass both base orders or neither");
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE((mask || n_edges == 0) && ent_edge && t_ent_edge && vals && t_vals, LTGNN_E_ARG,
                  "edge_mask_fwd: null pointer");
    LTGNN_USE_DEVICE(g->device);
    const int64_t rows = B * g->n;
    (base ? edge_mask_fwd_kernel<true> : edge_mask_fwd_kernel<false>)<<<grid_for(g, rows), 256, 0,
                                                                       static_cast<cudaStream_t>(stream_)>>>(
        g->rowptr[0], g->colval[0], g->rowptr[1], g->colval[1], ent_edge, t_ent_edge, mask, mask_stride, base, t_base,
        base_stride, g->n, g->nnz, rows, vals, t_vals);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_edge_mask_bwd(ltgnn_graph_t g, int64_t B, int32_t n_edges, const float* mask, int64_t mask_stride,
                                   const float* base, int64_t base_stride, const int32_t* ent_edge, const float* dvals,
                                   float* dmask, float* dmask_sum, float* dbase, float* dbase_sum, void* stream_) {
    LTGNN_REQUIRE(g != nullptr, LTGNN_E_ARG, "edge_mask_bwd: null graph handle");
    LTGNN_REQUIRE(B >= 0 && n_edges >= 0, LTGNN_E_ARG, "edge_mask_bwd: B=%lld E=%d", static_cast<long long>(B), n_edges);
    LTGNN_REQUIRE(mask_stride == 0 || mask_stride == n_edges, LTGNN_E_ARG, "edge_mask_bwd: mask_stride must be 0 or E");
    LTGNN_REQUIRE(base_stride == 0 || base_stride == g->nnz, LTGNN_E_ARG, "edge_mask_bwd: base_stride must be 0 or nnz");
    LTGNN_REQUIRE(!dbase || base, LTGNN_E_ARG, "edge_mask_bwd: d base needs per-call base values");
    LTGNN_REQUIRE(B < (1ll << 31), LTGNN_E_SHAPE, "edge_mask_bwd: B too large");
    if (B == 0 || n_edges == 0) return LTGNN_OK;
    LTGNN_REQUIRE(mask && ent_edge && dvals && dmask, LTGNN_E_ARG, "edge_mask_bwd: null pointer");
    LTGNN_USE_DEVICE(g->device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int64_t rows = B * g->n;
    LTGNN_CUDA_TRY(cudaMemsetAsync(dmask, 0, sizeof(float) * B * n_edges, stream));  // input self loops: no entry
    edge_mask_bwd_kernel<<<grid_for(g, rows), 256, 0, stream>>>(g->rowptr[0], g->colval[0], ent_edge, mask, mask_stride,
                                                                base, base_stride, g->n, g->nnz, n_edges, rows, dvals,
                                                                dmask, dbase);
    LTGNN_CUDA_TRY(cudaGetLastError());
    // a mask / base shared by every window: sum the B rows, fixed two-stage order
    if (dmask_sum) {
        const int rc = reduce_parts(dmask, n_edges, dmask_sum, static_cast<int>(B), n_edges, 0, stream);
        if (rc != LTGNN_OK) return rc;
    }
    if (dbase && dbase_sum) return reduce_parts(dbase, g->nnz, dbase_sum, static_cast<int>(B), g->nnz, 0, stream);
    return LTGNN_OK;
}

extern "C" int ltgnn_explain_step(int device, int64_t B, int32_t E, const float* g, float* m, float* s, float* exp_avg,
                                  float* exp_avg_sq, uint8_t* hard, int32_t* n_hard, int32_t* step, double lr,
                                  double beta1, double beta2, double eps, float edge_size, float edge_ent, int record,
                                  void* stream_) {
    LTGNN_REQUIRE(B >= 0 && E >= 0, LTGNN_E_ARG, "explain_step: B=%lld E=%d", static_cast<long long>(B), E);
    LTGNN_REQUIRE(lr > 0.0 && beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0, LTGNN_E_ARG,
                  "explain_step: lr %g, betas (%g, %g), eps %g", lr, beta1, beta2, eps);
    LTGNN_REQUIRE(g && m && s && exp_avg && exp_avg_sq && hard && n_hard && step, LTGNN_E_ARG, "explain_step: null pointer");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "explain_step: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_USE_DEVICE(device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (B > 0 && E > 0) {
        const int64_t cap = static_cast<int64_t>(di->sm_count) * 16;
        explain_step_kernel<<<static_cast<unsigned>(B < cap ? B : cap), 256, 0, stream>>>(
            B, E, g, m, s, exp_avg, exp_avg_sq, hard, n_hard, step, lr, beta1, beta2, eps, edge_size, edge_ent, record);
        LTGNN_CUDA_TRY(cudaGetLastError());
    }
    explain_step_count_kernel<<<1, 1, 0, stream>>>(step);  // after the update: a replayed epoch reads the next count
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}
