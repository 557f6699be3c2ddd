// gru_dx.cuh -- gradient of the shared sensor GRU encoder with respect to its inputs, for both hidden sizes (gru.cu: 64,
// gru_pred.cu: 128).  With g_r, g_z, g_n the gradients of the input pre-activations of sequence q = b S + s at step t,
//   dx[c] = sum_j g_r[j] W_ih[j, c] + g_z[j] W_ih[H + j, c] + g_n[j] W_ih[2H + j, c],   c = 0 .. F
// d residual[b, t, s] = dx[0] is written directly; the time-feature columns dx[1 .. F] go to per-sequence rows
// dxt[b, t, s, :] that the caller sums over s once every sequence is done (sequences may run in several launches).
// Thread = one (sequence, step) row: dG is streamed once, W_ih sits in shared memory zero-padded to 32 columns and is read
// as warp-wide float4 broadcasts, and the 1 + F dots are fp32 FMAs in a fixed order (group r, z, n; unit ascending):
// no atomics, bitwise deterministic.  At 1 + F <= 31 a tensor-core product would not pay for its hi / lo split.
#pragma once
#include "common.cuh"

namespace ltgnn {
namespace gru_dx {

constexpr int kCols = 32;      // W_ih columns held per row in shared memory: 1 + F <= 31, zero-padded
constexpr int kThreads = 256;
constexpr int kBlocksPerSm = 2;  // up to 128 registers: at 80 the 32 accumulators spill

// Layout: the dG storage of one caller.  rows = rows of the launch; decode(row, q, t) -> false for pad rows, else the
// global sequence q and step t; load(row, g, j4) = units 4 j4 .. 4 j4 + 3 of input group g (0 = r, 1 = z, 2 = n).
template <int H, class Layout>
__global__ void __launch_bounds__(kThreads, kBlocksPerSm)
gru_bwd_dx_kernel(const Layout lay, const float* __restrict__ w_ih, float* __restrict__ dr, float* __restrict__ dxt,
                  uint32_t S, int L, int F, uint64_t magic_s) {
    extern __shared__ float4 w_s[];  // [3H][kCols / 4]
    const int nc = 1 + F;
    for (int i = threadIdx.x; i < 3 * H * kCols; i += kThreads) {
        const int j = i / kCols, c = i - j * kCols;
        reinterpret_cast<float*>(w_s)[i] = c < nc ? __ldg(w_ih + j * nc + c) : 0.f;
    }
    __syncthreads();
    const int n4 = (nc + 3) / 4;  // float4 column chunks that hold data
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kThreads;
    for (int64_t row = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; row < lay.rows; row += stride) {
        uint32_t q, t;
        if (!lay.decode(row, q, t)) continue;
        float acc[kCols];
#pragma unroll
        for (int c = 0; c < kCols; ++c) acc[c] = 0.f;
#pragma unroll 1
        for (int g = 0; g < 3; ++g) {
#pragma unroll 4
            for (int j4 = 0; j4 < H / 4; ++j4) {
                const float4 v = lay.load(row, g, j4);
                const float gv[4] = {v.x, v.y, v.z, v.w};
                const float4* wr = w_s + (g * H + 4 * j4) * (kCols / 4);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
#pragma unroll
                    for (int c4 = 0; c4 < kCols / 4; ++c4) {
                        if (c4 < n4) {
                            const float4 w = wr[e * (kCols / 4) + c4];
                            acc[4 * c4 + 0] = fmaf(gv[e], w.x, acc[4 * c4 + 0]);
                            acc[4 * c4 + 1] = fmaf(gv[e], w.y, acc[4 * c4 + 1]);
                            acc[4 * c4 + 2] = fmaf(gv[e], w.z, acc[4 * c4 + 2]);
                            acc[4 * c4 + 3] = fmaf(gv[e], w.w, acc[4 * c4 + 3]);
                        }
                    }
                }
            }
        }
        const uint32_t b = magic_s ? ptx::fastdiv(q, magic_s) : q;
        const size_t o = (static_cast<size_t>(b) * L + t) * S + (q - b * S);  // (b, t, s) of the (B, L, S) input
        if (dr) dr[o] = acc[0];
        if (dxt) {
            float* dst = dxt + o * F;
#pragma unroll
            for (int c = 1; c < kCols; ++c)
                if (c <= F) dst[c - 1] = acc[c];
        }
    }
}

inline size_t smem_bytes(int H) { return static_cast<size_t>(3) * H * kCols * 4; }

// one wave of resident blocks at most: every block stages W_ih once
inline int grid_for(int64_t rows, int sm_count) {
    const int64_t blocks = (rows + kThreads - 1) / kThreads, cap = static_cast<int64_t>(sm_count) * kBlocksPerSm;
    return static_cast<int>(blocks < cap ? blocks : cap);
}

}  // namespace gru_dx
}  // namespace ltgnn
