// tcn_train.cu -- training of the TCN normal-state predictor on its dependency cone (reference models/predictor.py:17-81,
// train_predictor.py).  The loss reads only the last time step, so every parameter gradient depends only on the
// (window, position) rows of the cone that tcn.cu already evaluates: training runs the same gathered-row convolutions.
//
//   forward   ltgnn_tcn_conv_train: z = bias + sum_tap X[src[tap]] W_tap^T on tcn.cu's tensor-core pipeline (no LayerNorm),
//             then one row kernel: mean / rstd (the fused epilogue's two-pass order: bit-identical Y at drop_p = 0),
//             LayerNorm, ReLU, inverted dropout (Philox, launch seed + ltgnn_seed_source word), 1-bit live mask, residual.
//             z and (mean, rstd) are what LayerNorm's backward needs; x_hat is never rebuilt from Y (that divides by gamma).
//   epilogue backward  ltgnn_tcn_ln_bwd: dz = LN_bwd(dY * live / (1 - p)) with the column sums d gamma, d beta, d bias
//             (per-CTA partials of a fixed row range, added in CTA order: deterministic, no atomics).
//   input gradient  ltgnn_tcn_conv itself: dX[r] = sum_tap dz[inv[tap][r]] W_tap with the per-tap transposed weight and
//             the inverse index (a tap's row map is injective inside a window), plus the residual pass-through.
//   weight gradient  ltgnn_tcn_wgrad: dW[tap] = dz^T X[src[tap]] on tgrad.cuh's tensor-core kernel (per-chunk flush), the
//             X operand gathered through src while it is loaded -- no im2col.
#include "functors.cuh"
#include "tgrad.cuh"

using namespace ltgnn;
using ltgnn::ptx::launch_seed;
using ltgnn::ptx::philox4x32_7;

namespace {

constexpr int kC = 128;

// Thread = (row, 64-channel half), the mapping of tcn.cu's epilogue: the sums over a row's channels run in the same order
// and the two halves exchange them through shared memory, so that Y equals ltgnn_tcn_conv's bit for bit without dropout.
__global__ void __launch_bounds__(256)
tcn_ln_fwd_kernel(const float4* __restrict__ z, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                  const float4* __restrict__ res, const int32_t* __restrict__ res_row, uint32_t thresh, float keep_scale,
                  uint64_t drop_seed, const uint64_t* seed_src, float4* __restrict__ Y, float2* __restrict__ stats,
                  uint2* __restrict__ live, uint32_t M) {
    __shared__ float stat_s[2][2][128];
    __shared__ float4 prm_s[2][kC / 4];
    const int tid = threadIdx.x, rt = tid & 127, half = tid >> 7;
    if (tid < kC) {
        reinterpret_cast<float*>(prm_s[0])[tid] = __ldg(gamma + tid);
        reinterpret_cast<float*>(prm_s[1])[tid] = __ldg(beta + tid);
    }
    const uint32_t row = blockIdx.x * 128 + rt;
    const bool ok = row < M;
    const float4* zr = z + static_cast<size_t>(ok ? row : 0) * (kC / 4) + half * 16;
    float4 v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = ok ? __ldg(zr + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float inv_c = 1.f / static_cast<float>(kC);
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) s += v[j].x + v[j].y + v[j].z + v[j].w;
    stat_s[0][half][rt] = s;
    __syncthreads();
    const float mean = (stat_s[0][0][rt] + stat_s[0][1][rt]) * inv_c;
    float s2 = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float d0 = v[j].x - mean, d1 = v[j].y - mean, d2 = v[j].z - mean, d3 = v[j].w - mean;
        s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2); s2 = fmaf(d2, d2, s2); s2 = fmaf(d3, d3, s2);
    }
    stat_s[1][half][rt] = s2;
    __syncthreads();
    const float rstd = 1.f / sqrtf((stat_s[1][0][rt] + stat_s[1][1][rt]) * inv_c + eps);
    if (!ok) return;
    if (half == 0) stats[row] = make_float2(mean, rstd);
    const int32_t rr = res ? __ldg(res_row + row) : -1;
    const uint64_t seed = thresh ? launch_seed(drop_seed, seed_src) : 0;
    uint32_t bits[2] = {0u, 0u};
    float4* yr = Y + static_cast<size_t>(row) * (kC / 4) + half * 16;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const int c4 = half * 16 + j;
        const float4 g4 = prm_s[0][c4], e4 = prm_s[1][c4];
        float y[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
        const float gg[4] = {g4.x, g4.y, g4.z, g4.w}, ee[4] = {e4.x, e4.y, e4.z, e4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = fmaxf(fmaf((y[i] - mean) * rstd, gg[i], ee[i]), 0.f);
        if (thresh) {
            const uint64_t idx4 = static_cast<uint64_t>(row) * (kC / 4) + c4;
            const uint4 r = philox4x32_7(static_cast<uint32_t>(idx4), static_cast<uint32_t>(idx4 >> 32),
                                         static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
            const uint32_t rv[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) y[i] = rv[i] >= thresh ? y[i] * keep_scale : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) bits[j >> 3] |= (y[i] > 0.f ? 1u : 0u) << (4 * (j & 7) + i);
        const float4 a = rr >= 0 ? __ldg(res + static_cast<size_t>(rr) * (kC / 4) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        yr[j] = make_float4(y[0] + a.x, y[1] + a.y, y[2] + a.z, y[3] + a.w);
    }
    if (live) live[static_cast<size_t>(row) * 2 + half] = make_uint2(bits[0], bits[1]);
}

// Warp = row, lane = channels 4 lane .. 4 lane + 3.  CTA b takes the rows [b per, (b + 1) per), its warps every eighth;
// the per-lane column sums of the CTA's warps are added in warp order into part[b] = [d gamma | d beta | d bias].
constexpr int kLnBwdWarps = 8;
__global__ void __launch_bounds__(kLnBwdWarps * 32)
tcn_ln_bwd_kernel(const float4* __restrict__ dY, const uint32_t* __restrict__ live, const float4* __restrict__ z,
                  const float2* __restrict__ stats, const float4* __restrict__ gamma, float scale, float4* __restrict__ dz,
                  float4* __restrict__ part, uint32_t M, uint32_t per) {
    __shared__ float4 red_s[kLnBwdWarps][3][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float4 g4 = __ldg(gamma + lane);
    const float inv_c = 1.f / static_cast<float>(kC);
    float4 sg = make_float4(0.f, 0.f, 0.f, 0.f), sb = sg, sz = sg;
    const uint32_t r0 = blockIdx.x * per, r1 = r0 + per < M ? r0 + per : M;
    for (uint32_t row = r0 + warp; row < r1; row += kLnBwdWarps) {
        const size_t o = static_cast<size_t>(row) * (kC / 4) + lane;
        const float4 d = __ldg(dY + o), zv = __ldg(z + o);
        const float2 st = __ldg(stats + row);
        const uint32_t nib = __ldg(live + static_cast<size_t>(row) * 4 + (lane >> 3)) >> (4 * (lane & 7));
        const float g[4] = {nib & 1u ? d.x * scale : 0.f, nib & 2u ? d.y * scale : 0.f, nib & 4u ? d.z * scale : 0.f,
                            nib & 8u ? d.w * scale : 0.f};
        const float xh[4] = {(zv.x - st.x) * st.y, (zv.y - st.x) * st.y, (zv.z - st.x) * st.y, (zv.w - st.x) * st.y};
        const float gm[4] = {g4.x, g4.y, g4.z, g4.w};
        float dx[4], a = 0.f, b = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            dx[i] = g[i] * gm[i];
            a += dx[i];
            b = fmaf(dx[i], xh[i], b);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, off);
            b += __shfl_xor_sync(0xffffffffu, b, off);
        }
        a *= inv_c;
        b *= inv_c;
        float dzv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) dzv[i] = st.y * (dx[i] - a - xh[i] * b);
        dz[o] = make_float4(dzv[0], dzv[1], dzv[2], dzv[3]);
        sg.x = fmaf(g[0], xh[0], sg.x); sg.y = fmaf(g[1], xh[1], sg.y); sg.z = fmaf(g[2], xh[2], sg.z); sg.w = fmaf(g[3], xh[3], sg.w);
        sb.x += g[0]; sb.y += g[1]; sb.z += g[2]; sb.w += g[3];
        sz.x += dzv[0]; sz.y += dzv[1]; sz.z += dzv[2]; sz.w += dzv[3];
    }
    red_s[warp][0][lane] = sg;
    red_s[warp][1][lane] = sb;
    red_s[warp][2][lane] = sz;
    __syncthreads();
    if (threadIdx.x < 96) {
        const int q = threadIdx.x >> 5;
        float4 t = red_s[0][q][lane];
#pragma unroll
        for (int w = 1; w < kLnBwdWarps; ++w) {
            const float4 u = red_s[w][q][lane];
            t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w;
        }
        part[static_cast<size_t>(blockIdx.x) * 96 + q * 32 + lane] = t;
    }
}

int ln_bwd_grid(const DeviceInfo* di, int64_t M, uint32_t* per) {
    // at least 64 rows per CTA; at most 4 CTAs per SM
    int64_t grid = (M + 63) / 64;
    if (grid > 4ll * di->sm_count) grid = 4ll * di->sm_count;
    if (grid < 1) grid = 1;
    *per = static_cast<uint32_t>((M + grid - 1) / grid);
    return static_cast<int>((M + *per - 1) / *per);
}

// X operand of the weight gradient read through the gather index of one tap (-1 = the zero row of the left padding)
struct GatheredRows {
    static constexpr bool kRowFast = false;
    const float4* x;       // [x_rows, 32]
    const int32_t* src;    // [M]
    __device__ __forceinline__ float4 operator()(uint32_t row, int c) const {
        const int32_t s = __ldg(src + row);
        return s < 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : ptx::ldg_stream(x + static_cast<int64_t>(s) * (kC / 4) + c);
    }
};

}  // namespace

extern "C" int ltgnn_tcn_conv_train(int device, int64_t M, int32_t C, int32_t taps, const float* X, const int32_t* src,
                                    const float* W, const float* bias, const float* gamma, const float* beta, float eps,
                                    const float* res, const int32_t* res_row, float drop_p, uint64_t drop_seed, float* Y,
                                    float* Z, float* stats, uint32_t* live, float* ws, void* stream_) {
    LTGNN_REQUIRE(gamma && beta, LTGNN_E_ARG, "tcn_conv_train: gamma and beta are required (the training path is LayerNorm's)");
    LTGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, LTGNN_E_ARG, "tcn_conv_train: drop_p=%g", static_cast<double>(drop_p));
    LTGNN_REQUIRE(M >= 0 && M < (1ll << 31) - 512, LTGNN_E_ARG, "tcn_conv_train: M=%lld", static_cast<long long>(M));
    if (M == 0) return LTGNN_OK;
    LTGNN_REQUIRE((res == nullptr) == (res_row == nullptr), LTGNN_E_ARG, "tcn_conv_train: res and res_row come together");
    LTGNN_REQUIRE(Y && Z && stats && live, LTGNN_E_ARG, "tcn_conv_train: null output");
    LTGNN_REQUIRE(aligned16(Y) && aligned16(Z) && aligned16(stats) && aligned16(live) && aligned16(res), LTGNN_E_ALIGN,
                  "tcn_conv_train: 16-byte alignment");
    // z = bias + the gathered convolution, on tcn.cu's pipeline without its LayerNorm epilogue
    int rc = ltgnn_tcn_conv(device, M, C, taps, X, src, W, bias, nullptr, nullptr, 0.f, 0, nullptr, nullptr, Z, ws, stream_);
    if (rc) return rc;
    LTGNN_USE_DEVICE(device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const double t = static_cast<double>(drop_p) * 4294967296.0;
    const uint32_t thresh = drop_p > 0.f ? static_cast<uint32_t>(t < 4294967295.0 ? t : 4294967295.0) : 0u;
    const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    tcn_ln_fwd_kernel<<<static_cast<unsigned>((M + 127) / 128), 256, 0, stream>>>(
        reinterpret_cast<const float4*>(Z), gamma, beta, eps, reinterpret_cast<const float4*>(res), res_row, thresh,
        keep_scale, drop_seed, seed_source(), reinterpret_cast<float4*>(Y), reinterpret_cast<float2*>(stats),
        reinterpret_cast<uint2*>(live), static_cast<uint32_t>(M));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int64_t ltgnn_tcn_ln_bwd_ws_floats(int device) {
    const DeviceInfo* di = device_info(device);
    return di ? 4ll * di->sm_count * 3 * kC : -1;
}

extern "C" int ltgnn_tcn_ln_bwd(int device, int64_t M, int32_t C, const float* dY, const uint32_t* live, const float* Z,
                                const float* stats, const float* gamma, float scale, float* dZ, float* dprm, float* ws,
                                void* stream_) {
    LTGNN_REQUIRE(M >= 0 && M < (1ll << 31), LTGNN_E_ARG, "tcn_ln_bwd: M=%lld", static_cast<long long>(M));
    LTGNN_REQUIRE(C == kC, LTGNN_E_SHAPE, "tcn_ln_bwd: C=%d (built for %d channels)", C, kC);
    LTGNN_REQUIRE(dprm, LTGNN_E_ARG, "tcn_ln_bwd: null dprm");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    LTGNN_USE_DEVICE(device);
    if (M == 0) {
        LTGNN_CUDA_TRY(cudaMemsetAsync(dprm, 0, sizeof(float) * 3 * kC, stream));
        return LTGNN_OK;
    }
    LTGNN_REQUIRE(dY && live && Z && stats && gamma && dZ && ws, LTGNN_E_ARG, "tcn_ln_bwd: null tensor");
    LTGNN_REQUIRE(aligned16(dY) && aligned16(Z) && aligned16(gamma) && aligned16(dZ) && aligned16(ws), LTGNN_E_ALIGN,
                  "tcn_ln_bwd: 16-byte alignment");
    LTGNN_REQUIRE((reinterpret_cast<uintptr_t>(stats) & 7u) == 0 && (reinterpret_cast<uintptr_t>(live) & 3u) == 0,
                  LTGNN_E_ALIGN, "tcn_ln_bwd: stats 8-byte, live 4-byte alignment");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    uint32_t per = 0;
    const int grid = ln_bwd_grid(di, M, &per);
    tcn_ln_bwd_kernel<<<grid, kLnBwdWarps * 32, 0, stream>>>(
        reinterpret_cast<const float4*>(dY), live, reinterpret_cast<const float4*>(Z), reinterpret_cast<const float2*>(stats),
        reinterpret_cast<const float4*>(gamma), scale, reinterpret_cast<float4*>(dZ), reinterpret_cast<float4*>(ws),
        static_cast<uint32_t>(M), per);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return reduce_parts(ws, 3 * kC, dprm, grid, 3 * kC, 0, stream);
}

extern "C" int ltgnn_tcn_wgrad(int device, int64_t M, int32_t C, int32_t taps, const float* dZ, const float* X,
                               const int32_t* src, float* dW, float* ws, void* stream_) {
    LTGNN_REQUIRE(M >= 0, LTGNN_E_ARG, "tcn_wgrad: M=%lld", static_cast<long long>(M));
    LTGNN_REQUIRE(C == kC, LTGNN_E_SHAPE, "tcn_wgrad: C=%d (built for %d channels)", C, kC);
    LTGNN_REQUIRE(taps >= 1 && taps <= 8, LTGNN_E_SHAPE, "tcn_wgrad: taps=%d", taps);
    LTGNN_REQUIRE(dW, LTGNN_E_ARG, "tcn_wgrad: null dW");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (M == 0) {
        LTGNN_USE_DEVICE(device);
        LTGNN_CUDA_TRY(cudaMemsetAsync(dW, 0, sizeof(float) * taps * kC * kC, stream));
        return LTGNN_OK;
    }
    LTGNN_REQUIRE(dZ && X && src && ws, LTGNN_E_ARG, "tcn_wgrad: null tensor");
    LTGNN_REQUIRE(aligned16(dZ) && aligned16(X) && aligned16(ws), LTGNN_E_ALIGN, "tcn_wgrad: 16-byte alignment");
    functors::StackedRows g{reinterpret_cast<const float4*>(dZ), nullptr, kC / 4, 0};
    // one launch per tap, the workspace reused in stream order (the gather of tap t runs before the launch of tap t + 1)
    for (int tap = 0; tap < taps; ++tap) {
        GatheredRows x{reinterpret_cast<const float4*>(X), src + static_cast<size_t>(tap) * M};
        int grid = 0;
        int rc = tgrad::launch<1, 4, kC / 32>(device, g, x, ws, M, kC, &grid, stream, "tcn_wgrad");
        if (rc) return rc;
        rc = tgrad::gather(ws, grid, kC, 0, kC, 0, kC, dW + static_cast<size_t>(tap) * kC * kC, kC, 0, stream);
        if (rc) return rc;
    }
    return LTGNN_OK;
}
