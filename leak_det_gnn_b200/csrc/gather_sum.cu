// gather_sum.cu -- deterministic reduction of gathered rows:
//   out[p][r, :] = sum_{e = ptr[r]} ^ {ptr[r+1] - 1} src[p][idx[e], :]      (r < rows, p < planes)
//
// The input-gradient backward of the frozen predictor's shared windows: a row several windows read (a shared TCN row
// through one tap, a series row of the GRU's layer-0 projection) receives the sum of its readers' gradients.  ptr / idx
// are the transpose of the forward's gather as a CSR (``NormalPredictorTCN._shared_readers``, ``window_reader_csr``).
// Thread = 4 columns of one output row: consecutive threads cover a row (C = 128: one warp per row, 512-byte loads), the
// adds are fp32 in ascending e from zero -- no atomics, bitwise deterministic.  Four gathered float4 loads are in flight
// before they are added.  HBM-bound: every gathered row is read once per reader, every output row written once.
#include "common.cuh"

using namespace ltgnn;

namespace {

constexpr int kThreads = 256;
constexpr int kUnroll = 4;

__global__ void __launch_bounds__(kThreads)
row_gather_sum_kernel(int32_t rows, int32_t c4, const float4* __restrict__ src, int64_t src_stride4,
                      const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx, float4* __restrict__ out,
                      int64_t out_stride4) {
    const int64_t plane = blockIdx.y;
    src += plane * src_stride4;
    out += plane * out_stride4;
    const int64_t total = static_cast<int64_t>(rows) * c4;
    for (int64_t t = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; t < total;
         t += static_cast<int64_t>(gridDim.x) * kThreads) {
        const int32_t r = static_cast<int32_t>(t / c4);
        const int32_t c = static_cast<int32_t>(t - static_cast<int64_t>(r) * c4);
        const int32_t e1 = __ldg(ptr + r + 1);
        int32_t e = __ldg(ptr + r);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (; e + kUnroll <= e1; e += kUnroll) {
            float4 v[kUnroll];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) v[u] = __ldg(src + static_cast<int64_t>(__ldg(idx + e + u)) * c4 + c);
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                acc.x += v[u].x;
                acc.y += v[u].y;
                acc.z += v[u].z;
                acc.w += v[u].w;
            }
        }
        for (; e < e1; ++e) {
            const float4 v = __ldg(src + static_cast<int64_t>(__ldg(idx + e)) * c4 + c);
            acc.x += v.x;
            acc.y += v.y;
            acc.z += v.z;
            acc.w += v.w;
        }
        out[t] = acc;
    }
}

}  // namespace

extern "C" int ltgnn_row_gather_sum(int device, int64_t rows, int32_t C, int32_t planes, const float* src,
                                    int64_t src_plane_stride, const int32_t* ptr, const int32_t* idx, float* out,
                                    int64_t out_plane_stride, void* stream_) {
    LTGNN_REQUIRE(rows >= 0 && C > 0 && planes >= 1 && planes <= 65535 && src_plane_stride >= 0 && out_plane_stride >= 0,
                  LTGNN_E_ARG, "row_gather_sum: rows=%lld C=%d planes=%d strides %lld / %lld",
                  static_cast<long long>(rows), C, planes, static_cast<long long>(src_plane_stride),
                  static_cast<long long>(out_plane_stride));
    LTGNN_REQUIRE(C % 4 == 0, LTGNN_E_SHAPE, "row_gather_sum: C=%d is not a multiple of 4", C);
    LTGNN_REQUIRE(rows < (1ll << 31) - 1, LTGNN_E_SHAPE, "row_gather_sum: %lld rows exceed the 32-bit row index",
                  static_cast<long long>(rows));
    LTGNN_REQUIRE(src && ptr && idx && out, LTGNN_E_ARG, "row_gather_sum: null tensor");
    LTGNN_REQUIRE(aligned16(src) && aligned16(out) && src_plane_stride % 4 == 0 && out_plane_stride % 4 == 0 &&
                  reinterpret_cast<uintptr_t>(ptr) % 4 == 0 && reinterpret_cast<uintptr_t>(idx) % 4 == 0,
                  LTGNN_E_ALIGN, "row_gather_sum: src, out and the plane strides 16-byte aligned, ptr and idx 4-byte");
    if (rows == 0) return LTGNN_OK;
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "row_gather_sum: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_USE_DEVICE(device);
    const int32_t c4 = C / 4;
    const int64_t blocks = (rows * c4 + kThreads - 1) / kThreads;
    const dim3 grid(static_cast<unsigned>(std::min<int64_t>(blocks, static_cast<int64_t>(di->sm_count) * 16)),
                    static_cast<unsigned>(planes));
    row_gather_sum_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream_)>>>(
        static_cast<int32_t>(rows), c4, reinterpret_cast<const float4*>(src), src_plane_stride / 4, ptr, idx,
        reinterpret_cast<float4*>(out), out_plane_stride / 4);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}
