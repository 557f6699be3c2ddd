// linear.cu -- row-wise dense layer  Y = gate(act(X op(W) + b))  on tcgen05 tensor cores (3xTF32).
//
// Replaces the plain Linear layers of the detector's message-passing path that are not fused into a
// neighbouring kernel: GCNConv's `self.lin` (PyG Linear, models/detector.py:199) in the forward, its
// input-gradient GEMM dX = dXW * W in the backward (autograd of the same line), NoLeakHead
// (models/detector.py:94-99).  Built on the pipelined skeleton in rowgemm.cuh; also the validation
// vehicle for the tensor-core building blocks (tests/test_linear_gpu.py checks it against fp64).
#include "functors.cuh"
#include "rowgemm.cuh"
#include "rowgemm_ts.cuh"

using namespace ltgnn;
using namespace ltgnn::functors;

namespace {

// ---------------------------------------------------------------------------------------------------------
// Tensor-memory-operand form of the row GEMM for the streaming (HBM-bound) layers, K <= 128, N <= 128.
// In the shared-memory form (rowgemm.cuh) a 128-row tile moves ~270 KB through the SM's shared-memory pipe (hi and lo
// copies written by the loaders, read three times by the MMA, plus the epilogue patch): ncu showed the kernel at 73 % of
// the HBM peak with no other unit saturated.  Here the A operand goes to TENSOR memory: loader warps fetch rows
// cooperatively (8 lanes = 128 bytes of one row), transpose them to the row-per-thread form through a patch, split and
// tcgen05.st them; the MMA reads only the resident weight from shared memory.
//   warps 0-3   LOADERS   fill the A slots of the units (tile, 32-column K block) in order
//   warp  4     MMA       elected lane, 3xTF32
//   warps 5-12  EPILOGUE  StoreEpilogue (bias / ReLU / gate, coalesced stores through the patch); two warps per TMEM
//                         lane quadrant share the 32-column blocks -- a device-side timeline showed the epilogue, not
//                         the loads or the MMAs, setting the pace (3 300 clocks per tile with 4 warps).  Or
//                         GateSumEpilogue (node init's backward from the first layer's gradient: no product stored)
// ---------------------------------------------------------------------------------------------------------
namespace lt {
using namespace ltgnn::ptx;
using namespace ltgnn::umma;
constexpr int kLdWarps = 4, kMmaWarp = 4, kEpWarps = 8, kThreads = (kLdWarps + 1 + kEpWarps) * 32;  // 13 warps: 128 regs
constexpr int kSlots = 4, kSlotCols = 64;

template <class Epi>
__global__ void __launch_bounds__(kThreads, 1)
linear_ts_kernel(const float4* __restrict__ X, const Epi epilogue, const float* __restrict__ W, int ldw,
                 int transposed, uint32_t M, int K, int N, int depth) {
    constexpr bool kSums = std::is_same<Epi, GateSumEpilogue>::value;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_full[kSlots], bar_empty[kSlots], bar_tfull[2], bar_tempty[2];
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;
    uint8_t* b_lo = b_hi + N * K * 4;
    uint8_t* scratch = b_lo + N * K * 4;  // 4 loader rings of `depth` patches, then 8 epilogue patches
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_kg = K >> 5, k4 = K >> 2;

    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        for (int s = 0; s < kSlots; ++s) {
            mbar_init(&bar_full[s], 4);
            mbar_init(&bar_empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bar_tfull[a], 1);
            mbar_init(&bar_tempty[a], kEpWarps);
        }
        fence_mbar_init();
    }
    rowgemm_ts::fill_b(b_hi, b_lo, W, ldw, transposed, K, N, tid, kThreads);
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t acc_base = tmem_base, a_base = tmem_base + 256;  // 2 accumulators of <= 128 columns, 4 A slots
    const uint32_t n_tiles = (M + 127) / 128;
    const uint32_t per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;  // contiguous tile range per CTA
    const uint32_t t_begin = min(blockIdx.x * per_cta, n_tiles), t_end = min(t_begin + per_cta, n_tiles);
    const uint32_t n_units = (t_end - t_begin) * n_kg;

    if (warp < kLdWarps) {
        // Each loader warp owns a ring of `depth` patches that cp.async fills straight from global memory (no
        // registers in between): 4 warps x depth x 4 KB of loads are in flight per SM, which is what an HBM stream at
        // ~2 us of loaded latency needs (32 KB of register-staged loads capped this kernel at 73 % of the HBM peak).
        const int quad = warp & 3;
        uint8_t* ring = scratch + static_cast<size_t>(warp) * depth * patch::kPatchBytes;
        const uint32_t lane_base = a_base + (static_cast<uint32_t>(quad * 32) << 16);
        const int sub = lane >> 3, ch = lane & 7;
        auto fetch = [&](uint32_t unit, int slot_p) {  // 8 lanes copy the 128 bytes of one row: 4 rows per instruction
            const patch::Patch pt(ring + slot_p * patch::kPatchBytes, lane);
            if (unit < n_units) {
                const uint32_t tile = t_begin + unit / n_kg, kg = unit % n_kg;
                const uint32_t row0 = tile * 128 + quad * 32 + sub;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint32_t row = row0 + 4 * k;
                    const bool ok = row < M;  // rows past M are zero-filled (src-size 0)
                    const float4* src = X + static_cast<size_t>(ok ? row : 0) * k4 + kg * 8 + ch;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(pt.co(k))), "l"(src),
                                 "r"(ok ? 16 : 0)
                                 : "memory");
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");  // (an empty group keeps the wait count uniform)
        };
        for (int d = 0; d < depth; ++d) fetch(d, d);
        for (uint32_t unit = 0; unit < n_units; ++unit) {
            const int slot_p = static_cast<int>(unit % depth);
            if (depth == 8) asm volatile("cp.async.wait_group 7;" ::: "memory");
            else asm volatile("cp.async.wait_group 3;" ::: "memory");
            __syncwarp();
            float v[32];
            {
                const patch::Patch pt(ring + slot_p * patch::kPatchBytes, lane);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 t = *pt.row(j);
                    v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
                }
            }
            __syncwarp();
            fetch(unit + depth, slot_p);  // refill the patch just read
            const uint32_t slot = unit & 3;
            mbar_wait_relaxed(&bar_empty[slot], ((unit >> 2) & 1) ^ 1);
            fence_after_sync();
            const uint32_t st_addr = lane_base + slot * kSlotCols;
#pragma unroll
            for (int c = 0; c < 32; c += 8) {
                float hi[8], lo[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    hi[j] = tf32_hi(v[c + j]);
                    lo[j] = v[c + j] - hi[j];
                }
                asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(st_addr + c),
                             "f"(hi[0]), "f"(hi[1]), "f"(hi[2]), "f"(hi[3]), "f"(hi[4]), "f"(hi[5]), "f"(hi[6]), "f"(hi[7])
                             : "memory");
                asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(st_addr + 32 + c),
                             "f"(lo[0]), "f"(lo[1]), "f"(lo[2]), "f"(lo[3]), "f"(lo[4]), "f"(lo[5]), "f"(lo[6]), "f"(lo[7])
                             : "memory");
            }
            rowgemm_ts::tmem_wait_st();
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_full[slot]);
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if (warp == kMmaWarp) {
        const uint32_t idesc = idesc_tf32(128, N);
        const uint32_t bh = desc_lo(smem_u32(b_hi)), bl = desc_lo(smem_u32(b_lo));
        const uint32_t kg_units = static_cast<uint32_t>(N) * 128u >> 4;
        uint32_t unit = 0;
        for (uint32_t t = 0; t < t_end - t_begin; ++t) {
            const uint32_t a = t & 1;
            mbar_wait_relaxed(&bar_tempty[a], ((t >> 1) & 1) ^ 1);
            const uint32_t d = acc_base + a * 128;
            for (int kg = 0; kg < n_kg; ++kg, ++unit) {
                const uint32_t slot = unit & 3;
                mbar_wait_relaxed(&bar_full[slot], (unit >> 2) & 1);
                fence_after_sync();
                if (elect_one()) {
                    const uint32_t a_hi = a_base + slot * kSlotCols, a_lo = a_hi + 32;
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k) {
                        const uint32_t boff = kg * kg_units + 2 * k;
                        rowgemm_ts::mma_tf32_ts(d, a_lo + 8 * k, bh + boff, idesc, (kg == 0 && k == 0) ? 0u : 1u);
                        rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bl + boff, idesc, 1u);
                        rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bh + boff, idesc, 1u);
                    }
                    commit(&bar_empty[slot]);
                    if (kg == n_kg - 1) commit(&bar_tfull[a]);
                }
                __syncwarp();
            }
        }
    } else {
        const int q = warp & 3, half = (warp - kMmaWarp - 1) >> 2;  // TMEM lane quadrant = warp % 4
        uint8_t* const patch_mem = scratch + (kLdWarps * depth + warp - kMmaWarp - 1) * patch::kPatchBytes;
        const patch::Patch pt(patch_mem, lane);
        GateSumEpilogue::Cursor cur;
        if constexpr (kSums) epilogue.start(cur, t_begin * 128 + q * 32 + lane);
        for (uint32_t t = 0; t < t_end - t_begin; ++t) {
            const uint32_t a = t & 1;
            mbar_wait_relaxed(&bar_tfull[a], (t >> 1) & 1);
            fence_after_sync();
            const uint32_t taddr = acc_base + a * 128 + (static_cast<uint32_t>(q * 32) << 16);
            const uint32_t row = (t_begin + t) * 128 + q * 32 + lane;
            auto pull = [&](int c0, float* v, int w) { if (w == 32) tmem_ld32(taddr + c0, v); else tmem_ld16(taddr + c0, v); };
            if constexpr (kSums) {
                epilogue(cur, row < M, pull, lane, 32 * half, 64);
                epilogue.advance(cur, 128);
            } else {
                epilogue(row, M, 0, pull, pt, lane, 32 * half, 64);
            }
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_tempty[a]);
        }
        if constexpr (kSums) epilogue.warp_sums(cur, lane, 32 * half, 64, reinterpret_cast<float*>(patch_mem));
    }
    fence_before_sync();
    __syncthreads();
    if constexpr (kSums) {
        // this CTA's column sums: block c / 32 was handled by the four epilogue warps (one per lane quadrant) with
        // half = block & 1, as entry block >> 1 of their lists; added in warp order
        if (tid < N) {
            const int blk = tid >> 5, half = blk & 1;
            float s = 0.f;
            for (int e = 4 * half; e < 4 * half + 4; ++e)
                s += reinterpret_cast<const float*>(scratch + (kLdWarps * depth + e) * patch::kPatchBytes)[32 * (blk >> 1) + (tid & 31)];
            epilogue.part[static_cast<size_t>(blockIdx.x) * N + tid] = s;
        }
    }
    if (warp == kMmaWarp) {
        fence_after_sync();
        tmem_dealloc(tmem_base, 512);
    }
}
}  // namespace lt

// the tensor-memory form for the streaming shapes: K % 32 == 0, K <= 128, N % 32 == 0, N <= 128, M < 2^31 - 128
template <class Epi>
int launch_ts(int device, int64_t M, int K, int N, const float* X, const float* W, int w_transposed, const Epi& ep,
              int* grid_out, cudaStream_t stream) {
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "linear: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    const size_t wbytes = 2ull * N * K * 4;
    const int depth = 1024 + wbytes + (lt::kLdWarps * 8 + lt::kEpWarps) * patch::kPatchBytes <= static_cast<size_t>(di->smem_optin) ? 8 : 4;
    const size_t smem = 1024 + wbytes + (lt::kLdWarps * depth + lt::kEpWarps) * patch::kPatchBytes;
    LTGNN_REQUIRE(smem <= static_cast<size_t>(di->smem_optin), LTGNN_E_SHAPE, "linear: %zu B of shared memory", smem);
    LTGNN_USE_DEVICE(device);
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(lt::linear_ts_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    const int64_t tiles = (M + 127) / 128;
    const int grid = static_cast<int>(tiles < di->sm_count ? tiles : di->sm_count);
    lt::linear_ts_kernel<Epi><<<grid, lt::kThreads, smem, stream>>>(reinterpret_cast<const float4*>(X), ep, W,
                                                                    w_transposed ? N : K, w_transposed,
                                                                    static_cast<uint32_t>(M), K, N, depth);
    LTGNN_CUDA_TRY(cudaGetLastError());
    if (grid_out) *grid_out = grid;
    return LTGNN_OK;
}

}  // namespace

int ltgnn::functors::linear_gate_sums(int device, int64_t M, int K, const float* G, const float* W,
                                      const GateSumEpilogue& ep, int* parts, cudaStream_t stream) {
    LTGNN_REQUIRE(M > 0 && K % 32 == 0 && K > 0 && K <= 128 && (ep.n == 64 || ep.n == 128) && M < (1ll << 31) - 128,
                  LTGNN_E_SHAPE, "linear_gate_sums: M=%lld K=%d N=%d", static_cast<long long>(M), K, ep.n);
    return launch_ts(device, M, K, ep.n, G, W, 1, ep, parts, stream);
}

extern "C" int ltgnn_linear(int device, int64_t M, int32_t K, int32_t N, const float* X, const float* W,
                            int w_transposed, const float* bias, int relu, const float* gate, float gate_scale, float* Y,
                            void* stream_) {
    LTGNN_REQUIRE(M >= 0 && K > 0 && N > 0, LTGNN_E_ARG, "linear: M=%lld K=%d N=%d", static_cast<long long>(M), K, N);
    if (M == 0) return LTGNN_OK;
    LTGNN_REQUIRE(X && W && Y, LTGNN_E_ARG, "linear: null tensor");
    LTGNN_REQUIRE(aligned16(X) && aligned16(W) && aligned16(Y) && aligned16(gate), LTGNN_E_ALIGN,
                  "linear: 16-byte alignment required");
    StoreEpilogue ep{Y, bias, gate, gate_scale, N, relu};
    if (K % 32 == 0 && K <= 128 && N % 32 == 0 && N <= 128 && M < (1ll << 31) - 128)
        // the streaming shapes of the GCN layers: A operand in tensor memory (see linear_ts_kernel)
        return launch_ts(device, M, K, N, X, W, w_transposed, ep, nullptr, static_cast<cudaStream_t>(stream_));
    RowLoader ld{reinterpret_cast<const float4*>(X), K / 4};
    rowgemm::BSpec bs{W, w_transposed ? N : K, w_transposed, 1};
    return rowgemm::launch(device, ld, ep, bs, M, K, N, static_cast<cudaStream_t>(stream_), "linear");
}
