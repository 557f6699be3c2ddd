// gcn_layer.cu -- ONE kernel for a whole GCN layer forward:  Y = dropout(relu(A_hat (X W^T) + b))
//
// Reference: models/detector.py:198-201 -- `x = conv(x, edge_index); x = F.relu(x); x = self.dropout(x)` with
// conv = torch_geometric GCNConv (lin, propagate, + bias).  The unfused path of this library runs the dense part
// (linear.cu: X W^T written to HBM) and the aggregation (spmm.cu: read back, aggregate, epilogue) as two launches: four
// activation tensors of traffic per layer.  Here the product X W^T never leaves the SM: two tensors.
//
// Work unit = one window; the whole weight (D x K, TF32 hi/lo) is resident in shared memory.  Per window:
//   warps 0-3   LOADERS   stream the window's X rows ONCE (cp.async into a ring of transposition patches, 8 lanes = the
//                         128 bytes of one row), split fp32 -> TF32 hi/lo and tcgen05.st them into A slots in tensor
//                         memory (a slot = 16 K values: what is left of the 512 columns next to the accumulators)
//   warp  4     MMA       tcgen05.mma kind::tf32, 3xTF32, A from tensor memory, N = D: tile t of the window (128 node
//                         rows) accumulates into its own D tensor-memory columns -- the window's whole X W^T (up to
//                         7 x 128 rows x 64) sits in tensor memory when the window's last MMA commits
//   warps 5-16  CONSUMERS per 32-feature slice: drain that slice of the accumulators into a shared-memory stage
//                         [N][32] (XOR-swizzled 16-byte chunks: the row-per-lane writes and the 8-lanes-per-row reads
//                         are both conflict-free), then gather neighbour rows from it exactly like spmm_staged_kernel
//                         (same CSR order, one mul + one add per entry), add the bias, ReLU, Philox dropout, 1-bit live
//                         mask, 128-bit streaming stores.
// The tensor core starts the next window as soon as the last slice is drained, i.e. under that slice's aggregation.
// (A first version gave every CTA one 32-feature slice and let two CTAs read each window: correct, but the window's rows
// then cross every SM's load path twice, and with ~64 KB of loads in flight per SM that, not HBM, set the pace -- 0.58 ms
// per layer, no better than the two launches.)
// Arithmetic is the unfused path's, operation for operation (same MMA sequence per output element, same summation
// order, same dropout counter), so the result is BIT-IDENTICAL to ltgnn_linear + ltgnn_spmm_fused -- which stays as the
// path for shapes this kernel does not take (K > 128, more than 896 nodes, graphs that do not fit shared memory).
#include "patch.cuh"
#include "rowgemm_ts.cuh"

using namespace ltgnn;

namespace {
namespace gl {
using namespace ltgnn::ptx;
using namespace ltgnn::umma;

constexpr int kLdWarps = 4, kMmaWarp = 4, kCons = 24, kThreads = (kLdWarps + 1 + kCons) * 32;  // 29 warps: 64 registers
// (12 consumer warps were tried first: the gather is a chain of dependent shared-memory loads per row, and half the warps
// took twice as long -- 0.55 ms per layer; with 24 the aggregation runs at spmm.cu's pace and the GEMM hides under it)
constexpr int kMaxSlots = 4, kSlotCols = 32, kMaxTiles = 7, kSlice = 32;  // a slot: 16 K values as hi (16 columns) | lo (16)
constexpr int kRowsPerPass = kCons * 4;  // 8 lanes per row, 4 rows per warp; rows r and r + 96 share one Philox call, as in
                                         // spmm.cu: the dropout decisions are the unfused path's bit for bit

struct Params {
    const int32_t* rowptr;
    const int2* colval;
    const float4* X;
    float* Y;
    const float* W;       // [Dout, K] row-major (torch Linear layout)
    const float* bias;    // [Dout] or nullptr
    uint32_t* live_out;   // [B, Dout/32, N] or nullptr
    int64_t B;
    int32_t n, nnz, K, D, n_slices, T, depth, relu, n_slots;
    uint32_t drop_thresh;
    float keep_scale;
    uint64_t drop_seed;
    const uint64_t* seed_src;  // ltgnn_seed_source word or nullptr
    uint32_t off_stage, off_rowptr, off_colval, off_ring;  // byte offsets after the 1024-aligned base (W hi/lo first)
};

__device__ __forceinline__ void fma2(float4& acc, float w, const float4& x) {
    // two roundings per entry, as ATen's mul followed by index_add_ (and as spmm.cu)
    acc.x = __fadd_rn(acc.x, __fmul_rn(w, x.x));
    acc.y = __fadd_rn(acc.y, __fmul_rn(w, x.y));
    acc.z = __fadd_rn(acc.z, __fmul_rn(w, x.z));
    acc.w = __fadd_rn(acc.w, __fmul_rn(w, x.w));
}
__device__ __forceinline__ void cons_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kCons * 32) : "memory"); }

__global__ void __launch_bounds__(kThreads, 1)
gcn_layer_fwd_kernel(const Params p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_full[kMaxSlots], bar_empty[kMaxSlots], bar_acc_full, bar_acc_empty;
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;
    uint8_t* b_lo = b_hi + p.D * p.K * 4;
    float4* stage = reinterpret_cast<float4*>(smem + p.off_stage);
    int32_t* s_rowptr = reinterpret_cast<int32_t*>(smem + p.off_rowptr);
    int2* s_colval = reinterpret_cast<int2*>(smem + p.off_colval);
    uint8_t* rings = smem + p.off_ring;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_kg = p.K >> 5, k4 = p.K >> 2, d4 = p.D >> 2;

    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        for (int s = 0; s < kMaxSlots; ++s) {
            mbar_init(&bar_full[s], 4);
            mbar_init(&bar_empty[s], 1);
        }
        mbar_init(&bar_acc_full, 1);
        mbar_init(&bar_acc_empty, kCons);
        fence_mbar_init();
    }
    rowgemm_ts::fill_b(b_hi, b_lo, p.W, p.K, 0, p.K, p.D, tid, kThreads);
    for (int i = tid; i <= p.n; i += kThreads) s_rowptr[i] = __ldg(p.rowptr + i);
    for (int i = tid; i < p.nnz; i += kThreads) {
        // .x becomes the BYTE offset of chunk 0 of the neighbour's stage row, swizzle term included: chunk q of row c lives
        // at c * 128 + ((q ^ (c & 7)) << 4) = (c * 128 + ((c & 7) << 4)) ^ (q << 4) -- one XOR per entry in the gather loop
        int2 cv = __ldg(p.colval + i);
        cv.x = cv.x * 128 + ((cv.x & 7) << 4);
        s_colval[i] = cv;
    }
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t acc_base = tmem_base, a_base = tmem_base + p.T * p.D;  // T x D accumulator columns, then the A slots
    const uint32_t slot_mask = p.n_slots - 1, slot_log2 = p.n_slots == 4 ? 2u : 1u;  // 2 or 4 A slots in rotation
    const int64_t w_first = blockIdx.x, w_step = gridDim.x;
    const uint32_t n_win = w_first < p.B ? static_cast<uint32_t>((p.B - w_first + w_step - 1) / w_step) : 0;
    const uint32_t per_win = p.T * n_kg;  // patch fills (32 K values each = two A slots) per window

    if (warp < kLdWarps) {
        // ---------------- loaders: as linear.cu's tensor-memory form, rows = the nodes of this CTA's windows ----------------
        const int quad = warp & 3, depth = p.depth;
        uint8_t* ring = rings + static_cast<size_t>(warp) * depth * patch::kPatchBytes;
        const uint32_t lane_base = a_base + (static_cast<uint32_t>(quad * 32) << 16);
        const int sub = lane >> 3, ch = lane & 7;
        const uint32_t n_fills = n_win * per_win;
        auto fetch = [&](uint32_t f, int slot_p) {
            const patch::Patch pt(ring + slot_p * patch::kPatchBytes, lane);
            if (f < n_fills) {
                const uint32_t wi = f / per_win, rem = f - wi * per_win, tile = rem / n_kg, kg = rem - tile * n_kg;
                const float4* xb = p.X + (w_first + static_cast<int64_t>(wi) * w_step) * p.n * k4;
                const uint32_t row0 = tile * 128 + quad * 32 + sub;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint32_t row = row0 + 4 * k;
                    const bool ok = row < static_cast<uint32_t>(p.n);  // rows past N are zero-filled (src-size 0)
                    const float4* src = xb + static_cast<size_t>(ok ? row : 0) * k4 + kg * 8 + ch;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(pt.co(k))), "l"(src),
                                 "r"(ok ? 16 : 0)
                                 : "memory");
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");  // (an empty group keeps the wait count uniform)
        };
        for (int d = 0; d < depth; ++d) fetch(d, d);
        uint32_t sf = 0;  // running A-slot fill
        for (uint32_t f = 0; f < n_fills; ++f) {
            const int slot_p = static_cast<int>(f % depth);
            if (depth == 4) asm volatile("cp.async.wait_group 3;" ::: "memory");
            else asm volatile("cp.async.wait_group 1;" ::: "memory");
            __syncwarp();
            const patch::Patch pt(ring + slot_p * patch::kPatchBytes, lane);
#pragma unroll
            for (int h = 0; h < 2; ++h, ++sf) {  // the patch's 32 K values go out as two 16-value slots
                float v[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 t = *pt.row(4 * h + j);
                    v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
                }
                if (h == 1) {
                    __syncwarp();
                    fetch(f + depth, slot_p);  // the patch has been read: refill it
                }
                const uint32_t slot = sf & slot_mask;
                mbar_wait_relaxed(&bar_empty[slot], ((sf >> slot_log2) & 1) ^ 1);
                fence_after_sync();
                const uint32_t st_addr = lane_base + slot * kSlotCols;
#pragma unroll
                for (int c = 0; c < 16; c += 8) {
                    float hi[8], lo[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        hi[j] = tf32_hi(v[c + j]);
                        lo[j] = v[c + j] - hi[j];
                    }
                    tmem_st8(st_addr + c, hi);
                    tmem_st8(st_addr + 16 + c, lo);
                }
                rowgemm_ts::tmem_wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_full[slot]);
            }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if (warp == kMmaWarp) {
        // ---------------- MMA: tile t of a window -> accumulator columns [D t, D t + D) ----------------
        const uint32_t idesc = idesc_tf32(128, p.D);
        const uint32_t bh = desc_lo(smem_u32(b_hi)), bl = desc_lo(smem_u32(b_lo));
        const uint32_t kg_units = static_cast<uint32_t>(p.D) * 128u >> 4;
        uint32_t sf = 0;
        for (uint32_t wi = 0; wi < n_win; ++wi) {
            mbar_wait_relaxed(&bar_acc_empty, (wi & 1) ^ 1);  // the consumers drained the previous window
            fence_after_sync();
            for (int t = 0; t < p.T; ++t) {
                const uint32_t d = acc_base + t * p.D;
                if (p.n_slots == 4) {
                    // the two slots of one patch (32 K values) per hand-over: 12 MMAs back to back.  The tensor pipe only
                    // runs while this warp is issuing, and a wait + fence + election + commit round costs several times
                    // the 192 clocks of one slot's six MMAs -- taken slot by slot, the window's GEMM (24 slots) was longer
                    // than the aggregation of a slice it is meant to hide under
                    for (int kh = 0; kh < 2 * n_kg; kh += 2, sf += 2) {
                        const uint32_t slot = sf & 3, par = (sf >> 2) & 1;   // sf is even: slots (0, 1) or (2, 3), one parity
                        mbar_wait_relaxed(&bar_full[slot], par);
                        mbar_wait_relaxed(&bar_full[slot + 1], par);
                        fence_after_sync();
                        if (elect_one()) {
#pragma unroll
                            for (uint32_t h = 0; h < 2; ++h) {
                                const uint32_t a_hi = a_base + (slot + h) * kSlotCols, a_lo = a_hi + 16;
                                const uint32_t bbase = static_cast<uint32_t>(kh >> 1) * kg_units + 4 * h;
#pragma unroll
                                for (uint32_t k = 0; k < 2; ++k) {
                                    const uint32_t boff = bbase + 2 * k;
                                    rowgemm_ts::mma_tf32_ts(d, a_lo + 8 * k, bh + boff, idesc, (kh == 0 && h == 0 && k == 0) ? 0u : 1u);
                                    rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bl + boff, idesc, 1u);
                                    rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bh + boff, idesc, 1u);
                                }
                                commit(&bar_empty[slot + h]);
                            }
                            if (t == p.T - 1 && kh == 2 * n_kg - 2) commit(&bar_acc_full);
                        }
                        __syncwarp();
                    }
                    continue;
                }
                for (int kh = 0; kh < 2 * n_kg; ++kh, ++sf) {  // 16 K values per slot
                    const uint32_t slot = sf & slot_mask;
                    mbar_wait_relaxed(&bar_full[slot], (sf >> slot_log2) & 1);
                    fence_after_sync();
                    if (elect_one()) {
                        const uint32_t a_hi = a_base + slot * kSlotCols, a_lo = a_hi + 16;
                        const uint32_t bbase = static_cast<uint32_t>(kh >> 1) * kg_units + 4 * (kh & 1);
#pragma unroll
                        for (uint32_t k = 0; k < 2; ++k) {
                            const uint32_t boff = bbase + 2 * k;
                            rowgemm_ts::mma_tf32_ts(d, a_lo + 8 * k, bh + boff, idesc, (kh == 0 && k == 0) ? 0u : 1u);
                            rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bl + boff, idesc, 1u);
                            rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bh + boff, idesc, 1u);
                        }
                        commit(&bar_empty[slot]);
                        if (t == p.T - 1 && kh == 2 * n_kg - 1) commit(&bar_acc_full);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        // ---------------- consumers ----------------
        const int cw = warp - kMmaWarp - 1;          // 0 .. 23
        const int q4 = warp & 3, dj = cw >> 2;       // tensor-memory lane quadrant = warp % 4; this warp drains tiles dj, dj + 6
        const int g = lane >> 3, q = lane & 7;       // aggregation: row within the warp's group of 4, float4 of the slice
        const uint8_t* stage_b = reinterpret_cast<const uint8_t*>(stage);
        const int qx = q << 4;
        const uint64_t seed = launch_seed(p.drop_seed, p.seed_src);
        for (uint32_t wi = 0; wi < n_win; ++wi) {
            const int64_t b = w_first + static_cast<int64_t>(wi) * w_step;
            mbar_wait_relaxed(&bar_acc_full, wi & 1);   // 24 warps polling would take issue slots from the four loader warps
            fence_after_sync();
          for (int sl = 0; sl < p.n_slices; ++sl) {
            for (int t = dj; t < p.T; t += kCons / 4) {
                float v[32];
                tmem_ld32(acc_base + t * p.D + sl * kSlice + (static_cast<uint32_t>(q4 * 32) << 16), v);
                const int r = t * 128 + q4 * 32 + lane;
                if (r < p.n) {
#pragma unroll
                    for (int c = 0; c < 8; ++c)  // chunk c of row r lives at chunk c ^ (r & 7)
                        stage[r * 8 + (c ^ (r & 7))] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                }
            }
            if (sl == p.n_slices - 1) {  // accumulators free: the tensor core starts the next window
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_acc_empty);
            }
            cons_bar();                                  // the whole stage is written
            float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bias) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias) + sl * (kSlice / 4) + q);

            const int64_t u = b * p.n_slices + sl;       // unit index as in spmm.cu (dropout counter, live-mask row)
            const int64_t base4 = (b * p.n) * d4 + sl * (kSlice / 4) + q;
            float4* y = reinterpret_cast<float4*>(p.Y) + base4;
            for (int rb = cw * 4; rb < p.n; rb += 2 * kRowsPerPass) {
                const int r0 = rb + g, r1 = r0 + kRowsPerPass;
                int k0 = 0, e0 = 0, k1 = 0, e1 = 0;
                if (r0 < p.n) {
                    k0 = s_rowptr[r0];
                    e0 = s_rowptr[r0 + 1];
                }
                if (r1 < p.n) {
                    k1 = s_rowptr[r1];
                    e1 = s_rowptr[r1 + 1];
                }
                float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f);
                float4 a1 = a0;
                while (k0 < e0 && k1 < e1) {
                    const int2 c0 = s_colval[k0++];
                    const int2 c1 = s_colval[k1++];
                    const float4 x0 = *reinterpret_cast<const float4*>(stage_b + (c0.x ^ qx));
                    const float4 x1 = *reinterpret_cast<const float4*>(stage_b + (c1.x ^ qx));
                    fma2(a0, __int_as_float(c0.y), x0);
                    fma2(a1, __int_as_float(c1.y), x1);
                }
                for (; k0 < e0; ++k0) {
                    const int2 c0 = s_colval[k0];
                    fma2(a0, __int_as_float(c0.y), *reinterpret_cast<const float4*>(stage_b + (c0.x ^ qx)));
                }
                for (; k1 < e1; ++k1) {
                    const int2 c1 = s_colval[k1];
                    fma2(a1, __int_as_float(c1.y), *reinterpret_cast<const float4*>(stage_b + (c1.x ^ qx)));
                }
                if (p.bias) {
                    a0.x = __fadd_rn(a0.x, bias4.x); a0.y = __fadd_rn(a0.y, bias4.y);
                    a0.z = __fadd_rn(a0.z, bias4.z); a0.w = __fadd_rn(a0.w, bias4.w);
                    a1.x = __fadd_rn(a1.x, bias4.x); a1.y = __fadd_rn(a1.y, bias4.y);
                    a1.z = __fadd_rn(a1.z, bias4.z); a1.w = __fadd_rn(a1.w, bias4.w);
                }
                if (p.relu) {
                    a0.x = fmaxf(a0.x, 0.f); a0.y = fmaxf(a0.y, 0.f); a0.z = fmaxf(a0.z, 0.f); a0.w = fmaxf(a0.w, 0.f);
                    a1.x = fmaxf(a1.x, 0.f); a1.y = fmaxf(a1.y, 0.f); a1.z = fmaxf(a1.z, 0.f); a1.w = fmaxf(a1.w, 0.f);
                }
                if (p.drop_thresh) {  // one Philox call (16 random bits per element) decides both float4, as in spmm.cu
                    float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                    dropout8(v, static_cast<uint64_t>(base4 + static_cast<int64_t>(r0) * d4), seed, p.drop_thresh,
                             p.keep_scale);
                    a0 = make_float4(v[0], v[1], v[2], v[3]);
                    a1 = make_float4(v[4], v[5], v[6], v[7]);
                }
                if (r0 < p.n) stg_stream(y + static_cast<int64_t>(r0) * d4, a0);
                if (r1 < p.n) stg_stream(y + static_cast<int64_t>(r1) * d4, a1);
                if (p.live_out) {  // bit 8 c + q of the row's word <-> element 4 q + c of the 32-feature slice
                    const uint32_t sel = static_cast<uint32_t>(g) | (static_cast<uint32_t>(4 + g) << 4);
                    const uint32_t x0 = __ballot_sync(0xffffffffu, a0.x > 0.f), y0 = __ballot_sync(0xffffffffu, a0.y > 0.f);
                    const uint32_t z0 = __ballot_sync(0xffffffffu, a0.z > 0.f), w0 = __ballot_sync(0xffffffffu, a0.w > 0.f);
                    const uint32_t x1 = __ballot_sync(0xffffffffu, a1.x > 0.f), y1 = __ballot_sync(0xffffffffu, a1.y > 0.f);
                    const uint32_t z1 = __ballot_sync(0xffffffffu, a1.z > 0.f), w1 = __ballot_sync(0xffffffffu, a1.w > 0.f);
                    if (q == 0) {
                        uint32_t* lw = p.live_out + static_cast<size_t>(u) * p.n;
                        if (r0 < p.n) lw[r0] = __byte_perm(__byte_perm(x0, y0, sel), __byte_perm(z0, w0, sel), 0x5410);
                        if (r1 < p.n) lw[r1] = __byte_perm(__byte_perm(x1, y1, sel), __byte_perm(z1, w1, sel), 0x5410);
                    }
                }
            }
            cons_bar();  // every consumer is done with the stage: the next drain may overwrite it
          }
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == kMmaWarp) {
        fence_after_sync();
        tmem_dealloc(tmem_base, 512);
    }
}

inline uint32_t align_up(uint32_t x, uint32_t a) { return (x + a - 1) / a * a; }

// Shared memory a launch may ask for: the opt-in limit bounds dynamic + static bytes, and the kernel's barriers are
// static.  0 if the kernel's attributes cannot be read.
inline uint32_t dynamic_smem_limit(int smem_optin) {
    static const int static_bytes = [] {
        cudaFuncAttributes a{};
        if (cudaFuncGetAttributes(&a, gcn_layer_fwd_kernel) != cudaSuccess) {
            (void)cudaGetLastError();
            return -1;
        }
        return static_cast<int>(a.sharedSizeBytes);
    }();
    return static_bytes < 0 || static_bytes >= smem_optin ? 0u : static_cast<uint32_t>(smem_optin - static_bytes);
}

}  // namespace gl
}  // namespace

// 1 if ltgnn_gcn_layer_fwd takes this (graph, K = Din, D = Dout), else 0 (callers then run ltgnn_linear + ltgnn_spmm_fused)
extern "C" int ltgnn_gcn_layer_supported(ltgnn_graph_t g, int32_t K, int32_t D) {
    if (!g || K % 32 || K <= 0 || K > 128 || D % 32 || D <= 0 || D > 256) return 0;
    const int T = (g->n + 127) / 128;
    if (T > gl::kMaxTiles || T * D + 2 * gl::kSlotCols > 512) return 0;  // accumulators + at least two A slots
    const uint32_t fixed = gl::align_up(2u * D * K * 4 + gl::align_up(static_cast<uint32_t>(g->n) * 128, 128) +
                                            gl::align_up(4u * (g->n + 1), 16) + 8u * g->nnz, 1024);
    return 1024 + fixed + gl::kLdWarps * 2 * patch::kPatchBytes <= gl::dynamic_smem_limit(g->smem_optin);
}

extern "C" int ltgnn_gcn_layer_fwd(ltgnn_graph_t g, int64_t B, int32_t K, int32_t D, const float* X, const float* W,
                                   const float* bias, int relu, float drop_p, uint64_t drop_seed, float* Y,
                                   uint32_t* live_out, void* stream_) {
    LTGNN_REQUIRE(g != nullptr, LTGNN_E_ARG, "gcn_layer_fwd: null graph handle");
    LTGNN_REQUIRE(B >= 0 && B < (1ll << 31), LTGNN_E_ARG, "gcn_layer_fwd: B=%lld", static_cast<long long>(B));
    LTGNN_REQUIRE(ltgnn_gcn_layer_supported(g, K, D), LTGNN_E_SHAPE,
                  "gcn_layer_fwd: shape not taken by the fused kernel (K=%d, D=%d, %d nodes); use linear + spmm_fused", K, D, g->n);
    LTGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, LTGNN_E_ARG, "gcn_layer_fwd: dropout p=%f not in [0,1)", drop_p);
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(X && W && Y, LTGNN_E_ARG, "gcn_layer_fwd: null tensor");
    LTGNN_REQUIRE(X != Y, LTGNN_E_ARG, "gcn_layer_fwd: X and Y must not alias");
    LTGNN_REQUIRE(aligned16(X) && aligned16(W) && aligned16(Y) && aligned16(bias), LTGNN_E_ALIGN,
                  "gcn_layer_fwd: tensors must be 16-byte aligned");
    LTGNN_REQUIRE(B * g->n < (1ll << 31), LTGNN_E_SHAPE, "gcn_layer_fwd: B*N too large");
    LTGNN_USE_DEVICE(g->device);
    gl::Params p;
    p.rowptr = g->rowptr[0];
    p.colval = g->colval[0];
    p.X = reinterpret_cast<const float4*>(X);
    p.Y = Y;
    p.W = W;
    p.bias = bias;
    p.live_out = live_out;
    p.B = B;
    p.n = g->n;
    p.nnz = g->nnz;
    p.K = K;
    p.D = D;
    p.n_slices = D / gl::kSlice;
    p.T = (g->n + 127) / 128;
    p.relu = relu;
    p.drop_thresh = drop_p > 0.f ? static_cast<uint32_t>(static_cast<double>(drop_p) * 65536.0 + 0.5) : 0u;
    p.keep_scale = 1.f / (1.f - static_cast<float>(p.drop_thresh) / 65536.f);
    p.drop_seed = drop_seed;
    p.seed_src = seed_source();
    p.n_slots = (512 - p.T * D) / gl::kSlotCols >= gl::kMaxSlots ? gl::kMaxSlots : 2;  // a power of two
    p.off_stage = 2u * D * K * 4;
    p.off_rowptr = p.off_stage + gl::align_up(static_cast<uint32_t>(g->n) * 128, 128);
    p.off_colval = p.off_rowptr + gl::align_up(4u * (g->n + 1), 16);
    p.off_ring = gl::align_up(p.off_colval + 8u * g->nnz, 1024);  // patches address chunks by XOR: keep them aligned
    const uint32_t room = gl::dynamic_smem_limit(g->smem_optin) - 1024 - p.off_ring;
    p.depth = room >= gl::kLdWarps * 4 * patch::kPatchBytes ? 4 : 2;  // 64 KB (or 32 KB) of loads in flight
    const size_t smem = 1024 + p.off_ring + static_cast<size_t>(gl::kLdWarps) * p.depth * patch::kPatchBytes;
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(gl::gcn_layer_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    const int64_t grid = B < g->sm_count ? B : g->sm_count;
    gl::gcn_layer_fwd_kernel<<<static_cast<int>(grid), gl::kThreads, smem, static_cast<cudaStream_t>(stream_)>>>(p);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}
