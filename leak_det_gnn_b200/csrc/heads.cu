// heads.cu -- the two read-out heads of the detector on top of the last GCN layer.
//
//   pipe head  (models/detector.py:76-88, 204-211): for every class pipe p = (u, v)
//              feat = [h_u, h_v, |h_u - h_v|] -> Linear(3D, H) -> ReLU -> Dropout -> Linear(H, 1)
//              The reference gathers h_u / h_v into (B, P, D) tensors, concatenates a (B, P, 3D) feature
//              tensor (2.4 GB at B = 4096, P = 764) and runs cuBLAS on it.  Here the features are formed
//              on the fly by the loader warps straight from the node states; the hidden layer never leaves
//              the SM in the forward except as the saved post-activation the backward needs.
//   mean pool  (models/detector.py:214-215, PyG global_mean_pool over equal-sized graphs).
//
// Both head GEMMs keep the A operand in tensor memory (building blocks: rowgemm_ts.cuh): a thread owns one pipe
// row (= TMEM lane), splits it into TF32 hi/lo in registers and tcgen05.st's it, so shared memory only holds the
// whole weight W1 (192 KB as hi + lo) and every tile is produced exactly once.  Global memory is always touched
// in 128-byte row segments; the switch to / from the row-per-thread form goes through patch.cuh.
#include "patch.cuh"
#include "rowgemm_ts.cuh"

using namespace ltgnn;

namespace {

// ------------------------------------------------------------------ forward
constexpr int kD = 64;        // node width supported by the fused head
constexpr int kD4 = kD / 4;

// hidden = dropout(relu(acc + b1)) for hidden units [c_begin, c_end) of one pipe row; returns their share of
// the logit, sum of hidden * w2.  The inverted-dropout scale 1 / (1 - p) is folded into W1 and b1 by the kernel
// (relu commutes with a positive scale), so a kept unit costs add, max, compare, select, fma.
struct HeadFwdEpilogue {
    const float* b1;   // [H]
    const float* w2;   // [H]
    float* part;       // [M]
    float* hpost;      // blocked-32 [Mp, H] saved post-activation, or nullptr (inference)
    uint32_t* hmask;   // [Mp, H/32] 1 bit per hidden unit: hidden > 0 (ReLU-and-dropout gate of the backward), or nullptr;
                       // hidden unit j is bit 31 - j % 32 of word j / 32
    int H;
    uint32_t drop_thresh16;  // round(p * 2^16), 0 = no dropout
    float keep_scale;        // 1 / (1 - drop_thresh16 / 2^16)
    uint64_t drop_seed;
    const uint64_t* seed_src;  // ltgnn_seed_source word or nullptr
    template <class Pull>
    __device__ __forceinline__ float operator()(uint32_t row, int c_begin, int c_end, Pull&& pull) const {
        float acc = 0.f;
        const uint32_t thresh_hi = drop_thresh16 << 16;
        uint32_t bits = 0;
        for (int col = c_begin; col < c_end; col += 16) {
            float4 bb[4], ww[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {  // issued before the tcgen05.ld wait
                bb[j] = __ldg(reinterpret_cast<const float4*>(b1 + col) + j);
                ww[j] = __ldg(reinterpret_cast<const float4*>(w2 + col) + j);
            }
            float v[16];
            pull(col, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                v[4 * j + 0] = fmaxf(fmaf(bb[j].x, keep_scale, v[4 * j + 0]), 0.f);
                v[4 * j + 1] = fmaxf(fmaf(bb[j].y, keep_scale, v[4 * j + 1]), 0.f);
                v[4 * j + 2] = fmaxf(fmaf(bb[j].z, keep_scale, v[4 * j + 2]), 0.f);
                v[4 * j + 3] = fmaxf(fmaf(bb[j].w, keep_scale, v[4 * j + 3]), 0.f);
            }
            if (drop_thresh16) {
                const uint64_t i8 = static_cast<uint64_t>(row) * (H >> 3) + (col >> 3);
                const uint64_t seed = ptx::launch_seed(drop_seed, seed_src);
                ptx::dropout8_mask(v, i8, seed, thresh_hi);
                ptx::dropout8_mask(v + 8, i8 + 1, seed, thresh_hi);
            }
            if (hmask) {
                // v >= +0 here, so v > 0 <=> its bit pattern u != 0 <=> the top bit of -u is set; one funnel shift moves
                // that bit into the word: hidden unit j of a 32-unit group ends up at bit 31 - j
#pragma unroll
                for (int j = 0; j < 16; ++j) bits = __funnelshift_l(0u - __float_as_uint(v[j]), bits, 1);
                if ((col & 16) != 0) {  // a 32-unit word is complete
                    hmask[static_cast<size_t>(row) * (H >> 5) + (col >> 5)] = bits;
                    bits = 0;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (hpost)  // blocked-32 layout (rows padded to 128 by the caller): coalesced across the warp's rows
                    ptx::stg_stream(reinterpret_cast<float4*>(hpost) + ptx::b32(row, (col >> 2) + j, H >> 2),
                                    make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
                acc = fmaf(v[4 * j + 0], ww[j].x, acc);
                acc = fmaf(v[4 * j + 1], ww[j].y, acc);
                acc = fmaf(v[4 * j + 2], ww[j].z, acc);
                acc = fmaf(v[4 * j + 3], ww[j].w, acc);
            }
        }
        return acc;
    }
};

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "f"(v[0]), "f"(v[1]),
                 "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

// ------------------------------------------------------------------ forward kernel
// The generic tensor-memory skeleton (rowgemm_ts.cuh) lets every loader thread fetch its own row, which for
// gathered node states means 32 different 128-byte lines per load instruction: ncu showed the L1 data pipe
// (l1tex lsu wavefronts) at 70 % of peak and the tensor pipe at 29 %.  Here a warp fetches the rows
// cooperatively -- 8 lanes read the 128 B of one row, 4 rows per instruction, every line used in full -- and
// turns them into the row-per-thread form tcgen05.st needs through a 4 KB XOR-swizzled shared-memory patch
// (conflict-free both ways).  Each end-node row is fetched once per tile and reused for the |h_u - h_v| block.
//
//   warps 0-7   LOADERS   group g = warp / 4 owns feature columns [32 g, 32 g + 32) of every tile and emits
//                         three A stages: h_u, h_v, |h_u - h_v|  (K blocks 2 seg + g of W1)
//   warp  8     MMA       elected lane, 3xTF32, A from tensor memory, W1 resident in shared memory (192 KB)
//   warps 9-16  EPILOGUE  tcgen05.ld + bias / ReLU / dropout / w2 dot, double-buffered accumulators; two warps
//                         per TMEM lane quadrant, 64 hidden units each (the Philox chains are latency-bound)
namespace hf {
using namespace ltgnn::ptx;
using namespace ltgnn::umma;
constexpr int kLdWarps = 8, kMmaWarp = 8, kEpWarps = 8, kThreads = (kLdWarps + 1 + kEpWarps) * 32;
constexpr int kK = 192, kN = 128, kStages = 4, kStageCols = 64;
constexpr uint32_t kScrBytes = 4096;

__global__ void __launch_bounds__(kThreads, 1)
pipe_head_fwd_kernel(const float4* __restrict__ x, const int2* __restrict__ ends, uint32_t P, uint32_t N, uint64_t magic,
                     const HeadFwdEpilogue epilogue, const float* __restrict__ W1, uint32_t M, uint2* __restrict__ hsign) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_full[kStages], bar_empty[kStages], bar_tfull[2], bar_tempty[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ float part_s[2][128];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;
    uint8_t* b_lo = b_hi + kN * kK * 4;
    uint8_t* scratch = b_lo + kN * kK * 4;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&bar_full[s], 4);
            mbar_init(&bar_empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bar_tfull[a], 1);
            mbar_init(&bar_tempty[a], kEpWarps);
        }
        fence_mbar_init();
    }
    rowgemm_ts::fill_b(b_hi, b_lo, W1, kK, 0, kK, kN, tid, kThreads, epilogue.keep_scale);
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t acc_base = tmem_base, a_base = tmem_base + 2 * kN;
    const uint32_t n_tiles = (M + 127) / 128;
    // each CTA owns a contiguous range of tiles: consecutive tiles share a window, so its node states are fetched
    // from HBM once and the CTA's reads / writes / reductions stay local
    const uint32_t per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;
    const uint32_t t_begin = min(blockIdx.x * per_cta, n_tiles), t_end = min(t_begin + per_cta, n_tiles);

    if (warp < kLdWarps) {
        const int grp = warp >> 2, quad = warp & 3;
        const patch::Patch patch(scratch + warp * kScrBytes, lane);
        const uint32_t lane_base = a_base + (static_cast<uint32_t>(quad * 32) << 16);
        const int sub = lane >> 3, ch = lane & 7;
        uint32_t t = 0;
        for (uint32_t tile = t_begin; tile < t_end; ++tile, ++t) {
            const uint32_t row = tile * 128 + quad * 32 + lane;
            uint32_t iu = 0, iv = 0;  // node rows of the two ends (pad rows read node row 0; their results are unused)
            if (row < M) {
                const uint32_t b = magic ? fastdiv(row, magic) : row;
                const int2 e = __ldg(ends + (row - b * P));
                iu = b * N + e.x;
                iv = b * N + e.y;
            }
            float4 gu[8], gv[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t ru = __shfl_sync(0xffffffffu, iu, 4 * k + sub), rv = __shfl_sync(0xffffffffu, iv, 4 * k + sub);
                gu[k] = __ldg(x + static_cast<size_t>(ru) * kD4 + grp * 8 + ch);
                gv[k] = __ldg(x + static_cast<size_t>(rv) * kD4 + grp * 8 + ch);
            }
            // emit one A stage: split 32 values into TF32 hi / lo and store them to this thread's TMEM lane
            auto emit = [&](int seg, auto&& value) {
                const uint32_t stage = 6 * t + 3 * grp + seg, slot = stage & 3;
                mbar_wait_relaxed(&bar_empty[slot], ((stage >> 2) & 1) ^ 1);  // slot consumed by the tensor core
                fence_after_sync();
                const uint32_t st_addr = lane_base + slot * kStageCols;
#pragma unroll
                for (int c = 0; c < 32; c += 8) {
                    float hi[8], lo[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float a = value(c + j);
                        hi[j] = tf32_hi(a);
                        lo[j] = a - hi[j];
                    }
                    tmem_st8(st_addr + c, hi);
                    tmem_st8(st_addr + 32 + c, lo);
                }
                rowgemm_ts::tmem_wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_full[slot]);
            };
            float u[32], v[32];
            patch::transpose_in(patch, gu, u);
            emit(0, [&](int j) { return u[j]; });   // h_v still in flight
            patch::transpose_in(patch, gv, v);
            emit(1, [&](int j) { return v[j]; });
            if (hsign && row < M) {
                // sign(h_u - h_v) of this row's 32 features for the backward (d|x| = sign(x), 0 at 0): two words, feature
                // j at bit 31 - j.  d < 0 <=> the top bit of its pattern; d > 0 <=> the top bit of minus its pattern
                // taken as an integer (h >= +0, so d is never -0).  One funnel shift each.
                uint32_t pos = 0, neg = 0;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const uint32_t bits = __float_as_uint(u[j] - v[j]);
                    neg = __funnelshift_l(bits, neg, 1);
                    pos = __funnelshift_l(0u - bits, pos, 1);
                }
                hsign[static_cast<size_t>(row) * 2 + grp] = make_uint2(pos, neg);
            }
            emit(2, [&](int j) { return fabsf(u[j] - v[j]); });
        }
    } else if (warp == kMmaWarp) {
        const uint32_t idesc = idesc_tf32(128, kN);
        const uint32_t bh = desc_lo(smem_u32(b_hi)), bl = desc_lo(smem_u32(b_lo));
        constexpr uint32_t kg_units = static_cast<uint32_t>(kN) * 128u >> 4;
        uint32_t t = 0;
        for (uint32_t tile = t_begin; tile < t_end; ++tile, ++t) {
            const uint32_t a = t & 1;
            mbar_wait_relaxed(&bar_tempty[a], ((t >> 1) & 1) ^ 1);
            const uint32_t d = acc_base + a * kN;
            // two stages (24 MMAs) per hand-over: the tensor pipe only runs while this warp is issuing (its queue is
            // shallow), so waits, fence, election and commits are paid once per pair.  6 t + s is even: the pair sits in
            // slots (0, 1) or (2, 3) and shares the ring parity.
#pragma unroll 1
            for (uint32_t s = 0; s < 6; s += 2) {
                const uint32_t stage = 6 * t + s, slot = stage & 3, par = (stage >> 2) & 1;
                mbar_wait_relaxed(&bar_full[slot], par);
                mbar_wait_relaxed(&bar_full[slot + 1], par);
                fence_after_sync();
                if (elect_one()) {
#pragma unroll
                    for (uint32_t h = 0; h < 2; ++h) {
                        const uint32_t sh = s + h;
                        const uint32_t kg = sh < 3 ? 2 * sh : 2 * (sh - 3) + 1;  // K block of W1 this stage multiplies
                        const uint32_t a_hi = a_base + (slot + h) * kStageCols, a_lo = a_hi + 32;
#pragma unroll
                        for (uint32_t k = 0; k < 4; ++k) {
                            const uint32_t boff = kg * kg_units + 2 * k;
                            rowgemm_ts::mma_tf32_ts(d, a_lo + 8 * k, bh + boff, idesc, (sh == 0 && k == 0) ? 0u : 1u);
                            rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bl + boff, idesc, 1u);
                            rowgemm_ts::mma_tf32_ts(d, a_hi + 8 * k, bh + boff, idesc, 1u);
                        }
                        commit(&bar_empty[slot + h]);
                    }
                    if (s == 4) commit(&bar_tfull[a]);
                }
                __syncwarp();
            }
        }
    } else {
        const int q = warp & 3, half = (warp - kMmaWarp - 1) >> 2;  // TMEM lane quadrant = warp % 4
        uint32_t t = 0;
        for (uint32_t tile = t_begin; tile < t_end; ++tile, ++t) {
            const uint32_t a = t & 1;
            mbar_wait_relaxed(&bar_tfull[a], (t >> 1) & 1);
            fence_after_sync();
            const uint32_t taddr = acc_base + a * kN + (static_cast<uint32_t>(q * 32) << 16);
            const uint32_t row = tile * 128 + q * 32 + lane;
            const float acc = epilogue(row, half * (kN / 2), (half + 1) * (kN / 2),
                                       [&](int c0, float (&v)[16]) { tmem_ld16(taddr + c0, v); });
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_tempty[a]);
            // the two warps of a quadrant add their halves of the logit in a fixed order
            if (half == 1) part_s[a][q * 32 + lane] = acc;
            asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
            if (half == 0 && row < M) epilogue.part[row] = acc + part_s[a][q * 32 + lane];
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == kMmaWarp) {
        fence_after_sync();
        tmem_dealloc(tmem_base, 512);
    }
}
}  // namespace hf

// ------------------------------------------------------------------ backward (input gradient)
// d loss / d pre[row, j] = g[row] * w2[j] * live[row, j] with g = dlogit * scale is rank one up to the 0 / 1 gate, so
//      dfeat[row, c] = g[row] * sum_j live[row, j] * (w2[j] * W1[j, c]):
// the A operand is the gate itself (exact in TF32: no lo copy, two MMAs per K step instead of three), the resident B
// operand is W1 with its rows scaled by w2, and g multiplies the accumulator row in the epilogue.
struct DpreLoader {
    const uint4* hmask;    // [Mp] rows of 128 bits: hidden unit j of a row is live <=> bit 31 - j % 32 of word j / 32
    const float* dlogit;   // [M]
    const float* w2;       // [H]
    float scale;
};

// dfeat goes back to the two end nodes: +u for the h_u block, +v for the h_v block, +-sign(h_u - h_v) for the |.| block
// (torch: d|x| = sign(x), 0 at 0; the signs come as 2 bits per feature from the forward, `hsign` -- re-reading the node
// states for them cost a third of this kernel).  Several pipes share a node, and the reference adds them with index_add_
// (atomics on a GPU).  Here the sum is a GATHER in a fixed order, so the gradient is bit-reproducible: a CTA works through
// whole windows; the epilogue warps park the per-pipe-end rows of the window in a CTA-private scratch (reused window
// after window: it lives in L2) at the position the end has in the node-sorted incidence list, so the ends of a node are
// contiguous.  When the window is complete the scratch comes back through 1-D bulk copies (TMA) in chunks of whole nodes
// and every node adds its rows in list order:
//     dx[b, i, :] = dpooled[b, :] / N + sum over the pipe ends at node i,        written exactly once
// (the mean-pool gradient rides along: no separate fill pass, no read-modify-write of dx).
//
// The gather must not sit on the epilogue warps' critical path: done by them at the end of every window it cost as much
// as the GEMM (45 000 clocks per window as a per-thread gather from L2; still 20 000 with bulk copies, the loop around
// them and the refill of the drained MMA pipeline), and done by the loader warps in between their tiles it held up the A
// operand.  So the scratch is double-buffered by window parity and four GATHER warps work on window w - 1 while the tiles
// of window w are in flight (chunks are warp-private: no barrier inside the gather).  The staging buffers do not fit next
// to a resident [192 x 128] hi + lo weight, so a CTA owns one HALF of the 64 node features (32 columns of each of the
// three blocks: B is [96 x 128], 96 KB) and two CTAs share a window range.
//
//   warps 0-3   LOADERS   thread = pipe row = TMEM lane: gate bits -> 0 / 1 floats -> tcgen05.st, four K blocks per tile
//                         into a ring two tiles deep
//   warp  4     MMA       elected lane, A from tensor memory, B resident
//   warps 5-8   EPILOGUE  one per TMEM lane quadrant, thread = pipe row: g * (u + s c) and g * (v - s c) of its 32
//                         features (the row's own 64 sign bits come with one load, the shifts are constants), written as
//                         two 128-byte rows into a shared-memory staging area (row pitch 144 B: row-per-thread stores and
//                         8-lanes-per-row loads are both conflict-free), read back as coalesced row segments and stored
//                         to their node-sorted scratch positions, 4 full lines per instruction.  (The first version
//                         transposed the three accumulator blocks separately and applied the signs afterwards: 850
//                         instructions per tile and warp, and the four epilogue warps were the kernel's pace.  One
//                         128-byte bulk store per row instead of the read-back was slower still: 1.21 ms.)
//   warps 9-15  GATHER    bulk copies scratch -> shared memory, node sums, dx   (16 warps: still 128 registers each)
namespace hb {
using namespace ltgnn::ptx;
using namespace ltgnn::umma;
constexpr int kLdWarps = 4, kMmaWarp = 4, kEpWarps = 4, kGaWarps = 7;
constexpr int kThreads = (kLdWarps + 1 + kEpWarps + kGaWarps) * 32;  // 16 warps: 128 registers
constexpr int kK = 128, kHalf = 32, kN = 3 * kHalf, kStages = 8, kStageCols = 32;  // A ring: two tiles deep
constexpr uint32_t kRowPitch = 144;                          // staging row: 128 B + 16 (bank spread)
constexpr uint32_t kScrBytes = 2 * 32 * kRowPitch;           // per epilogue warp: the u rows, then the v rows
constexpr uint32_t kRowBytes = kHalf * 4;                    // one pipe end's share of this CTA: 128 B
constexpr uint32_t kBufs = 2 * kGaWarps, kCapRows = 48;   // gather buffers: two per gather warp, 6 KB each
constexpr uint32_t kBufBytes = kCapRows * kRowBytes;      // (a chunk: <= 32 nodes, <= 48 pipe ends)
constexpr uint32_t kTblWords = 2048;           // shared-memory copy of the chunk table and of inc_ptr, when they fit
constexpr int kH4 = kHalf / 4;

// Index tables of the gather, rebuilt per call (microseconds):
//   end_pos[2 p + end] = position of that pipe end in the node-sorted incidence list `inc` (its inverse permutation)
//   chunks: tbl[0] = number of chunks C, tbl[1 .. C + 1] = first node of every chunk (tbl[C + 1] = N); a chunk is a run
//   of at most kCapNodes nodes with at most kCapRows pipe ends (a node with more ends than that is a chunk of its own)
__global__ void __launch_bounds__(256)
prep_incidence_kernel(const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc, int32_t* __restrict__ end_pos,
                      int32_t* __restrict__ tbl, int n_ends, uint32_t N) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n_ends) end_pos[__ldg(inc + e)] = e;
    if (blockIdx.x == 0 && threadIdx.x < 32) {
        const uint32_t lane = threadIdx.x;
        uint32_t n0 = 0, c = 0;
        while (n0 < N) {
            if (lane == 0) tbl[1 + c] = static_cast<int32_t>(n0);
            const uint32_t r0 = static_cast<uint32_t>(__ldg(inc_ptr + n0)), i = n0 + 1 + lane;
            const uint32_t re = i <= N ? static_cast<uint32_t>(__ldg(inc_ptr + i)) : 0xffffffffu;
            const uint32_t cnt = __popc(__ballot_sync(0xffffffffu, i <= N && re - r0 <= kCapRows));
            n0 += cnt ? cnt : 1;
            ++c;
        }
        if (lane == 0) {
            tbl[1 + c] = static_cast<int32_t>(N);
            tbl[0] = static_cast<int32_t>(c);
        }
    }
}

__global__ void __launch_bounds__(kThreads, 1)
pipe_head_bwd_dx_kernel(const DpreLoader loader, float4* __restrict__ dx, const int2* __restrict__ end_pos,
                        const int32_t* __restrict__ tbl, const int32_t* __restrict__ inc_ptr,
                        const uint2* __restrict__ hsign, const float4* __restrict__ dpooled, float4* __restrict__ scratch,
                        uint32_t P, uint32_t N, uint32_t B, const float* __restrict__ W1) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t bar_full[kStages], bar_empty[kStages], bar_tfull[2], bar_tempty[2], bar_gather[kBufs];
    __shared__ uint64_t bar_wdone[2], bar_wfree[2];   // scratch of window parity p: complete (epilogue) / gathered
    __shared__ uint32_t tmem_base_s;
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_hi = smem;  // B[n][k] = w2[k] * W1[k][column n of this CTA's half], n = 32 * block + feature
    uint8_t* b_lo = b_hi + kN * kK * 4;
    uint8_t* scr_patch = b_lo + kN * kK * 4;
    uint8_t* gbuf = scr_patch + kEpWarps * kScrBytes;
    int32_t* tbl_s = reinterpret_cast<int32_t*>(gbuf + kBufs * kBufBytes);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t fh = blockIdx.x & 1;  // which half of the node features this CTA produces

    if (warp == kMmaWarp) tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&bar_full[s], 4);
            mbar_init(&bar_empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bar_tfull[a], 1);
            mbar_init(&bar_tempty[a], 4);   // the four quadrant warps that drain this accumulator
        }
        for (uint32_t b = 0; b < kBufs; ++b) mbar_init(&bar_gather[b], 1);
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bar_wdone[a], kEpWarps);
            mbar_init(&bar_wfree[a], kGaWarps);
        }
        fence_mbar_init();
    }
    // the gather's index tables (first_node -> inc_ptr -> rows: dependent loads) fit shared memory for any graph this
    // head is used on
    const uint32_t n_chunks = static_cast<uint32_t>(__ldg(tbl));
    const bool tbl_fits = n_chunks + 2 + N + 1 <= kTblWords;
    if (tbl_fits) {
        for (uint32_t i = tid; i < n_chunks + 1; i += kThreads) tbl_s[i] = __ldg(tbl + 1 + i);
        for (uint32_t i = tid; i <= N; i += kThreads) tbl_s[n_chunks + 1 + i] = __ldg(inc_ptr + i);
    }
    const int32_t* first_node = tbl_fits ? tbl_s : tbl + 1;
    const int32_t* node_ptr = tbl_fits ? tbl_s + n_chunks + 1 : inc_ptr;
    for (int i = tid; i < kN * kK; i += kThreads) {   // resident B, K-major SW128, hi / lo
        const int k = i / kN, n = i - k * kN;
        const float w = __ldg(W1 + static_cast<size_t>(k) * (3 * kD) + (n >> 5) * kD + fh * kHalf + (n & 31)) * __ldg(loader.w2 + k);
        const float hi = tf32_hi(w), lo = w - hi;
        const uint32_t off = sw128_offset(n, k >> 2, kN) + (k & 3) * 4;
        *reinterpret_cast<float*>(b_hi + off) = hi;
        *reinterpret_cast<float*>(b_lo + off) = lo;
    }
    fence_proxy_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t acc_base = tmem_base, a_base = tmem_base + 2 * kN;
    // two CTAs (the two feature halves) share a contiguous range of windows; a window is T tiles of 128 pipe rows
    const uint32_t T = (P + 127) / 128;
    const uint32_t n_ranges = gridDim.x >> 1;
    const uint32_t per_cta = (B + n_ranges - 1) / n_ranges;
    const uint32_t w_begin = min((blockIdx.x >> 1) * per_cta, B), w_end = min(w_begin + per_cta, B);
    const uint32_t n_tiles = (w_end - w_begin) * T;

    // scratch: [window parity][2 P pipe ends, node-sorted][8] float4 per CTA
    float4* scr_cta = scratch + static_cast<size_t>(blockIdx.x) * 2 * P * 2 * kH4;
    const size_t scr_par = static_cast<size_t>(P) * 2 * kH4;
    if (warp < kLdWarps) {
        const int quad = warp & 3;
        const uint32_t st_base = a_base + (static_cast<uint32_t>(quad * 32) << 16);
        uint32_t stage = 0;
        uint4 m_next = make_uint4(0, 0, 0, 0);
        auto fetch = [&](uint32_t t) {
            const uint32_t w = w_begin + t / T, p = (t % T) * 128 + quad * 32 + lane;
            m_next = (t < n_tiles && p < P) ? __ldg(loader.hmask + static_cast<size_t>(w) * P + p) : make_uint4(0, 0, 0, 0);
        };
        fetch(0);
        for (uint32_t t = 0; t < n_tiles; ++t) {
            const uint4 m = m_next;
            fetch(t + 1);
#pragma unroll 1
            for (int kg = 0; kg < 4; ++kg) {
                const uint32_t slot = stage & (kStages - 1);
                mbar_wait_relaxed(&bar_empty[slot], ((stage / kStages) & 1) ^ 1);   // the MMA that read it two tiles ago is done
                ++stage;
                fence_after_sync();
                const uint32_t bits = kg == 0 ? m.x : (kg == 1 ? m.y : (kg == 2 ? m.z : m.w));
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = static_cast<int32_t>(bits << j) < 0 ? 1.f : 0.f;
                rowgemm_ts::tmem_st32(st_base + slot * kStageCols, v);
                rowgemm_ts::tmem_wait_st();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_full[slot]);
            }
        }
    } else if (warp == kMmaWarp) {
        const uint32_t idesc = idesc_tf32(128, kN);
        const uint32_t bh = desc_lo(smem_u32(b_hi)), bl = desc_lo(smem_u32(b_lo));
        constexpr uint32_t kg_units = static_cast<uint32_t>(kN) * 128u >> 4;
        for (uint32_t t = 0; t < n_tiles; ++t) {
            const uint32_t a = t & 1;
            mbar_wait_relaxed(&bar_tempty[a], ((t >> 1) & 1) ^ 1);
            const uint32_t d = acc_base + a * kN;
            // the four stages of a tile per hand-over (32 MMAs back to back; the ring is two tiles deep, so the loaders
            // fill the next tile meanwhile): the tensor pipe only runs while this warp is issuing
            const uint32_t stage0 = 4 * t, slot0 = stage0 & (kStages - 1), par = (stage0 / kStages) & 1;
#pragma unroll
            for (uint32_t kg = 0; kg < 4; ++kg) mbar_wait_relaxed(&bar_full[slot0 + kg], par);
            fence_after_sync();
            if (elect_one()) {
#pragma unroll
                for (uint32_t kg = 0; kg < 4; ++kg) {
                    const uint32_t a_op = a_base + (slot0 + kg) * kStageCols;
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k) {
                        const uint32_t boff = kg * kg_units + 2 * k;
                        rowgemm_ts::mma_tf32_ts(d, a_op + 8 * k, bl + boff, idesc, (kg == 0 && k == 0) ? 0u : 1u);
                        rowgemm_ts::mma_tf32_ts(d, a_op + 8 * k, bh + boff, idesc, 1u);
                    }
                    commit(&bar_empty[slot0 + kg]);
                }
                commit(&bar_tfull[a]);
            }
            __syncwarp();
        }
    } else if (warp > kMmaWarp + kEpWarps) {
        // ---- gather: this warp owns chunks j, j + 4, ... of every window and two staging buffers; a chunk's bulk copy
        // travels while the previous chunk is added up; 8 lanes = the 128 bytes of a node, 4 nodes per pass
        const uint32_t j = static_cast<uint32_t>(warp - kMmaWarp - kEpWarps - 1);
        const uint32_t n_win = w_end - w_begin;
        const uint32_t own = n_chunks > j ? (n_chunks - j + kGaWarps - 1) / kGaWarps : 0;   // chunks per window
        const float inv_n = 1.f / static_cast<float>(N);
        const uint32_t f = lane & 7;
        uint8_t* my_buf = gbuf + 2 * j * kBufBytes;
        uint64_t* my_bar = bar_gather + 2 * j;
        uint32_t cnt = 0;                                     // chunks so far: buffer = cnt & 1, phase = (cnt >> 1) & 1
        auto chunk_rows = [&](uint32_t k, uint32_t& n0, uint32_t& n1, uint32_t& r0, uint32_t& r1) {
            const uint32_t c = j + k * kGaWarps;
            n0 = static_cast<uint32_t>(first_node[c]);
            n1 = static_cast<uint32_t>(first_node[c + 1]);
            r0 = static_cast<uint32_t>(node_ptr[n0]);
            r1 = static_cast<uint32_t>(node_ptr[n1]);
        };
        auto issue = [&](uint32_t k, uint32_t idx, const float4* scr) {
            uint32_t n0, n1, r0, r1;
            chunk_rows(k, n0, n1, r0, r1);
            if (lane == 0) {
                uint64_t* bar = my_bar + (idx & 1);
                if (r1 > r0 && r1 - r0 <= kCapRows) {
                    const uint32_t bytes = (r1 - r0) * kRowBytes;
                    fence_proxy_async_smem();   // my reads of this buffer (two chunks ago), before the async proxy refills it
                    mbar_arrive_expect_tx(bar, bytes);
                    bulk_load(my_buf + (idx & 1) * kBufBytes, scr + static_cast<size_t>(r0) * kH4, bytes, bar);
                } else {
                    mbar_arrive(bar);   // nothing to stage (no pipe ends, or one node above the cap): keeps the phase in step
                }
            }
        };
        for (uint32_t win = 0; win < n_win; ++win) {
            const uint32_t w = w_begin + win;
            float4 base = make_float4(0.f, 0.f, 0.f, 0.f);
            if (dpooled) {
                const float4 pl = __ldg(dpooled + static_cast<size_t>(w) * kD4 + fh * kH4 + f);
                base = make_float4(pl.x * inv_n, pl.y * inv_n, pl.z * inv_n, pl.w * inv_n);
            }
            const float4* scr = scr_cta + (win & 1) * scr_par;
            mbar_wait_relaxed(&bar_wdone[win & 1], (win >> 1) & 1);   // the epilogue has parked all rows of the window
            if (own) issue(0, cnt, scr);
            for (uint32_t k = 0; k < own; ++k, ++cnt) {
                __syncwarp();
                if (k + 1 < own) issue(k + 1, cnt + 1, scr);
                uint32_t n0, n1, r0, r1;
                chunk_rows(k, n0, n1, r0, r1);
                const bool staged = r1 > r0 && r1 - r0 <= kCapRows;
                mbar_wait(my_bar + (cnt & 1), (cnt >> 1) & 1);
                const float4* stage = reinterpret_cast<const float4*>(my_buf + (cnt & 1) * kBufBytes) + f;
                // The row range of a lane's node is read one pass ahead.  The row loop is warp-uniform (it runs to the
                // longest of the pass's four nodes, shorter ones add zeros): as a per-lane loop the compiler unrolled it
                // into a thicket of divergent remainders, 120 instructions and 650 clocks per pass.  Two rows per trip,
                // two partial sums: the order of the additions is a fixed function of the graph.
                uint32_t node = n0 + (lane >> 3);
                uint32_t e0 = 0, rows = 0;
                if (node < n1) {
                    e0 = static_cast<uint32_t>(node_ptr[node]);
                    rows = static_cast<uint32_t>(node_ptr[node + 1]) - e0;
                }
                const uint32_t n_pass = (n1 - n0 + 3) >> 2;
#pragma unroll 1
                for (uint32_t ps = 0; ps < n_pass; ++ps) {
                    const uint32_t nxt = node + 4;
                    uint32_t f0 = 0, frows = 0;
                    if (nxt < n1) {
                        f0 = static_cast<uint32_t>(node_ptr[nxt]);
                        frows = static_cast<uint32_t>(node_ptr[nxt + 1]) - f0;
                    }
                    float4 acc = base, acc2 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (staged) {
                        const uint32_t longest = __reduce_max_sync(0xffffffffu, rows);
                        const float4* row = stage + static_cast<int32_t>(e0 - r0) * kH4;   // (never read when rows == 0)
#pragma unroll 1
                        for (uint32_t i = 0; i < longest; i += 2, row += 2 * kH4) {
                            float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
                            if (i < rows) v0 = row[0];
                            if (i + 1 < rows) v1 = row[kH4];
                            acc.x += v0.x; acc.y += v0.y; acc.z += v0.z; acc.w += v0.w;
                            acc2.x += v1.x; acc2.y += v1.y; acc2.z += v1.z; acc2.w += v1.w;
                        }
                    } else {
                        for (uint32_t e = e0; e < e0 + rows; ++e) {
                            const float4 v = __ldcg(scr + static_cast<size_t>(e) * kH4 + f);
                            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
                        }
                    }
                    if (node < n1)
                        stg_stream(dx + (static_cast<size_t>(w) * N + node) * kD4 + fh * kH4 + f,
                                   make_float4(acc.x + acc2.x, acc.y + acc2.y, acc.z + acc2.z, acc.w + acc2.w));
                    node = nxt;
                    e0 = f0;
                    rows = frows;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_wfree[win & 1]);   // this warp is done with the window's scratch
        }
    } else {
        const int e_warp = warp - kMmaWarp - 1;
        const int q = warp & 3;                                     // TMEM lane quadrant = warp % 4
        constexpr uint32_t kGroups = kEpWarps / 4;                  // 1: every warp takes every tile; 2: even / odd tiles
        const uint32_t par = static_cast<uint32_t>(e_warp >> 2);    // this warp's group
        uint8_t* row_u = scr_patch + e_warp * kScrBytes + lane * kRowPitch;   // this thread's two staging rows
        uint8_t* row_v = row_u + 32 * kRowPitch;
        const int sub = lane >> 3, ch = lane & 7;
        const uint8_t* seg = scr_patch + e_warp * kScrBytes + sub * kRowPitch + ch * 16;   // read-back: row 4 k + sub, chunk ch
        // per tile, fetched one of this warp's tiles ahead: g, the scratch positions of the two ends and the 2 x 32 sign bits
        // of this thread's pipe row
        float g_next = 0.f;
        int2 pos_next = make_int2(-1, -1);
        uint2 sg_next = make_uint2(0u, 0u);
        auto fetch = [&](uint32_t t) {
            const uint32_t w = w_begin + t / T, p = (t % T) * 128 + q * 32 + lane;
            if (t < n_tiles && p < P) {
                const size_t row = static_cast<size_t>(w) * P + p;
                g_next = __ldg(loader.dlogit + row) * loader.scale;
                pos_next = __ldg(end_pos + p);
                sg_next = __ldg(hsign + row * 2 + fh);
            } else {
                g_next = 0.f;
                pos_next = make_int2(-1, -1);
                sg_next = make_uint2(0u, 0u);
            }
        };
        fetch(par);
        for (uint32_t t = 0; t < n_tiles; ++t) {
            const uint32_t a = t & 1, widx = t / T, tt = t % T;
            float4* scr = scr_cta + (widx & 1) * scr_par;
            // the gather of the window that used this half of the scratch two windows ago must be over
            if (tt == 0 && widx >= 2) mbar_wait(&bar_wfree[widx & 1], ((widx >> 1) - 1) & 1);
            if (t % kGroups == par) {
                const float g = g_next;
                const int2 pos = pos_next;
                const uint2 sg = sg_next;    // .x: x_u > x_v, .y: x_u < x_v; feature j of the half at bit 31 - j
                fetch(t + kGroups);
                mbar_wait_relaxed(&bar_tfull[a], (t >> 1) & 1);
                fence_after_sync();
                const uint32_t taddr = acc_base + a * kN + (static_cast<uint32_t>(q * 32) << 16);
                float c[32], e[32];
                tmem_ld32(taddr + 2 * kHalf, c);     // d / d |x_u - x_v|  ->  g * sign * c
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float gc = g * c[j];
                    c[j] = static_cast<int32_t>(sg.x << j) < 0 ? gc : (static_cast<int32_t>(sg.y << j) < 0 ? -gc : 0.f);
                }
                tmem_ld32(taddr, e);                 // d / d x_u
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(row_u + 4 * j) = make_float4(fmaf(g, e[j], c[j]), fmaf(g, e[j + 1], c[j + 1]),
                                                                            fmaf(g, e[j + 2], c[j + 2]), fmaf(g, e[j + 3], c[j + 3]));
                tmem_ld32(taddr + kHalf, e);         // d / d x_v
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_tempty[a]);  // accumulator drained
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(row_v + 4 * j) = make_float4(fmaf(g, e[j], -c[j]), fmaf(g, e[j + 1], -c[j + 1]),
                                                                            fmaf(g, e[j + 2], -c[j + 2]), fmaf(g, e[j + 3], -c[j + 3]));
                __syncwarp();
#pragma unroll
                for (int k = 0; k < 8; ++k) {        // rows 4 k + sub: 8 lanes = one 128-byte row
                    const int pu = __shfl_sync(0xffffffffu, pos.x, 4 * k + sub), pv = __shfl_sync(0xffffffffu, pos.y, 4 * k + sub);
                    if (pu >= 0) {
                        __stcg(scr + static_cast<size_t>(pu) * kH4 + ch, *reinterpret_cast<const float4*>(seg + 4 * k * kRowPitch));
                        __stcg(scr + static_cast<size_t>(pv) * kH4 + ch,
                               *reinterpret_cast<const float4*>(seg + (32 + 4 * k) * kRowPitch));
                    }
                }
                __syncwarp();                        // the staging rows may be overwritten
            }
            if (tt == T - 1) {
                // my rows of this window are parked: hand the scratch to the gather warps
                fence_proxy_async_all();   // my scratch stores, before the async proxy reads them
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_wdone[widx & 1]);
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
}  // namespace hb

// ------------------------------------------------------------------ mean pool and its adjoint
// out[u, :] = (sum of rows [r_lo, r_hi) of window b) / div, u = b * units_per_b + block (one unit per window and
// div = N for the L-TOWN sizes; large graphs are split into row blocks and a second call sums the partials).  A divide,
// not a multiply by 1 / N: the rounded reciprocal is off by up to 6e-8 in one direction for every output (-3.6e-8 at
// N = 661), a bias that tests/test_bench_sizes_gpu.py::test_mean_pool_at_bench_rows sees on same-sign inputs
__global__ void __launch_bounds__(256)
mean_pool_kernel(const float4* __restrict__ x, float4* __restrict__ pooled, int64_t B, int N, int d4, int units_per_b,
                 int rows_per_unit, float div) {
    __shared__ float4 red[256];
    const int tid = threadIdx.x;
    const int c = tid % d4, r0 = tid / d4, rstep = 256 / d4;
    for (int64_t u = blockIdx.x; u < B * units_per_b; u += gridDim.x) {
        const int64_t b = u / units_per_b;
        const int r_lo = static_cast<int>(u - b * units_per_b) * rows_per_unit;
        const int r_hi = r_lo + rows_per_unit < N ? r_lo + rows_per_unit : N;
        const float4* xb = x + b * N * d4 + c;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int r = r_lo + r0; r < r_hi; r += rstep) {
            const float4 v = ptx::ldg_stream(xb + static_cast<int64_t>(r) * d4);
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        red[tid] = s;
        __syncthreads();
        if (tid < d4) {
            float4 t = red[tid];
            for (int k = tid + d4; k < 256; k += d4) {
                const float4 o = red[k];
                t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
            }
            pooled[u * d4 + tid] = make_float4(t.x / div, t.y / div, t.z / div, t.w / div);
        }
        __syncthreads();
    }
}

// dx[b, i, :] = dpooled[b, :] / N   (adjoint of the mean; also the initial value the pipe-head scatter adds onto)
__global__ void __launch_bounds__(256)
pool_bwd_fill_kernel(const float4* __restrict__ dpooled, float4* __restrict__ dx, int64_t total4, int N, int d4) {
    const float inv = 1.f / static_cast<float>(N);
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    const int64_t per_b = static_cast<int64_t>(N) * d4;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total4; i += stride) {
        const int64_t b = i / per_b;
        const int c = static_cast<int>(i % d4);
        const float4 g = __ldg(dpooled + b * d4 + c);
        ptx::stg_stream(dx + i, make_float4(g.x * inv, g.y * inv, g.z * inv, g.w * inv));
    }
}

uint64_t magic_of(int P) { return P >= 2 ? (~0ull / static_cast<uint64_t>(P)) + 1 : 0ull; }

int head_shape_check(int D, int H, const char* who) {
    LTGNN_REQUIRE(D == 64, LTGNN_E_SHAPE, "%s: node width D=%d not supported by the fused head (64 only)", who, D);
    LTGNN_REQUIRE(H == 128, LTGNN_E_SHAPE, "%s: hidden width H=%d not supported by the fused head (128 only)", who, H);
    return LTGNN_OK;
}

}  // namespace

extern "C" int ltgnn_pipe_head_fwd(int device, int64_t B, int32_t N, int32_t P, int32_t D, int32_t H, const float* X,
                                   const int32_t* ends, const float* W1, const float* b1, const float* w2,
                                   float drop_p, uint64_t drop_seed, float* part, float* hpost, uint32_t* hmask,
                                   uint32_t* hsign, void* stream_) {
    LTGNN_REQUIRE(B >= 0 && N > 0 && P > 0, LTGNN_E_ARG, "pipe_head_fwd: B=%lld N=%d P=%d", static_cast<long long>(B), N, P);
    int rc = head_shape_check(D, H, "pipe_head_fwd");
    if (rc) return rc;
    LTGNN_REQUIRE(drop_p >= 0.f && drop_p < 1.f, LTGNN_E_ARG, "pipe_head_fwd: dropout p=%f", drop_p);
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(X && ends && W1 && b1 && w2 && part, LTGNN_E_ARG, "pipe_head_fwd: null tensor");
    LTGNN_REQUIRE(aligned16(X) && aligned16(W1) && aligned16(b1) && aligned16(w2) && aligned16(hpost) && aligned16(hmask) &&
                      aligned16(hsign),
                  LTGNN_E_ALIGN, "pipe_head_fwd: 16-byte alignment required");
    const int64_t M = B * P;
    LTGNN_REQUIRE(M < (1ll << 31), LTGNN_E_SHAPE, "pipe_head_fwd: B*P too large");
    const uint32_t t16 = drop_p > 0.f ? static_cast<uint32_t>(static_cast<double>(drop_p) * 65536.0 + 0.5) : 0u;
    HeadFwdEpilogue ep{b1, w2, part, hpost, hmask, H, t16, 1.f / (1.f - static_cast<float>(t16) / 65536.f), drop_seed,
                       seed_source()};
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "pipe_head_fwd: device is sm_%d%d, need sm_100", di->cc_major,
                  di->cc_minor);
    LTGNN_REQUIRE(B * N < (1ll << 31), LTGNN_E_SHAPE, "pipe_head_fwd: B*N too large");
    const size_t smem = 1024 + 2ull * hf::kN * hf::kK * 4 + hf::kLdWarps * hf::kScrBytes;
    LTGNN_REQUIRE(smem <= static_cast<size_t>(di->smem_optin), LTGNN_E_SHAPE, "pipe_head_fwd: %zu B of shared memory", smem);
    LTGNN_USE_DEVICE(device);
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(hf::pipe_head_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    const int64_t tiles = (M + 127) / 128;
    const int grid = static_cast<int>(tiles < di->sm_count ? tiles : di->sm_count);
    hf::pipe_head_fwd_kernel<<<grid, hf::kThreads, smem, static_cast<cudaStream_t>(stream_)>>>(
        reinterpret_cast<const float4*>(X), reinterpret_cast<const int2*>(ends), static_cast<uint32_t>(P),
        static_cast<uint32_t>(N), magic_of(P), ep, W1, static_cast<uint32_t>(M), reinterpret_cast<uint2*>(hsign));
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

// index tables (2 P end positions, the chunk table: 1 + N + 1 entries) + per CTA two windows' 2 P rows of 32 floats
static int64_t dx_table_words(int32_t N, int32_t P) { return (2ll * P + N + 2 + 3) / 4 * 4; }
extern "C" int64_t ltgnn_pipe_head_dx_ws_floats(int device, int32_t N, int32_t P) {
    const DeviceInfo* di = device_info(device);
    return di ? dx_table_words(N, P) + static_cast<int64_t>(di->sm_count) * 2 * 2 * P * hb::kHalf : -1;
}

extern "C" int ltgnn_pipe_head_bwd_dx(int device, int64_t B, int32_t N, int32_t P, int32_t D, int32_t H,
                                      const int32_t* inc_ptr, const int32_t* inc, const float* W1, const float* w2,
                                      const uint32_t* hmask, const uint32_t* hsign, const float* dlogit, float gate_scale,
                                      const float* dpooled, float* ws, float* dX, void* stream_) {
    LTGNN_REQUIRE(B >= 0 && N > 0 && P > 0, LTGNN_E_ARG, "pipe_head_bwd_dx: B=%lld N=%d P=%d", static_cast<long long>(B), N, P);
    int rc = head_shape_check(D, H, "pipe_head_bwd_dx");
    if (rc) return rc;
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(inc_ptr && inc && W1 && w2 && hmask && hsign && dlogit && ws && dX, LTGNN_E_ARG,
                  "pipe_head_bwd_dx: null tensor");
    LTGNN_REQUIRE(aligned16(W1) && aligned16(hmask) && aligned16(hsign) && aligned16(dX) && aligned16(ws) && aligned16(dpooled),
                  LTGNN_E_ALIGN, "pipe_head_bwd_dx: 16-byte alignment required");
    DpreLoader ld{reinterpret_cast<const uint4*>(hmask), dlogit, w2, gate_scale};
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_REQUIRE(di->cc_major == 10, LTGNN_E_UNSUPPORTED, "pipe_head_bwd_dx: device is sm_%d%d, need sm_100",
                  di->cc_major, di->cc_minor);
    LTGNN_REQUIRE(B * P < (1ll << 31) && B * N < (1ll << 28), LTGNN_E_SHAPE, "pipe_head_bwd_dx: B*P or B*N too large");
    const size_t smem = 1024 + 2ull * hb::kN * hb::kK * 4 + hb::kEpWarps * hb::kScrBytes + hb::kBufs * hb::kBufBytes + hb::kTblWords * 4;
    LTGNN_REQUIRE(smem <= static_cast<size_t>(di->smem_optin), LTGNN_E_SHAPE, "pipe_head_bwd_dx: %zu B of shared memory", smem);
    LTGNN_USE_DEVICE(device);
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int32_t* end_pos = reinterpret_cast<int32_t*>(ws);
    int32_t* tbl = end_pos + 2 * P;
    float* scratch = ws + dx_table_words(N, P);
    hb::prep_incidence_kernel<<<(2 * P + 255) / 256, 256, 0, stream>>>(inc_ptr, inc, end_pos, tbl, 2 * P, static_cast<uint32_t>(N));
    LTGNN_CUDA_TRY(cudaGetLastError());
    LTGNN_CUDA_TRY(cudaFuncSetAttribute(hb::pipe_head_bwd_dx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        static_cast<int>(smem)));
    // two CTAs (feature halves) per window range
    const int64_t ranges = B < di->sm_count / 2 ? B : di->sm_count / 2;
    hb::pipe_head_bwd_dx_kernel<<<static_cast<int>(2 * ranges), hb::kThreads, smem, stream>>>(
        ld, reinterpret_cast<float4*>(dX), reinterpret_cast<const int2*>(end_pos), tbl, inc_ptr,
        reinterpret_cast<const uint2*>(hsign), reinterpret_cast<const float4*>(dpooled), reinterpret_cast<float4*>(scratch),
        static_cast<uint32_t>(P), static_cast<uint32_t>(N), static_cast<uint32_t>(B), W1);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}

extern "C" int ltgnn_mean_pool_fwd(int device, int64_t B, int32_t N, int32_t D, const float* X, float* pooled,
                                   void* stream_) {
    LTGNN_REQUIRE(B >= 0 && N > 0 && D > 0, LTGNN_E_ARG, "mean_pool_fwd: B=%lld N=%d D=%d", static_cast<long long>(B), N, D);
    LTGNN_REQUIRE(D % 4 == 0 && 256 % (D / 4) == 0, LTGNN_E_SHAPE, "mean_pool_fwd: D=%d must be 4 * a divisor of 256", D);
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(X && pooled, LTGNN_E_ARG, "mean_pool_fwd: null tensor");
    LTGNN_REQUIRE(aligned16(X) && aligned16(pooled), LTGNN_E_ALIGN, "mean_pool_fwd: 16-byte alignment required");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_USE_DEVICE(device);
    const int64_t cap = static_cast<int64_t>(di->sm_count) * 8;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const float n_f = static_cast<float>(N);
    int units_per_b = static_cast<int>((cap + B - 1) / B);
    const int max_units = (N + 2047) / 2048;  // at least 2048 rows per unit
    if (units_per_b > max_units) units_per_b = max_units;
    if (units_per_b <= 1) {
        mean_pool_kernel<<<static_cast<int>(B < cap ? B : cap), 256, 0, stream>>>(
            reinterpret_cast<const float4*>(X), reinterpret_cast<float4*>(pooled), B, N, D / 4, 1, N, n_f);
        LTGNN_CUDA_TRY(cudaGetLastError());
        return LTGNN_OK;
    }
    // few windows over a large graph: partial sums per (window, row block) in a stream-ordered temporary, then the same
    // kernel over the partials ([B, units_per_b, D] seen as B windows of units_per_b rows); fixed order, no atomics
    const int rows_per_unit = (N + units_per_b - 1) / units_per_b;
    const int64_t n_units = B * units_per_b;
    float4* part = nullptr;
    LTGNN_CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&part), sizeof(float) * n_units * D, stream));
    mean_pool_kernel<<<static_cast<int>(n_units < cap ? n_units : cap), 256, 0, stream>>>(
        reinterpret_cast<const float4*>(X), part, B, N, D / 4, units_per_b, rows_per_unit, 1.f);
    mean_pool_kernel<<<static_cast<int>(B < cap ? B : cap), 256, 0, stream>>>(part, reinterpret_cast<float4*>(pooled), B,
                                                                              units_per_b, D / 4, 1, units_per_b, n_f);
    cudaError_t e = cudaGetLastError();
    cudaFreeAsync(part, stream);
    LTGNN_CUDA_TRY(e);
    return LTGNN_OK;
}

extern "C" int ltgnn_mean_pool_bwd_fill(int device, int64_t B, int32_t N, int32_t D, const float* dpooled, float* dX,
                                        void* stream_) {
    LTGNN_REQUIRE(B >= 0 && N > 0 && D > 0 && D % 4 == 0, LTGNN_E_ARG, "mean_pool_bwd_fill: B=%lld N=%d D=%d",
                  static_cast<long long>(B), N, D);
    if (B == 0) return LTGNN_OK;
    LTGNN_REQUIRE(dpooled && dX, LTGNN_E_ARG, "mean_pool_bwd_fill: null tensor");
    LTGNN_REQUIRE(aligned16(dpooled) && aligned16(dX), LTGNN_E_ALIGN, "mean_pool_bwd_fill: 16-byte alignment required");
    const DeviceInfo* di = device_info(device);
    if (!di) return LTGNN_E_CUDA;
    LTGNN_USE_DEVICE(device);
    const int64_t total4 = B * N * (D / 4);
    int64_t blocks = (total4 + 255) / 256;
    const int64_t cap = static_cast<int64_t>(di->sm_count) * 16;
    if (blocks > cap) blocks = cap;
    pool_bwd_fill_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream_)>>>(
        reinterpret_cast<const float4*>(dpooled), reinterpret_cast<float4*>(dX), total4, N, D / 4);
    LTGNN_CUDA_TRY(cudaGetLastError());
    return LTGNN_OK;
}
