// spmm.cu -- batched aggregation  Y[b] = A_hat * X[b]  (or A_hat^T * X[b]) over a fixed graph.
//
// Replaces torch_geometric's GCNConv.propagate as the reference runs it for the B-times
// replicated graph (models/detector.py:199): index_select of (B*nnz, D) messages, multiply
// by norm, scatter_add_ with atomics -- and its autograd adjoint (index_add_ with atomics).
// Here: CSR gather for the forward, CSR-of-the-transpose gather for the backward, no atomics,
// fixed summation order (edge order, self loop last), one fp32 mul + one fp32 add per entry
// so the result is bit-identical to a sequential CPU scatter-add.
//
// Two kernels:
//   STAGED  (graphs whose 32-feature slice fits shared memory, e.g. L-TOWN 661/785 nodes):
//           persistent CTAs, one per SM.  Topology (rowptr + packed col/weight) is staged in
//           shared memory once per CTA.  A work unit is (window b, 32-feature slice): the
//           N x 128 B slice is pulled HBM -> smem by TMA (3-D tensor map, zero-filled rows
//           past N) into a multi-stage ring by one producer thread; 16 consumer warps gather
//           neighbour rows from smem with conflict-free LDS.128 (8 lanes = one 128 B row),
//           and stream the result out with 128-bit stores.  HBM traffic = read X once +
//           write Y once; every re-read of a neighbour row is a shared-memory hit.
//   GATHER  (any size, e.g. the 100k-node network): one thread per float4 of output, neighbour
//           rows read through L2; topology read through the read-only path.
#include "common.cuh"

using namespace ltgnn;
using namespace ltgnn::ptx;

namespace {

constexpr int kSliceFloats = 32;  // 128 B of each node row per work unit
constexpr int kSliceBytes = kSliceFloats * 4;
constexpr int kConsumerWarps = 24;
constexpr int kStagedThreads = (kConsumerWarps + 1) * 32;  // + 1 producer warp
constexpr int kMaxStages = 4;
constexpr int kRowsPerPass = kConsumerWarps * 4;  // 8 lanes per row, 4 rows per warp
constexpr int kMaxGateRows = 11;  // rows per thread in the gate pass: graphs up to 1056 nodes

struct StagedParams {
    const int32_t* rowptr;
    const int2* colval;
    float* Y;
    int64_t n_units;  // B * n_slices
    int32_t n, nnz, d4, n_slices;
    int32_t box_rows, n_boxes, n_stages;
    uint32_t stage_bytes, off_rowptr, off_colval, off_stage0;
    // output epilogue (kEpi): y = dropout(relu(acc + bias))
    const float* bias;
    int32_t relu;
    uint32_t drop_thresh;  // round(p * 2^16), 0 = no dropout (16 random bits per element)
    float keep_scale;      // 1 / (1 - drop_thresh / 2^16): exactly unbiased
    uint64_t drop_seed;
    const uint64_t* seed_src;  // ltgnn_seed_source word or nullptr
    // input gate (kGate): x *= gate > 0 ? gate_scale : 0 before aggregation; column sums of the gated x
    const float* gate;
    float gate_scale;
    float* colsum_ws;  // [gridDim.x][32] per-CTA partial column sums, or nullptr
    // 1-bit-per-element form of the gate: word (b, slice, node), bit 8 c + q <-> element (b, node, 32 slice + 4 q + c)
    uint32_t* live_out;       // written by the output epilogue (kEpi), or nullptr
    const uint32_t* live_in;  // read by the input gate (kGate) instead of `gate`, or nullptr
    // per-call entry values (kVals): entry k of window b weighs vals[b * vals_stride + k] instead of the handle's value
    const float* vals;
    int64_t vals_stride;  // 0: one set shared by every window
};

__device__ __forceinline__ void fma2(float4& acc, float w, const float4& x) {
    // two roundings per entry, as ATen's mul followed by index_add_ (see file header)
    acc.x = __fadd_rn(acc.x, __fmul_rn(w, x.x));
    acc.y = __fadd_rn(acc.y, __fmul_rn(w, x.y));
    acc.z = __fadd_rn(acc.z, __fmul_rn(w, x.z));
    acc.w = __fadd_rn(acc.w, __fmul_rn(w, x.w));
}

__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kConsumerWarps * 32) : "memory"); }

template <bool kEpi, bool kGate, bool kVals = false>
__global__ void __launch_bounds__(kStagedThreads, 1)
spmm_staged_kernel(const __grid_constant__ CUtensorMap tmap, const StagedParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* empty = full + kMaxStages;
    int32_t* s_rowptr = reinterpret_cast<int32_t*>(smem + p.off_rowptr);
    int2* s_colval = reinterpret_cast<int2*>(smem + p.off_colval);
    uint8_t* s_stage = smem + p.off_stage0;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int S = p.n_stages;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, kConsumerWarps);
        }
        fence_mbar_init();
    }
    for (int i = threadIdx.x; i <= p.n; i += kStagedThreads) s_rowptr[i] = __ldg(p.rowptr + i);
    for (int i = threadIdx.x; i < p.nnz; i += kStagedThreads) s_colval[i] = __ldg(p.colval + i);
    __syncthreads();

    if (warp == kConsumerWarps) {
        // ---------------- producer: one thread drives TMA ----------------
        if (lane == 0) {
            tma_prefetch_desc(&tmap);
            int it = 0;
            for (int64_t u = blockIdx.x; u < p.n_units; u += gridDim.x, ++it) {
                const int s = it % S;
                const uint32_t ph = (it / S) & 1;
                mbar_wait(empty + s, ph ^ 1);  // slot free (passes at once on first use)
                mbar_arrive_expect_tx(full + s, p.stage_bytes);
                const int64_t b = u / p.n_slices;
                const int sl = static_cast<int>(u - b * p.n_slices);
                uint8_t* dst = s_stage + static_cast<size_t>(s) * p.stage_bytes;
                for (int bx = 0; bx < p.n_boxes; ++bx)
                    tma_load_3d(dst + static_cast<size_t>(bx) * p.box_rows * kSliceBytes, &tmap, full + s,
                                sl * kSliceFloats, bx * p.box_rows, static_cast<int>(b));
            }
        }
        return;
    }

    // ---------------- consumers: (gate,) gather from smem, (epilogue,) stream out ----------------
    const int g = lane >> 3;  // row within the warp's group of 4
    const int q = lane & 7;   // float4 within the 128 B slice
    float4 csum = make_float4(0.f, 0.f, 0.f, 0.f);
    int it = 0;
    for (int64_t u = blockIdx.x; u < p.n_units; u += gridDim.x, ++it) {
        const int s = it % S;
        const uint32_t ph = (it / S) & 1;
        const int64_t b = u / p.n_slices;
        const int sl = static_cast<int>(u - b * p.n_slices);
        constexpr int kStepG = kConsumerWarps * 4;  // rows covered by the consumer threads per gate pass
        uint32_t live[kMaxGateRows];
        if (kGate && p.live_in) {
            // this thread's rows of the 1-bit gate: 4 bytes per row, all in flight before the stage is even waited for
            const uint32_t* lw = p.live_in + static_cast<size_t>(u) * p.n + (threadIdx.x >> 3);
#pragma unroll
            for (int k = 0; k < kMaxGateRows; ++k) live[k] = (threadIdx.x >> 3) + k * kStepG < p.n ? __ldg(lw + k * kStepG) : 0u;
        }
        mbar_wait(full + s, ph);
        float4* stage = reinterpret_cast<float4*>(s_stage + static_cast<size_t>(s) * p.stage_bytes);
        const float4* xs = stage + q;
        const int64_t base4 = (b * p.n) * p.d4 + sl * (kSliceFloats / 4) + q;  // float4 index of (b, row 0, this lane)

        if (kGate && p.live_in) {
#pragma unroll
            for (int k = 0; k < kMaxGateRows; ++k) {
                const int r = (threadIdx.x >> 3) + k * kStepG;
                if (r < p.n) {
                    const uint32_t m = live[k] >> q;  // bit 8 c of m <-> component c of this lane's float4
                    float4 x = stage[r * 8 + q];
                    x.x = (m & 0x1u) ? x.x * p.gate_scale : 0.f;
                    x.y = (m & 0x100u) ? x.y * p.gate_scale : 0.f;
                    x.z = (m & 0x10000u) ? x.z * p.gate_scale : 0.f;
                    x.w = (m & 0x1000000u) ? x.w * p.gate_scale : 0.f;
                    stage[r * 8 + q] = x;
                    csum.x += x.x; csum.y += x.y; csum.z += x.z; csum.w += x.w;
                }
            }
            consumer_bar();
        } else if (kGate) {
            // backward of the upstream ReLU(+dropout): its OUTPUT `gate` says which entries were live.
            // Each thread owns column group q for rows tid/8, tid/8 + 64, ...; then all consumers sync.
            const float4* gt = reinterpret_cast<const float4*>(p.gate) + base4;
            constexpr int kStep = kConsumerWarps * 4;  // rows covered by the consumer threads per pass
            for (int r0 = threadIdx.x >> 3; r0 < p.n; r0 += 4 * kStep) {
                float4 m[4];  // 4 gate loads in flight per thread: this pass streams a whole tensor from HBM
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (r0 + u * kStep < p.n) m[u] = ldg_stream(gt + static_cast<int64_t>(r0 + u * kStep) * p.d4);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int r = r0 + u * kStep;
                    if (r < p.n) {
                        float4 x = stage[r * 8 + q];
                        x.x = m[u].x > 0.f ? x.x * p.gate_scale : 0.f;
                        x.y = m[u].y > 0.f ? x.y * p.gate_scale : 0.f;
                        x.z = m[u].z > 0.f ? x.z * p.gate_scale : 0.f;
                        x.w = m[u].w > 0.f ? x.w * p.gate_scale : 0.f;
                        stage[r * 8 + q] = x;
                        csum.x += x.x; csum.y += x.y; csum.z += x.z; csum.w += x.w;
                    }
                }
            }
            consumer_bar();
        }

        float4* y = reinterpret_cast<float4*>(p.Y) + base4;
        const float* vb = kVals ? p.vals + b * p.vals_stride : nullptr;
        // an entry's weight: the handle's packed value, or the per-call one (same summation order either way)
        auto wt = [&](const int2 c, int k) { return kVals ? __ldg(vb + k) : __int_as_float(c.y); };
        float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (kEpi && p.bias) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias) + sl * (kSliceFloats / 4) + q);

        // two rows in flight per lane group for memory-level parallelism on the LDS chain
        // (the trip count is warp-uniform so that the epilogue may use warp votes)
        for (int rb = warp * 4; rb < p.n; rb += 2 * kRowsPerPass) {
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
                const float4 x0 = xs[c0.x * 8];
                const float4 x1 = xs[c1.x * 8];
                fma2(a0, wt(c0, k0 - 1), x0);
                fma2(a1, wt(c1, k1 - 1), x1);
            }
            for (; k0 < e0; ++k0) {
                const int2 c0 = s_colval[k0];
                fma2(a0, wt(c0, k0), xs[c0.x * 8]);
            }
            for (; k1 < e1; ++k1) {
                const int2 c1 = s_colval[k1];
                fma2(a1, wt(c1, k1), xs[c1.x * 8]);
            }
            if (kEpi) {
                a0.x = __fadd_rn(a0.x, bias4.x); a0.y = __fadd_rn(a0.y, bias4.y);
                a0.z = __fadd_rn(a0.z, bias4.z); a0.w = __fadd_rn(a0.w, bias4.w);
                a1.x = __fadd_rn(a1.x, bias4.x); a1.y = __fadd_rn(a1.y, bias4.y);
                a1.z = __fadd_rn(a1.z, bias4.z); a1.w = __fadd_rn(a1.w, bias4.w);
                if (p.relu) {
                    a0.x = fmaxf(a0.x, 0.f); a0.y = fmaxf(a0.y, 0.f); a0.z = fmaxf(a0.z, 0.f); a0.w = fmaxf(a0.w, 0.f);
                    a1.x = fmaxf(a1.x, 0.f); a1.y = fmaxf(a1.y, 0.f); a1.z = fmaxf(a1.z, 0.f); a1.w = fmaxf(a1.w, 0.f);
                }
                if (p.drop_thresh) {  // one Philox call (16 random bits per element) decides both float4
                    float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                    dropout8(v, static_cast<uint64_t>(base4 + static_cast<int64_t>(r0) * p.d4), launch_seed(p.drop_seed, p.seed_src),
                             p.drop_thresh, p.keep_scale);
                    a0 = make_float4(v[0], v[1], v[2], v[3]);
                    a1 = make_float4(v[4], v[5], v[6], v[7]);
                }
            }
            if (r0 < p.n) stg_stream(y + static_cast<int64_t>(r0) * p.d4, a0);
            if (r1 < p.n) stg_stream(y + static_cast<int64_t>(r1) * p.d4, a1);
            if (kEpi && p.live_out) {
                // 1-bit record of y > 0: one vote per float4 component, then byte g of each vote (the 8 lanes of
                // this row) forms the row's word: bit 8 c + q  <->  element 4 q + c of the 32-feature slice
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
        if (kGate) fence_proxy_async_smem();  // our generic-proxy writes to the stage precede the next TMA fill
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + s);
    }

    if (kGate && p.colsum_ws) {
        // lanes q, q+8, q+16, q+24 share a column group; then 16 warps through shared memory, fixed order
        csum.x += __shfl_xor_sync(0xffffffffu, csum.x, 8);  csum.y += __shfl_xor_sync(0xffffffffu, csum.y, 8);
        csum.z += __shfl_xor_sync(0xffffffffu, csum.z, 8);  csum.w += __shfl_xor_sync(0xffffffffu, csum.w, 8);
        csum.x += __shfl_xor_sync(0xffffffffu, csum.x, 16); csum.y += __shfl_xor_sync(0xffffffffu, csum.y, 16);
        csum.z += __shfl_xor_sync(0xffffffffu, csum.z, 16); csum.w += __shfl_xor_sync(0xffffffffu, csum.w, 16);
        consumer_bar();  // every consumer is done with the stage buffers (all its units consumed)
        float4* red = reinterpret_cast<float4*>(s_stage);
        if (lane < 8) red[warp * 8 + lane] = csum;
        consumer_bar();
        if (warp == 0 && lane < 8) {
            float4 t = red[lane];
            for (int w = 1; w < kConsumerWarps; ++w) {
                const float4 o = red[w * 8 + lane];
                t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
            }
            reinterpret_cast<float4*>(p.colsum_ws)[blockIdx.x * 8 + lane] = t;
        }
    }
}

// colsum[sl*32 + c] = sum over CTAs that worked on slice sl (cta % n_slices == sl) of ws[cta][c], fixed order
__global__ void colsum_reduce_kernel(const float* __restrict__ ws, float* __restrict__ colsum, int n_ctas, int n_slices) {
    const int col = threadIdx.x;  // 0 .. D-1
    const int sl = col >> 5, c = col & 31;
    float t = 0.f;
    for (int cta = sl; cta < n_ctas; cta += n_slices) t += ws[cta * 32 + c];
    colsum[col] = t;
}

// kEpi: y = dropout(relu(acc + bias)) as in the STAGED kernel (same Philox counter: the float4 pair (r, r + 96) of a
// window shares one call there; here a thread owns one float4, so it draws for its own index with dropout4h -- the two
// paths are statistically, not bitwise, the same stream).  kGate: every neighbour value is gated on the fly, either by the
// float gate tensor (the upstream layer's output): x * (gate > 0 ? gate_scale : 0), or -- D % 32 == 0 -- by its 1-bit
// form live_in [B, D/32, N] (4 bytes per neighbour and 32-feature slice instead of a second 16-byte gather per float4).
// live_out: the same record of y > 0, written by the q == 0 lane of every 8-lane slice group (word layout of new_live_mask:
// bit 8 c + q <-> element 4 q + c of the slice).  Lanes of a warp stay together (the ballots need all 32).
template <bool kEpi, bool kGate, bool kVals = false>
__global__ void __launch_bounds__(256)
spmm_gather_kernel(const int32_t* __restrict__ rowptr, const int2* __restrict__ colval, const float4* __restrict__ X,
                   float4* __restrict__ Y, int32_t n, int32_t d4, int64_t total, const float4* __restrict__ bias, int relu,
                   uint32_t drop_thresh, float keep_scale, uint64_t drop_seed_arg, const uint64_t* seed_src,
                   const float4* __restrict__ gate, float gate_scale, uint32_t* __restrict__ live_out,
                   const uint32_t* __restrict__ live_in, const float* __restrict__ vals, int64_t vals_stride) {
    const uint64_t drop_seed = launch_seed(drop_seed_arg, seed_src);
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    const int lane = threadIdx.x & 31, n_slices = d4 >> 3;
    for (int64_t e0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + (threadIdx.x & ~31); e0 < total; e0 += stride) {
        const int64_t e = e0 + lane;
        const bool valid = e < total;
        const int64_t row = (valid ? e : 0) / d4;
        const int c4 = static_cast<int>((valid ? e : 0) - row * d4);
        const int64_t b = row / n;
        const int r = static_cast<int>(row - b * n);
        const float4* xb = X + b * n * d4 + c4;
        const float4* gb = (kGate && gate) ? gate + b * n * d4 + c4 : nullptr;
        const uint32_t* lb = (kGate && live_in) ? live_in + (b * n_slices + (c4 >> 3)) * n : nullptr;
        const int q = c4 & 7;
        const float* vb = kVals ? vals + b * vals_stride : nullptr;
        auto wt = [&](const int2 c, int kk) { return kVals ? __ldg(vb + kk) : __int_as_float(c.y); };
        auto fetch = [&](int col) {
            float4 x = __ldg(xb + static_cast<int64_t>(col) * d4);
            if (kGate) {
                if (lb) {
                    const uint32_t w = __ldg(lb + col) >> q;
                    x.x = (w & 1u) ? x.x * gate_scale : 0.f; x.y = (w & 0x100u) ? x.y * gate_scale : 0.f;
                    x.z = (w & 0x10000u) ? x.z * gate_scale : 0.f; x.w = (w & 0x1000000u) ? x.w * gate_scale : 0.f;
                } else {
                    const float4 m = __ldg(gb + static_cast<int64_t>(col) * d4);
                    x.x = m.x > 0.f ? x.x * gate_scale : 0.f; x.y = m.y > 0.f ? x.y * gate_scale : 0.f;
                    x.z = m.z > 0.f ? x.z * gate_scale : 0.f; x.w = m.w > 0.f ? x.w * gate_scale : 0.f;
                }
            }
            return x;
        };
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid) {
            int k = __ldg(rowptr + r);
            const int end = __ldg(rowptr + r + 1);
            for (; k + 1 < end; k += 2) {
                const int2 c0 = __ldg(colval + k);
                const int2 c1 = __ldg(colval + k + 1);
                const float4 x0 = fetch(c0.x);
                const float4 x1 = fetch(c1.x);
                fma2(acc, wt(c0, k), x0);
                fma2(acc, wt(c1, k + 1), x1);
            }
            if (k < end) {
                const int2 c0 = __ldg(colval + k);
                fma2(acc, wt(c0, k), fetch(c0.x));
            }
            if (kEpi) {
                if (bias) {
                    const float4 bb = __ldg(bias + c4);
                    acc.x = __fadd_rn(acc.x, bb.x); acc.y = __fadd_rn(acc.y, bb.y);
                    acc.z = __fadd_rn(acc.z, bb.z); acc.w = __fadd_rn(acc.w, bb.w);
                }
                if (relu) {
                    acc.x = fmaxf(acc.x, 0.f); acc.y = fmaxf(acc.y, 0.f); acc.z = fmaxf(acc.z, 0.f); acc.w = fmaxf(acc.w, 0.f);
                }
                if (drop_thresh) dropout4h(acc, static_cast<uint64_t>(e), drop_seed, drop_thresh, keep_scale);
            }
            stg_stream(Y + e, acc);
        }
        if (kEpi && live_out) {   // d4 % 8 == 0: an 8-lane group is one 32-feature slice of one row, valid as a whole
            const uint32_t bx = __ballot_sync(0xffffffffu, acc.x > 0.f), by = __ballot_sync(0xffffffffu, acc.y > 0.f);
            const uint32_t bz = __ballot_sync(0xffffffffu, acc.z > 0.f), bw = __ballot_sync(0xffffffffu, acc.w > 0.f);
            const uint32_t g8 = static_cast<uint32_t>(lane >> 3), sel = g8 | ((4u + g8) << 4);
            if (valid && q == 0)
                live_out[(b * n_slices + (c4 >> 3)) * n + r] =
                    __byte_perm(__byte_perm(bx, by, sel), __byte_perm(bz, bw, sel), 0x5410);
        }
    }
}

// colsum[c] = sum over all rows of gate(x): per-CTA partials, fixed order (the d bias of the gather path); the gate as
// floats or as the 1-bit record `live` [B, D/32, N]
__global__ void __launch_bounds__(256)
gated_colsum_kernel(const float4* __restrict__ X, const float4* __restrict__ gate, const uint32_t* __restrict__ live,
                    float gate_scale, int64_t rows, int d4, int n, float* __restrict__ part) {
    __shared__ float4 red[256];
    const int tid = threadIdx.x, c = tid % d4, rstep = 256 / d4, q = c & 7, n_slices = d4 >> 3;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t step = static_cast<int64_t>(gridDim.x) * rstep;
    const int64_t step_b = step / n;                     // (window, node) of a thread's row advance without divisions
    const int step_r = static_cast<int>(step - step_b * n);
    int64_t r = static_cast<int64_t>(blockIdx.x) * rstep + tid / d4;
    int64_t b = r / n;
    int rl = static_cast<int>(r - b * n);
    for (; r < rows; r += step) {
        const float4 x = ldg_stream(X + r * d4 + c);
        if (live) {
            const uint32_t w = __ldg(live + (b * n_slices + (c >> 3)) * n + rl) >> q;
            s.x += (w & 1u) ? x.x * gate_scale : 0.f; s.y += (w & 0x100u) ? x.y * gate_scale : 0.f;
            s.z += (w & 0x10000u) ? x.z * gate_scale : 0.f; s.w += (w & 0x1000000u) ? x.w * gate_scale : 0.f;
        } else {
            const float4 m = ldg_stream(gate + r * d4 + c);
            s.x += m.x > 0.f ? x.x * gate_scale : 0.f; s.y += m.y > 0.f ? x.y * gate_scale : 0.f;
            s.z += m.z > 0.f ? x.z * gate_scale : 0.f; s.w += m.w > 0.f ? x.w * gate_scale : 0.f;
        }
        b += step_b;
        rl += step_r;
        if (rl >= n) {
            rl -= n;
            ++b;
        }
    }
    red[tid] = s;
    __syncthreads();
    if (tid < d4) {
        float4 t = red[tid];
        for (int k = tid + d4; k < 256; k += d4) {
            const float4 o = red[k];
            t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
        }
        reinterpret_cast<float4*>(part)[static_cast<size_t>(blockIdx.x) * d4 + tid] = t;
    }
}

struct StagedPlan {
    bool ok = false;
    int box_rows = 0, n_boxes = 0, n_stages = 0;
    uint32_t stage_bytes = 0, off_rowptr = 0, off_colval = 0, off_stage0 = 0, smem_bytes = 0;
};

inline uint32_t align_up(uint32_t x, uint32_t a) { return (x + a - 1) / a * a; }

StagedPlan plan_staged(const ltgnn_graph* g, int32_t D) {
    StagedPlan pl;
    if (D % kSliceFloats != 0) return pl;
    pl.n_boxes = (g->n + 255) / 256;
    pl.box_rows = (g->n + pl.n_boxes - 1) / pl.n_boxes;
    pl.stage_bytes = static_cast<uint32_t>(pl.n_boxes) * pl.box_rows * kSliceBytes;
    pl.off_rowptr = 128;  // after the barriers
    pl.off_colval = align_up(pl.off_rowptr + 4u * (g->n + 1), 16);
    pl.off_stage0 = align_up(pl.off_colval + 8u * g->nnz, 128);
    const int64_t avail = static_cast<int64_t>(g->smem_optin) - 128 /*alignment slack*/ - pl.off_stage0;
    if (avail < static_cast<int64_t>(pl.stage_bytes)) return pl;
    pl.n_stages = static_cast<int>(avail / pl.stage_bytes);
    if (pl.n_stages > kMaxStages) pl.n_stages = kMaxStages;
    pl.smem_bytes = 128 + pl.off_stage0 + pl.n_stages * pl.stage_bytes;
    pl.ok = true;
    return pl;
}

struct FusedArgs {
    const float* bias = nullptr;
    int relu = 0;
    float drop_p = 0.f;
    uint64_t drop_seed = 0;
    const float* gate = nullptr;
    float gate_scale = 1.f;
    float* colsum = nullptr;
    float* ws = nullptr;
    uint32_t* live_out = nullptr;
    const uint32_t* live_in = nullptr;
    const float* vals = nullptr;  // per-call entry values [1 or B][nnz], in the order of the chosen orientation
    int64_t vals_stride = 0;
};

int spmm_impl(ltgnn_graph_t g, int transpose, int64_t B, int32_t D, const float* X, float* Y, int algo,
              const FusedArgs& f, cudaStream_t stream, const char* who) {
    LTGNN_REQUIRE(g != nullptr, LTGNN_E_ARG, "%s: null graph handle", who);
    LTGNN_REQUIRE(transpose == 0 || transpose == 1, LTGNN_E_ARG, "%s: transpose must be 0 or 1", who);
    LTGNN_REQUIRE(B >= 0 && D > 0, LTGNN_E_ARG, "%s: B=%lld D=%d", who, static_cast<long long>(B), D);
    LTGNN_REQUIRE(D % 4 == 0, LTGNN_E_SHAPE, "%s: D=%d must be a multiple of 4", who, D);
    LTGNN_REQUIRE(B < (1ll << 31), LTGNN_E_SHAPE, "%s: B too large", who);
    LTGNN_REQUIRE(f.drop_p >= 0.f && f.drop_p < 1.f, LTGNN_E_ARG, "%s: dropout p=%f not in [0,1)", who, f.drop_p);
    const bool epi = f.bias || f.relu || f.drop_p > 0.f;
    const bool gated = f.gate != nullptr || f.live_in != nullptr;
    LTGNN_REQUIRE(!(f.gate && f.live_in), LTGNN_E_ARG, "%s: pass the gate as floats or as bits, not both", who);
    LTGNN_REQUIRE(!f.live_out || epi, LTGNN_E_ARG, "%s: live_out needs the output epilogue", who);
    LTGNN_REQUIRE(!f.colsum || (gated && f.ws), LTGNN_E_ARG, "%s: colsum needs gate and workspace", who);
    if (B == 0) {
        if (f.colsum) LTGNN_CUDA_TRY(cudaMemsetAsync(f.colsum, 0, sizeof(float) * D, stream));
        return LTGNN_OK;
    }
    LTGNN_REQUIRE(X && Y, LTGNN_E_ARG, "%s: null tensor", who);
    LTGNN_REQUIRE(X != Y, LTGNN_E_ARG, "%s: X and Y must not alias", who);
    LTGNN_REQUIRE(aligned16(X) && aligned16(Y) && aligned16(f.bias) && aligned16(f.gate), LTGNN_E_ALIGN,
                  "%s: tensors must be 16-byte aligned", who);
    LTGNN_USE_DEVICE(g->device);

    const StagedPlan pl = plan_staged(g, D);
    const bool fused = epi || gated;
    const bool want_staged = (algo == LTGNN_SPMM_STAGED) || (fused && pl.ok && algo != LTGNN_SPMM_GATHER) ||
                             (algo == LTGNN_SPMM_AUTO && pl.ok && pl.n_stages >= 2);
    if (algo == LTGNN_SPMM_STAGED)
        LTGNN_REQUIRE(pl.ok, LTGNN_E_SHAPE, "%s: the STAGED kernel needs D %% 32 == 0 and a 32-feature slice of the "
                      "graph (%d rows) to fit shared memory", who, g->n);
    if (fused && !want_staged) {  // large graphs: the L2-gather kernel carries the same epilogue / gate
        LTGNN_REQUIRE((!f.live_in && !f.live_out) || D % 32 == 0, LTGNN_E_SHAPE, "%s: 1-bit gates need D %% 32 == 0", who);
        LTGNN_REQUIRE(256 % (D / 4) == 0 || !f.colsum, LTGNN_E_SHAPE, "%s: colsum on the gather path needs D/4 | 256", who);
    }

    if (want_staged) {
        PFN_tmapEncodeTiled enc = tmap_encode_fn();
        LTGNN_REQUIRE(enc != nullptr, LTGNN_E_CUDA, "%s: cuTensorMapEncodeTiled not available from the driver", who);
        CUtensorMap tmap;
        const cuuint64_t gdim[3] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(g->n),
                                    static_cast<cuuint64_t>(B)};
        const cuuint64_t gstr[2] = {static_cast<cuuint64_t>(D) * 4, static_cast<cuuint64_t>(g->n) * D * 4};
        const cuuint32_t box[3] = {kSliceFloats, static_cast<cuuint32_t>(pl.box_rows), 1};
        const cuuint32_t estr[3] = {1, 1, 1};
        CUresult cr = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(X), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        LTGNN_REQUIRE(cr == CUDA_SUCCESS, LTGNN_E_CUDA, "%s: cuTensorMapEncodeTiled failed with CUresult %d", who,
                      static_cast<int>(cr));
        StagedParams p;
        p.rowptr = g->rowptr[transpose];
        p.colval = g->colval[transpose];
        p.Y = Y;
        p.n = g->n;
        p.nnz = g->nnz;
        p.d4 = D / 4;
        p.n_slices = D / kSliceFloats;
        p.n_units = B * p.n_slices;
        p.box_rows = pl.box_rows;
        p.n_boxes = pl.n_boxes;
        p.n_stages = pl.n_stages;
        p.stage_bytes = pl.stage_bytes;
        p.off_rowptr = pl.off_rowptr;
        p.off_colval = pl.off_colval;
        p.off_stage0 = pl.off_stage0;
        p.bias = f.bias;
        p.relu = f.relu;
        p.drop_thresh = f.drop_p > 0.f ? static_cast<uint32_t>(static_cast<double>(f.drop_p) * 65536.0 + 0.5) : 0u;
        p.keep_scale = 1.f / (1.f - static_cast<float>(p.drop_thresh) / 65536.f);
        p.drop_seed = f.drop_seed;
        p.seed_src = seed_source();
        p.gate = f.gate;
        p.gate_scale = f.gate_scale;
        p.colsum_ws = f.colsum ? f.ws : nullptr;
        p.live_out = f.live_out;
        p.live_in = f.live_in;
        p.vals = f.vals;
        p.vals_stride = f.vals_stride;
        LTGNN_REQUIRE(!f.live_in || g->n <= kMaxGateRows * kConsumerWarps * 4, LTGNN_E_SHAPE,
                      "%s: the 1-bit gate supports graphs up to %d nodes", who, kMaxGateRows * kConsumerWarps * 4);
        // a CTA must keep one feature slice for its whole life when it accumulates column sums
        int64_t grid = p.n_units < g->sm_count ? p.n_units : g->sm_count;
        grid -= grid % p.n_slices;
        LTGNN_REQUIRE(grid > 0, LTGNN_E_SHAPE, "%s: fewer SMs (%d) than feature slices (%d)", who, g->sm_count,
                      p.n_slices);
        auto launch = [&](auto kern) -> int {
            LTGNN_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                static_cast<int>(pl.smem_bytes)));
            kern<<<static_cast<int>(grid), kStagedThreads, pl.smem_bytes, stream>>>(tmap, p);
            LTGNN_CUDA_TRY(cudaGetLastError());
            return LTGNN_OK;
        };
        int rc;
        if (f.vals) {
            if (gated) rc = epi ? launch(spmm_staged_kernel<true, true, true>) : launch(spmm_staged_kernel<false, true, true>);
            else rc = epi ? launch(spmm_staged_kernel<true, false, true>) : launch(spmm_staged_kernel<false, false, true>);
        } else if (gated) rc = epi ? launch(spmm_staged_kernel<true, true>) : launch(spmm_staged_kernel<false, true>);
        else rc = epi ? launch(spmm_staged_kernel<true, false>) : launch(spmm_staged_kernel<false, false>);
        if (rc) return rc;
        if (f.colsum) {
            colsum_reduce_kernel<<<1, D, 0, stream>>>(f.ws, f.colsum, static_cast<int>(grid), p.n_slices);
            LTGNN_CUDA_TRY(cudaGetLastError());
        }
        return LTGNN_OK;
    }

    const int64_t total = B * g->n * (D / 4);
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = static_cast<int64_t>(g->sm_count) * 16;
    if (blocks > cap) blocks = cap;
    const uint32_t thresh = f.drop_p > 0.f ? static_cast<uint32_t>(static_cast<double>(f.drop_p) * 65536.0 + 0.5) : 0u;
    const float keep = 1.f / (1.f - static_cast<float>(thresh) / 65536.f);
    auto launch_g = [&](auto kern) -> int {
        kern<<<static_cast<int>(blocks), 256, 0, stream>>>(
            g->rowptr[transpose], g->colval[transpose], reinterpret_cast<const float4*>(X), reinterpret_cast<float4*>(Y),
            g->n, D / 4, total, reinterpret_cast<const float4*>(f.bias), f.relu, thresh, keep, f.drop_seed, seed_source(),
            reinterpret_cast<const float4*>(f.gate), f.gate_scale, f.live_out, f.live_in, f.vals, f.vals_stride);
        LTGNN_CUDA_TRY(cudaGetLastError());
        return LTGNN_OK;
    };
    int rc;
    if (f.vals) {
        if (gated) rc = epi ? launch_g(spmm_gather_kernel<true, true, true>) : launch_g(spmm_gather_kernel<false, true, true>);
        else rc = epi ? launch_g(spmm_gather_kernel<true, false, true>) : launch_g(spmm_gather_kernel<false, false, true>);
    } else if (gated) rc = epi ? launch_g(spmm_gather_kernel<true, true>) : launch_g(spmm_gather_kernel<false, true>);
    else rc = epi ? launch_g(spmm_gather_kernel<true, false>) : launch_g(spmm_gather_kernel<false, false>);
    if (rc) return rc;
    if (f.colsum) {
        const int n_parts = g->sm_count * 8;  // 8 CTAs per SM keep enough loads in flight; ws is too small for this: use our own
        float* part = nullptr;
        LTGNN_CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&part), sizeof(float) * n_parts * D, stream));
        gated_colsum_kernel<<<n_parts, 256, 0, stream>>>(reinterpret_cast<const float4*>(X),
                                                          reinterpret_cast<const float4*>(f.gate), f.live_in, f.gate_scale,
                                                          B * g->n, D / 4, g->n, part);
        cudaError_t e = cudaGetLastError();
        int rr = e == cudaSuccess ? reduce_parts(part, D, f.colsum, n_parts, D, 0, stream) : LTGNN_OK;
        cudaFreeAsync(part, stream);
        LTGNN_CUDA_TRY(e);
        return rr;
    }
    return LTGNN_OK;
}

}  // namespace

extern "C" int ltgnn_spmm(ltgnn_graph_t g, int transpose, int64_t B, int32_t D, const float* X, float* Y, int algo,
                          void* stream_) {
    return spmm_impl(g, transpose, B, D, X, Y, algo, FusedArgs{}, static_cast<cudaStream_t>(stream_), "spmm");
}

extern "C" int64_t ltgnn_spmm_ws_floats(ltgnn_graph_t g) { return g ? static_cast<int64_t>(g->sm_count) * 32 : 0; }

extern "C" int ltgnn_spmm_fused(ltgnn_graph_t g, int transpose, int64_t B, int32_t D, const float* X, float* Y,
                                const float* bias, int relu, float drop_p, uint64_t drop_seed, const float* gate,
                                float gate_scale, float* colsum, float* ws, uint32_t* live_out, const uint32_t* live_in,
                                void* stream_) {
    FusedArgs f;
    f.live_out = live_out;
    f.live_in = live_in;
    f.bias = bias;
    f.relu = relu;
    f.drop_p = drop_p;
    f.drop_seed = drop_seed;
    f.gate = gate;
    f.gate_scale = gate_scale;
    f.colsum = colsum;
    f.ws = ws;
    return spmm_impl(g, transpose, B, D, X, Y, LTGNN_SPMM_AUTO, f, static_cast<cudaStream_t>(stream_), "spmm_fused");
}

extern "C" int ltgnn_spmm_fused_vals(ltgnn_graph_t g, int transpose, int64_t B, int32_t D, const float* X, float* Y,
                                     const float* vals, int64_t vals_stride, int algo, const float* bias, int relu,
                                     float drop_p, uint64_t drop_seed, const float* gate, float gate_scale, float* colsum,
                                     float* ws, uint32_t* live_out, const uint32_t* live_in, void* stream_) {
    LTGNN_REQUIRE(vals != nullptr, LTGNN_E_ARG, "spmm_fused_vals: null vals");
    LTGNN_REQUIRE(g == nullptr || vals_stride == 0 || vals_stride == g->nnz, LTGNN_E_ARG,
                  "spmm_fused_vals: vals_stride %lld must be 0 (shared) or nnz", static_cast<long long>(vals_stride));
    LTGNN_REQUIRE(algo == LTGNN_SPMM_AUTO || algo == LTGNN_SPMM_STAGED || algo == LTGNN_SPMM_GATHER, LTGNN_E_ARG,
                  "spmm_fused_vals: unknown algo %d", algo);
    FusedArgs f;
    f.live_out = live_out;
    f.live_in = live_in;
    f.bias = bias;
    f.relu = relu;
    f.drop_p = drop_p;
    f.drop_seed = drop_seed;
    f.gate = gate;
    f.gate_scale = gate_scale;
    f.colsum = colsum;
    f.ws = ws;
    f.vals = vals;
    f.vals_stride = vals_stride;
    return spmm_impl(g, transpose, B, D, X, Y, algo, f, static_cast<cudaStream_t>(stream_), "spmm_fused_vals");
}
