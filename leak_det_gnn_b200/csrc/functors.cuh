// functors.cuh -- loader / epilogue functors shared by the GEMM skeletons (rowgemm.cuh, tgrad.cuh).
#pragma once

#include "common.cuh"
#include "patch.cuh"

namespace ltgnn {
namespace functors {

struct RowLoader {
    const float4* x;
    int k4;
    __device__ __forceinline__ float4 operator()(uint32_t row, int c) const {
        return ptx::ldg_stream(x + static_cast<int64_t>(row) * k4 + c);
    }
};

// bias -> ReLU -> optional gate: y *= (gate[row, col] > 0) ? gate_scale : 0
// (the gate is the output of an upstream ReLU(+dropout): its positivity IS that layer's backward mask)
// The accumulator arrives row-per-thread; 32-column blocks go through the warp's transposition patch so that the
// stores (and gate loads) are 128-byte row segments, 4 rows per instruction, instead of 32 scattered 16-byte pieces.
struct StoreEpilogue {
    float* y;
    const float* bias;
    const float* gate;
    float gate_scale;
    int n;
    int relu;
    template <class Pull>
    __device__ __forceinline__ void operator()(uint32_t row, uint32_t M, int /*var*/, Pull&& pull, const patch::Patch& pt,
                                               int lane, int c_first = 0, int c_stride = 32) const {
        // (c_first, c_stride): the 32-column blocks this warp handles when several warps share the rows
        const bool valid = row < M;
        const uint32_t row0 = row - lane;  // first row of this warp's 32
        const int sub = lane >> 3, ch = lane & 7;
        int c0 = c_first;
        for (; c0 + 32 <= n; c0 += c_stride) {
            float v[32];
            pull(c0, v, 32);
            if (bias) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] += __ldg(bias + c0 + j);
            }
            if (relu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            float4 g[8];
            patch::transpose_out(pt, v, g);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t r = row0 + 4 * k + sub;
                if (r < M) {
                    const size_t o = static_cast<size_t>(r) * n + c0 + 4 * ch;
                    if (gate) {
                        const float4 m = ptx::ldg_stream(reinterpret_cast<const float4*>(gate + o));
                        g[k].x = m.x > 0.f ? g[k].x * gate_scale : 0.f;
                        g[k].y = m.y > 0.f ? g[k].y * gate_scale : 0.f;
                        g[k].z = m.z > 0.f ? g[k].z * gate_scale : 0.f;
                        g[k].w = m.w > 0.f ? g[k].w * gate_scale : 0.f;
                    }
                    *reinterpret_cast<float4*>(y + o) = g[k];
                }
            }
        }
        if (c_first != 0) return;
        for (c0 = n & ~31; c0 < n; c0 += 16) {  // a trailing 16-column block keeps the row-per-thread form
            float v[16];
            pull(c0, v, 16);
            if (valid) chunk(row, c0, v);
        }
    }
    __device__ __forceinline__ void chunk(int64_t row, int c0, float (&v)[16]) const {
        if (bias) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] += __ldg(bias + c0 + j);
        }
        if (relu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (gate) {
            const float4* g = reinterpret_cast<const float4*>(gate + row * n + c0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 m = ptx::ldg_stream(g + j);
                v[4 * j + 0] = m.x > 0.f ? v[4 * j + 0] * gate_scale : 0.f;
                v[4 * j + 1] = m.y > 0.f ? v[4 * j + 1] * gate_scale : 0.f;
                v[4 * j + 2] = m.z > 0.f ? v[4 * j + 2] * gate_scale : 0.f;
                v[4 * j + 3] = m.w > 0.f ? v[4 * j + 3] * gate_scale : 0.f;
            }
        }
        float4* out = reinterpret_cast<float4*>(y + row * n + c0);
#pragma unroll
        for (int j = 0; j < 4; ++j) out[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
};


// Epilogue of the first GCN layer's input-gradient GEMM dX0 = G1 W1 when node init's backward is its only reader: of dX0
// that backward needs just the gated column sums (-> d bias) and the gated sensor rows (-> dz [B, S, D]), so dX0 itself is
// never stored.  Gate exactly as gate_extract_kernel<true> (node_init.cu): live bit ? v * gate_scale : 0, with element j
// of a 32-column slice at bit 8 (j & 3) + (j >> 2) of the word [b][D/32][node].  Works in row form (lane = row): column
// sums accumulate per lane pair (the first round of a shuffle tree per tile: 16 sums per 32 columns, so that two blocks
// fit the kernel's 128 registers) over its rows, and are reduced once at the end (warp_sums: the rest of the tree; the
// kernel then adds its warps in a fixed order into part[cta][D]) -- no atomics, the same bits on every run.
struct GateSumEpilogue {
    float* dz;             // [B, S, n]: gated gradient of the sensor rows
    float* part;           // [CTAs, n]: column-sum partials
    const uint32_t* live;  // [B, n/32, N]
    const int32_t* slot;   // [N]: sensor slot of node i, or -1
    float gate_scale;
    int n;                 // D: 64 or 128 (one or two 32-column blocks per epilogue warp)
    uint32_t N, S;
    struct Cursor {        // per thread, carried over its tiles
        uint32_t b, node;  // its row as (window, node), advanced without a division per tile
        float sum[2][16];  // column sums of its blocks c_first, c_first + c_stride: column j + 16 (lane >> 4)
    };
    __device__ __forceinline__ void start(Cursor& cur, uint32_t row) const {
        cur.b = row / N;
        cur.node = row - cur.b * N;
#pragma unroll
        for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int j = 0; j < 16; ++j) cur.sum[k][j] = 0.f;
    }
    __device__ __forceinline__ void advance(Cursor& cur, uint32_t rows) const {
        cur.node += rows;
        while (cur.node >= N) {
            cur.node -= N;
            ++cur.b;
        }
    }
    template <class Pull>
    __device__ __forceinline__ void operator()(Cursor& cur, bool valid, Pull&& pull, int lane, int c_first,
                                               int c_stride) const {
        const int sl = valid ? __ldg(slot + cur.node) : -1;
        const bool up = lane & 16;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int c0 = c_first + k * c_stride;
            if (c0 >= n) break;
            float v[32];
            pull(c0, v, 32);
            const uint32_t w = valid ? __ldg(live + (static_cast<size_t>(cur.b) * (n >> 5) + (c0 >> 5)) * N + cur.node) : 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (w >> (8 * (j & 3) + (j >> 2))) & 1u ? v[j] * gate_scale : 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float send = up ? v[j] : v[j + 16], keep = up ? v[j + 16] : v[j];
                cur.sum[k][j] += keep + __shfl_xor_sync(0xffffffffu, send, 16);
            }
            if (sl >= 0) {
                float4* o = reinterpret_cast<float4*>(dz + (static_cast<size_t>(cur.b) * S + sl) * n + c0);
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
        }
    }
    // the warp's column sums: out[32 k + l] = column l of block k, summed over the 32 lanes.  Each round of the tree
    // halves the columns a lane holds: it keeps the half selected by its lane bit and adds the partner's copy of it.
    __device__ __forceinline__ void warp_sums(Cursor& cur, int lane, int c_first, int c_stride, float* out) const {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (c_first + k * c_stride >= n) break;
            float* s = cur.sum[k];
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1) {
                const bool up = lane & o;
#pragma unroll
                for (int j = 0; j < o; ++j) {
                    const float send = up ? s[j] : s[j + o], keep = up ? s[j + o] : s[j];
                    s[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                }
            }
            out[32 * k + lane] = s[0];
        }
    }
};

// dX = G W (W [K, N] row-major, N = ep.n) on linear.cu's tensor-memory row GEMM with a GateSumEpilogue; *parts: the number
// of rows of ep.part written (one per CTA).  K a multiple of 32 up to 128; M < 2^31 - 128.
int linear_gate_sums(int device, int64_t M, int K, const float* G, const float* W, const GateSumEpilogue& ep, int* parts,
                     cudaStream_t stream);


// ---- plain row-major operands, optionally two matrices stacked side by side to fill the 128 accumulator rows
struct StackedRows {
    static constexpr bool kRowFast = false;
    const float4* a;  // [M, wa4]
    const float4* b;  // [M, wb4] (columns wa4.. of the stacked operand) or nullptr
    int wa4, wb4;
    __device__ __forceinline__ float4 operator()(uint32_t row, int c) const {
        if (c < wa4) return ptx::ldg_stream(a + static_cast<int64_t>(row) * wa4 + c);
        if (b && c - wa4 < wb4) return ptx::ldg_stream(b + static_cast<int64_t>(row) * wb4 + (c - wa4));
        return make_float4(0.f, 0.f, 0.f, 0.f);
    }
};


// [a | 1 | 0 ...]: operand rows followed by a ones column (its product column is the column sum of the other operand)
struct RowsThenOne {
    static constexpr bool kRowFast = false;
    const float4* a;  // [M, wa4]
    int wa4;
    __device__ __forceinline__ float4 operator()(uint32_t row, int c) const {
        if (c < wa4) return ptx::ldg_stream(a + static_cast<int64_t>(row) * wa4 + c);
        return make_float4(c == wa4 ? 1.f : 0.f, 0.f, 0.f, 0.f);
    }
};

}  // namespace functors
}  // namespace ltgnn
