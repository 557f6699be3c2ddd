/* ltgnn.h -- C ABI of libltgnn.so: sm_100a kernels for the pipe-graph message-passing path
 * of Mateng0228/Leak-det-gnn's leak detector.
 *
 * The reference has NO native code and no FFI; the boundary it offers is the Python
 * operator API of torch_geometric (GCNConv / global_mean_pool) called from
 * models/detector.py:170-218.  Each entry point below names the reference lines it
 * replaces.  INTEGRATION.md shows the ctypes binding and the 3-line reference patch.
 *
 * Conventions
 *   - plain C types only; every function returns an ltgnn_status (0 = ok, <0 = error);
 *     ltgnn_last_error() returns the thread's last message.  No exception crosses the ABI.
 *   - the caller owns every tensor: device pointers to fp32, contiguous, row-major,
 *     16-byte aligned.  The library never allocates activations; it owns only the device
 *     copy of the graph held by a handle (immutable after create -> shareable by threads).
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Calls are
 *     asynchronous on that stream.  Safe to call from any host thread (torch's autograd
 *     worker calls the *_bwd functions).
 *   - activations are [B, N, D]: B independent windows over the SAME N-node graph
 *     (the reference's B-times replicated disjoint union, detector.py:105-114, kept dense).
 *   - there is no CPU fallback: without a CUDA device every compute call fails with
 *     LTGNN_E_CUDA.
 */
#ifndef LTGNN_H_
#define LTGNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LTGNN_VERSION 200 /* major*10000 + minor*100 + patch : 0.2.0 */

typedef enum ltgnn_status {
    LTGNN_OK = 0,
    LTGNN_E_ARG = -1,         /* null pointer / negative size / bad flag                 */
    LTGNN_E_SHAPE = -2,       /* shape not supported by the kernels (see each function)  */
    LTGNN_E_ALIGN = -3,       /* pointer not 16-byte aligned                             */
    LTGNN_E_CUDA = -4,        /* CUDA runtime / driver error (message has the detail)    */
    LTGNN_E_UNSUPPORTED = -5  /* device is not sm_100                                    */
} ltgnn_status;

typedef struct ltgnn_graph* ltgnn_graph_t;

int ltgnn_version(void);
/* Copies the calling thread's last error message (NUL terminated) into buf; returns its length. */
size_t ltgnn_last_error(char* buf, size_t cap);

/* Device-resident dropout seed, for CUDA-graph capture of a TRAINING step (the reference draws fresh dropout masks on
 * every call of train_detector.py:310; a captured launch would otherwise replay the drop_seed it was captured with).
 * After ltgnn_seed_source(w), every dropout-bearing launch made FROM THE CALLING THREAD (ltgnn_node_init_fwd,
 * ltgnn_gcn_layer_fwd, ltgnn_spmm_fused, ltgnn_pipe_head_fwd, ltgnn_tcn_conv_train, ltgnn_gru_dropout) keys its random stream with drop_seed + *w, where the
 * 64-bit device word *w is read when the kernel runs: bump it between replays (on the stream) and every replay draws
 * new masks.  ltgnn_seed_source(NULL) (the default) restores drop_seed alone.  The word must outlive the launches. */
void ltgnn_seed_source(const uint64_t* dev_word);

/* ---- graph handle -------------------------------------------------------------------
 * Replaces the per-forward work of detector.py:195-196 (_batchify_edge_index) and of
 * torch_geometric gcn_norm inside every GCNConv.forward (detector.py:199): the normalised
 * adjacency A_hat of ONE graph is uploaded once, as CSR (row = message target) and as the
 * CSR of A_hat^T ("CSC transpose", row = message source) used by every backward.
 * Host arrays: rowptr int32[N+1], col int32[nnz], val fp32[nnz]; same for t_*.
 * Row entries are consumed in array order (the summation order is part of the contract).
 */
int ltgnn_graph_create(int device, int32_t n_nodes, int32_t nnz,
                       const int32_t* rowptr, const int32_t* col, const float* val,
                       const int32_t* t_rowptr, const int32_t* t_col, const float* t_val,
                       ltgnn_graph_t* out);
int ltgnn_graph_destroy(ltgnn_graph_t g);
int ltgnn_graph_info(ltgnn_graph_t g, int32_t* n_nodes, int32_t* nnz, int32_t* device, int32_t* sm_count);

/* ---- aggregation (SpMM) ---------------------------------------------------------------
 * Y[b,i,:] = sum_k val[k] * X[b, col[k], :]   over row i of A_hat (transpose=0)
 *                                              or of A_hat^T        (transpose=1).
 * transpose=0 replaces GCNConv.propagate (gather x_j, multiply by norm, scatter_add at the
 * target; detector.py:199) for all B windows; transpose=1 is its adjoint, i.e. the
 * backward of propagate wrt x, as a deterministic gather (no atomics).
 * Each entry is one fp32 multiply then one fp32 add in row order -- bit-identical to a
 * sequential scatter-add over PyG's edge list.
 * D must be a multiple of 4.  X and Y must not alias.
 * algo: LTGNN_SPMM_AUTO picks; the others force a kernel (testing / benchmarking).
 */
enum {
    LTGNN_SPMM_AUTO = 0,
    LTGNN_SPMM_STAGED = 1, /* whole-graph feature slices staged in shared memory by TMA    */
    LTGNN_SPMM_GATHER = 2  /* neighbour rows gathered straight from L2 (any graph size)    */
};
int ltgnn_spmm(ltgnn_graph_t g, int transpose, int64_t B, int32_t D, const float* X, float* Y, int algo,
               void* stream);

/* Fused variant of the STAGED kernel (D % 32 == 0 and the graph slice must fit shared memory,
 * otherwise LTGNN_E_SHAPE and the caller composes the unfused pieces):
 *   input gate   (gate != NULL): X is multiplied by (gate > 0 ? gate_scale : 0) BEFORE aggregation --
 *                the backward of an upstream ReLU(+inverted dropout) whose output is `gate`
 *                (detector.py:200-201); colsum[D] (optional) receives the column sums of the gated X
 *                over all B*N rows, i.e. d loss / d bias of that layer.  `ws` must hold
 *                ltgnn_spmm_ws_floats(g) floats.  Deterministic (fixed reduction order).
 *   output epilogue: Y = dropout(relu(A X + bias)); bias NULL / relu 0 / drop_p 0 switch parts off
 *                (GCNConv's `out + bias`, F.relu, nn.Dropout: detector.py:199-201).  Dropout is
 *                inverted dropout from a counter-based Philox stream keyed by drop_seed:
 *                statistically equivalent to torch's, not bit-identical.
 *   1-bit gates: live_out (optional, with the output epilogue) receives one bit per element of Y,
 *                word [b][D/32][N]: bit 8 c + q of word (b, s, i) = (Y[b, i, 32 s + 4 q + c] > 0), c < 4, q < 8
 *                (the order in which a warp vote delivers them).  live_in (instead of
 *                `gate`) feeds such a tensor to the input gate: the backward then streams 1/32 of the
 *                bytes of the float gate.  Graphs up to 1024 nodes.
 */
int64_t ltgnn_spmm_ws_floats(ltgnn_graph_t g);
int ltgnn_spmm_fused(ltgnn_graph_t g, int transpose, int64_t B, int32_t D, const float* X, float* Y,
                     const float* bias, int relu, float drop_p, uint64_t drop_seed, const float* gate,
                     float gate_scale, float* colsum, float* ws, uint32_t* live_out, const uint32_t* live_in,
                     void* stream);

/* ---- weighted adjacency: per-call edge weights (PyG's GCNConv edge_weight) ------------------------------------
 * ltgnn_spmm_fused_vals: ltgnn_spmm_fused (and ltgnn_spmm through algo, with no fused part) with the entry values
 *   read from vals[b * vals_stride + k] instead of the handle: vals [1 or B][nnz] in the order of the chosen orientation
 *   (A_hat's rows for transpose = 0, A_hat^T's for transpose = 1), vals_stride 0 (one set shared by every window) or
 *   nnz.  Column indices and the summation order are the handle's.  algo as in ltgnn_spmm (a fused call honours
 *   LTGNN_SPMM_GATHER).
 * ltgnn_edge_norm_fwd: PyG gcn_norm(edge_index, w, add_self_loops=True) of Bw sets of edge weights w [Bw][E]
 *   (w_stride 0 = one set read for every row of the output, or E): ent_edge [nnz] / t_ent_edge [nnz] give for every
 *   entry of A_hat / A_hat^T the edge it comes from (an appended self loop: the position of the loop it replaces, or -1
 *   for weight 1).  Writes dis [Bw][N] = deg^-1/2 (inf -> 0; deg summed in row order, self loop last), vals [Bw][nnz]
 *   (A_hat order) and t_vals [Bw][nnz] (A_hat^T order), each (dis[src] * w) * dis[dst].
 * ltgnn_edge_norm_bwd: dw [Bw][E] from dvals [Bw][nnz] (A_hat order) through the normalisation above; t_perm [nnz]:
 *   A_hat position of each A_hat^T entry; ddeg: workspace of Bw * N floats.  Edges no entry comes from (a node's
 *   earlier duplicate self loops) get 0.
 * ltgnn_gcn_adj_grad: dA[b][k] (+)= sum_d Gg[b, row_k, d] XW[b, col_k, d] over A_hat's entries (A_hat order): the
 *   gradient of Y = A_hat XW with respect to the entry values.  Gg = G gated as in ltgnn_spmm_fused (gate or live_in,
 *   times gate_scale; both NULL: G itself).  accumulate = 1 adds to dA (several layers sharing one adjacency).
 *   dA_sum (NULL or [nnz]): weights shared by every window -- dA is then scratch, written afresh, and dA_sum (+)= the
 *   sum of its B rows (fixed two-stage order).
 *   D % 4 == 0 and D <= 256.  All four: fixed summation order, no atomics, no allocation, no host synchronisation.
 */
int ltgnn_spmm_fused_vals(ltgnn_graph_t g, int transpose, int64_t B, int32_t D, const float* X, float* Y,
                          const float* vals, int64_t vals_stride, int algo, const float* bias, int relu, float drop_p,
                          uint64_t drop_seed, const float* gate, float gate_scale, float* colsum, float* ws,
                          uint32_t* live_out, const uint32_t* live_in, void* stream);
int ltgnn_edge_norm_fwd(ltgnn_graph_t g, int64_t Bw, int32_t n_edges, const float* w, int64_t w_stride,
                        const int32_t* ent_edge, const int32_t* t_ent_edge, float* dis, float* vals, float* t_vals,
                        void* stream);
int ltgnn_edge_norm_bwd(ltgnn_graph_t g, int64_t Bw, int32_t n_edges, const float* w, int64_t w_stride,
                        const int32_t* ent_edge, const int32_t* t_ent_edge, const int32_t* t_perm, const float* dis,
                        const float* dvals, float* ddeg, float* dw, void* stream);
int ltgnn_gcn_adj_grad(ltgnn_graph_t g, int64_t B, int32_t D, const float* G, const float* gate, const uint32_t* live_in,
                       float gate_scale, const float* XW, float* dA, int accumulate, float* dA_sum, void* stream);

/* ---- explainer edge masks (PyG's MessagePassing.explain_message, GNNExplainer) --------------------------------------
 * ltgnn_edge_mask_fwd: vals [B][nnz] (A_hat order) and t_vals [B][nnz] (A_hat^T order) = base * f, f = mask[b][edge(k)]
 *   for an off-diagonal entry k and 1 for gcn_norm's self loops: the mask scales the message after the normalisation.
 *   mask [1 or B][E] (mask_stride 0 or E); base / t_base [1 or B][nnz] in the two orders (base_stride 0 or nnz), e.g.
 *   ltgnn_edge_norm_fwd's vals / t_vals, or both NULL for the handle's own values.  ent_edge / t_ent_edge as in
 *   ltgnn_edge_norm_fwd.
 * ltgnn_edge_mask_bwd: from dvals [B][nnz] (A_hat order): dmask [B][E] = dvals[k] * base[k] at edge(k) (0 for edges no
 *   entry comes from: input self loops); dbase (NULL, or [B][nnz] with per-call base) = dvals * f.  dmask_sum /
 *   dbase_sum (NULL or [E] / [nnz]): a mask / base shared by every window -- the row results are then scratch and the
 *   sums of their B rows (fixed two-stage order) are written there.
 * ltgnn_explain_step: one GNNExplainer epoch (PyG 2.x, edge_mask_type='object', edge_reduction='sum') on the mask
 *   logits m [B][E] of s = sigmoid(m) [B][E], from g = d loss / d s [B][E]:
 *     dm = g s(1-s) + hard [edge_size + edge_ent / n_hard[b] * dH/ds] s(1-s),
 *     H(s) = -s log(s + 1e-15) - (1-s) log(1-s + 1e-15), the entropy term 0 for a window without hard entries;
 *   then torch.optim.Adam (lr, beta1, beta2, eps; state exp_avg / exp_avg_sq [B][E]; *step = steps taken, read and then
 *   incremented on the device, so a captured epoch replays with the right bias corrections) and the new m and s.
 *   record = 1 (epoch 0): no regulariser; writes hard [B][E] (bytes, dm != 0) and n_hard [B] (int32 counts).
 *   All three: no atomics, no allocation, no host synchronisation.
 */
int ltgnn_edge_mask_fwd(ltgnn_graph_t g, int64_t B, int32_t n_edges, const float* mask, int64_t mask_stride,
                        const float* base, const float* t_base, int64_t base_stride, const int32_t* ent_edge,
                        const int32_t* t_ent_edge, float* vals, float* t_vals, void* stream);
int ltgnn_edge_mask_bwd(ltgnn_graph_t g, int64_t B, int32_t n_edges, const float* mask, int64_t mask_stride,
                        const float* base, int64_t base_stride, const int32_t* ent_edge, const float* dvals, float* dmask,
                        float* dmask_sum, float* dbase, float* dbase_sum, void* stream);
int ltgnn_explain_step(int device, int64_t B, int32_t E, const float* g, float* m, float* s, float* exp_avg,
                       float* exp_avg_sq, uint8_t* hard, int32_t* n_hard, int32_t* step, double lr, double beta1,
                       double beta2, double eps, float edge_size, float edge_ent, int record, void* stream);

/* ---- PGExplainer's edge network (PyG 2.x, torch_geometric/explain/algorithm/pg_explainer.py) ----------------
 * The MLP Linear(2D, 64) -> ReLU -> Linear(64, 1) on [z[src] | z[dst]], factored per node: pq [B*N][128] = [P | Q]
 * = z [W1a; W1b]^T (one ltgnn_linear), then per edge e of window b (src / dst [E] int32 node indices)
 *   pre = (P[b, src[e]] + Q[b, dst[e]]) + b1,  logit = w2 . relu(pre) + *b2   (b1, w2 [64] and b2 [1] on the device).
 * ltgnn_pg_edge_fwd: inv_t NULL (explaining): mask [B][E] = sigmoid(logit), nothing else written.
 *   inv_t (device scalar 1 / T, training): the concrete sample s [B][E] = (log eps - log(1 - eps) + logit) * (1 / T),
 *   eps = (1 - 2 bias) U + bias, U in [0, 1) from Philox keyed by seed (+ the ltgnn_seed_source word when one is set)
 *   and the edge's index b * E + e; mask = sigmoid(s); gate [B][E][2] uint32: bit l of word j = (pre of unit 2l + j
 *   > 0); uniform (NULL or [B][E]) receives U.  bias in [0, 0.5]; 0.5 is noise-free.
 * ltgnn_pg_edge_bwd: from dmask [B][E] (the gradient at fwd's mask) and fwd's mask, gate and inv_t:
 *   dlogit = dmask s(1 - s) / T,  gh[u] = dlogit w2[u] [pre_u > 0];  R [B*N][128]: R[b, n, :64] = sum of gh over the
 *   edges with src = n, R[b, n, 64:] over those with dst = n, in ascending edge order (out_ptr / out_edge [N+1] / [E]:
 *   the edges by source, in_ptr / in_edge by target, each ascending) -- d pq; dparams [129] = d b1 [64] | d w2 [64] |
 *   d b2 (relu(pre) recomputed in the forward's order), per-CTA partials (ws: ltgnn_pg_edge_bwd_ws_floats floats)
 *   summed in a fixed order.  Both: no atomics, no allocation, no host synchronisation; any N (gathers through L2).
 */
int ltgnn_pg_edge_fwd(int device, int64_t B, int32_t N, int32_t E, const int32_t* src, const int32_t* dst,
                      const float* pq, const float* b1, const float* w2, const float* b2, const float* inv_t, float bias,
                      uint64_t seed, float* mask, float* s, uint32_t* gate, float* uniform, void* stream);
int64_t ltgnn_pg_edge_bwd_ws_floats(int device);
int ltgnn_pg_edge_bwd(int device, int64_t B, int32_t N, int32_t E, const int32_t* out_ptr, const int32_t* out_edge,
                      const int32_t* in_ptr, const int32_t* in_edge, const int32_t* dst, const float* pq, const float* b1,
                      const float* w2, const float* inv_t, const float* mask, const float* dmask, const uint32_t* gate,
                      float* R, float* dparams, float* ws, void* stream);

/* ---- dense row-wise layer on tensor cores --------------------------------------------------
 * Y[M,N] = gate( act( X[M,K] op(W) + bias[N] ) )
 *   op(W) = W^T with W [N,K] row-major (w_transposed = 0, torch.nn.Linear layout)
 *         = W   with W [K,N] row-major (w_transposed = 1; the input-gradient GEMM dX = dY W)
 *   bias may be NULL; relu = 0/1;
 *   gate (NULL or [M,N]): Y *= gate > 0 ? gate_scale : 0 -- the backward of an upstream
 *   ReLU(+inverted dropout) whose OUTPUT is `gate` (detector.py:189-190,200-201).
 * tcgen05 3xTF32 with fp32 accumulation in tensor memory: fp32-faithful (the reference runs these in
 * full fp32: GCNConv.lin detector.py:199; NoLeakHead detector.py:94-99).
 * K multiple of 32 (<= 256), N multiple of 16 (<= 256), operands must fit shared memory.
 */
int ltgnn_linear(int device, int64_t M, int32_t K, int32_t N, const float* X, const float* W, int w_transposed,
                 const float* bias, int relu, const float* gate, float gate_scale, float* Y, void* stream);

/* ---- weight gradient of a row-wise linear map ---------------------------------------------
 * dW[Do,Di] (+)= sum over the M rows of G[row,:]^T X[row,:]   (accumulate = 0/1)
 * Replaces autograd's grad_weight of GCNConv.lin (detector.py:199) over the B*N node rows.
 * (Do/8)*(Di/8) must divide 256 (64x64, 128x128, 64x128, ...).  ws: ltgnn_wgrad_ws_floats() floats.
 * Deterministic: per-CTA partials are added in a fixed order.
 */
int64_t ltgnn_wgrad_ws_floats(int device, int32_t Do, int32_t Di);
int ltgnn_wgrad(int device, int64_t M, int32_t Do, int32_t Di, const float* G, const float* X, float* dW,
                int accumulate, float* ws, void* stream);

/* ---- node-feature initialisation (detector.py:178-190) and its backward ---------------------
 * fwd: X0[b,i,:] = dropout(relu(W[:, :ds] h + W[:, ds] m + bias)), (h, m) = (hs[b, slot[i], :], 1) for a
 *      sensor node (slot[i] >= 0) and (0, 0) otherwise.  hs [B,S,ds]; W [D, ds+1] (sensor_to_node.weight);
 *      slot int32[N] on the device.  Never builds the zero-padded (B,N,ds+1) tensor.
 * bwd: gate = (X0 > 0) * gate_scale applied to dX0; dhs [B,S,ds], dW [D, ds+1], dbias [D].
 *      ws: ltgnn_node_init_ws_floats() floats, 16-byte aligned.  Deterministic.
 *      live_out (fwd, optional, D % 32 == 0) / live_in (bwd, instead of X0): the gate as 1 bit per element,
 *      word [b][D/32][N] as in ltgnn_spmm_fused.
 */
int ltgnn_node_init_fwd(int device, int64_t B, int32_t N, int32_t S, int32_t ds, int32_t D, const float* hs,
                        const int32_t* slot, const float* W, const float* bias, float drop_p, uint64_t drop_seed,
                        float* X0, uint32_t* live_out, void* stream);
int64_t ltgnn_node_init_ws_floats(int device, int64_t B, int32_t S, int32_t ds, int32_t D);
int ltgnn_node_init_bwd(int device, int64_t B, int32_t N, int32_t S, int32_t ds, int32_t D, const float* hs,
                        const int32_t* slot, const float* W, const float* dX0, const float* X0,
                        const uint32_t* live_in, float gate_scale, float* dhs, float* dW, float* dbias, float* ws,
                        void* stream);
/* bwd_from_layer: the same three gradients for dX0 = G1 W1, the input gradient of the first GCN layer -- G1 [B,N,K] its
 *      aggregated output gradient, W1 [K, D] its weight (GCNConv.lin.weight) -- without forming dX0: the tensor-core GEMM
 *      gates it with live_in (required) in its epilogue and keeps only the column sums and the sensor rows.  dhs and dW
 *      carry the bits of ltgnn_node_init_bwd on the same dX0; dbias differs by summation order.  K a multiple of 32 up to
 *      128, D 64 or 128, B*N < 2^31 - 128.  ws: ltgnn_node_init_ws_floats() floats.  Deterministic.
 */
int ltgnn_node_init_bwd_from_layer(int device, int64_t B, int32_t N, int32_t S, int32_t ds, int32_t D, int32_t K,
                                   const float* hs, const int32_t* slot, const float* W, const float* G1,
                                   const float* W1, const uint32_t* live_in, float gate_scale, float* dhs, float* dW,
                                   float* dbias, float* ws, void* stream);

/* ---- one GCN layer forward as ONE kernel (detector.py:198-201: conv -> relu -> dropout) ---------
 * Y = dropout(relu(A_hat (X W^T) + bias)) with the dense product on tcgen05 and never written to HBM: the window's
 * X W^T slice goes from tensor memory to shared memory and is aggregated there.  X [B,N,K], W [D,K] (torch Linear
 * layout, GCNConv.lin.weight), bias [D] or null, Y [B,N,D]; dropout / live_out as in ltgnn_spmm_fused.  Bit-identical to
 * ltgnn_linear followed by ltgnn_spmm_fused.  ltgnn_gcn_layer_supported: 1 if the kernel takes (graph, K, D) -- K a
 * multiple of 32 up to 128, D a multiple of 32, at most 896 nodes, the slice of the graph fits shared memory.
 */
int ltgnn_gcn_layer_supported(ltgnn_graph_t g, int32_t K, int32_t D);
int ltgnn_gcn_layer_fwd(ltgnn_graph_t g, int64_t B, int32_t K, int32_t D, const float* X, const float* W,
                        const float* bias, int relu, float drop_p, uint64_t drop_seed, float* Y, uint32_t* live_out,
                        void* stream);

/* ---- read-out heads (detector.py:76-102, 204-216) ---------------------------------------------
 * pipe_head_fwd: for every window b and class pipe p with end nodes ends[p] = (u, v):
 *      hidden = dropout(relu(W1 [x_u, x_v, |x_u - x_v|] + b1)),   W1 [H, 3D] (edge_head.mlp.0.weight)
 *      part[b*P + p] = sum over the H hidden units of hidden * w2
 *   so pipe_logit = part + b2 (edge_head.mlp.3).  hpost (optional; logical [Mp, H], Mp = B*P rounded up to 128,
 *   stored blocked-32 as [Mp/32][H/4][32][4]) receives `hidden` for the backward.  X [B,N,D] node states; ends int32 [P,2] on the device.  D = 64, H = 128.
 *   hmask (optional; uint32 [Mp, H/32]) receives the 1-bit form of hidden > 0: bit 31 - j % 32 of word j / 32 of a row.
 *   hsign (optional; uint32 [Mp, 4]) receives sign(x_u - x_v) as two bits per feature: words 2 g / 2 g + 1 of a row hold
 *   the `> 0` / `< 0` bits of features 32 g .. 32 g + 31 (feature j at bit 31 - j % 32).  The backward needs both.
 * pipe_head_bwd_dx: dX[b, i, :] = dpooled[b, :] / N (the mean-pool gradient; dpooled may be null) + the input gradient
 *   of the pipe head given dlogit [B*P], summed over the pipe ends at node i -- the entries of the incidence lists
 *   inc_ptr int32 [N+1], inc int32 [2P] (entry = pipe << 1 | end, grouped by node) -- in a fixed order (the even and
 *   the odd positions of a node's list as two partial sums): a gather, bit-reproducible, dX is written exactly once.  The node states are not read: hmask and hsign carry everything the forward knew.
 *   ws: ltgnn_pipe_head_dx_ws_floats(device, N, P) floats.
 * mean_pool_fwd / mean_pool_bwd_fill: pooled[b,:] = mean_i X[b,i,:];  dX[b,i,:] = dpooled[b,:] / N.
 */
int ltgnn_pipe_head_fwd(int device, int64_t B, int32_t N, int32_t P, int32_t D, int32_t H, const float* X,
                        const int32_t* ends, const float* W1, const float* b1, const float* w2, float drop_p,
                        uint64_t drop_seed, float* part, float* hpost, uint32_t* hmask, uint32_t* hsign, void* stream);
int64_t ltgnn_pipe_head_dx_ws_floats(int device, int32_t N, int32_t P);
int ltgnn_pipe_head_bwd_dx(int device, int64_t B, int32_t N, int32_t P, int32_t D, int32_t H, const int32_t* inc_ptr,
                           const int32_t* inc, const float* W1, const float* w2, const uint32_t* hmask,
                           const uint32_t* hsign, const float* dlogit, float gate_scale, const float* dpooled, float* ws,
                           float* dX, void* stream);
/* ---- the pipe head for node widths the fused kernels above do not take (csrc/heads_wide.cu) -------------------------
 * Same reference lines (detector.py:76-88,204-211) at D = 128 (BASELINE configs[4]): the features are materialised,
 * F [3][B*P][D] = h_u | h_v | |h_u - h_v|; Linear(3D, H) + ReLU runs as the three-tap gathered-row GEMM ltgnn_tcn_conv
 * (tap t reads row t*B*P + m of F against W1[:, tD:(t+1)D]); these four streaming kernels do the rest.
 *   ltgnn_pipe_feat_fwd   X [B,N,D], ends int32 [P,2] -> F
 *   ltgnn_head_out_fwd    h [M,H] = relu(pre) -> (in place) hd = dropout(h);  part[m] = sum_j hd[m,j] w2[j]
 *   ltgnn_head_out_bwd    gq[m,j] = hd[m,j] > 0 ? dlogit[m] scale : 0;  dh = gq * w2;  cs[j] = sum_m gq[m,j];
 *                         ws: ltgnn_head_out_ws_floats(device, H) floats
 *   ltgnn_head_wide_finish  T [3][H][D] = gq^T F[t] (three ltgnn_wgrad_tc products) -> dW1 [H,3D] = w2[j] T,
 *                         db1 = w2 * cs,  dw2[j] = b1[j] cs[j] + sum W1[j,:] . T[:,j,:]  (the hidden layer is linear in
 *                         W1, b1 under the gate, so dw2 needs no pass over the hidden activations)
 *   ltgnn_pipe_feat_bwd   dX[b,n] = dpooled[b]/N (if given) + sum over the pipe ends at n, in the order of inc
 *                         (inc_ptr int32 [N+1], inc int32 [2P]: pipe << 1 | end), of  end u: dF0[m] + s dF2[m],
 *                         end v: dF1[m] - s dF2[m],  s = sign(x_u - x_v).  dX written once; deterministic.
 */
int ltgnn_pipe_feat_fwd(int device, int64_t B, int32_t N, int32_t P, int32_t D, const float* X, const int32_t* ends,
                        float* F, void* stream);
int ltgnn_head_out_fwd(int device, int64_t M, int32_t H, float* h, const float* w2, float drop_p, uint64_t drop_seed,
                       float* part, void* stream);
int64_t ltgnn_head_out_ws_floats(int device, int32_t H);
int ltgnn_head_out_bwd(int device, int64_t M, int32_t H, const float* hd, const float* w2, const float* dlogit, float scale,
                       float* dh, float* gq, float* cs, float* ws, void* stream);
int ltgnn_head_wide_finish(int device, int32_t H, int32_t D, const float* T, const float* W1, const float* b1,
                           const float* w2, const float* cs, float* dW1, float* db1, float* dw2, void* stream);
int ltgnn_pipe_feat_bwd(int device, int64_t B, int32_t N, int32_t P, int32_t D, const float* X, const int32_t* ends,
                        const int32_t* inc_ptr, const int32_t* inc, const float* dF, const float* dpooled, float* dX,
                        void* stream);

int ltgnn_mean_pool_fwd(int device, int64_t B, int32_t N, int32_t D, const float* X, float* pooled, void* stream);
int ltgnn_mean_pool_bwd_fill(int device, int64_t B, int32_t N, int32_t D, const float* dpooled, float* dX, void* stream);

/* ---- weight gradients on tensor cores (tcgen05, MN-major operands, 3xTF32) ---------------------
 * wgrad_tc: same contract as ltgnn_wgrad for Do in {64, 128}, Di a multiple of 32 (<= 256); ~3x faster.
 * pipe_head_bwd_w: dW1 [H, 3D] = dpre^T [x_u, x_v, |x_u - x_v|] and db1 [H] = column sums of dpre, where
 *   dpre[r, j] = dlogit[r] * w2[j] * (hidden[r, j] > 0 ? gate_scale : 0), with the gate read as 1 bit per unit from
 *   hmask (ltgnn_pipe_head_fwd) and the operands formed on the fly; dw2 [H] = sum_r dlogit[r] * hidden[r, :] is
 *   recovered from the same accumulators (hidden is linear in W1, b1 under the gate), so the forward need not save
 *   the hidden activations.
 * ws: ltgnn_tgrad_ws_floats(device, Di) floats; pipe head: ltgnn_pipe_head_ws_floats(device).  Deterministic.
 */
int64_t ltgnn_tgrad_ws_floats(int device, int32_t No);
int ltgnn_wgrad_tc(int device, int64_t M, int32_t Do, int32_t Di, const float* G, const float* X, float* dW,
                   int accumulate, float* ws, void* stream);
int ltgnn_pipe_head_bwd_w(int device, int64_t B, int32_t N, int32_t P, int32_t D, int32_t H, const float* X,
                          const int32_t* ends, const float* W1, const float* b1, const float* w2, const uint32_t* hmask,
                          const float* dlogit, float gate_scale, float* dW1, float* db1, float* dw2, float* ws,
                          void* stream);
int64_t ltgnn_pipe_head_ws_floats(int device);

/* ---- frozen TCN predictor, one dilated causal convolution over gathered rows (SURVEY 8f rank 1) ---------
 * Reference: models/predictor.py:17-52 (CausalConv1d -> LayerNorm -> ReLU, residual add), evaluated only on the
 * (window, position) rows the last time step depends on (models/utils.py:169-216 reads nothing else).
 *   Y[m, :] = [res[res_row[m], :] +] relu(LayerNorm(bias + sum_tap X[src[tap * M + m], :] W[tap]^T))
 * X [x_rows, C], src int32 [taps, M] (-1 = zero row: the left padding), W [taps, C, C] (tap 0 = the oldest input;
 * torch's conv weight permuted (2, 0, 1)), bias / gamma / beta [C] (gamma = beta = null: no LayerNorm), res [r_rows, C]
 * with res_row int32 [M] or both null, Y [M, C].  C = 128.  tcgen05, 3xTF32; the weight is split into TF32 hi / lo and laid
 * out as shared-memory operand stages once per call (into ws: ltgnn_tcn_ws_floats(taps) floats) and streamed by bulk copies.
 * res_row[m] = -1 adds nothing to row m (the input gradient below uses it for block-input rows no output row keeps).
 */
int64_t ltgnn_tcn_ws_floats(int32_t taps);
int ltgnn_tcn_conv(int device, int64_t M, int32_t C, int32_t taps, const float* X, const int32_t* src, const float* W,
                   const float* bias, const float* gamma, const float* beta, float eps, int relu, const float* res,
                   const int32_t* res_row, float* Y, float* ws, void* stream);

/* ---- training of the TCN predictor on the same cone (reference train_predictor.py; csrc/tcn_train.cu) ---------
 * The loss reads only the last time step (predictor.py:80), so every parameter gradient depends only on the cone rows.
 * tcn_conv_train: the forward of one training convolution of a TCN block,
 *     Y[m, :] = [res[res_row[m], :] +] dropout(relu(LayerNorm(Z[m, :]))),  Z = bias + sum_tap X[src[tap * M + m], :] W[tap]^T
 *   with everything as in ltgnn_tcn_conv (gamma, beta required).  Also writes Z [M, C] (pre-norm rows), stats [M, 2]
 *   (mean, rstd per row) and live uint32 [M, 4]: bit b of word w = (output channel 32 w + b is > 0 after ReLU and
 *   dropout).  Dropout is inverted dropout from Philox keyed by drop_seed (+ the ltgnn_seed_source word); drop_p = 0
 *   gives Y bit-identical to ltgnn_tcn_conv with relu = 1.  ws: ltgnn_tcn_ws_floats(taps) floats.
 * tcn_ln_bwd: dZ = the LayerNorm backward of g = dY * live * scale (scale = 1 / (1 - drop_p)) from Z, stats and gamma;
 *   dprm [3, C] = column sums over the M rows of g * x_hat (d gamma), g (d beta) and dZ (d bias).  Fixed-order partials:
 *   deterministic.  ws: ltgnn_tcn_ln_bwd_ws_floats(device) floats.
 * Input gradient of a training convolution: ltgnn_tcn_conv with X = dZ, src = inv, W[tap] = W[tap]^T, a zero bias, no
 *   LayerNorm, relu = 0, where inv int32 [taps, x_rows] is the inverse index: inv[tap * x_rows + r] = the m with
 *   src[tap * M + m] = r, or -1 if there is none (it must be unique: a tap's row map is injective).  A block input also
 *   receives the block output's gradient on the rows it keeps: res = dY of the block, res_row = the kept-row inverse.
 * tcn_wgrad: dW [taps, C, C], dW[tap] = dZ^T X[src[tap]] (row -1 of X = zeros), summed over the M rows on the tensor cores
 *   (3xTF32, fp32 per-chunk flush; X rows gathered while loaded).  ws: ltgnn_tgrad_ws_floats(device, C) floats.
 *   Deterministic.  C = 128 for all three.
 */
int ltgnn_tcn_conv_train(int device, int64_t M, int32_t C, int32_t taps, const float* X, const int32_t* src, const float* W,
                         const float* bias, const float* gamma, const float* beta, float eps, const float* res,
                         const int32_t* res_row, float drop_p, uint64_t drop_seed, float* Y, float* Z, float* stats,
                         uint32_t* live, float* ws, void* stream);
int64_t ltgnn_tcn_ln_bwd_ws_floats(int device);
int ltgnn_tcn_ln_bwd(int device, int64_t M, int32_t C, const float* dY, const uint32_t* live, const float* Z,
                     const float* stats, const float* gamma, float scale, float* dZ, float* dprm, float* ws, void* stream);
int ltgnn_tcn_wgrad(int device, int64_t M, int32_t C, int32_t taps, const float* dZ, const float* X, const int32_t* src,
                    float* dW, float* ws, void* stream);

/* ---- shared per-sensor GRU encoder (detector.py:28-73; SURVEY 8f rank 2) -----------------------
 * Sequence q = b*S + s has input [r[b,t,s], tf[b,t,0..F)] at step t (the reference's cat([rr, tf]) order);
 * weights in torch.nn.GRU layout (gate order r, z, n): w_ih [3H, 1+F], w_hh [3H, H], b_ih, b_hh [3H].  H = 64
 * (H = 128: ltgnn_gru_sensor_fwd below).
 * gru_fwd:       h_last [B*S, H] = hidden state after step L-1 (h_0 = 0).  For training also pass hseq (every state,
 *                logical [L*Qp, H]) and gates (r, z, n; logical [L*Qp, 3H]), Qp = B*S rounded up to 128, both in the
 *                kernels' blocked-32 layout [rows/32][W/4][32][4]; NULL otherwise.
 *                State lives in tensor memory; recurrent + input GEMM fused on tcgen05 (3xTF32).
 * gru_bwd_dg_hn: back-propagation through time given dh_last [B*S, H] and the forward's hseq and gates3 (r, z, n):
 *                writes dG (blocked-32, [L*Qp, 4H]), the gradient wrt the four pre-activation groups
 *                (r, z, W_hn h + b_hn, W_in x + b_in).  W_hn h_{t-1} + b_hn is rebuilt per step by one 64-column
 *                tensor-core GEMM instead of being saved: 8.75 GB less written and read at B*S = 118 784, L = 288.
 * gru_bwd_w:     dBfused [4H, 96] = sum_(t,q) dG^T [h_{t-1} | x | tf | 1 | 0]: columns 0..H-1 are d w_hh, H..H+F
 *                d w_ih, H+F+1 the bias gradients (rows: r, z, hn-part, in-part).  ws: ltgnn_gru_ws_floats() floats.
 * gru_bwd_dx:    the gradient wrt the inputs from gru_bwd_dg_hn's dG: dx[q,t,:] = dG_r W_ih[r] + dG_z W_ih[z] + dG_in W_ih[n]
 *                ([1+F] per sequence and step, fp32 FMAs in a fixed order).  dr [B, L, S] = dx[:, :, 0] at (b, t, s);
 *                dxt [B, L, S, F] = dx[:, :, 1..F] per sequence, which the caller sums over s for d tf.  Either output may
 *                be NULL (not both; dxt needs F > 0).  H = 64 and 1 + F <= 31 (else LTGNN_E_SHAPE); dG 16-byte aligned,
 *                w_ih, dr and dxt 4-byte aligned (else LTGNN_E_ALIGN).  No atomics, allocation or host synchronisation.
 */
int ltgnn_gru_fwd(int device, int64_t B, int32_t L, int32_t S, int32_t F, int32_t H, const float* r, const float* tf,
                  const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, float* h_last,
                  float* hseq, float* gates, void* stream);
int ltgnn_gru_bwd_dg_hn(int device, int64_t Q, int32_t L, int32_t H, const float* w_hh, const float* b_hh,
                        const float* gates3, const float* hseq, const float* dh_last, float* dG, void* stream);
int64_t ltgnn_gru_ws_floats(int device);
int ltgnn_gru_bwd_w(int device, int64_t B, int32_t L, int32_t S, int32_t F, int32_t H, const float* r, const float* tf,
                    const float* hseq, const float* dG, float* dBfused, float* ws, void* stream);
int ltgnn_gru_bwd_dx(int device, int64_t B, int32_t L, int32_t S, int32_t F, int32_t H, const float* w_ih,
                     const float* dG, float* dr, float* dxt, void* stream);

/* ---- one layer of the GRU normal-state predictor (predictor.py:84-111), forward only (csrc/gru_pred.cu) -------------
 * Q sequences of L steps, torch.nn.GRU equations and gate order (r, z, n), h_0 = 0.  The input projection is computed
 * beforehand (ltgnn_linear, one launch per gate group):
 *   gx [3][Q*L][H]: gx[g][q*L + t] = x_(q,t) W_ih[g]^T + b_ih[g], plus b_hh[g] for g = r, z (not for n)
 * w_hh [3H, H] and b_hn = b_hh[2H:3H] in torch layout.  Writes h_last [Q, H] (the state after step L-1) and, if hseq is
 * not NULL, every state: hseq [Q, L, H] (the next layer's input).  H = 128 only (else LTGNN_E_SHAPE); Q, L > 0 and
 * gx, w_hh, b_hn, h_last non-NULL (else LTGNN_E_ARG); gx, w_hh, hseq, h_last 16-byte aligned (else LTGNN_E_ALIGN).
 * Clusters of 4 CTAs per 128 sequences exchange the state through distributed shared memory; 3xTF32 tcgen05 products.
 * Deterministic, no allocation or host synchronisation: capturable into a CUDA graph.
 */
int ltgnn_gru_layer_fwd(int device, int64_t Q, int32_t L, int32_t H, const float* gx, const float* w_hh, const float* b_hn,
                        float* hseq, float* h_last, void* stream);
/* gru_layer_fwd_windows: ltgnn_gru_layer_fwd on Q windows that share one input projection (overlapping windows of a
 * series, e.g. every window of a segment): gx [3][gx_rows][H] is projected once per series row, and window q reads its
 * step-t row at row_base[q] + t (int32 [Q]) instead of q*L + t.  h_last [Q, H] and hseq [Q, L, H] are the planar form's,
 * bit for bit.  The caller guarantees 0 <= row_base[q] and row_base[q] + L <= gx_rows (the entry point does not read
 * device memory).  H = 128 only, Q < 2^31 - 128 and gx_rows < 2^31 (else LTGNN_E_SHAPE); Q, L > 0, gx_rows >= L and gx,
 * row_base, w_hh, b_hn, h_last non-NULL (else LTGNN_E_ARG); gx, w_hh, hseq, h_last 16-byte aligned and row_base 4-byte
 * aligned (else LTGNN_E_ALIGN).  Deterministic, no allocation or host synchronisation: capturable into a CUDA graph.
 */
int ltgnn_gru_layer_fwd_windows(int device, int64_t Q, int32_t L, int32_t H, const float* gx, int64_t gx_rows,
                                const int32_t* row_base, const float* w_hh, const float* b_hn, float* hseq, float* h_last,
                                void* stream);

/* ---- training of the GRU normal-state predictor (predictor.py:84-111, train_predictor.py), same file ----------------
 * gru_layer_fwd_train: ltgnn_gru_layer_fwd (same kernel, same h_last and hseq bit for bit) that also stores every step's
 *   gates [4][Q*L][H] = r | z | n | hn, hn = W_hn h_{t-1} + b_hn, in gx's planar layout.  hseq and gates are required.
 * gru_layer_bwd: back-propagation through time of one layer from what gru_layer_fwd_train saved.  dh_last [Q, H] is the
 *   gradient of h_last (the top layer's, from the head) and dh_seq [Q*L, H] the gradient of every state (a lower layer's,
 *   from the layer above; its row L-1 covers h_last); either may be NULL, not both.  Writes
 *   dG [4][Q*L][H] = dr_pre | dz_pre | dn_pre | dhn (gradients of the r, z pre-activations, of gx_n and of hn), from which
 *   the weight gradients are ltgnn_wgrad_tc products: dW_hh rows r, z, n = planes 0, 1, 3 against h_{t-1}, dW_ih rows
 *   r, z, n = planes 0, 1, 2 against the layer input.  Clusters of 4 CTAs: each multiplies its own 96 gate columns by its
 *   96 x 128 slice of W_hh (3xTF32 tcgen05) and sends its peers their 32-column blocks of the partial through distributed
 *   shared memory; the owner adds the four partials in rank order.  Deterministic, capturable into a CUDA graph.
 * gru_dropout: the inter-layer dropout of nn.GRU in train mode, y [M, H] = x * keep / (1 - drop_p), keep from Philox keyed
 *   by drop_seed (+ the ltgnn_seed_source word); live uint32 [M, H/32]: bit b of word w = unit 32 (w % (H/32)) + b kept.
 *   drop_p = 0 copies x bit for bit (every bit set).
 * gru_dropout_bwd: dx [M, H] = (dy[0] + ... + dy[n_parts - 1]) * keep / (1 - drop_p), dy [n_parts][M][H] added in index
 *   order (the input gradient of the layer above, one part per gate group), keep read from live (NULL: no dropout).
 * All four: H = 128 only (else LTGNN_E_SHAPE); Q, L, M > 0, drop_p in [0, 1), 1 <= n_parts <= 4 and the required tensors
 * non-NULL (else LTGNN_E_ARG); tensors 16-byte aligned (else LTGNN_E_ALIGN); sm_100 (else LTGNN_E_UNSUPPORTED).
 */
int ltgnn_gru_layer_fwd_train(int device, int64_t Q, int32_t L, int32_t H, const float* gx, const float* w_hh,
                              const float* b_hn, float* hseq, float* h_last, float* gates, void* stream);
int ltgnn_gru_layer_bwd(int device, int64_t Q, int32_t L, int32_t H, const float* w_hh, const float* gates,
                        const float* hseq, const float* dh_last, const float* dh_seq, float* dG, void* stream);
int ltgnn_gru_dropout(int device, int64_t M, int32_t H, const float* x, float drop_p, uint64_t drop_seed, float* y,
                      uint32_t* live, void* stream);
int ltgnn_gru_dropout_bwd(int device, int64_t M, int32_t H, const float* dy, int32_t n_parts, const uint32_t* live,
                          float drop_p, float* dx, void* stream);

/* ---- the shared sensor GRU encoder at hidden 128 (detector.py:28-73 with sensor_hidden = 128), same file -------------
 * gru_sensor_fwd: the cluster recurrence of ltgnn_gru_layer_fwd / _fwd_train with the encoder's input formed in the
 *   kernel.  Sequence q = b*S + s has input [r[b,t,s], tf[b,t,:]] at step t; the time features are the same for the S
 *   sensors of a window, so their projection is computed once per (window, step) beforehand (ltgnn_linear):
 *     tproj [3][B*L][H]: tproj[g][b*L + t] = tf[b,t,:] W_ih[g][:, 1:]^T + b_ih[g], plus b_hh[g] for g = r, z (not n)
 *   and the gate thread adds w_r[g] * r[b,t,s], w_r [3][H] = W_ih[:, 0] (the residual column).  One call runs the
 *   sequences q0 .. q0+Q-1 of the B*S (so a caller can run them in slabs); its outputs are those of the planar form for
 *   these Q sequences, local sequence i = sequence q0 + i: h_last [Q, H]; if hseq is not NULL, hseq [Q*L, H]; if gates is
 *   not NULL (training: hseq required), gates [4][Q*L][H] = r | z | n | hn, which ltgnn_gru_layer_bwd reads unchanged.
 *   The weight gradients are the ltgnn_wgrad_tc products of ltgnn_gru_layer_bwd's comment, the layer input being
 *   [r | tf | 1] per row.  H = 128 only and B*S < 2^31 - 128 (else LTGNN_E_SHAPE); B, L, S, Q > 0, q0 >= 0,
 *   q0 + Q <= B*S and r, tproj, w_r, w_hh, b_hn, h_last non-NULL (else LTGNN_E_ARG); tproj, w_r, w_hh, hseq, h_last,
 *   gates 16-byte aligned (else LTGNN_E_ALIGN).  Deterministic, no allocation or host synchronisation: capturable.
 * gru_resident_tiles: *tiles = how many 128-sequence tiles (4-CTA clusters) of these recurrences the device runs at
 *   once (cudaOccupancyMaxActiveClusters): one wave.  Callers size their slabs in whole waves.
 * gru_sensor_bwd_dx: ltgnn_gru_bwd_dx for the sequences q0 .. q0+Q-1 of the B*S, from ltgnn_gru_layer_bwd's dG
 *   [4][Q*L][H] of those sequences (input planes r, z, n): writes their elements of dr [B, L, S] and dxt [B, L, S, F].
 *   Every element is written by one thread whatever the slab split, so the caller's sum of dxt over s (after the last
 *   slab) does not depend on it.  H = 128 and 1 + F <= 31 (else LTGNN_E_SHAPE); B, L, S, Q > 0, F >= 0, q0 >= 0,
 *   q0 + Q <= B*S, w_ih and dG non-NULL, dr or dxt non-NULL, dxt only with F > 0 (else LTGNN_E_ARG); alignment as
 *   ltgnn_gru_bwd_dx (else LTGNN_E_ALIGN).  No atomics, allocation or host synchronisation.
 */
int ltgnn_gru_sensor_fwd(int device, int64_t B, int32_t L, int32_t S, int64_t q0, int64_t Q, int32_t H, const float* r,
                         const float* tproj, const float* w_r, const float* w_hh, const float* b_hn, float* hseq,
                         float* h_last, float* gates, void* stream);
int ltgnn_gru_resident_tiles(int device, int32_t* tiles);
int ltgnn_gru_sensor_bwd_dx(int device, int64_t B, int32_t L, int32_t S, int32_t F, int64_t q0, int64_t Q, int32_t H,
                            const float* w_ih, const float* dG, float* dr, float* dxt, void* stream);

/* ---- deterministic sum of gathered rows (csrc/gather_sum.cu) -------------------------------------------------------
 * For every plane p < planes and row r < rows:
 *   out[p * out_plane_stride + r * C + c] = sum_{e = ptr[r]} ^ {ptr[r+1] - 1} src[p * src_plane_stride + idx[e] * C + c]
 * fp32 adds in ascending e from zero (an empty row is zeros): no atomics, bitwise deterministic.  ptr int32 [rows + 1]
 * non-decreasing and idx int32 [ptr[rows]] are the transpose of a gather as a CSR; the caller guarantees that every idx
 * is a row of src (the entry point does not read device memory).  The input-gradient backward of rows several readers
 * gathered (the frozen predictor's shared windows).  C % 4 == 0 and rows < 2^31 - 1 (else LTGNN_E_SHAPE); rows >= 0,
 * C > 0, 1 <= planes <= 65535, strides >= 0 and src, ptr, idx, out non-NULL (else LTGNN_E_ARG); src and out 16-byte
 * aligned, the plane strides (in floats) multiples of 4, ptr and idx 4-byte aligned (else LTGNN_E_ALIGN).  No
 * allocation or host synchronisation: capturable into a CUDA graph.
 */
int ltgnn_row_gather_sum(int device, int64_t rows, int32_t C, int32_t planes, const float* src, int64_t src_plane_stride,
                         const int32_t* ptr, const int32_t* idx, float* out, int64_t out_plane_stride, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LTGNN_H_ */
