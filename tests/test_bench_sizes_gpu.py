"""Parity at the sizes bench.py runs: the long reductions at the benchmark's row counts and one step of the `lta4096`
and `scaled100k` workloads themselves, all against plain fp64 torch on the GPU (cuBLAS DGEMM, fp64 `index_add_`,
fp64 cuDNN: no code shared with the kernels under test).

Why these sizes: the tensor-memory accumulator adds with truncation (DESIGN section 2, csrc/tgrad.cuh), a bias that grows
linearly with the rows one accumulator sums.  One accumulator for a CTA's whole range measured 4e-6 at 570 rows per CTA
(under the 1e-5 bar) but 1.2e-4 at the 18 000 rows per CTA of `lta4096`.  So the reductions are run here at the row
counts the benchmark gives them, on three operand kinds:
  relu  X = relu(randn), G = randn * (rand > 0.5): the shape of real activations and gradients;
  same  X, G uniform in [0, 1): every product is positive, the worst case for a biased accumulator;
  real  the operands of a B = 4096 cross-entropy step (ill-conditioned: the sum of |terms| is ~100 x |sum|).

Two checks per tensor:
  error  max|ours - truth| / max|truth| <= 1e-5 (GRU BPTT 5e-5); where the sum is ill-conditioned, <= 3 x torch fp32's
         own distance on the same operands (TF32 off) and never above 3e-5, the rule of tests/test_benchscale_gpu.py;
  bias   on same-sign operands every truth entry is far from zero, so a biased sum shows as a mean signed relative
         deviation (|ours| - |truth|) / |truth| away from zero, long before it reaches the 1e-5 bar.  Round-to-nearest
         sums (CUDA cores) must also leave |ours| < |truth| for about half of the entries: [0.35, 0.65] (tensors with
         >= 1 000 entries).  Tensor-core sums cannot: tcgen05 truncates inside every MMA, so the few MMAs that
         accumulate between two round-to-nearest flushes leave a small bias of their own.  Measured on the B200 at
         M/16, M/4 and M (same-sign, wgrad 64 x 64 at M = 2 707 456 and 128 x 128 at M = 1 600 000): the mean deviation
         is -1.2e-7 at every M (fraction below 0.975-0.99, max error 3.1e-7, torch fp32 7e-7 to 1.5e-6), so it is set by
         the flush interval, not by the rows a CTA sums; TC_BIAS holds it to 5e-7.  One accumulator for a CTA's whole
         range gives -1.3e-4 at lta4096.  The GRU weight gradient uses the cheaper segmented form (kSeg = 16: 192
         truncating MMAs per flush, csrc/tgrad.cuh): -4.9e-6 at B = 256, 1024 and 4096 alike (max error 2.7e-6), held by
         GRU_BIAS to 7.5e-6; a range-long accumulator there gives -1.7e-3.
Every comparison is logged with conftest.parity_log, torch fp32's distance next to ours."""
import copy

import numpy as np
import pytest
import torch

import bench
from conftest import parity_log, rel_err
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.models import LeakDetector
from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder
from oracle.detector_oracle import OracleLeakDetector
from test_benchscale_gpu import _assert_within, _head_ref, _replay

pytestmark = pytest.mark.gpu
TOL, GRU_TOL, SLACK, ILL = 1e-5, 5e-5, 3.0, 3e-5
BIAS_LO, BIAS_HI, BIAS_MIN_ENTRIES = 0.35, 0.65, 1000
# the kernels draw 16 random bits per element (keep probability 1 - round(0.1 * 2^16) / 2^16) and scale the kept
# gradients by this fp32 constant; the truth uses the same constant, so its own rounding is not counted as a bias
TC_BIAS, GRU_BIAS = 5e-7, 7.5e-6    # see the module docstring
SCALE = float(np.float32(1.0) / (np.float32(1.0) - np.float32(round(0.1 * 65536) / 65536)))

LTA_ROWS = 4096 * 661          # lta4096: rows of one GCN layer's weight gradient and d bias
SYN_ROWS = 16 * 100_000        # scaled100k: the same at hidden 128
_NETS = {}


def _net(name, pipes):
    if (name, pipes) not in _NETS:
        _NETS[(name, pipes)] = bench.network(name, pipes)
    return _NETS[(name, pipes)]


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _operands(kind, shape_g, shape_x, seed):
    gen = _gen(seed)
    if kind == "relu":
        g = torch.randn(shape_g, device="cuda", generator=gen)
        g *= torch.rand(shape_g, device="cuda", generator=gen) > 0.5
        x = torch.randn(shape_x, device="cuda", generator=gen).relu_()
    else:
        g = torch.rand(shape_g, device="cuda", generator=gen)
        x = torch.rand(shape_x, device="cuda", generator=gen)
    return g, x


def _below(got, truth):
    """Fraction of entries with |ours| < |truth| (same-sign operands: every truth entry is a sum of positive terms)."""
    return (got.detach().double().abs() < truth.abs()).double().mean().item()


def _entry(got, truth, fp32, bias=None):
    """Errors of ours and of torch fp32 against the truth; with `bias` (same-sign operands) also the mean signed relative
    deviation (|ours| - |truth|) / |truth| and, with >= 1 000 entries, the fraction of entries with |ours| < |truth|.
    bias = "rn": a sum of round-to-nearest adds, held to TC_BIAS and the fraction bounds; bias = a number: a tensor-core
    sum, held to |mean deviation| <= that number."""
    e = {"ours": rel_err(got, truth), "torch_fp32": rel_err(fp32, truth)}
    if bias is not None:
        t = truth.detach().double()
        assert (t.abs() > 0).all()
        e["rel_bias"] = ((got.detach().double().abs() - t.abs()) / t.abs()).mean().item()
        e["bias_rule"] = bias
        if truth.numel() >= BIAS_MIN_ENTRIES:
            e["below_truth"] = _below(got, t)
    return e


def _assert_report(tag, rep, tol=TOL):
    parity_log(tag, rep)
    for name, e in rep.items():
        assert e["ours"] <= max(tol, min(SLACK * e["torch_fp32"], ILL)), (tag, name, e)
        if "bias_rule" in e:
            rn = e["bias_rule"] == "rn"
            assert abs(e["rel_bias"]) <= (TC_BIAS if rn else e["bias_rule"]), (tag, name, e)
            if rn and "below_truth" in e:
                assert BIAS_LO <= e["below_truth"] <= BIAS_HI, (tag, name, e)


# ------------------------------------------------------------------------------------------------ weight gradients
@pytest.mark.parametrize("kind", ["relu", "same"])
@pytest.mark.parametrize("m,do,di", [(LTA_ROWS, 64, 64), (SYN_ROWS, 128, 128), (SYN_ROWS, 64, 128)])
def test_wgrad_at_bench_rows(m, do, di, kind):
    """64 x 64: the register-total form (kSeg = -1) of the GCN layers at lta4096, ~18 300 rows per CTA; 128 x 128 and
    64 x 128: the generic per-chunk form at the scaled100k layer size."""
    _assert_report(f"bench_rows wgrad {kind} M={m} {do}x{di}", {"dW": _wgrad_entry(kind, m, do, di)})


def _wgrad_entry(kind, m, do, di):
    g, x = _operands(kind, (m, do), (m, di), m + do + di + (kind == "same"))
    truth = g.double().t() @ x.double()
    return _entry(ops.wgrad(g, x), truth, g.t() @ x, bias=TC_BIAS if kind == "same" else None)


# ------------------------------------------------------------------------------------------------ d bias, mean pool
_SHAPES = {"lta4096": ("LTA", 764, 4096, 64), "scaled100k": ("SYN100K", 2000, 16, 128)}


@pytest.mark.parametrize("kind", ["relu", "same"])
@pytest.mark.parametrize("workload", ["lta4096", "scaled100k"])
def test_bias_colsum_at_bench_rows(workload, kind):
    """d bias of a GCN layer = column sums of the gated gradient over B*N rows, fused into the transpose aggregation:
    STAGED path at lta4096 (2.7 M rows), GATHER path at scaled100k (1.6 M rows).  The gate is the 1-bit live mask a
    fused forward (ReLU + dropout 0.1) wrote, as in the model."""
    name, pipes, b, d = _SHAPES[workload]
    net = _net(name, pipes)
    graph = ops.PipeGraph(torch.from_numpy(net["edge_index"]), net["n_nodes"])
    n = net["n_nodes"]
    assert ops._staged_ok(graph, d) == (workload == "lta4096")
    gen = _gen(7 + b)
    live = ops.new_live_mask(b, n, d, "cuda")
    ops.spmm_fused(graph, torch.randn(b, n, d, device="cuda", generator=gen), bias=torch.zeros(d, device="cuda"),
                   relu=True, drop_p=0.1, drop_seed=11, live_out=live)
    gate = ops.unpack_live_mask(live)
    x, _ = _operands(kind, (b, n, d), (1,), 8 + b + (kind == "same"))
    _, colsum = ops.spmm_fused(graph, x, transpose=True, live_in=live, gate_scale=SCALE, want_colsum=True)
    truth = (x.double() * gate * SCALE).sum((0, 1))
    rep = {"colsum": _entry(colsum, truth, (x * gate * SCALE).sum((0, 1)), bias="rn" if kind == "same" else None)}
    _assert_report(f"bench_rows colsum {kind} {workload} B={b} N={n} D={d}", rep)


@pytest.mark.parametrize("kind", ["relu", "same"])
@pytest.mark.parametrize("workload", ["lta4096", "scaled100k"])
def test_mean_pool_at_bench_rows(workload, kind):
    """The no-leak head's mean pool: 661 rows per window x 4096 windows, and 100 000 rows per window (the two-pass
    partial-sum form)."""
    name, pipes, b, d = _SHAPES[workload]
    n = _net(name, pipes)["n_nodes"]
    x, _ = _operands(kind, (b, n, d), (1,), 9 + b + (kind == "same"))
    truth = x.double().mean(1)
    rep = {"pooled": _entry(ops.mean_pool(x), truth, x.mean(1), bias="rn" if kind == "same" else None)}
    _assert_report(f"bench_rows mean_pool {kind} {workload} B={b} N={n} D={d}", rep)


# ------------------------------------------------------------------------------------------------ node init
def _node_init_grads(h_s, idx, n, w, b, dx0, live):
    """Gradients of detector.py:178-189 (gate = the ReLU / dropout decisions of the forward that ran) in h_s's dtype."""
    h_s, w, b = (t.detach().clone().requires_grad_(True) for t in (h_s, w, b))
    bsz, _, ds = h_s.shape
    h0 = torch.zeros(bsz, n, ds, dtype=h_s.dtype, device=h_s.device).index_copy(1, idx, h_s)
    mask = torch.zeros(n, 1, dtype=h_s.dtype, device=h_s.device)
    mask[idx, 0] = 1.0
    pre = torch.nn.functional.linear(torch.cat([h0, mask.unsqueeze(0).expand(bsz, -1, -1)], dim=-1), w, b)
    (pre * live.to(h_s.dtype)).backward(dx0.to(h_s.dtype))
    return h_s.grad, w.grad, b.grad


@pytest.mark.parametrize("kind", ["relu", "same"])
def test_node_init_bwd_at_bench_rows(kind):
    """node_init backward at lta4096: dW over B*S = 118 784 sensor rows, d bias over B*N = 2.7 M rows."""
    net = _net("LTA", 764)
    bsz, n, ds, d = 4096, net["n_nodes"], 64, 64
    idx = torch.from_numpy(net["sensor_idx"]).cuda()
    s = idx.numel()
    slot = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    slot[idx] = torch.arange(s, dtype=torch.int32, device="cuda")
    gen = _gen(13 + (kind == "same"))
    dx0, h_s = _operands(kind, (bsz, n, d), (bsz, s, ds), 14 + (kind == "same"))
    if kind == "same":   # positive weights and bias: every unit is live, every product of the sums positive
        w = torch.rand(d, ds + 1, device="cuda", generator=gen) * 0.2
        b = torch.rand(d, device="cuda", generator=gen)
    else:
        w = torch.randn(d, ds + 1, device="cuda", generator=gen) * 0.2
        b = torch.randn(d, device="cuda", generator=gen) * 0.5
    live = ops.new_live_mask(bsz, n, d, "cuda")
    x0 = ops.node_init_fwd(h_s, slot, n, w, b, 0.1, 21, live_out=live)
    gate = ops.unpack_live_mask(live)
    got = ops.node_init_bwd(h_s, slot, w, dx0, x0, SCALE, live=live)
    truth = _node_init_grads(h_s.double(), idx, n, w.double(), b.double(), dx0.double() * SCALE, gate)
    fp32 = _node_init_grads(h_s, idx, n, w, b, dx0 * SCALE, gate)
    # dh_s is a 64-term product, not a long reduction: only its error is checked
    rep = {nm: _entry(a, t, f, bias=TC_BIAS if kind == "same" and nm == "dW" else None)
           for nm, a, t, f in zip(("dh_s", "dW", "db"), got, truth, fp32)}
    _assert_report(f"bench_rows node_init_bwd {kind} B={bsz} S={s}", rep)


# ------------------------------------------------------------------------------------------------ pipe head
def test_heads_same_sign_at_bench_rows():
    """Pipe head at lta4096 (B*P = 3.1 M pipe rows) on same-sign operands: x >= 0 makes every feature >= 0, and
    dlogit >= 0 with w2 >= 0 makes every gradient of the hidden layer >= 0, so dW1 (and db1, dw2) are sums of positive
    terms.  W1 and b1 keep both signs, so the ReLU gate is a real mix.  The fp64 truth replays the captured gate."""
    bsz, n, p = 4096, 661, 764
    gen = _gen(17)
    x = torch.rand(bsz, n, 64, device="cuda", generator=gen)
    ends = torch.from_numpy(_net("LTA", 764)["pipe_ends"]).cuda()
    w1 = torch.randn(128, 192, device="cuda", generator=gen) * 0.1
    b1 = torch.randn(128, device="cuda", generator=gen) * 0.1
    w2 = torch.rand(1, 128, device="cuda", generator=gen)
    b2 = torch.rand(1, device="cuda", generator=gen)
    dlog = torch.rand(bsz, p, device="cuda", generator=gen)
    dpool = torch.rand(bsz, 64, device="cuda", generator=gen)

    o = [v.clone().requires_grad_(True) for v in (x, w1, b1, w2)]
    cap = {}
    ops.DEBUG_CAPTURE = cap
    try:
        part, pooled = ops.heads(o[0], ends.to(torch.int32), o[1], o[2], o[3], 0.1, False)
    finally:
        ops.DEBUG_CAPTURE = None
    logits = part.sum(0) + b2
    ((logits * dlog).sum() + (pooled * dpool).sum()).backward()
    live = cap.pop("head_live").view(bsz, p, 128)

    def ref(dt):
        t = [v.to(dt, copy=True).requires_grad_(True) for v in (x, w1, b1, w2, b2)]
        lr, pr = _head_ref(t[0], ends, *t[1:], live.to(dt))
        ((lr * dlog.to(dt)).sum() + (pr * dpool.to(dt)).sum()).backward()
        return lr.detach(), [v.grad for v in t[:4]]

    l64, g64 = ref(torch.float64)
    l32, g32 = ref(torch.float32)
    rep = {"logits": _entry(logits, l64, l32)}
    for nm, a, t, f in zip(("dx", "dw1", "db1", "dw2"), o, g64, g32):
        rep[nm] = _entry(a.grad, t, f, bias=TC_BIAS if nm != "dx" else None)
    _assert_report(f"bench_rows heads same B={bsz} N={n} P={p}", rep)


# ------------------------------------------------------------------------------------------------ GRU
GRU_NAMES = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")


def _blocked(logical):
    """(L, Qp, W) -> the kernels' blocked-32 storage [L * Qp / 32, W / 4, 32, 4] (inverse of ops.unblock32)."""
    l, qp, w = logical.shape
    return logical.reshape(l * qp // 32, 32, w // 4, 4).permute(0, 2, 1, 3).contiguous()


def test_gru_weight_gradient_same_sign_at_bench_rows():
    """The GRU weight-gradient GEMM (ltgnn_gru_bwd_w) alone at e2e lta4096: 4096 windows x 29 sensors x 288 steps =
    34.2 M rows, fed uniform [0, 1) states, inputs and gate gradients so that every product is positive.
    dBfused[4H, 96] = sum over (t, q) of dG(t, q)^T [h_{t-1}(q) | r | tf | 1 | 0]."""
    _assert_report("bench_rows gru_bwd_w same B=4096 L=288 S=29 F=9", {"dBfused": _gru_bwd_w_entry(4096)})


def _gru_bwd_w_entry(b):
    l, s, f, hd = 288, 29, 9, 64
    q = b * s
    assert q % 128 == 0
    gen = _gen(19)
    r = torch.rand(b, l, s, device="cuda", generator=gen)
    tf = torch.rand(b, l, f, device="cuda", generator=gen)
    hseq = torch.rand(l * q // 32, hd // 4, 32, 4, device="cuda", generator=gen)
    dg = torch.rand(l * q // 32, hd, 32, 4, device="cuda", generator=gen)
    fused = torch.empty(4 * hd, 96, device="cuda")
    lib = _lib.load()
    dev = torch.cuda.current_device()
    ws = torch.empty(int(lib.ltgnn_gru_ws_floats(dev)), device="cuda")
    _lib.check(lib.ltgnn_gru_bwd_w(dev, b, l, s, f, hd, r.data_ptr(), tf.data_ptr(),
                                   hseq.data_ptr(), dg.data_ptr(), fused.data_ptr(), ws.data_ptr(), ops._stream(r)))
    h_log, g_log = ops.unblock32(hseq, l, q), ops.unblock32(dg, l, q)
    kb = hd + 1 + f + 1
    truth = torch.zeros(4 * hd, kb, dtype=torch.float64, device="cuda")
    fp32 = torch.zeros(4 * hd, kb, device="cuda")
    a = torch.empty(q, kb, device="cuda")
    for t in range(l):
        a[:, :hd] = h_log[t - 1] if t else 0.0
        a[:, hd] = r[:, t, :].reshape(q)
        a[:, hd + 1:hd + 1 + f] = tf[:, t, :].repeat_interleave(s, dim=0)
        a[:, hd + 1 + f] = 1.0
        truth += g_log[t].double().t() @ a.double()
        fp32 += g_log[t].t() @ a
    return _entry(fused[:, :kb], truth, fp32, bias=GRU_BIAS)


def test_gru_bptt_at_bench_size():
    """The native GRU encoder, forward and BPTT, on all 118 784 sequences of lta4096's e2e (L = 288) in one call, against
    torch.nn.GRU through cuDNN in fp64 (the truth) and fp32 (for scale), run in slabs of 256 windows with forward and
    backward per slab so that one slab's reserve space is alive at a time."""
    b, l, s = 4096, 288, 29
    residual, tfeat, _ = bench.synthetic_batch(b, l, s, 765, 198)
    r, tf = residual.cuda(), tfeat.cuda()
    torch.manual_seed(42)
    enc = SharedSensorGRUEncoder(hidden_size=64).cuda().train()
    ref64, ref32 = copy.deepcopy(enc).double(), copy.deepcopy(enc)
    dh = torch.randn(b, s, 64, device="cuda", generator=_gen(23))
    (enc(r, tf) * dh).sum().backward()
    for m, dt in ((ref64, torch.float64), (ref32, torch.float32)):
        m.use_native = False
        for i in range(0, b, 256):
            sl = slice(i, i + 256)
            (m(r[sl].to(dt), tf[sl].to(dt)) * dh[sl].to(dt)).sum().backward()
    rep = {nm: _entry(getattr(enc.gru, nm).grad, getattr(ref64.gru, nm).grad, getattr(ref32.gru, nm).grad)
           for nm in GRU_NAMES}
    _assert_report(f"bench_rows gru_bptt real B={b} L={l} S={s}", rep, tol=GRU_TOL)


# ------------------------------------------------------------------------------------------------ the workloads
_STEPS = {}


def _bench_step(workload):
    """One train-mode step (dropout 0.1) of bench.py's `value` scope -- h_s from the sensor encoder, gnn_stack, CE,
    backward -- built as bench.py builds it, and the same step of the fp64 / fp32 oracle on the GPU replaying the
    captured ReLU / dropout masks.  Also returns the operands of every ops.wgrad call of the step.  Cached per module."""
    if workload in _STEPS:
        return _STEPS[workload]
    wl = bench.WORKLOADS[workload]
    net = _net(wl["net"], wl["pipes"])
    torch.manual_seed(42)
    ours = LeakDetector(net["inp"], net["sensors"], net["pipe_ids"], sensor_hidden=64, node_hidden=wl["hidden"],
                        gnn_layers=2, dropout=0.1, use_time=True).cuda().train()
    state = {k: v.detach().clone() for k, v in ours.state_dict().items()}

    def oracle(dtype):
        m = OracleLeakDetector(len(ours.node_names), ours.edge_index_single, ours.pipe_ends,
                               ours.sensor_node_idx.tolist(), 64, wl["hidden"], 2, 0.1, True).to(dtype)
        m.load_state_dict({k: v.to(dtype) for k, v in state.items()}, strict=True)
        m = m.cuda().train()
        # plain attributes, not buffers: .cuda() leaves them on the host
        m.edge_index_single, m.pipe_ends = m.edge_index_single.cuda(), m.pipe_ends.cuda()
        m.sensor_node_idx = m.sensor_node_idx.cuda()
        return m

    n_classes = len(net["pipe_ids"]) + 1
    residual, tfeat, label = bench.synthetic_batch(wl["batch"], wl["l_det"], len(net["sensors"]), n_classes, 198)
    label = label.cuda()
    with torch.no_grad():
        h_s = ours.sensor_encoder(residual.cuda(), tfeat.cuda())
    leaf = h_s.detach().clone().requires_grad_(True)

    cap, keep, calls = {}, {}, []

    def hook(_m, inp, out):
        keep["v"] = torch.where(inp[0] != 0, out / inp[0], torch.ones((), device=out.device)).detach()

    def spy(g, x, out=None):
        calls.append((g.detach().clone(), x.detach().clone()))
        return orig(g, x, out)

    orig = ops.wgrad
    ops.wgrad = spy
    h = ours.noleak_head.mlp[2].register_forward_hook(hook)
    ops.DEBUG_CAPTURE = cap
    try:
        torch.manual_seed(3)
        lo = ours.gnn_stack(leaf)
        torch.nn.functional.cross_entropy(lo, label).backward()
    finally:
        ops.DEBUG_CAPTURE = None
        ops.wgrad = orig
        h.remove()
    # 1-bit live masks where the kernels wrote them; node states too large for the staged node init keep x0 as the gate
    masks = [ops.unpack_live_mask(lv) if lv is not None else x > 0 for lv, x in zip(cap["lives"], cap["xs"])]
    assert 0.02 < 1.0 - masks[1].double().mean().item() < 0.98
    n = len(ours.node_names)
    rep = {}
    outs = {}
    for dt in (torch.float64, torch.float32):
        orc = oracle(dt)
        h_in = leaf.detach().to(dt).requires_grad_(True)
        lr = _replay(orc, h_in, masks, cap["head_live"], keep["v"], SCALE, n)
        torch.nn.functional.cross_entropy(lr, label).backward()
        outs[dt] = (lr.detach(), h_in.grad, {k: p.grad for k, p in orc.named_parameters() if p.grad is not None})
        del orc, lr, h_in
    (l64, dh64, g64), (l32, dh32, g32) = outs[torch.float64], outs[torch.float32]
    rep["logits"] = (rel_err(lo, l64), rel_err(l32, l64))
    for name, p in ours.named_parameters():
        if p.grad is not None:
            rep[name] = (rel_err(p.grad, g64[name]), rel_err(g32[name], g64[name]))
    rep["d_h_s"] = (rel_err(leaf.grad, dh64), rel_err(dh32, dh64))
    parity_log(f"bench_step {workload} B={wl['batch']} N={n} P={wl['pipes']} hidden={wl['hidden']} train",
               {k: {"ours": a, "oracle_fp32": c} for k, (a, c) in rep.items()})
    del ours, cap, masks, outs
    torch.cuda.empty_cache()
    _STEPS[workload] = (rep, calls)
    return _STEPS[workload]


@pytest.mark.parametrize("workload", ["lta4096", "scaled100k"])
def test_bench_workload_step_vs_oracle(workload):
    """bench.py's `value` step at its own size: logits, the 14 parameter gradients of the GNN stack (the sensor GRU is
    behind the detached h_s, as in the benchmark; its gradients at this size are test_gru_bptt_at_bench_size) and d h_s
    against the fp64 oracle, with the rule of test_benchscale_gpu."""
    rep, _ = _bench_step(workload)
    assert len(rep) == 16
    _assert_within(rep)


@pytest.mark.parametrize("workload,rows,width", [("lta4096", LTA_ROWS, 64), ("scaled100k", SYN_ROWS, 128)])
def test_wgrad_real_operands_at_bench_rows(workload, rows, width):
    """The GCN weight gradients on the operands of the benchmark step itself (G = the gated transpose aggregation of a
    cross-entropy gradient, X = the layer input), captured through a spy on ops.wgrad."""
    _, calls = _bench_step(workload)
    layers = [(g.reshape(-1, g.shape[-1]), x.reshape(-1, x.shape[-1])) for g, x in calls if g.numel() == rows * width]
    assert len(layers) == 2
    rep = {}
    for i, (g, x) in enumerate(layers):
        rep[f"conv{1 - i}.dW"] = _entry(ops.wgrad(g, x), g.double().t() @ x.double(), g.t() @ x)
    _assert_report(f"bench_rows wgrad real {workload} M={rows} {width}x{width}", rep)
