"""The one-kernel GCN layer (csrc/gcn_layer.cu) at every plan it picks -- tile count, k-groups, consumer slices, A slots,
loader ring depth, one or many windows per CTA -- on synthetic pipe networks against
``relu(A_hat (X W^T) + b)`` in fp64 (A_hat from the PyG restatement's gcn_norm), elementwise.  Plus: its support
predicate against the Python restatement of the plan (tests/gcn_plans.py), the refusals and the two-launch path that
carries them, window independence, the bit-identity with ltgnn_linear + ltgnn_spmm_fused that the kernel documents,
and the detector body on both sides of each switch.  Margins go to conftest.parity_log."""
import functools

import pytest
import torch

import gcn_plans as G
from conftest import parity_log, rel_err
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.lib import LtgnnError

pytestmark = pytest.mark.gpu
CASES = G.cases()
REFUSED = G.refused_cases()
P, SEED = 0.1, 4242
KEEP_SCALE = torch.tensor(1.0) / (1.0 - torch.tensor(round(P * 65536) / 65536, dtype=torch.float32))


@functools.lru_cache(maxsize=None)
def _graph(n, nnz):
    ei = G.pipe_edges(n, nnz)
    return ops.PipeGraph(ei, n), ei


@functools.lru_cache(maxsize=8)
def _a_hat(n, nnz):
    return G.gcn_dense(_graph(n, nnz)[1], n, device="cuda")


def _supported(graph, k, d):
    return ops.gcn_layer_supported(graph, torch.empty(1, device="cuda"), torch.empty(d, k))


def test_supported_matches_the_plan():
    """The kernel's predicate == the restatement, at +-1 node around every tile boundary and +-1 entry around every
    shared-memory limit."""
    checked = 0
    ns = sorted({1, 2, 95, 96} | {t * 128 + e for t in range(1, 8) for e in (-1, 0, 1)})
    for n in ns:
        graph, _ = _graph(n, None if n > 2 else G.min_nnz(n))
        for k, d in ((32, 32), (64, 64), (96, 64), (128, 64), (64, 96), (128, 128), (64, 160), (96, 224), (64, 256),
                     (128, 256), (160, 64)):
            assert _supported(graph, k, d) == G.plan(n, graph.nnz, k, d).supported, (n, graph.nnz, k, d)
            checked += 1
    for n, k, d in G.LIMIT_SHAPES:
        for depth in (2, 4):
            last = G.last_nnz(n, k, d, depth)
            for nnz in (last - 1, last, last + 1):
                if nnz < G.min_nnz(n):
                    continue
                graph, _ = _graph(n, nnz)
                want = G.plan(n, nnz, k, d)
                assert _supported(graph, k, d) == want.supported, (n, nnz, k, d, want)
                checked += 1
    for c in CASES + REFUSED:
        assert _supported(_graph(c.n, c.nnz)[0], c.K, c.D) == G.plan(c.n, c.nnz, c.K, c.D).supported, c
    print(f"{checked} shapes")


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_layer_vs_fp64(case):
    """No bias; bias + ReLU; bias + ReLU + dropout, with the live mask; and, where the tensor-core linear takes the
    shape, bit for bit the two-launch path."""
    graph, _ = _graph(case.n, case.nnz)
    assert graph.nnz == case.nnz and _supported(graph, case.K, case.D)
    bsz = 3
    x, w, b = (t.cuda() for t in G.inputs(case, bsz))
    a = _a_hat(case.n, case.nnz)
    rep = {}

    y64, s = G.reference(a, x, w, None)
    y = ops.gcn_layer_fwd(graph, x, w)
    rep["plain"] = (G.bound_ratio(y, y64, s), rel_err(y, y64))

    y64, s = G.reference(a, x, w, b)
    live = ops.new_live_mask(bsz, case.n, case.D, x.device)
    yr = ops.gcn_layer_fwd(graph, x, w, bias=b, relu=True, live_out=live)
    rep["bias_relu"] = (G.bound_ratio(yr, y64.relu(), s), rel_err(yr, y64.relu()))
    assert torch.equal(ops.unpack_live_mask(live), yr > 0)

    yd = ops.gcn_layer_fwd(graph, x, w, bias=b, relu=True, drop_p=P, drop_seed=SEED, live_out=live)
    assert torch.equal(ops.unpack_live_mask(live), yd > 0)
    scaled = yr * KEEP_SCALE.item()
    assert bool(((yd == 0) | (yd == scaled)).all())
    dropped = ((yd == 0) & (yr > 0)).sum().item() / max((yr > 0).sum().item(), 1)
    assert 0.06 < dropped < 0.14, dropped
    parity_log(f"gcn_layer_plans {case.name}", {k: {"bound": r, "rel": e} for k, (r, e) in rep.items()})
    for r, e in rep.values():
        assert r <= 1.0 and e <= 1e-5, rep

    if ops._linear_tc_ok(case.K, case.D):
        xw = ops.linear_tc(x, w)
        assert torch.equal(ops.gcn_layer_fwd(graph, x, w), ops.spmm(graph, xw))   # no epilogue: plain aggregation
        for bias, relu, p in ((b, False, 0.0), (b, True, 0.0), (b, True, P)):
            la = ops.new_live_mask(bsz, case.n, case.D, x.device)
            lb = ops.new_live_mask(bsz, case.n, case.D, x.device)
            want = ops.spmm_fused(graph, xw, bias=bias, relu=relu, drop_p=p, drop_seed=SEED, live_out=la)
            got = ops.gcn_layer_fwd(graph, x, w, bias=bias, relu=relu, drop_p=p, drop_seed=SEED, live_out=lb)
            assert torch.equal(got, want), (relu, p, (got - want).abs().max().item())
            assert torch.equal(la, lb)


def _one_per_plan():
    seen, out = set(), []
    for c in CASES:
        p = G.plan(c.n, c.nnz, c.K, c.D)
        if (p.T, p.n_slots, p.depth) not in seen:
            seen.add((p.T, p.n_slots, p.depth))
            out.append(c)
    return out


@pytest.mark.parametrize("case", _one_per_plan(), ids=lambda c: c.name)
def test_windows_are_independent(case):
    """B = 3 SMs + 5 windows (a CTA runs three or four): sampled windows -- first, last, and ones that share a CTA --
    equal the same window run alone, bit for bit."""
    graph, _ = _graph(case.n, case.nnz)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    bsz = 3 * sms + 5
    gen = torch.Generator().manual_seed(case.n + case.K)
    x = torch.randn(bsz, case.n, case.K, generator=gen).cuda()
    w = (torch.randn(case.D, case.K, generator=gen) * case.K ** -0.5).cuda()
    b = (torch.randn(case.D, generator=gen) * 0.1).cuda()
    y = ops.gcn_layer_fwd(graph, x, w, bias=b, relu=True)
    for i in (0, 1, sms - 1, sms, 2 * sms, 3 * sms, 3 * sms + 4, 4, sms + 4, 2 * sms + 4, bsz - 1):
        alone = ops.gcn_layer_fwd(graph, x[i:i + 1].contiguous(), w, bias=b, relu=True)
        assert torch.equal(y[i:i + 1], alone), i


@pytest.mark.parametrize("case", REFUSED, ids=lambda c: c.name)
def test_refused_shapes_take_the_two_launch_path(case):
    graph, _ = _graph(case.n, case.nnz)
    assert not _supported(graph, case.K, case.D)
    x, w, b = (t.cuda() for t in G.inputs(case, 2))
    with pytest.raises(LtgnnError):
        ops.gcn_layer_fwd(graph, x, w, bias=b, relu=True)
    y = ops.spmm_fused(graph, ops._linear_any(x, w), bias=b, relu=True)   # what gnn_body runs for this layer
    y64, s = G.reference(_a_hat(case.n, case.nnz), x, w, b)
    r, e = G.bound_ratio(y, y64.relu(), s), rel_err(y, y64.relu())
    parity_log(f"gcn_layer_plans refused {case.name}", {"bound": r, "rel": e})
    assert r <= 1.0 and e <= 1e-5


# ------------------------------------------------------------------------------------------------ the detector body
def _body_ref(h_s, idx, n, a, w0, b0, convs, gates):
    """node init + GCN layers in fp64 with the ReLU decisions of the forward that ran (eval mode: no dropout)."""
    bsz, _, ds = h_s.shape
    h0 = torch.zeros(bsz, n, ds, dtype=h_s.dtype, device=h_s.device).index_copy(1, idx, h_s)
    mark = torch.zeros(n, 1, dtype=h_s.dtype, device=h_s.device)
    mark[idx] = 1.0
    x = torch.nn.functional.linear(torch.cat([h0, mark.expand(bsz, n, 1)], dim=-1), w0, b0) * gates[0]
    for (w, b), g in zip(convs, gates[1:]):
        x = (a @ (x @ w.t()) + b) * g
    return x


@pytest.mark.parametrize("n,nnz,width", [(384, None, 128), (385, None, 128), (896, None, 64), (897, None, 64),
                                         (785, G.last_nnz(785, 64, 64, 2) + 1, 64)],
                         ids=["n384_w128", "n385_w128", "n896_w64", "n897_w64", "exact_n785_w64"])
def test_body_at_the_switches(n, nnz, width, monkeypatch):
    """gnn_body forward and every gradient against fp64, on both sides of the fused layer's node and shared-memory
    limits; where the layer is fused, FUSED_LAYER on and off give the same bits."""
    graph, ei = _graph(n, nnz)
    fused = _supported(graph, width, width)
    assert fused == G.plan(n, graph.nnz, width, width).supported
    bsz, s, ds = 5, 29, 64
    gen = torch.Generator().manual_seed(n + width)
    idx = torch.randperm(n, generator=gen)[:s]
    slot = torch.full((n,), -1, dtype=torch.int32)
    slot[idx] = torch.arange(s, dtype=torch.int32)
    h_s = torch.randn(bsz, s, ds, generator=gen)
    prm = [torch.randn(width, ds + 1, generator=gen) * 0.2, torch.randn(width, generator=gen) * 0.1]
    for _ in range(2):
        prm += [torch.randn(width, width, generator=gen) * width ** -0.5, torch.randn(width, generator=gen) * 0.1]
    dy = torch.randn(bsz, n, width, generator=gen).cuda()

    runs = []
    for on in ((True, False) if fused else (True,)):
        monkeypatch.setattr(ops, "FUSED_LAYER", on)
        leaves = [t.cuda().requires_grad_(True) for t in [h_s] + prm]
        ops.DEBUG_CAPTURE = cap = {}
        try:
            y = ops.gnn_body(leaves[0], slot.cuda(), graph, 0.1, False, leaves[1], leaves[2], leaves[3:])
        finally:
            ops.DEBUG_CAPTURE = None
        (y * dy).sum().backward()
        runs.append(([y.detach()] + [t.grad for t in leaves], [(x > 0).double() for x in cap["xs"]]))
    if fused:
        for a_, b_ in zip(runs[0][0], runs[1][0]):
            assert torch.equal(a_, b_)
    outs, gates = runs[0]

    t64 = [t.double().cuda().requires_grad_(True) for t in [h_s] + prm]
    convs = [(t64[3], t64[4]), (t64[5], t64[6])]
    y64 = _body_ref(t64[0], idx.cuda(), n, G.gcn_dense(ei, n, device="cuda"), t64[1], t64[2], convs, gates)
    (y64 * dy.double()).sum().backward()
    names = ["y", "h_s", "w0", "b0", "w1", "b1", "w2", "b2"]
    rep = {nm: rel_err(o, r) for nm, o, r in zip(names, outs, [y64] + [t.grad for t in t64])}
    parity_log(f"gcn_layer_plans body n={n} nnz={graph.nnz} width={width} fused={fused}", rep)
    assert all(v <= 1e-5 for v in rep.values()), rep
