"""Weighted message passing on the GPU: device normalisation of per-call edge weights, aggregation with per-call entry
values (STAGED on L-TOWN-A, GATHER on a 100 000-node graph), the adjacency-value gradient, GCNConv in both signatures
and LeakDetector with shared (E,) and per-window (B, E) weights -- all against fp64.  Tolerance as everywhere here:
max|a - b| <= 1e-5 max|b| against fp64, or no further than 3x the fp32 oracle's own distance where a long reduction is
ill-conditioned."""
import numpy as np
import pytest
import torch

from conftest import TOPO, parity_log, rel_err
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.graph import build_wdn_graph_from_inp, parse_epanet_inp
from oracle.pyg_weighted import GCNConv as OracleConv
from oracle.pyg_weighted import gcn_norm

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _pipes(n):
    return [ln.split()[0] for ln in parse_epanet_inp(TOPO["LTA"])["PIPES"]][:n]


@pytest.fixture(scope="module")
def lta():
    ei = build_wdn_graph_from_inp(TOPO["LTA"], [], _pipes(4), add_self_loops=False).edge_index
    return ei, ops.PipeGraph(ei, 661)


@pytest.fixture(scope="module")
def big():
    """100 000 nodes: a chain plus 15 000 chords, both directions of each link, no self loops -- too large for STAGED."""
    n = 100_000
    gen = torch.Generator().manual_seed(5)
    a = torch.cat([torch.arange(n - 1), torch.randint(0, n - 100, (15_000,), generator=gen)])
    b = torch.cat([torch.arange(1, n), a[n - 1:] + torch.randint(2, 100, (15_000,), generator=gen)])
    ei = torch.stack([torch.stack([a, b], 1).reshape(-1), torch.stack([b, a], 1).reshape(-1)])
    return ei, ops.PipeGraph(ei, n)


def _entries(graph, transpose=False):
    c = graph.csr
    ptr, col = (c.t_rowptr, c.t_col) if transpose else (c.rowptr, c.col)
    rows = torch.from_numpy(np.repeat(np.arange(c.num_nodes), np.diff(ptr))).cuda()
    return rows, torch.from_numpy(col.astype(np.int64)).cuda()


def _dense(graph, vals_row):
    rows, cols = _entries(graph)
    a = torch.zeros(graph.num_nodes, graph.num_nodes, dtype=torch.float64, device="cuda")
    return a.index_put_((rows, cols), vals_row.double(), accumulate=True)


def _oracle_dense(ei, w, n):
    out_ei, norm = gcn_norm(ei, n, dtype=torch.float64, edge_weight=w.double().cpu())
    a = torch.zeros(n, n, dtype=torch.float64)
    return a.index_put_((out_ei[1], out_ei[0]), norm, accumulate=True).cuda()


def _ref_spmm(graph, vals, x, transpose=False):
    """fp64 Y[b] = A_b x[b] with A_b the entries `vals` (1 or B rows) in the orientation's order, index_add_ on the GPU."""
    rows, cols = _entries(graph, transpose)
    x = x.double()
    v = vals.double().expand(x.shape[0], -1)
    y = torch.zeros_like(x)
    for b in range(x.shape[0]):
        y[b].index_add_(0, rows, v[b][:, None] * x[b][cols])
    return y


def _ref_adj(graph, gg, xw):
    rows, cols = _entries(graph)
    out = torch.empty(gg.shape[0], graph.nnz, dtype=torch.float64, device="cuda")
    for s in range(0, gg.shape[0], 256):
        out[s:s + 256] = (gg[s:s + 256].double()[:, rows] * xw[s:s + 256].double()[:, cols]).sum(-1)
    return out


# ---------------------------------------------------------------------------------------------------------------- norm
def test_device_norm_matches_fp64_and_host_values(lta):
    ei, g = lta
    gen = torch.Generator().manual_seed(1)
    w = (torch.rand(3, g.num_edges, generator=gen) * 2 + 0.05).cuda()
    vals, t_vals, _ = ops.edge_norm(g, w)
    assert vals.shape == t_vals.shape == (3, g.nnz)
    t_perm = torch.from_numpy(g.csr.t_perm.astype(np.int64)).cuda()
    for b in range(3):
        truth = _oracle_dense(ei, w[b], 661)
        assert rel_err(_dense(g, vals[b]), truth) <= 1e-6
        assert torch.equal(t_vals[b], vals[b][t_perm])
    shared, _, _ = ops.edge_norm(g, w[1])
    assert shared.shape == (1, g.nnz) and torch.equal(shared[0], vals[1])
    ones, t_ones, _ = ops.edge_norm(g, torch.ones(g.num_edges, device="cuda"))
    for dev, host in ((ones, g.csr.val), (t_ones, g.csr.t_val)):
        ulp = (dev[0].cpu().view(torch.int32).long() - torch.from_numpy(host).view(torch.int32).long()).abs().max().item()
        assert ulp <= 1, ulp


def test_device_norm_keeps_existing_self_loop_weights():
    ei = torch.tensor([[0, 1, 1, 2, 3, 1, 2, 4, 3, 1], [1, 0, 1, 1, 3, 2, 4, 2, 0, 1]])
    g = ops.PipeGraph(ei, 5)
    w = torch.tensor([0.5, 1.5, 2.0, 0.7, 3.0, 1.1, 0.9, 1.3, 0.6, 2.5], device="cuda")
    vals, _, _ = ops.edge_norm(g, w)
    assert rel_err(_dense(g, vals[0]), _oracle_dense(ei, w, 5)) <= 1e-6
    w64 = w.double().cpu().requires_grad_(True)
    out_ei, norm = gcn_norm(ei, 5, dtype=torch.float64, edge_weight=w64)
    dvals = torch.randn(1, g.nnz, generator=torch.Generator().manual_seed(2)).cuda()
    # the oracle's entries in A_hat order: same (dst, src) pairs, unique here
    rows, cols = _entries(g)
    key = {(int(d), int(s)): k for k, (s, d) in enumerate(out_ei.t().tolist())}
    perm = torch.tensor([key[(int(r), int(c))] for r, c in zip(rows.tolist(), cols.tolist())])
    (norm[perm] * dvals[0].double().cpu()).sum().backward()
    dw = ops.edge_norm_bwd(g, w, ops.edge_norm(g, w)[2], dvals)
    assert rel_err(dw, w64.grad) <= TOL
    assert dw[2].item() == 0.0  # node 1's first loop is replaced by its last one: no gradient


# --------------------------------------------------------------------------------------------------------- aggregation
@pytest.mark.parametrize("which", ["lta", "big"])
@pytest.mark.parametrize("shared", [True, False])
def test_weighted_aggregation_matches_fp64(request, which, shared):
    """Forward epilogue (bias + ReLU, live bits out) and the gated transposed backward (live bits in, column sums) with
    per-call values: STAGED on L-TOWN-A, GATHER on the 100k graph (and forced GATHER on L-TOWN-A)."""
    ei, g = request.getfixturevalue(which)
    b, d = (3, 64) if which == "lta" else (2, 128)
    gen = torch.Generator().manual_seed(7 + b)
    w = (torch.rand(1 if shared else b, g.num_edges, generator=gen) + 0.2).cuda()
    vals, t_vals, _ = ops.edge_norm(g, w[0] if shared else w)
    x = torch.randn(b, g.num_nodes, d, generator=gen).cuda()
    bias = torch.randn(d, generator=gen).cuda()
    algos = [_lib.SPMM_AUTO] + ([_lib.SPMM_GATHER] if which == "lta" else [])
    rep = {}
    for algo in algos:
        live = ops.new_live_mask(b, g.num_nodes, d, x.device)
        y = ops.spmm_fused(g, x, bias=bias, relu=True, live_out=live, vals=vals, algo=algo)
        ref = torch.relu(_ref_spmm(g, vals, x) + bias.double())
        rep[f"fwd algo={algo}"] = rel_err(y, ref)
        assert torch.equal(ops.unpack_live_mask(live), y > 0)
        gy = torch.randn(b, g.num_nodes, d, generator=gen).cuda()
        gz, cs = ops.spmm_fused(g, gy, transpose=True, live_in=live, gate_scale=1.25, want_colsum=True, vals=t_vals,
                                algo=algo)
        gated = gy.double() * (y > 0) * 1.25
        rep[f"bwd algo={algo}"] = rel_err(gz, _ref_spmm(g, t_vals, gated, transpose=True))
        rep[f"colsum algo={algo}"] = rel_err(cs, gated.sum((0, 1)))
        plain = ops.spmm_fused(g, x, vals=vals, algo=algo)
        rep[f"plain algo={algo}"] = rel_err(plain, _ref_spmm(g, vals, x))
    parity_log(f"weighted aggregation {which} shared={shared}", rep)
    assert all(e <= TOL for e in rep.values()), rep


@pytest.mark.parametrize("which,b", [("lta", 1), ("lta", 3), ("lta", 4096), ("big", 16)])
def test_adj_grad_matches_fp64_einsum(request, which, b):
    ei, g = request.getfixturevalue(which)
    d = 64 if which == "lta" else 128
    gen = torch.Generator().manual_seed(b)
    gy = torch.randn(b, g.num_nodes, d, generator=gen).cuda()
    xw = torch.randn(b, g.num_nodes, d, generator=gen).cuda()
    gate = torch.randn(b, g.num_nodes, d, generator=gen).cuda()
    live = ops.new_live_mask(b, g.num_nodes, d, gy.device)
    ops.spmm_fused(g, gate, bias=torch.zeros(d, device="cuda"), live_out=live)  # any tensor's own > 0 record
    act = ops.unpack_live_mask(live)
    rep = {
        "plain": rel_err(ops.gcn_adj_grad(g, gy, xw), _ref_adj(g, gy, xw)),
        "live": rel_err(ops.gcn_adj_grad(g, gy, xw, live_in=live, gate_scale=1.5), _ref_adj(g, gy * act * 1.5, xw)),
        "float gate": rel_err(ops.gcn_adj_grad(g, gy, xw, gate=gate, gate_scale=2.0), _ref_adj(g, gy * (gate > 0) * 2, xw)),
    }
    full = ops.gcn_adj_grad(g, gy, xw)
    acc = ops.gcn_adj_grad(g, gy, xw, out=full.clone(), accumulate=True)
    assert torch.equal(acc, full + full)
    shared = ops.gcn_adj_grad(g, gy, xw, shared=True)
    rep["shared"] = rel_err(shared, _ref_adj(g, gy, xw).sum(0, keepdim=True))
    parity_log(f"adj grad {which} B={b}", rep)
    assert all(e <= TOL for e in rep.values()), rep
    assert torch.equal(ops.gcn_adj_grad(g, gy, xw, shared=True), shared)


# ----------------------------------------------------------------------------------------------------------- GCNConv
# the PyG signature has one graph: its (B E,) weights are the shared case of the replicated graph
@pytest.mark.parametrize("signature,shape", [("pipegraph", "shared"), ("pipegraph", "per_window"), ("edge_index", "shared")])
def test_gcnconv_matches_fp64_restatement(lta, signature, shape):
    from leak_det_gnn_b200.nn import GCNConv

    ei, g = lta
    b, n, d = 3, 661, 64
    torch.manual_seed(3)
    conv = GCNConv(d, d).cuda()
    with torch.no_grad():
        conv.bias.normal_()
    ref = OracleConv(d, d).double()
    ref.load_state_dict({k: v.double().cpu() for k, v in conv.state_dict().items()})
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(b, n, d, generator=gen)
    w = torch.rand(b, g.num_edges, generator=gen) + 0.1
    r = torch.randn(b, n, d, generator=gen)
    big_ei = ei.repeat(1, b) + (torch.arange(b).repeat_interleave(ei.shape[1]) * n)[None]
    w_ours = w[0] if shape == "shared" else w
    w_ref = w[0].repeat(b) if shape == "shared" else w.reshape(-1)

    xc = x.cuda().requires_grad_(True)
    wc = w_ours.cuda().requires_grad_(True)
    if signature == "pipegraph":
        y = conv(xc, g, wc)
    else:
        xc2 = xc.view(b * n, d)
        wc2 = wc.repeat(b) if shape == "shared" else wc
        y = conv(xc2, big_ei.cuda(), wc2).view(b, n, d)
    (y * r.cuda()).sum().backward()

    x64 = x.double().view(b * n, d).requires_grad_(True)
    w64 = w_ref.double().requires_grad_(True)
    y64 = ref(x64, big_ei, w64).view(b, n, d)
    (y64 * r.double()).sum().backward()
    dw64 = w64.grad.view(b, -1).sum(0) if shape == "shared" else w64.grad.view(b, -1)
    rep = {"y": rel_err(y, y64), "dx": rel_err(xc.grad, x64.grad.view(b, n, d)),
           "dW": rel_err(conv.lin.weight.grad, ref.lin.weight.grad), "db": rel_err(conv.bias.grad, ref.bias.grad),
           "d_edge_weight": rel_err(wc.grad, dw64)}
    parity_log(f"GCNConv {signature} {shape}", rep)
    assert all(e <= TOL for e in rep.values()), rep


def test_gcnconv_without_weights_is_unchanged(lta):
    from leak_det_gnn_b200.nn import GCNConv

    ei, g = lta
    torch.manual_seed(4)
    conv = GCNConv(64, 64).cuda()
    x = torch.randn(2, 661, 64, device="cuda")
    assert rel_err(conv(x, g, torch.ones(g.num_edges, device="cuda")), conv(x, g)) <= 1e-6
    assert torch.equal(conv(x, g, None), ops.gcn_conv(x, g, conv.lin.weight, conv.bias))


# ---------------------------------------------------------------------------------------------------------- detector
def _detector(sensor_hidden, node_hidden, n_pipes=40, seed=19):
    from leak_det_gnn_b200.models import LeakDetector

    z = np.load(TOPO["LTA"].parent / "graph_LTA.npz")
    torch.manual_seed(seed)
    m = LeakDetector(TOPO["LTA"], [str(x) for x in z["sensor_node_ids"]], _pipes(n_pipes), sensor_hidden=sensor_hidden,
                     node_hidden=node_hidden)
    return m


def _oracle_detector(ours, state, dtype, train):
    from oracle.pyg_weighted import WeightedOracleLeakDetector

    m = WeightedOracleLeakDetector(len(ours.node_names), ours.edge_index_single, ours.pipe_ends, ours.sensor_node_idx.tolist(),
                           ours.sensor_encoder.hidden_size, ours.sensor_to_node.out_features, 2, 0.0, True).to(dtype)
    m.load_state_dict({k: v.to(dtype) for k, v in state.items()}, strict=True)
    return m.train(train)


@pytest.mark.parametrize("sensor_hidden,node_hidden", [(64, 64), (128, 128)])
@pytest.mark.parametrize("shape", ["shared", "per_window"])
@pytest.mark.parametrize("mode", ["eval", "train_p0"])
def test_detector_with_edge_weights_matches_oracle(sensor_hidden, node_hidden, shape, mode):
    """Logits, loss, all 18 parameter gradients, d edge_weight, d residual and d tfeat against the fp64 oracle."""
    ours = _detector(sensor_hidden, node_hidden)
    state = {k: v.clone() for k, v in ours.state_dict().items()}
    assert len(state) == 18
    ours = ours.cuda()
    for mod in ours.modules():  # the detector's own and the two head MLPs' dropouts
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    ours.train(mode != "eval")
    gen = torch.Generator().manual_seed(8)
    b, l, s, e = 6, 36, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen), torch.randn(b, l, 9, generator=gen)
    w = torch.rand(e, generator=gen) + 0.2 if shape == "shared" else torch.rand(b, e, generator=gen) + 0.2
    label = torch.randint(0, 41, (b,), generator=gen)

    def run(model, dtype, device):
        x = residual.to(device, dtype, copy=True).requires_grad_(True)
        t = tfeat.to(device, dtype, copy=True).requires_grad_(True)
        ew = w.to(device, dtype, copy=True).requires_grad_(True)
        logits = model(x, t, edge_weight=ew)
        loss = torch.nn.functional.cross_entropy(logits, label.to(device))
        loss.backward()
        grads = {k: p.grad for k, p in model.named_parameters()}
        return logits, loss, grads, ew.grad, x.grad, t.grad

    o64 = run(_oracle_detector(ours, state, torch.float64, mode != "eval"), torch.float64, "cpu")
    o32 = run(_oracle_detector(ours, state, torch.float32, mode != "eval"), torch.float32, "cpu")
    got = run(ours, torch.float32, "cuda")
    rep = {"logits": (rel_err(got[0], o64[0]), rel_err(o32[0], o64[0])),
           "loss": (rel_err(got[1].view(1), o64[1].view(1)), rel_err(o32[1].view(1), o64[1].view(1)))}
    for k in o64[2]:
        rep[k] = (rel_err(got[2][k], o64[2][k]), rel_err(o32[2][k], o64[2][k]))
    for i, k in ((3, "d_edge_weight"), (4, "d_residual"), (5, "d_tfeat")):
        rep[k] = (rel_err(got[i], o64[i]), rel_err(o32[i], o64[i]))
    assert got[3].shape == w.shape
    parity_log(f"detector edge weights {shape} {mode} sensor={sensor_hidden} node={node_hidden}",
               {k: {"ours": a, "oracle_fp32": c} for k, (a, c) in rep.items()})
    assert len(rep) == 18 + 5
    for k, (a, c) in rep.items():
        tol = 1e-4 if k.startswith("sensor_encoder.") else TOL  # BPTT over the window, as in test_detector_gpu
        assert a <= max(tol, 3.0 * c), (k, a, c)


def test_window_rows_are_batch_independent_and_deterministic():
    """Row b of a (B, E) gradient equals the (E,) gradient of a B = 1 call on window b, bit for bit; a second run gives
    the same bits.  (The logits pass through the no-leak MLP in torch, whose GEMM may change with B: to rounding.)"""
    ours = _detector(64, 64).cuda().eval().requires_grad_(False)
    gen = torch.Generator().manual_seed(12)
    b, s, e = 5, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    h_s = torch.randn(b, s, 64, generator=gen).cuda()
    target = torch.randint(0, 41, (b,), generator=gen).cuda()

    def grad(h, t, ew):
        ew = ew.clone().requires_grad_(True)
        logits = ours.gnn_stack(h, ew)
        return torch.autograd.grad(logits.gather(1, t[:, None]).sum(), ew)[0], logits.detach()

    ones = torch.ones(b, e, device="cuda")
    full, logits = grad(h_s, target, ones)
    again, logits2 = grad(h_s, target, ones)
    assert torch.equal(full, again) and torch.equal(logits, logits2)
    for i in range(b):
        one, lg = grad(h_s[i:i + 1], target[i:i + 1], torch.ones(e, device="cuda"))
        assert one.shape == (e,)
        assert torch.equal(one, full[i]), i
        assert rel_err(lg, logits[i:i + 1]) <= 1e-6, i
    assert torch.equal(ours.gnn_stack(h_s, torch.ones(e, device="cuda")), ours.gnn_stack(h_s, ones))


def test_lta4096_pipe_attribution_matches_fp64_on_sampled_windows():
    """The per-pipe attribution recipe at the lta4096 shape (B = 4096, L = 288, all 764 pipes, frozen, eval): d target
    logit / d (B, E) ones, one backward; sampled windows against the fp64 oracle run on those windows alone."""
    ours = _detector(64, 64, n_pipes=764, seed=23)
    state = {k: v.clone() for k, v in ours.state_dict().items()}
    ours = ours.cuda().eval().requires_grad_(False)
    gen = torch.Generator().manual_seed(9)
    b, l, s, e = 4096, 288, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen), torch.randn(b, l, 9, generator=gen)
    target = torch.randint(0, 765, (b,), generator=gen)
    ew = torch.ones(b, e, device="cuda", requires_grad=True)
    logits = ours(residual.cuda(), tfeat.cuda(), edge_weight=ew)
    (dw,) = torch.autograd.grad(logits.gather(1, target.cuda()[:, None]).sum(), ew)
    pipe_score = dw.view(b, -1, 2).sum(-1)  # link p = edges 2p and 2p + 1
    assert pipe_score.shape == (b, e // 2)
    sample = [0, 1, 2047, 4095]
    rep = {}
    for dtype in (torch.float64, torch.float32):
        m = _oracle_detector(ours, state, dtype, False)
        ew_o = torch.ones(len(sample), e, dtype=dtype, requires_grad=True)
        lo = m(residual[sample].to(dtype), tfeat[sample].to(dtype), edge_weight=ew_o)
        (g,) = torch.autograd.grad(lo.gather(1, target[sample][:, None]).sum(), ew_o)
        rep[str(dtype)] = g
    ours_e, o32_e = rel_err(dw[sample], rep["torch.float64"]), rel_err(rep["torch.float32"], rep["torch.float64"])
    parity_log("lta4096 pipe attribution", {"ours": ours_e, "oracle_fp32": o32_e})
    assert ours_e <= max(TOL, 3.0 * o32_e), (ours_e, o32_e)


def test_weighted_step_replays_in_a_cuda_graph():
    """Weighted forward and backward (parameter and edge-weight gradients) captured in a torch.cuda.graph replay equal
    to eager, bit for bit."""
    ours = _detector(64, 64).cuda().eval()
    gen = torch.Generator().manual_seed(14)
    b, s, e = 8, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    h_s = torch.randn(b, s, 64, generator=gen).cuda()
    ew = (torch.rand(b, e, generator=gen) + 0.5).cuda().requires_grad_(True)
    label = torch.randint(0, 41, (b,), generator=gen).cuda()
    params = [p for n, p in ours.named_parameters() if not n.startswith("sensor_encoder.")]

    def step():
        loss = torch.nn.functional.cross_entropy(ours.gnn_stack(h_s, ew), label)
        return torch.autograd.grad(loss, [ew] + params)

    eager = [t.clone() for t in step()]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    graph.replay()
    torch.cuda.synchronize()
    for a, c in zip(static, eager):
        assert torch.equal(a, c)
