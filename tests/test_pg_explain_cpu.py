"""PGExplainer, host side: the per-node factorisation of the edge MLP and its node-centric backward against PyG's
concatenated form in fp64, the temperature schedule and concrete sample, the batched oracle step against PyG's loss on
the disjoint union taken apart window by window, the new C symbols, and the argument checks."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import TOPO
from leak_det_gnn_b200.graph import build_wdn_graph_from_inp, parse_epanet_inp
from oracle.pyg_explain import MaskedOracleLeakDetector
from oracle.pyg_pg_explainer import PGExplainerOracle

NEW_SYMBOLS = ("ltgnn_pg_edge_fwd", "ltgnn_pg_edge_bwd", "ltgnn_pg_edge_bwd_ws_floats")


def _graph(n=23, e=60, seed=0):
    gen = torch.Generator().manual_seed(seed)
    ei = torch.randint(0, n, (2, e), generator=gen)
    ei[:, 5] = torch.tensor([3, 3])  # an input self loop
    return ei, n


def _mlp(d, seed=1):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(2 * d, 64), torch.nn.ReLU(), torch.nn.Linear(64, 1)).double()


@pytest.mark.parametrize("d", [64, 128])
def test_factorised_mlp_and_node_centric_backward_equal_pyg_form(d):
    from leak_det_gnn_b200.ops import pg_edge_index

    ei, n = _graph()
    b = 3
    gen = torch.Generator().manual_seed(2)
    z = torch.randn(b, n, d, generator=gen, dtype=torch.float64)
    mlp = _mlp(d)
    w1, b1, w2, b2 = mlp[0].weight, mlp[0].bias, mlp[2].weight, mlp[2].bias
    # PyG: the concatenated input, one row per (window, edge)
    inputs = torch.cat([z[:, ei[0]], z[:, ei[1]]], -1)                  # (B, E, 2D)
    logit = mlp(inputs).squeeze(-1)
    dl = torch.randn(logit.shape, generator=gen, dtype=torch.float64)
    grads = torch.autograd.grad((logit * dl).sum(), [w1, b1, w2, b2])
    # the factorisation: [P | Q] = z [W1a; W1b]^T, per edge (P[src] + Q[dst]) + b1
    with torch.no_grad():
        pq = z @ torch.cat([w1[:, :d], w1[:, d:]], 0).t()              # (B, N, 128)
        pre = (pq[:, ei[0], :64] + pq[:, ei[1], 64:]) + b1
        h = pre.clamp(min=0)
        fact = h @ w2[0] + b2
        assert (fact - logit).abs().max().item() <= 1e-12
        # the node-centric backward: gated hidden gradient summed by source / target in ascending edge order
        src, dst, out_ptr, out_edge, in_ptr, in_edge = (t.long() for t in pg_edge_index(ei, n, torch.device("cpu")))
        assert torch.equal(out_edge, torch.sort(ei[0], stable=True).indices)
        gh = dl[..., None] * w2[0] * (pre > 0)
        r = torch.zeros(b, n, 128, dtype=torch.float64)
        for i in range(n):
            for k in range(int(out_ptr[i]), int(out_ptr[i + 1])):
                r[:, i, :64] += gh[:, out_edge[k]]
            for k in range(int(in_ptr[i]), int(in_ptr[i + 1])):
                r[:, i, 64:] += gh[:, in_edge[k]]
        dws = r.reshape(-1, 128).t() @ z.reshape(-1, d)                 # wgrad: R^T z
        ours = [torch.cat([dws[:64], dws[64:]], 1), gh.sum((0, 1)), (dl[..., None] * h).sum((0, 1)).view(1, 64),
                dl.sum().view(1)]
    for name, a, c in zip(("dW1", "db1", "dw2", "db2"), ours, grads):
        assert (a - c).abs().max().item() <= 1e-12 * max(1.0, c.abs().max().item()), name


def test_temperature_and_concrete_sample():
    ex = PGExplainerOracle(64, epochs=30)
    assert ex._get_temperature(0) == 5.0
    for ep in (1, 17, 29):
        assert ex._get_temperature(ep) == pytest.approx(5.0 * (2.0 / 5.0) ** (ep / 30), rel=1e-15)
    gen = torch.Generator().manual_seed(3)
    logits = torch.randn(4, 9, generator=gen, dtype=torch.float64)
    u = torch.rand(4, 9, generator=gen, dtype=torch.float64)
    eps = 0.98 * u + 0.01
    want = (torch.log(eps) - torch.log(1 - eps) + logits) / 3.0
    assert (ex._concrete_sample(logits, 3.0, u) - want).abs().max().item() <= 1e-15
    flat = PGExplainerOracle(64, epochs=30, bias=0.5)
    assert torch.equal(flat._concrete_sample(logits, 3.0, u), logits / 3.0)


def _small_detector(d=64, n_pipes=6):
    sec = parse_epanet_inp(TOPO["LTA"])
    z = np.load(TOPO["LTA"].parent / "graph_LTA.npz")
    sensors = [str(x) for x in z["sensor_node_ids"]]
    g = build_wdn_graph_from_inp(TOPO["LTA"], sensors, [ln.split()[0] for ln in sec["PIPES"]][:n_pipes],
                                 add_self_loops=False)
    torch.manual_seed(0)
    m = MaskedOracleLeakDetector(len(g.node_names), g.edge_index, torch.tensor(g.pipe_ends),
                                 [g.node_to_idx[s] for s in sensors], sensor_hidden=d, node_hidden=d,
                                 dropout=0.0).double().eval()
    return m, len(sensors)


def test_batched_step_is_pyg_on_the_disjoint_union():
    """B windows in one step are PyG's step on their disjoint union: mean cross-entropy over the windows, the size
    term over all B E edges, the entropy mean over all B E edges -- taken apart here window by window (each window's
    own PyG loss pieces on its own graph), gradients to 1e-12."""
    model, s = _small_detector()
    gen = torch.Generator().manual_seed(4)
    b, e = 3, model.edge_index_single.shape[1]
    h_s = torch.randn(b, s, 64, generator=gen, dtype=torch.float64)
    target = torch.tensor([2, 6, 0])  # 6: the no-leak class
    u = torch.rand(b, e, generator=gen, dtype=torch.float64)
    ex = PGExplainerOracle(64, epochs=5).double()
    twin = PGExplainerOracle(64, epochs=5).double()
    twin.load_state_dict(ex.state_dict())
    loss = ex.train(2, model, h_s, target, u)
    temp = ex._get_temperature(2)
    # window by window on a one-window graph
    total = 0.0
    for i in range(b):
        z = twin.get_embeddings(model, h_s[i:i + 1])
        sm = twin._concrete_sample(twin.mlp(twin._get_inputs(z, model.edge_index_single)).view(-1), temp, u[i])
        y_hat = model.gnn_stack(h_s[i:i + 1], edge_mask=sm.sigmoid())
        m = 0.99 * sm.sigmoid() + 0.005
        ent = (-m * m.log() - (1 - m) * (1 - m).log()).sum()
        total = total + F.cross_entropy(y_hat, target[i:i + 1]) / b + 0.05 * sm.sigmoid().sum() + ent / (b * e)
    grads = torch.autograd.grad(total, list(twin.mlp.parameters()))
    assert abs(total.item() - loss.item()) <= 1e-12
    for p, g in zip(ex.mlp.parameters(), grads):
        assert (p.grad - g).abs().max().item() <= 1e-12
    assert ex._curr_epoch == 2
    with pytest.raises(ValueError, match="not yet fully trained"):
        ex(model, h_s)
    ex.train(4, model, h_s, target, u)
    assert ex(model, h_s).shape == (b, e)


def test_new_symbols_are_exported():
    from leak_det_gnn_b200 import lib as _lib

    so = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in NEW_SYMBOLS:
        assert hasattr(so, name), name
        assert name in _lib.SIGNATURES


def _cpu_detector():
    from leak_det_gnn_b200.models import LeakDetector

    sec = parse_epanet_inp(TOPO["LTA"])
    z = np.load(TOPO["LTA"].parent / "graph_LTA.npz")
    torch.manual_seed(0)
    return LeakDetector(TOPO["LTA"], [str(x) for x in z["sensor_node_ids"]], [ln.split()[0] for ln in sec["PIPES"]][:6])


def test_bad_arguments_raise():
    from leak_det_gnn_b200 import explain, instrument, ops

    det = _cpu_detector()
    s, e = len(det.sensor_node_ids), det.edge_index_single.shape[1]
    with pytest.raises(ValueError, match="epochs"):
        explain.PGExplainer(det, epochs=0)
    with pytest.raises(ValueError, match="unknown coefficients"):
        explain.PGExplainer(det, epochs=3, edge_sz=0.1)
    with pytest.raises(ValueError, match="bias"):
        explain.PGExplainer(det, epochs=3, bias=0.7)
    ex = explain.PGExplainer(det, epochs=3)
    assert list(ex.state_dict()) == ["mlp.0.weight", "mlp.0.bias", "mlp.2.weight", "mlp.2.bias"]
    assert tuple(ex.mlp[0].weight.shape) == (64, 128)
    r, t = torch.randn(2, 12, s), torch.randn(2, 12, 9)
    instrument.reset()
    for bad in (-1, 3, 1.0, True):
        with pytest.raises(ValueError, match="epoch"):
            ex.train(bad, r, t, torch.zeros(2, dtype=torch.long))
    for bad in (None, torch.zeros(3, dtype=torch.long), torch.zeros(2), torch.tensor([0, 7])):
        with pytest.raises(ValueError, match="target"):
            ex.train(0, r, t, bad)
    with pytest.raises(ValueError, match="CUDA"):  # CPU tensors: no CPU path
        ex.train(0, r, t, torch.zeros(2, dtype=torch.long))
    with pytest.raises(ValueError, match="not yet fully trained"):
        ex.explain(r, t)
    assert det.training and all(p.requires_grad for p in det.parameters())  # restored after the failures
    assert ex.eval() is ex and not ex.training  # nn.Module.train(False) still works
    ex.load_state_dict({k: v.clone() for k, v in ex.state_dict().items()})  # a loaded MLP counts as trained
    with pytest.raises(ValueError, match="CUDA"):
        ex.explain(r, t)
    idx = ops.pg_edge_index(det.edge_index_single, len(det.node_names), torch.device("cpu"))
    w = [p.detach() for p in ex.mlp.parameters()]
    with pytest.raises(ValueError, match="CUDA"):
        ops.pg_edge_mask(torch.zeros(2, len(det.node_names), 64), idx, *w)
    with pytest.raises(ValueError, match="edge_index"):
        ops.pg_edge_index(torch.tensor([[0, 1], [1, len(det.node_names)]]), len(det.node_names), torch.device("cpu"))
    assert instrument.launches == 0 and e > 0


def test_pinned_against_torch_geometric():
    tg = pytest.importorskip("torch_geometric")
    from torch_geometric.explain.algorithm import PGExplainer

    from conftest import parity_log

    real = PGExplainer(epochs=30, lr=0.003)
    ours = PGExplainerOracle(64, epochs=30)
    assert dict(real.coeffs) == {k: list(v) if isinstance(v, tuple) else v for k, v in ours.coeffs.items()}
    for ep in (0, 7, 29):
        assert real._get_temperature(ep) == pytest.approx(ours._get_temperature(ep), rel=1e-15)
    logits = torch.randn(50, dtype=torch.float64)
    torch.manual_seed(5)
    got = real._concrete_sample(logits, 2.5)
    torch.manual_seed(5)
    u = torch.rand_like(logits)
    assert (got - ours._concrete_sample(logits, 2.5, u)).abs().max().item() <= 1e-12
    parity_log("pyg_pin PGExplainer", {"torch_geometric": tg.__version__})
