"""Explainer edge masks, host side: the oracle's message mask against a dense formula on a graph with an input self
loop, the batched GNNExplainer restatement against B single-window runs of PyG's loop, the new C symbols, and the mask
checks that run before any device work."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import TOPO
from leak_det_gnn_b200.graph import build_wdn_graph_from_inp, parse_epanet_inp
from oracle.pyg_explain import GCNConv, MaskedOracleLeakDetector, explain_batched, explain_single, initial_logits

NEW_SYMBOLS = ("ltgnn_edge_mask_fwd", "ltgnn_edge_mask_bwd", "ltgnn_explain_step")


def _loop_graph():
    """5 nodes, both directions of four links, and edge 4 an input self loop at node 2."""
    return torch.tensor([[0, 1, 1, 2, 2, 2, 3, 3, 4],
                         [1, 0, 2, 1, 2, 3, 2, 4, 3]])


def test_oracle_mask_matches_dense_formula():
    ei, n = _loop_graph(), 5
    gen = torch.Generator().manual_seed(0)
    conv = GCNConv(4, 3).double()
    with torch.no_grad():
        conv.bias.normal_(generator=gen)
    x = torch.randn(n, 4, generator=gen, dtype=torch.float64)
    w = torch.rand(ei.shape[1], generator=gen, dtype=torch.float64) + 0.2
    mask = torch.rand(ei.shape[1], generator=gen, dtype=torch.float64).requires_grad_(True)
    for weight in (None, w):
        # dense: A[dst, src] = w (input loop dropped, its weight kept on the appended loop), deg over rows, then the
        # normalised value of every off-diagonal edge times its mask; the diagonal unmasked
        a = torch.zeros(n, n, dtype=torch.float64)
        m = torch.zeros(n, n, dtype=torch.float64)
        loop = torch.ones(n, dtype=torch.float64)
        for e in range(ei.shape[1]):
            s, d = int(ei[0, e]), int(ei[1, e])
            we = 1.0 if weight is None else weight[e]
            if s == d:
                loop[s] = we
            else:
                a[d, s] += we
        a = a + torch.diag(loop)
        dis = a.sum(1).pow(-0.5)
        for e in range(ei.shape[1]):
            s, d = int(ei[0, e]), int(ei[1, e])
            if s != d:
                m[d, s] += dis[d] * (1.0 if weight is None else weight[e]) * dis[s] * mask[e]
        m = m + torch.diag(dis * loop * dis)
        want = m @ (x @ conv.lin.weight.t()) + conv.bias
        got = conv(x, ei, weight, mask)
        assert (got - want).abs().max().item() <= 1e-14
        (g,) = torch.autograd.grad(got.sum(), mask)
        assert g[4].item() == 0.0 and (g[[0, 1, 2, 3, 5, 6, 7, 8]] != 0).all()
    assert torch.equal(conv(x, ei, None, torch.ones(ei.shape[1], dtype=torch.float64)), conv(x, ei))


def _small_detector():
    sec = parse_epanet_inp(TOPO["LTA"])
    z = np.load(TOPO["LTA"].parent / "graph_LTA.npz")
    sensors = [str(x) for x in z["sensor_node_ids"]]
    g = build_wdn_graph_from_inp(TOPO["LTA"], sensors, [ln.split()[0] for ln in sec["PIPES"]][:6], add_self_loops=False)
    torch.manual_seed(0)
    m = MaskedOracleLeakDetector(len(g.node_names), g.edge_index, torch.tensor(g.pipe_ends),
                                 [g.node_to_idx[s] for s in sensors], dropout=0.0).double().eval()
    return m, len(sensors)


def test_batched_loop_equals_single_window_runs():
    """The batched restatement (loss summed over windows, per-window regularisers on per-window hard masks) is B
    independent runs of PyG's loop: an epoch 0 with the regulariser, or a hard mask not taken from epoch 0's gradient,
    would move the masks far beyond rounding."""
    model, s = _small_detector()
    gen = torch.Generator().manual_seed(1)
    b, e, n = 3, model.edge_index_single.shape[1], model.num_nodes
    h_s = torch.randn(b, s, 64, generator=gen, dtype=torch.float64)
    target = torch.tensor([2, 6, 0])  # 6 = the no-leak class
    m0 = initial_logits(b, e, n, torch.Generator().manual_seed(2))
    mask, hard, logits = explain_batched(model, h_s, target, m0, epochs=8)
    assert mask.shape == (b, e) and hard.any(1).all()
    for i in range(b):
        one, one_hard, one_logits = explain_single(model, h_s[i:i + 1], int(target[i]), m0[i], epochs=8)
        assert torch.equal(one_hard, hard[i])
        assert (one - mask[i]).abs().max().item() <= 1e-12
        assert (one_logits - logits[i]).abs().max().item() <= 1e-12
    # the regularisers act from epoch 1 on: one epoch is plain Adam on the cross-entropy, two are not
    first, _, _ = explain_batched(model, h_s, target, m0, epochs=1)
    p = torch.nn.Parameter(m0.clone().double())
    opt = torch.optim.Adam([p], lr=0.01)
    torch.nn.functional.cross_entropy(model.gnn_stack(h_s, edge_mask=p.sigmoid()), target, reduction="sum").backward()
    opt.step()
    assert (first - torch.where(hard, p.detach().sigmoid(), 0.0)).abs().max().item() <= 1e-15


def test_new_symbols_are_exported():
    from leak_det_gnn_b200 import lib as _lib

    so = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in NEW_SYMBOLS:
        assert hasattr(so, name), name
        assert name in _lib.SIGNATURES


def test_bad_masks_raise_before_any_launch():
    from leak_det_gnn_b200 import instrument, ops
    from leak_det_gnn_b200.nn import GCNConv as Conv

    g = ops.PipeGraph(_loop_graph(), 5)
    instrument.reset()
    with pytest.raises(ValueError, match="CUDA"):
        ops.normalized_edge_values(g, None, 1, torch.ones(g.num_edges))
    conv = Conv(8, 8)
    with pytest.raises(ValueError, match="CUDA"):
        conv(torch.randn(1, 5, 8), g, edge_mask=torch.ones(g.num_edges))
    for bad in (torch.ones(g.num_edges + 1), torch.ones(2, g.num_edges), torch.ones(1, 1, g.num_edges)):
        with pytest.raises(ValueError, match=r"edge_mask must be \(9,\)"):
            ops.normalized_edge_values(g, None, 3, bad)
    assert instrument.launches == 0
