"""Weighted message passing, host side: the weighted restatement of PyG's gcn_norm against the unweighted one and a
dense fp64 construction, the entry -> edge maps of build_gcn_csr, the new C symbols, and the argument checks that run
before any device work."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import TOPO
from leak_det_gnn_b200.graph import build_gcn_csr, build_wdn_graph_from_inp, gcn_norm_edges, parse_epanet_inp
from oracle.pyg_weighted import gcn_norm

NEW_SYMBOLS = ("ltgnn_spmm_fused_vals", "ltgnn_edge_norm_fwd", "ltgnn_edge_norm_bwd", "ltgnn_gcn_adj_grad")


def _lta_edge_index():
    sec = parse_epanet_inp(TOPO["LTA"])
    pipes = [ln.split()[0] for ln in sec["PIPES"]][:4]
    return build_wdn_graph_from_inp(TOPO["LTA"], [], pipes, add_self_loops=False).edge_index


def _with_loops():
    """A small graph with existing self loops: node 1 twice (the last one counts), node 3 once, nodes 0, 2, 4 none."""
    return torch.tensor([[0, 1, 1, 2, 3, 1, 2, 4, 3, 1],
                         [1, 0, 1, 1, 3, 2, 4, 2, 0, 1]])


def _dense_norm(ei: torch.Tensor, w: torch.Tensor, n: int) -> torch.Tensor:
    """D^-1/2 (A_w + I') D^-1/2 in fp64, A[dst, src]: I' carries each node's (last) existing loop weight, else 1."""
    a = torch.zeros(n, n, dtype=torch.float64)
    loop = torch.ones(n, dtype=torch.float64)
    for e in range(ei.shape[1]):
        s, d = int(ei[0, e]), int(ei[1, e])
        if s == d:
            loop[s] = w[e]
        else:
            a[d, s] += w[e]
    a += torch.diag(loop)
    dis = a.sum(1).pow(-0.5)
    dis[torch.isinf(dis)] = 0
    return dis[:, None] * a * dis[None, :]


def _sparse_to_dense(ei: torch.Tensor, norm: torch.Tensor, n: int) -> torch.Tensor:
    a = torch.zeros(n, n, dtype=torch.float64)
    a.index_put_((ei[1], ei[0]), norm.double(), accumulate=True)
    return a


def test_weighted_oracle_at_ones_is_bitwise_the_unweighted_norm():
    for ei, n in ((_lta_edge_index(), 661), (_with_loops(), 5)):
        ref_ei, ref = gcn_norm_edges(ei, n)
        out_ei, out = gcn_norm(ei, n, edge_weight=torch.ones(ei.shape[1]))
        assert torch.equal(out_ei, ref_ei)
        assert torch.equal(out.view(torch.int32), ref.view(torch.int32))
        _, unweighted = gcn_norm(ei, n)
        assert torch.equal(unweighted.view(torch.int32), ref.view(torch.int32))


@pytest.mark.parametrize("case", ["lta", "loops"])
def test_weighted_oracle_matches_dense_fp64(case):
    ei, n = (_lta_edge_index(), 661) if case == "lta" else (_with_loops(), 5)
    w = torch.rand(ei.shape[1], generator=torch.Generator().manual_seed(3), dtype=torch.float64) * 2 + 0.1
    out_ei, norm = gcn_norm(ei, n, dtype=torch.float64, edge_weight=w)
    dense = _dense_norm(ei, w, n)
    assert (_sparse_to_dense(out_ei, norm, n) - dense).abs().max().item() <= 1e-14 * dense.abs().max().item()


@pytest.mark.parametrize("case", ["lta", "loops"])
def test_entry_edge_maps_reproduce_the_csr_orders(case):
    """Entry k of A_hat / A_hat^T comes from edge `edge[k]` / `t_edge[k]`: its endpoints are the entry's row and
    column, every non-loop edge owns exactly one entry, an appended loop points at the node's last loop or -1, and the
    transposed map is the forward map through t_perm."""
    ei, n = (_lta_edge_index(), 661) if case == "lta" else (_with_loops(), 5)
    c = build_gcn_csr(ei, n)
    assert c.num_edges == ei.shape[1] and c.edge.dtype == np.int32 and c.t_edge.dtype == np.int32
    rows = np.repeat(np.arange(n), np.diff(c.rowptr))
    src, dst = ei[0].numpy(), ei[1].numpy()
    for k in range(c.nnz):
        e = c.edge[k]
        if rows[k] == c.col[k]:
            loops = np.nonzero((src == rows[k]) & (dst == rows[k]))[0]
            assert e == (loops[-1] if len(loops) else -1)
        else:
            assert e >= 0 and src[e] == c.col[k] and dst[e] == rows[k]
    assert np.array_equal(c.edge[c.t_perm], c.t_edge)
    kept = np.sort(c.edge[(c.edge >= 0) & (rows != c.col)])
    assert np.array_equal(kept, np.nonzero(src != dst)[0])


def test_weighted_oracle_detector_at_ones_is_the_unweighted_one():
    """The weighted restatement adds to the unweighted oracle without changing it: at weight 1, shared or per window,
    the logits are those of the unweighted oracle detector bit for bit, and without weights it is that detector."""
    from leak_det_gnn_b200.graph import build_wdn_graph_from_inp as build
    from oracle.detector_oracle import OracleLeakDetector
    from oracle.pyg_weighted import WeightedOracleLeakDetector

    sec = parse_epanet_inp(TOPO["LTA"])
    z = np.load(TOPO["LTA"].parent / "graph_LTA.npz")
    sensors = [str(x) for x in z["sensor_node_ids"]]
    g = build(TOPO["LTA"], sensors, [ln.split()[0] for ln in sec["PIPES"]][:6], add_self_loops=False)
    args = (len(g.node_names), g.edge_index, torch.tensor(g.pipe_ends), [g.node_to_idx[s] for s in sensors])
    torch.manual_seed(0)
    ref = OracleLeakDetector(*args).eval()
    ours = WeightedOracleLeakDetector(*args).eval()
    ours.load_state_dict(ref.state_dict(), strict=True)
    gen = torch.Generator().manual_seed(1)
    b, e = 3, g.edge_index.shape[1]
    r, tf = torch.randn(b, 12, len(sensors), generator=gen), torch.randn(b, 12, 9, generator=gen)
    want = ref(r, tf)
    assert torch.equal(ours(r, tf), want)
    assert torch.equal(ours(r, tf, edge_weight=torch.ones(e)), want)
    assert torch.equal(ours(r, tf, edge_weight=torch.ones(b, e)), want)


def test_weighted_oracle_gives_replaced_duplicate_loops_no_gradient():
    w = torch.rand(10, generator=torch.Generator().manual_seed(4), dtype=torch.float64).add_(0.5).requires_grad_(True)
    _, norm = gcn_norm(_with_loops(), 5, dtype=torch.float64, edge_weight=w)
    norm.sum().backward()
    assert w.grad[2].item() == 0.0 and w.grad[9].item() != 0.0  # node 1's loops: edge 2 is replaced by edge 9


def test_new_symbols_are_exported():
    from leak_det_gnn_b200 import lib as _lib

    so = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in NEW_SYMBOLS:
        assert hasattr(so, name), name
        assert name in _lib.SIGNATURES


def test_cpu_tensors_and_bad_shapes_raise():
    from leak_det_gnn_b200 import ops
    from leak_det_gnn_b200.nn import GCNConv

    g = ops.PipeGraph(_with_loops(), 5)
    with pytest.raises(ValueError, match="CUDA"):
        ops.normalized_edge_values(g, torch.ones(g.num_edges), 1)
    with pytest.raises(ValueError, match="CUDA"):
        ops.edge_norm(g, torch.ones(g.num_edges))
    conv = GCNConv(8, 8)
    with pytest.raises(ValueError, match="CUDA"):
        conv(torch.randn(1, 5, 8), g, torch.ones(g.num_edges))
    for bad in (torch.ones(g.num_edges + 1), torch.ones(2, g.num_edges), torch.ones(1, 1, g.num_edges)):
        with pytest.raises(ValueError, match=r"edge_weight must be \(10,\)"):
            ops.normalized_edge_values(g, bad, 3)
