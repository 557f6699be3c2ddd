"""Host graph construction: bit-exact against goldens minted by the reference's own builder
(tests/golden/make_goldens.py; reference models/utils.py:84-166)."""
import hashlib

import numpy as np
import pytest
import torch

from conftest import TOPO
from leak_det_gnn_b200.graph import batchify_edge_index, build_gcn_csr, build_wdn_graph_from_inp, parse_epanet_inp
from oracle import pyg_restatement as pyg


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("net,n,e,p", [("LTA", 661, 1532, 764), ("LT", 785, 1818, 905)])
def test_graph_matches_reference_golden(graph_golden, net, n, e, p):
    g0 = graph_golden(net)
    sensors = [str(s) for s in g0["sensor_node_ids"]]
    pipes = [str(s) for s in g0["pipe_ids"]]
    g = build_wdn_graph_from_inp(TOPO[net], sensors, pipes, add_self_loops=False, make_undirected=True)
    assert len(g.node_names) == n and g.edge_index.shape == (2, e) and g.pipe_ends.shape == (p, 2)
    assert g.node_names == [str(s) for s in g0["node_names"]]
    assert g.edge_index.dtype == torch.long and g.pipe_ends.dtype == np.int64
    assert np.array_equal(g.edge_index.numpy(), g0["edge_index"])
    assert np.array_equal(g.pipe_ends, g0["pipe_ends"])
    assert _sha(g.edge_index.numpy()) == str(g0["sha_edge_index"])
    assert _sha(g.pipe_ends) == str(g0["sha_pipe_ends"])
    assert [g.node_to_idx[s] for s in sensors] == g0["sensor_node_idx"].tolist()
    assert g.pipe_ids == pipes and g.pipe_to_idx[pipes[3]] == 3


def test_survey_known_answers(graph_golden):
    """SURVEY.md F5 / 8a-a2 facts for L-TOWN-A."""
    g0 = graph_golden("LTA")
    sensors = [str(s) for s in g0["sensor_node_ids"]]
    pipes = [str(s) for s in g0["pipe_ids"]]
    g = build_wdn_graph_from_inp(TOPO["LTA"], sensors, pipes, add_self_loops=False)
    assert g.node_names[:8] == ["R1", "R2", "n100", "n101", "n102", "n103", "n104", "n105"]
    assert g.edge_index[:, :6].tolist() == [[465, 454, 505, 483, 647, 651], [454, 465, 483, 505, 651, 647]]
    assert g.pipe_ends[:3].tolist() == [[465, 454], [505, 483], [647, 651]]
    deg = np.bincount(g.edge_index[1].numpy(), minlength=661)
    assert np.bincount(deg).tolist() == [0, 24, 427, 187, 22, 1]
    assert (g.edge_index[0] != g.edge_index[1]).all()


def test_builder_options_and_errors(tmp_path):
    inp = tmp_path / "t.inp"
    inp.write_text("""
pre-header junk is ignored
[junctions]
 b 1 2 ; comment
 a
[RESERVOIRS]
 R
[PIPES]
;ID n1 n2
 p1 a b 10
 p2 b R 10 ; trailing
 bad a
 p1 R a 10
[PUMPS]
 u1 a c
[VALVES]
""")
    sec = parse_epanet_inp(inp)
    assert list(sec) == ["JUNCTIONS", "RESERVOIRS", "PIPES", "PUMPS", "VALVES"]
    assert sec["JUNCTIONS"] == ["b 1 2", "a"] and len(sec["PIPES"]) == 4
    g = build_wdn_graph_from_inp(inp, ["s9"], ["p2", "p1"], add_self_loops=True)
    # lexicographic order; 'c' only appears as a pump endpoint, 's9' only as a sensor
    assert g.node_names == ["R", "a", "b", "c", "s9"]
    # p1 redefined: keeps first position, takes last endpoints (R, a)
    assert g.edge_index.tolist() == [[0, 1, 2, 0, 1, 3, 0, 1, 2, 3, 4], [1, 0, 0, 2, 3, 1, 0, 1, 2, 3, 4]]
    assert g.pipe_ends.tolist() == [[2, 0], [0, 1]]
    g = build_wdn_graph_from_inp(inp, [], ["p1"], add_self_loops=False, make_undirected=False, include_links=("PIPES",))
    assert g.node_names == ["R", "a", "b"] and g.edge_index.tolist() == [[0, 2], [1, 0]]
    with pytest.raises(ValueError, match="not found"):
        build_wdn_graph_from_inp(inp, [], ["nope"])
    with pytest.raises(ValueError, match="No link endpoints"):
        build_wdn_graph_from_inp(inp, [], ["p1"], include_links=("VALVES",))
    (tmp_path / "e.inp").write_text("[PUMPS]\n u a b\n")
    with pytest.raises(ValueError, match="PIPES"):
        build_wdn_graph_from_inp(tmp_path / "e.inp", [], [])


@pytest.mark.parametrize("net", ["LTA", "LT"])
def test_csr_bit_exact_vs_pyg_restatement(graph_golden, net):
    g0 = graph_golden(net)
    ei = torch.from_numpy(g0["edge_index"])
    n = len(g0["node_names"])
    csr = build_gcn_csr(ei, n)
    ei2, norm = pyg.gcn_norm(ei, n)
    assert csr.nnz == ei.shape[1] + n == ei2.shape[1]
    # CSR -> COO multiset == PyG edge list (+ self loops); values bitwise
    rows = np.repeat(np.arange(n), np.diff(csr.rowptr))
    got = sorted(zip(csr.col.tolist(), rows.tolist(), csr.val.view(np.int32).tolist()))
    want = sorted(zip(ei2[0].tolist(), ei2[1].tolist(), norm.numpy().view(np.int32).tolist()))
    assert got == want
    # inside a row: edge order, self loop last
    for i in (0, 1, 17, n - 1):
        seg = csr.col[csr.rowptr[i]:csr.rowptr[i + 1]]
        assert seg[-1] == i
        assert seg[:-1].tolist() == ei[0][ei[1] == i].tolist()
    # the transposed arrays are the exact transpose, linked by t_perm
    t_rows = np.repeat(np.arange(n), np.diff(csr.t_rowptr))
    assert np.array_equal(csr.col[csr.t_perm], t_rows)
    assert np.array_equal(rows[csr.t_perm], csr.t_col)
    assert np.array_equal(csr.val.view(np.int32)[csr.t_perm], csr.t_val.view(np.int32))
    assert csr.rowptr.dtype == np.int32 and csr.col.dtype == np.int32 and csr.val.dtype == np.float32


def test_csr_batched_equals_single(graph_golden):
    """gcn_norm of the B-times replicated graph (what the reference feeds PyG) is B copies of the
    single-graph weights -- the fact the dense-batch design rests on (SURVEY F4)."""
    g0 = graph_golden("LTA")
    ei = torch.from_numpy(g0["edge_index"])
    n, b = 661, 3
    big, norm_big = pyg.gcn_norm(batchify_edge_index(ei, n, b), n * b)
    one, norm_one = pyg.gcn_norm(ei, n)
    e = ei.shape[1]
    for k in range(b):
        assert torch.equal(norm_big[k * e:(k + 1) * e], norm_one[:e])
        assert torch.equal(norm_big[b * e + k * n: b * e + (k + 1) * n], norm_one[e:])
        assert torch.equal(big[:, k * e:(k + 1) * e], one[:, :e] + k * n)


def test_csr_edge_cases():
    # existing self loop is replaced by exactly one; isolated node gets weight 1; duplicates kept
    ei = torch.tensor([[0, 1, 1, 2, 2, 0], [1, 0, 1, 0, 0, 2]])
    csr = build_gcn_csr(ei, 4)
    assert csr.nnz == 5 + 4
    assert csr.col[csr.rowptr[3]:csr.rowptr[4]].tolist() == [3] and csr.val[csr.rowptr[3]] == 1.0
    assert csr.col[csr.rowptr[0]:csr.rowptr[1]].tolist() == [1, 2, 2, 0]
    with pytest.raises(ValueError):
        build_gcn_csr(torch.tensor([[0], [5]]), 4)
    with pytest.raises(ValueError):
        build_gcn_csr(torch.zeros(3, 2, dtype=torch.long), 4)
    empty = build_gcn_csr(torch.zeros(2, 0, dtype=torch.long), 3)
    assert empty.nnz == 3 and empty.val.tolist() == [1.0, 1.0, 1.0]
