"""The oracle itself: pinned against the goldens produced by the reference's own LeakDetector code
(PyG operators supplied by the restatement -- 'parity unpinned' for those two, see
oracle/pyg_restatement.py) and internally cross-checked (C scatter-add == torch restatement)."""
import numpy as np
import pytest
import torch

from leak_det_gnn_b200.graph import build_gcn_csr
from oracle import c_oracle
from oracle import pyg_restatement as pyg
from oracle.detector_oracle import OracleLeakDetector


def _oracle_from_golden(graph_golden, g):
    g0 = graph_golden(g["net"])
    names = [str(s) for s in g0["node_names"]]
    idx = {n: i for i, n in enumerate(names)}
    pipe_row = {str(p): i for i, p in enumerate(g0["pipe_ids"])}
    ends = torch.from_numpy(g0["pipe_ends"][[pipe_row[p] for p in g["pipe_ids"]]])
    hp = g["hparams"]
    m = OracleLeakDetector(len(names), torch.from_numpy(g0["edge_index"]), ends,
                           [idx[s] for s in g["sensor_node_ids"]], hp["sensor_hidden"], hp["node_hidden"],
                           hp["gnn_layers"], hp["dropout"], hp["use_time"])
    m.load_state_dict(g["state_dict"], strict=True)
    return m.eval()


@pytest.fixture
def golden_threads():
    """The detector goldens were minted on 8 CPU threads.  Some of torch's fp32 CPU kernels split their sums by the
    thread count, so a bitwise reproduction runs on that count whatever the machine has."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("case", ["LTA_P2", "LTA_Pall", "LT_Pall", "LTA_D128_L3"])
def test_oracle_reproduces_reference_module(graph_golden, detector_golden, case, golden_threads):
    g = detector_golden(case)
    assert g["oracle_equals_reference_module_bitwise"] is True
    m = _oracle_from_golden(graph_golden, g)
    logits = m(g["residual"], g["tfeat"])
    loss = torch.nn.functional.cross_entropy(logits, g["label"])
    loss.backward()
    assert torch.equal(logits, g["logits"])
    assert torch.equal(loss, g["loss"])
    grads = {k: p.grad for k, p in m.named_parameters()}
    assert set(grads) == set(g["grads"]) and len(grads) == len(g["state_dict"])
    for k, v in g["grads"].items():
        assert torch.allclose(grads[k], v, rtol=0, atol=1e-7 * max(1.0, v.abs().max().item())), k


def test_fp64_oracle_close_to_fp32(graph_golden, detector_golden):
    g = detector_golden("LTA_Pall")
    m = _oracle_from_golden(graph_golden, g).double()
    logits = m(g["residual"].double(), g["tfeat"].double())
    err = (logits.float() - g["logits"]).abs().max() / g["logits"].abs().max()
    assert err < 1e-5


@pytest.mark.parametrize("net", ["LTA", "LT"])
def test_c_spmm_equals_torch_scatter_add_bitwise(graph_golden, net):
    g0 = graph_golden(net)
    ei = torch.from_numpy(g0["edge_index"])
    n = len(g0["node_names"])
    csr = build_gcn_csr(ei, n)
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(3, n, 32, generator=gen)
    y_c = c_oracle.spmm(csr.rowptr, csr.col, csr.val, x.numpy())
    ei2, norm = pyg.gcn_norm(ei, n)
    for b in range(3):
        y_t = pyg.propagate_add(ei2, norm, x[b])
        assert np.array_equal(y_c[b].view(np.int32), y_t.numpy().view(np.int32))
        y_e = c_oracle.scatter_add(ei2[0].numpy(), ei2[1].numpy(), norm.numpy(), x[b].numpy())
        assert np.array_equal(y_c[b].view(np.int32), y_e.view(np.int32))
    # transpose arrays give the adjoint: <A x, y> == <x, A^T y> (fp64 check of structure)
    yt = c_oracle.spmm(csr.t_rowptr, csr.t_col, csr.t_val, x.numpy())
    lhs = (torch.from_numpy(y_c).double() * x.flip(0).double()).sum()
    rhs = (x.double() * torch.from_numpy(c_oracle.spmm(csr.t_rowptr, csr.t_col, csr.t_val, x.flip(0).numpy())).double()).sum()
    assert abs(lhs - rhs) < 1e-6 * abs(lhs)
    assert yt.shape == x.shape


def test_gcnconv_restatement_properties():
    torch.manual_seed(0)
    conv = pyg.GCNConv(8, 5)
    assert list(conv.state_dict()) == ["bias", "lin.weight"]
    assert conv.lin.weight.shape == (5, 8) and torch.count_nonzero(conv.bias) == 0
    assert conv.lin.weight.abs().max() <= (6.0 / 13.0) ** 0.5
    # init draws glorot twice: second draw of the same stream
    torch.manual_seed(0)
    a = (6.0 / 13.0) ** 0.5
    _ = torch.empty(5, 8).uniform_(-a, a)
    second = torch.empty(5, 8).uniform_(-a, a)
    assert torch.equal(conv.lin.weight.detach(), second)
    # path graph 0-1-2: hand-computed normalisation
    ei = torch.tensor([[0, 1, 1, 2], [1, 0, 2, 1]])
    _, norm = pyg.gcn_norm(ei, 3)
    d = torch.tensor([2.0, 3.0, 2.0]).pow(-0.5)
    want = torch.stack([d[0] * d[1], d[1] * d[0], d[1] * d[2], d[2] * d[1], d[0] * d[0], d[1] * d[1], d[2] * d[2]])
    assert torch.equal(norm, want)
    x = torch.randn(6, 4)
    pooled = pyg.global_mean_pool(x, torch.tensor([0, 0, 0, 1, 1, 1]))
    assert torch.allclose(pooled, x.view(2, 3, 4).mean(1))
