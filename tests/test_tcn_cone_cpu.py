"""The host side of TCN predictor training: the inverse gather indices (every input row is read by at most one output
row per tap) and the torch-op cone that ``forward_cone`` uses off the native shapes, against the dense model."""
import torch

from leak_det_gnn_b200.models import NormalPredictorTCN


def test_inverse_indices_invert_the_gathers():
    m = NormalPredictorTCN(29, 9)
    rows, inv = m._native_rows(36, 3, "cpu"), m._native_inverse(36, 3, "cpu")
    n_in = 3 * 36
    for (src1, src2, keep), (inv1, inv2, keep_inv) in zip(rows, inv):
        for src, iv in ((src1, inv1), (src2, inv2)):
            assert iv.dtype == torch.int32 and iv.shape[0] == src.shape[0]
            for t in range(src.shape[0]):
                ok = src[t] >= 0
                assert torch.equal(iv[t, src[t][ok].long()], torch.arange(src.shape[1], dtype=torch.int32)[ok])
                assert int((iv[t] >= 0).sum()) == int(ok.sum())
        assert inv1.shape[1] == n_in and torch.equal(keep_inv[keep.long()], torch.arange(keep.numel(), dtype=torch.int32))
        n_in = keep.numel()


def test_cone_torch_gradients_equal_dense():
    torch.manual_seed(0)
    m = NormalPredictorTCN(29, 9).double().eval()
    x, xt, y = torch.randn(4, 36, 29).double(), torch.randn(4, 36, 9).double(), torch.randn(4, 29).double()
    torch.nn.functional.mse_loss(m.forward_cone(x, xt), y).backward()
    g_cone = [p.grad.clone() for p in m.parameters()]
    m.zero_grad()
    torch.nn.functional.mse_loss(m(x, xt), y).backward()
    for a, p in zip(g_cone, m.parameters()):
        assert torch.allclose(a, p.grad, rtol=1e-10, atol=1e-12)
