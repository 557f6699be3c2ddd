"""NormalPredictorGRU.forward_cone off the native shapes (here: on the CPU) is the dense ``forward``, in value and in every
parameter gradient."""
import torch

from leak_det_gnn_b200.models import NormalPredictorGRU


def test_forward_cone_on_cpu_is_the_dense_forward():
    torch.manual_seed(0)
    m = NormalPredictorGRU(29, 9).double().eval()
    x, xt, y = torch.randn(4, 36, 29).double(), torch.randn(4, 36, 9).double(), torch.randn(4, 29).double()
    pred = m.forward_cone(x, xt)
    assert torch.equal(pred, m(x, xt))
    torch.nn.functional.mse_loss(pred, y).backward()
    g_cone = [p.grad.clone() for p in m.parameters()]
    m.zero_grad()
    torch.nn.functional.mse_loss(m(x, xt), y).backward()
    assert len(g_cone) == 10
    for a, p in zip(g_cone, m.parameters()):
        assert torch.equal(a, p.grad)
