"""NormalPredictorGRU.forward_last off the native shapes / devices: on CPU it is the dense forward, and like the TCN's it
refuses train mode."""
import pytest
import torch

from leak_det_gnn_b200.models import NormalPredictorGRU


def test_forward_last_on_cpu_is_the_dense_forward():
    torch.manual_seed(0)
    m = NormalPredictorGRU(29, 9).eval()
    x, tf = torch.randn(5, 12, 29), torch.randn(5, 12, 9)
    assert not m._native_ok(x)
    with torch.no_grad():
        ref = m(x, tf)
    assert torch.equal(m.forward_last(x, tf), ref)
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.forward_last(x, tf)


def test_state_dict_keys_unchanged():
    m = NormalPredictorGRU(29, 9)
    keys = [f"gru.{k}_l{i}" for i in range(2) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
    assert sorted(m.state_dict()) == sorted(keys + ["head.weight", "head.bias"])
