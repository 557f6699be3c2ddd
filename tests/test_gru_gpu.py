"""Sensor GRU encoder kernel vs torch.nn.GRU in fp64 on the CPU (the reference calls nn.GRU; detector.py:50-73)."""
import pytest
import torch

from conftest import rel_err
from leak_det_gnn_b200 import ops

pytestmark = pytest.mark.gpu


def _ref(r, tf, gru):
    b, l, s = r.shape
    seq = r.transpose(1, 2).reshape(b * s, l, 1)
    if tf is not None:
        seq = torch.cat([seq, tf.unsqueeze(1).expand(b, s, l, tf.shape[-1]).reshape(b * s, l, -1)], dim=-1)
    out, _ = gru(seq)
    return out  # (B*S, L, H)


@pytest.mark.parametrize("b,l,s,f", [(1, 1, 1, 0), (3, 36, 29, 9), (10, 36, 29, 9), (2, 288, 29, 9), (5, 12, 7, 3),
                                     (40, 5, 29, 0)])
def test_gru_forward(b, l, s, f):
    torch.manual_seed(b * 100 + l)
    gru = torch.nn.GRU(input_size=1 + f, hidden_size=64, num_layers=1, batch_first=True).double()
    r = torch.randn(b, l, s)
    tf = torch.randn(b, l, f) if f else None
    out = _ref(r.double(), None if tf is None else tf.double(), gru)
    w = [getattr(gru, n).detach().float().cuda() for n in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")]
    h_last, hseq, gates = ops.gru_fwd(r.cuda(), None if tf is None else tf.cuda(), *w, save=True)
    hseq = ops.unblock32(hseq, l, b * s)
    assert h_last.shape == (b, s, 64) and hseq.shape == (l, b * s, 64)
    assert rel_err(hseq.permute(1, 0, 2), out) <= 2e-5
    assert rel_err(h_last.reshape(b * s, 64), out[:, -1, :]) <= 2e-5
    h2 = ops.gru_fwd(r.cuda(), None if tf is None else tf.cuda(), *w)
    assert torch.equal(h2, h_last)


@pytest.mark.parametrize("b,l,s,f", [(2, 5, 3, 2), (3, 36, 29, 9), (7, 20, 29, 9), (2, 100, 29, 9), (9, 8, 11, 0)])
def test_gru_backward(b, l, s, f):
    """BPTT from the saved r | z | n and states (hn rebuilt per step) + the weight-gradient pass, against fp64 nn.GRU."""
    torch.manual_seed(7 * b + l)
    gru = torch.nn.GRU(input_size=1 + f, hidden_size=64, num_layers=1, batch_first=True).double()
    r = torch.randn(b, l, s)
    tf = torch.randn(b, l, f) if f else None
    dh = torch.randn(b * s, 64)
    out = _ref(r.double(), None if tf is None else tf.double(), gru)
    (out[:, -1, :] * dh.double()).sum().backward()
    names = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")
    w = [getattr(gru, n).detach().float().cuda().requires_grad_(True) for n in names]
    h = ops.gru_encode(r.cuda(), None if tf is None else tf.cuda(), *w)
    (h.reshape(b * s, 64) * dh.cuda()).sum().backward()
    for n, p in zip(names, w):
        ref = getattr(gru, n).grad
        assert rel_err(p.grad, ref) <= 5e-5, (n, rel_err(p.grad, ref))


def test_encoder_module_native_matches_cudnn():
    from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder
    torch.manual_seed(3)
    enc = SharedSensorGRUEncoder(hidden_size=64).cuda().train()
    r = torch.randn(6, 36, 29, device="cuda")
    tf = torch.randn(6, 36, 9, device="cuda")
    dh = torch.randn(6, 29, 64, device="cuda")
    (enc(r, tf) * dh).sum().backward()
    native = [p.grad.clone() for p in enc.parameters()]
    h_native = enc(r, tf).detach()
    enc.zero_grad()
    enc.use_native = False
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        h_cudnn = enc(r, tf)
        (h_cudnn * dh).sum().backward()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert rel_err(h_native, h_cudnn) <= 2e-5
    for a, p in zip(native, enc.parameters()):
        assert rel_err(a, p.grad) <= 1e-4
