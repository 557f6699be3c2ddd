"""``forward_windows`` on the sm_100a kernels: every window of a series from rows computed once, bit for bit what
``forward_last`` gives the materialised windows; the windowed GRU recurrence against the planar one; and the two
callers (residual builder, scenario scoring) and the graphed detector step with sharing on against sharing off."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import TOPO
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.event_windows import scenario_window_logits
from leak_det_gnn_b200.models import (LeakDetector, NormalPredictorGRU, NormalPredictorTCN,
                                      build_residual_sequence_from_segment)
from leak_det_gnn_b200.models.predictor import windows_of
from leak_det_gnn_b200.models.utils import residual_series

pytestmark = pytest.mark.gpu
ARCH = {"tcn": NormalPredictorTCN, "gru": NormalPredictorGRU}


def _pred(arch, seed=0):
    torch.manual_seed(seed)
    return ARCH[arch](29, 9).cuda().eval()


def _series(b, t, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, t, 29, generator=g).cuda(), torch.randn(b, t, 9, generator=g).cuda()


@pytest.mark.parametrize("arch", ["tcn", "gru"])
@pytest.mark.parametrize("b,t,window,count", [(256, 72, 36, 36), (1, 2017, 36, None), (3, 300, 20, None),
                                              (3, 300, 64, None), (2, 64, 64, None), (4, 72, 36, 1)])
def test_forward_windows_equals_forward_last(arch, b, t, window, count):
    m = _pred(arch)
    x, xt = _series(b, t, t + window)
    n = count or t - window + 1
    got = m.forward_windows(x, xt, window, count=count)
    want = m.forward_last(windows_of(x, window, n), windows_of(xt, window, n)).view(b, n, -1)
    assert got.shape == (b, n, 29)
    assert torch.equal(got, want)
    m.share_windows = False
    assert torch.equal(m.forward_windows(x, xt, window, count=count), want)


@pytest.mark.parametrize("q", [1, 127, 128, 129, 9216])
def test_gru_windowed_kernel_equals_planar(q):
    l, rows, hd = 36, q + 50, 128
    g = torch.Generator().manual_seed(q)
    gx = torch.randn(3, rows, hd, generator=g).cuda()
    base = torch.randint(0, rows - l + 1, (q,), generator=g, dtype=torch.int32).cuda()
    w_hh = (torch.randn(3 * hd, hd, generator=g) * 0.1).cuda()
    b_hn = (torch.randn(hd, generator=g) * 0.1).cuda()
    layer = (None, None, w_hh, b_hn)
    h_w, seq_w = ops.gru_layer_fwd_windows(gx, base, l, layer, seq=True)
    planar = gx[:, (base.long().unsqueeze(1) + torch.arange(l, device="cuda")).reshape(-1)].contiguous()  # (3, q l, H)
    h_p = torch.empty(q, hd, device="cuda")
    seq_p = torch.empty(q * l, hd, device="cuda")
    _lib.check(_lib.load().ltgnn_gru_layer_fwd(0, q, l, hd, planar.data_ptr(), w_hh.data_ptr(), b_hn.data_ptr(),
                                               seq_p.data_ptr(), h_p.data_ptr(),
                                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert torch.equal(h_w, h_p) and torch.equal(seq_w, seq_p)
    h_only, none = ops.gru_layer_fwd_windows(gx, base, l, layer)
    assert none is None and torch.equal(h_only, h_p)


def test_gru_windowed_entry_rejects_bad_arguments():
    lib = _lib.load()
    q, l, rows = 4, 3, 10
    gx = torch.zeros(3, rows, 128, device="cuda")
    base = torch.zeros(q + 1, dtype=torch.int32, device="cuda")
    w = torch.zeros(384, 128, device="cuda")
    bh = torch.zeros(128, device="cuda")
    h = torch.zeros(q, 128, device="cuda")
    hs = torch.zeros(q * l, 128, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(q_=q, l_=l, hd=128, gx_=gx.data_ptr(), rows_=rows, base_=base.data_ptr(), w_=w.data_ptr(),
             bh_=bh.data_ptr(), hs_=hs.data_ptr(), h_=h.data_ptr()):
        return lib.ltgnn_gru_layer_fwd_windows(0, q_, l_, hd, gx_, rows_, base_, w_, bh_, hs_, h_, stream)

    assert call() == 0 and call(hs_=None) == 0 and call(rows_=l) == 0
    assert call(hd=64) == -2 and call(q_=1 << 31) == -2 and call(rows_=1 << 31) == -2      # LTGNN_E_SHAPE
    assert call(q_=0) == -1 and call(l_=0) == -1 and call(rows_=l - 1) == -1                # LTGNN_E_ARG
    for k in ("gx_", "base_", "w_", "bh_", "h_"):
        assert call(**{k: None}) == -1, k
    for k, p in (("gx_", gx), ("w_", w), ("hs_", hs), ("h_", h)):                           # LTGNN_E_ALIGN
        assert call(**{k: p.data_ptr() + 4}) == -3, k
    assert call(base_=base.data_ptr() + 2) == -3 and call(base_=base.data_ptr() + 4) == 0
    with pytest.raises(_lib.LtgnnError) as e:
        _lib.check(call(hd=64))
    assert e.value.code == -2 and "128" in str(e.value)
    torch.cuda.synchronize()


@pytest.mark.parametrize("arch", ["tcn", "gru"])
def test_residual_builder_sharing_on_equals_off(arch):
    m = _pred(arch, 1)
    noisy, tf = _series(256, 72, 7)
    with torch.no_grad():
        on = build_residual_sequence_from_segment(m, noisy, tf, 36, 36)
        one = build_residual_sequence_from_segment(m, noisy[5], tf[5], 36, 36)
        m.share_windows = False
        off = build_residual_sequence_from_segment(m, noisy, tf, 36, 36)
    assert on.shape == off.shape == (256, 36, 29) and torch.equal(on, off) and torch.equal(one, off[5])


def test_residual_builder_sharing_matches_the_golden():
    from test_residual import TOL, rel_err
    gold = torch.load(TOPO["LTA"].parent / "residual_TCN.pt", map_location="cpu")
    m = NormalPredictorTCN(gold["noisy_seg"].shape[-1], 9)
    m.load_state_dict(gold["state_dict"], strict=True)
    m = m.cuda().eval()
    with torch.no_grad():
        r = build_residual_sequence_from_segment(m, gold["noisy_seg"], gold["time_seg"], 36, 36, device="cuda")
        m.share_windows = False
        off = build_residual_sequence_from_segment(m, gold["noisy_seg"], gold["time_seg"], 36, 36, device="cuda")
    assert torch.equal(r, off)
    assert rel_err(r.cpu(), gold["residual64"]) <= TOL


@pytest.mark.parametrize("arch", ["tcn", "gru"])
def test_residual_series_equals_the_builder(arch):
    m = _pred(arch, 2)
    x, xt = _series(2, 300, 3)
    r = residual_series(m, x, xt, 36, max_windows=100)                  # several chunks per series
    assert r.shape == (2, 264, 29)
    with torch.no_grad():
        seg = build_residual_sequence_from_segment(m, x[:, 40:112], xt[:, 40:112], 36, 36)
    assert torch.equal(r[:, 40:76], seg)
    assert torch.equal(residual_series(m, x[1], xt[1], 36), r[1])


def _scenario_per_segment(predictor, detector, pressure, tfeat, l_pred, l_det, stride, batch):
    """The per-segment scoring loop: every window's segment through the residual builder."""
    p, f = torch.as_tensor(pressure), torch.as_tensor(tfeat)
    seg_len = l_pred + l_det
    starts = list(range(0, p.shape[0] - seg_len + 1, stride))
    seg_p, seg_f = p.unfold(0, seg_len, 1).permute(0, 2, 1), f.unfold(0, seg_len, 1).permute(0, 2, 1)
    out = []
    with torch.no_grad():
        for lo in range(0, len(starts), batch):
            sel = torch.tensor(starts[lo:lo + batch])
            noisy, tseg = seg_p[sel].contiguous().cuda(), seg_f[sel].contiguous().cuda()
            res = build_residual_sequence_from_segment(predictor, noisy, tseg, l_pred, l_det)
            out.append(detector(res, tseg[:, l_pred:].contiguous()))
    return [s + seg_len for s in starts], torch.cat(out).cpu()


@pytest.mark.parametrize("arch", ["tcn", "gru"])
@pytest.mark.parametrize("t", [200, 2017])
def test_scenario_scoring_sharing_on_equals_off(graph_golden, arch, t):
    g = graph_golden("LTA")
    sensors, pipes = [str(s) for s in g["sensor_node_ids"]], [str(p) for p in g["pipe_ids"]][:60]
    torch.manual_seed(11)
    det = LeakDetector(TOPO["LTA"], sensors, pipes).cuda().eval()
    pred = _pred(arch, 4)
    rng = np.random.default_rng(t)
    pressure, tfeat = rng.standard_normal((t, 29)).astype(np.float32), rng.standard_normal((t, 9)).astype(np.float32)
    for stride in (1, 3, 12, 48):
        pred.share_windows = True
        ends, on = scenario_window_logits(pred, det, pressure, tfeat, 36, 36, stride, "cuda", batch=256)
        pred.share_windows = False
        want_ends, off = _scenario_per_segment(pred, det, pressure, tfeat, 36, 36, stride, 256)
        assert ends == want_ends and on.shape == off.shape and torch.equal(on, off), stride


@pytest.mark.parametrize("arch", ["tcn", "gru"])
def test_graphed_ltown_step_equals_eager_step(arch):
    """A graphed ltown_dp256-shaped step (full L-TOWN, B = 256, l_pred = l_det = 36) with the predictor sharing its
    windows, against eager steps with sharing off; dropout off, so the results agree bit for bit."""
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.parallel import FlatGradBucket

    z = np.load(TOPO["LT"].parent / "graph_LT.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    b, l_det, l_pred = 256, 36, 36
    gen = torch.Generator().manual_seed(198)
    data = [(torch.randn(b, l_pred + l_det, len(sensors), generator=gen).cuda(),
             torch.randn(b, l_pred + l_det, 9, generator=gen).cuda(),
             torch.randint(0, len(pipes) + 1, (b,), generator=gen).cuda()) for _ in range(3)]
    pred = ARCH[arch](len(sensors), 9)
    torch.manual_seed(5)
    pred = pred.cuda().eval()

    def fresh():
        torch.manual_seed(42)
        m = LeakDetector(TOPO["LT"], sensors, pipes, sensor_hidden=64, node_hidden=64, gnn_layers=2, dropout=0.0,
                         use_time=True).cuda().train()
        return m, FlatGradBucket(m.parameters()), torch.optim.AdamW(m.parameters(), lr=1e-3, capturable=True)

    m_e, bucket_e, opt_e = fresh()
    pred.share_windows = False
    losses_e = []
    for noisy, tf, label in data:
        with torch.no_grad():
            residual = build_residual_sequence_from_segment(pred, noisy, tf, l_pred, l_det)
        bucket_e.zero()
        loss = torch.nn.functional.cross_entropy(m_e(residual, tf[:, l_pred:].contiguous()), label)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m_e.parameters(), 1.0)
        opt_e.step()
        losses_e.append(loss.item())

    pred.share_windows = True
    m_g, bucket_g, opt_g = fresh()
    step = GraphedTrainStep(m_g, opt_g, bucket_g, b, l_det, predictor=pred, l_pred=l_pred, grad_clip=1.0)
    losses_g = [step(*d).item() for d in data]
    assert losses_g == losses_e, (losses_g, losses_e)
    for (n, a), c in zip(m_e.named_parameters(), m_g.parameters()):
        assert torch.equal(a, c), n
