"""Gradients with respect to the raw sensor series through the frozen predictor's shared windows on the sm_100a kernels:
the deterministic row gather-sum (ltgnn_row_gather_sum), the differentiable ``forward_windows`` of both predictors
(forward bits, input gradients against fp64, determinism, no weight-gradient kernel), the input gradients of
``forward_cone``, and the whole pipeline noisy segment -> residual builder -> LeakDetector against the fp64 oracle."""
import copy
import ctypes

import pytest
import torch

from conftest import TOPO, parity_log, rel_err
from leak_det_gnn_b200 import instrument
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.models import NormalPredictorGRU, NormalPredictorTCN, build_residual_sequence_from_segment
from leak_det_gnn_b200.models.predictor import shared_cone_plan, windows_of

pytestmark = pytest.mark.gpu
ARCH = {"tcn": NormalPredictorTCN, "gru": NormalPredictorGRU}
WEIGHT_KERNELS = {"tcn_wgrad", "wgrad", "wgrad_tc", "gru_bwd_w"}
TOL = 1e-5


def _random_csr(g, rows, n_src, max_deg):
    deg = torch.randint(0, max_deg + 1, (rows,), generator=g)
    deg[torch.randperm(rows, generator=g)[: rows // 4]] = 0                     # empty rows give zeros
    ptr = torch.zeros(rows + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(deg, 0)
    idx = torch.randint(0, n_src, (int(ptr[-1]),), generator=g)
    return ptr, idx


def _loop_sum(src, ptr, idx):
    """fp32 reference in the kernel's order: out[r] = ((0 + src[idx[e0]]) + src[idx[e0 + 1]]) + ..."""
    rows = ptr.numel() - 1
    out = torch.zeros(*src.shape[:-2], rows, src.shape[-1], dtype=torch.float32)
    deg = ptr[1:] - ptr[:-1]
    for k in range(int(deg.max()) if rows else 0):
        have = (deg > k).nonzero().view(-1)
        out[..., have, :] += src[..., idx[ptr[have] + k], :]
    return out


@pytest.mark.parametrize("c", [4, 128])
@pytest.mark.parametrize("planes", [1, 3])
@pytest.mark.parametrize("rows,n_src,max_deg", [(1, 3, 2), (1000, 700, 9), (20011, 5000, 40)])
def test_row_gather_sum_equals_ordered_fp32_loop(c, planes, rows, n_src, max_deg):
    g = torch.Generator().manual_seed(rows + c + planes)
    ptr, idx = _random_csr(g, rows, n_src, max_deg)
    src = torch.randn(planes, n_src, c, generator=g) if planes > 1 else torch.randn(n_src, c, generator=g)
    got = ops.row_gather_sum(src.cuda(), ptr.to(torch.int32).cuda(), idx.to(torch.int32).cuda())
    want = _loop_sum(src, ptr, idx)
    assert got.shape == want.shape and torch.equal(got.cpu(), want)


def test_row_gather_sum_rejects_bad_arguments():
    lib = _lib.load()
    rows, c, n_src, planes = 5, 8, 7, 3
    src = torch.zeros(planes, n_src, c, device="cuda")
    out = torch.zeros(planes, rows, c, device="cuda")
    ptr = torch.zeros(rows + 1, dtype=torch.int32, device="cuda")
    idx = torch.zeros(4, dtype=torch.int32, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(r=rows, c_=c, p=planes, s=src.data_ptr(), ss=n_src * c, pt=ptr.data_ptr(), ix=idx.data_ptr(),
             o=out.data_ptr(), os_=rows * c):
        return lib.ltgnn_row_gather_sum(0, r, c_, p, s, ss, pt, ix, o, os_, stream)

    assert call() == 0 and call(r=0) == 0 and call(p=1, ss=0, os_=0) == 0
    assert call(c_=6) == -2 and call(r=1 << 31) == -2                                       # LTGNN_E_SHAPE
    assert call(r=-1) == -1 and call(c_=0) == -1 and call(p=0) == -1 and call(p=65536) == -1  # LTGNN_E_ARG
    assert call(ss=-4) == -1 and call(os_=-4) == -1
    for k in ("s", "pt", "ix", "o"):
        assert call(**{k: None}) == -1, k
    assert call(s=src.data_ptr() + 4) == -3 and call(o=out.data_ptr() + 8) == -3              # LTGNN_E_ALIGN
    assert call(ss=n_src * c + 2) == -3 and call(os_=rows * c + 1) == -3
    assert call(pt=ptr.data_ptr() + 2) == -3 and call(ix=idx.data_ptr() + 2) == -3
    with pytest.raises(_lib.LtgnnError) as e:
        _lib.check(call(c_=6))
    assert e.value.code == -2 and "multiple of 4" in str(e.value)
    torch.cuda.synchronize()


def _pred(arch, seed=0):
    torch.manual_seed(seed)
    m = ARCH[arch](29, 9)
    if arch == "tcn":
        with torch.no_grad():
            for blk in m.tcn:                               # LayerNorm parameters off their (1, 0) initialisation
                for nm in (blk.norm1, blk.norm2):
                    nm.weight.add_(0.1 * torch.randn_like(nm.weight))
                    nm.bias.add_(0.1 * torch.randn_like(nm.bias))
    return m.eval().requires_grad_(False)


def _series(b, t, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, t, 29, generator=g), torch.randn(b, t, 9, generator=g)


@pytest.mark.parametrize("arch", ["tcn", "gru"])
@pytest.mark.parametrize("b,t,window,count", [(256, 72, 36, 36), (1, 2017, 36, None), (3, 300, 20, None),
                                              (3, 300, 64, None), (2, 64, 64, None), (4, 72, 36, 1)])
def test_differentiable_forward_windows_keeps_the_bits(arch, b, t, window, count):
    """Window 36: the head row (p = 35 < R = 60) is windowed; window 64: it is shared."""
    m = _pred(arch).cuda()
    x, xt = (v.cuda() for v in _series(b, t, t + window))
    with torch.no_grad():
        want = m.forward_windows(x, xt, window, count=count)
    xg = x.clone().requires_grad_(True)
    assert m.differentiable_windows(xg, xt)
    got = m.forward_windows(xg, xt, window, count=count)
    assert got.requires_grad and torch.equal(got.detach(), want)


def _unpack(live):
    bits = (live.unsqueeze(-1).long() >> torch.arange(32)) & 1
    return bits.reshape(live.shape[0], -1).double()


def _tcn_plan_replay64(m64, x, xt, window, count, lives):
    """fp64 evaluation of the shared plan (what the kernels compute) with every ReLU decision taken from the kernels' live
    bits: a pre-activation within fp32 rounding of zero may land on the other side in fp64, which says nothing about
    the kernels."""
    b, length, _ = x.shape
    plan, _ = shared_cone_plan(length, window, count, b, 3, [blk.conv1.conv.dilation[0] for blk in m64.tcn])
    h = torch.nn.functional.linear(torch.cat([x, xt], -1).reshape(b * length, -1), m64.input_proj.weight[:, :, 0],
                                   m64.input_proj.bias)
    k = 0
    for blk, (src1, src2, res) in zip(m64.tcn, plan):
        y = h
        for conv, norm, src in ((blk.conv1, blk.norm1, src1), (blk.conv2, blk.norm2, src2)):
            w = conv.conv.weight.permute(0, 2, 1).reshape(conv.conv.weight.shape[0], -1)
            padded = torch.cat([y, y.new_zeros(1, y.shape[1])])
            taps = torch.where(src < 0, torch.full_like(src, y.shape[0]), src)
            y = norm(torch.nn.functional.linear(padded[taps.t()].reshape(src.shape[1], -1), w, conv.conv.bias))
            y = y * _unpack(lives[k].cpu())
            k += 1
        h = h[res] + y
    return m64.head(h).view(b, count, -1)


def _dense64(m64, x, xt, window, count):
    b = x.shape[0]
    return m64(windows_of(x, window, count), windows_of(xt, window, count)).view(b, count, -1)


@pytest.mark.parametrize("arch", ["tcn", "gru"])
@pytest.mark.parametrize("b,t,window,count", [(2, 72, 36, 36), (3, 41, 20, None), (2, 130, 64, None), (1, 40, 36, 2)])
def test_forward_windows_input_grads_match_fp64(arch, b, t, window, count):
    n = count or t - window + 1
    m = _pred(arch, 3).cuda()
    m64 = _pred(arch, 3).double()
    x, xt = _series(b, t, 5 * t + window)
    dy = torch.randn(b, n, 29, generator=torch.Generator().manual_seed(t))
    xg, xtg = x.cuda().requires_grad_(True), xt.cuda().requires_grad_(True)
    ops.DEBUG_CAPTURE = {}
    try:
        out = m.forward_windows(xg, xtg, window, count=n)
        lives = ops.DEBUG_CAPTURE.get("tcn_lives")
    finally:
        ops.DEBUG_CAPTURE = None
    (out * dy.cuda()).sum().backward()
    x64, xt64 = x.double().requires_grad_(True), xt.double().requires_grad_(True)
    ref = _tcn_plan_replay64(m64, x64, xt64, window, n, lives) if arch == "tcn" else _dense64(m64, x64, xt64, window, n)
    with torch.no_grad():         # the replayed gates changed ~nothing: the truth is the dense model's function
        assert (ref - _dense64(m64, x.double(), xt.double(), window, n)).abs().max() <= 1e-4
    (ref * dy.double()).sum().backward()
    rep = {"d_x": rel_err(xg.grad, x64.grad), "d_x_time": rel_err(xtg.grad, xt64.grad)}
    parity_log(f"forward_windows input grad {arch} B={b} T={t} window={window} count={n}", rep)
    assert all(v <= TOL for v in rep.values()), rep


@pytest.mark.parametrize("arch", ["tcn", "gru"])
def test_windows_backward_is_deterministic_and_frozen(arch, monkeypatch):
    m = _pred(arch, 4).cuda()
    x, xt = (v.cuda() for v in _series(16, 72, 9))
    dy = torch.randn(16, 36, 29, device="cuda")
    launched = []
    monkeypatch.setattr(instrument, "begin", lambda name: launched.append(name))

    def run():
        xg, xtg = x.clone().requires_grad_(True), xt.clone().requires_grad_(True)
        launched.clear()
        (m.forward_windows(xg, xtg, 36, count=36) * dy).sum().backward()
        return xg.grad, xtg.grad, set(launched)

    a, b = run(), run()
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert all(p.grad is None for p in m.parameters())
    assert "row_gather_sum" in a[2] and not a[2] & WEIGHT_KERNELS, a[2]
    # only x asks for a gradient: same d x
    xg = x.clone().requires_grad_(True)
    (m.forward_windows(xg, xt, 36, count=36) * dy).sum().backward()
    assert torch.equal(xg.grad, a[0])
    # a trainable predictor keeps today's no-grad forward_windows
    m.requires_grad_(True)
    assert not m.differentiable_windows(x.clone().requires_grad_(True), xt)


def _tcn_cone_replay64(model, x, xt, lives):
    """fp64 cone with every ReLU replaced by the kernels' live bits (eval mode: no dropout)."""
    b, length, _ = x.shape
    gather = model._cone_plan(length, x.device)
    h = torch.nn.functional.linear(torch.cat([x, xt], -1), model.input_proj.weight[:, :, 0], model.input_proj.bias)
    zero = h.new_zeros(b, 1, h.shape[-1])
    k = 0
    for blk, (taps1, taps2, keep) in zip(model.tcn, gather):
        yv = h
        for conv, norm, taps in ((blk.conv1, blk.norm1, taps1), (blk.conv2, blk.norm2, taps2)):
            w = conv.conv.weight.permute(0, 2, 1).reshape(conv.conv.weight.shape[0], -1)
            rows = torch.cat([yv, zero], 1).index_select(1, taps).view(b, -1, w.shape[1])
            yv = norm(torch.nn.functional.linear(rows, w, conv.conv.bias)) * _unpack(lives[k].cpu()).view(b, rows.shape[1], -1)
            k += 1
        h = h.index_select(1, keep) + yv
    return model.head(h[:, 0, :])


@pytest.mark.parametrize("arch", ["tcn", "gru"])
def test_forward_cone_input_grads(arch):
    """d x and d x_time of forward_cone within 1e-5 of fp64 (x.grad stayed None before); with input gradients asked for,
    the parameter gradients equal those of the parameter-only backward bit for bit."""
    m = _pred(arch, 6).cuda().requires_grad_(True)
    m64 = _pred(arch, 6).double()
    x, xt = _series(64, 36, 8)
    dy = torch.randn(64, 29, generator=torch.Generator().manual_seed(1))

    def native(inputs_grad):
        m.zero_grad(set_to_none=True)
        xg, xtg = x.cuda().requires_grad_(inputs_grad), xt.cuda().requires_grad_(inputs_grad)
        ops.DEBUG_CAPTURE = {}
        try:
            out = m.forward_cone(xg, xtg)
            lives = ops.DEBUG_CAPTURE.get("tcn_lives")
        finally:
            ops.DEBUG_CAPTURE = None
        (out * dy.cuda()).sum().backward()
        return xg.grad, xtg.grad, [p.grad.clone() for p in m.parameters()], lives

    dx, dxt, g_in, lives = native(True)
    _, _, g_only, _ = native(False)
    for a, c in zip(g_in, g_only):
        assert torch.equal(a, c)
    x64, xt64 = x.double().requires_grad_(True), xt.double().requires_grad_(True)
    ref = _tcn_cone_replay64(m64, x64, xt64, lives) if arch == "tcn" else m64(x64, xt64)
    with torch.no_grad():
        assert (ref - m64(x.double(), xt.double())).abs().max() <= 1e-4
    (ref * dy.double()).sum().backward()
    rep = {"d_x": rel_err(dx, x64.grad), "d_x_time": rel_err(dxt, xt64.grad)}
    parity_log(f"forward_cone input grad {arch} B=64 L=36", rep)
    assert all(v <= TOL for v in rep.values()), rep


def _pipes(n):
    from leak_det_gnn_b200.graph import parse_epanet_inp
    return [ln.split()[0] for ln in parse_epanet_inp(TOPO["LTA"])["PIPES"]][:n]


@pytest.mark.parametrize("arch", ["tcn", "gru"])
@pytest.mark.parametrize("sensor_hidden", [64, 128])
def test_raw_series_grad_through_builder_and_detector(graph_golden, arch, sensor_hidden):
    """Frozen predictor -> build_residual_sequence_from_segment -> frozen LeakDetector (L-TOWN-A, eval mode, B = 8,
    l_pred = l_det = 36): the gradient of each window's target logit with respect to noisy_seg and time_seg within 1e-5
    of the fp64 truth (dense double predictor through the same builder on the CPU, then the oracle detector in double),
    or no further than 3x the same pipeline in fp32 on the CPU; for the TCN the dense route (share_windows = False)
    meets the same bound."""
    from leak_det_gnn_b200.models import LeakDetector
    from oracle.detector_oracle import OracleLeakDetector

    g = graph_golden("LTA")
    pipes = _pipes(40)
    torch.manual_seed(19)
    det = LeakDetector(TOPO["LTA"], [str(v) for v in g["sensor_node_ids"]], pipes, sensor_hidden=sensor_hidden,
                       node_hidden=64)
    state = {k: v.clone() for k, v in det.state_dict().items()}
    det = det.cuda().eval().requires_grad_(False)
    pred = _pred(arch, 7)
    b, l_pred, l_det = 8, 36, 36
    noisy, tseg = _series(b, l_pred + l_det, 21)
    near = [p for p, (u, v) in enumerate(det.pipe_ends.tolist())
            if u in det.sensor_node_idx.tolist() or v in det.sensor_node_idx.tolist()]
    classes = torch.tensor(near + [len(pipes)])
    target = classes[torch.randint(0, len(classes), (b,), generator=torch.Generator().manual_seed(2))]

    def grads(p, d, dtype, device):
        n_, t_ = noisy.to(device, dtype).requires_grad_(True), tseg.to(device, dtype).requires_grad_(True)
        res = build_residual_sequence_from_segment(p, n_, t_, l_pred, l_det)
        logits = d(res, t_[:, l_pred:])
        return torch.autograd.grad(logits.gather(1, target.to(device)[:, None]).sum(), (n_, t_))

    def truth(dtype):
        o = OracleLeakDetector(len(det.node_names), det.edge_index_single, det.pipe_ends, det.sensor_node_idx.tolist(),
                               sensor_hidden, 64, 2, 0.1, True).to(dtype)
        o.load_state_dict({k: v.to(dtype) for k, v in state.items()}, strict=True)
        return grads(copy.deepcopy(pred).to(dtype), o.eval(), dtype, "cpu")

    t64, t32 = truth(torch.float64), truth(torch.float32)
    pg = pred.cuda()
    native = grads(pg, det, torch.float32, "cuda")
    rep = {n: {"ours": rel_err(native[i], t64[i]), "cpu_fp32": rel_err(t32[i], t64[i])}
           for i, n in enumerate(("d_noisy_seg", "d_time_seg"))}
    if arch == "tcn":
        pg.share_windows = False
        old = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            dense = grads(pg, det, torch.float32, "cuda")
        finally:
            torch.backends.cudnn.allow_tf32 = old
            pg.share_windows = True
        for i, n in enumerate(("d_noisy_seg", "d_time_seg")):
            rep[n]["dense_route"] = rel_err(dense[i], t64[i])
            rep[n]["shared_vs_dense"] = rel_err(native[i], dense[i])
    parity_log(f"raw series grad {arch} sensor_hidden={sensor_hidden}", rep)
    assert all(t.abs().max() > 0 for t in t64)
    for n, e in rep.items():
        bound = max(TOL, 3.0 * e["cpu_fp32"])
        assert e["ours"] <= bound, (n, e)
        if "dense_route" in e:
            assert e["dense_route"] <= bound and e["shared_vs_dense"] <= bound, (n, e)
