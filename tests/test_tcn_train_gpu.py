"""Training of the TCN predictor on the cone (csrc/tcn_train.cu, ops.tcn_cone, NormalPredictorTCN.forward_cone) against
fp64 truth.  Tolerance: rel <= 1e-5 (fp32 path, 3xTF32 products).  Where dropout or a ReLU decides, the fp64 side replays
the kernels' captured live bits (a unit at the ReLU boundary may flip between fp32 and fp64: DESIGN section 2)."""
import pytest
import torch

from conftest import parity_log, rel_err
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.models import NormalPredictorTCN
from leak_det_gnn_b200.models.predictor import cone_positions

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _unpack(live):
    """int32 (M, 4) -> float (M, 128): bit b of word w <-> channel 32 w + b."""
    bits = (live.unsqueeze(-1) >> torch.arange(32, device=live.device, dtype=torch.int32)) & 1
    return bits.reshape(live.shape[0], -1).double()


def _injective_src(g, taps, m, rows):
    src = torch.stack([torch.randperm(rows, generator=g)[:m] for _ in range(taps)])
    src[torch.rand(taps, m, generator=g) < 0.1] = -1
    if m > 3:
        src[:, 2] = -1                                   # a row with only zero padding
    return src.to(torch.int32)


def _invert(idx, n_rows):
    inv = torch.full((idx.shape[0], n_rows), -1, dtype=torch.int64, device=idx.device)
    m = torch.arange(idx.shape[1], device=idx.device)
    for t in range(idx.shape[0]):
        ok = idx[t] >= 0
        inv[t, idx[t][ok].long()] = m[ok]
    return inv.to(torch.int32).contiguous()


def _case(m, rows, taps, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, 128, generator=g).cuda()
    src = _injective_src(g, taps, m, rows).cuda()
    w = (torch.randn(taps, 128, 128, generator=g) / (128 * taps) ** 0.5).cuda()
    bias = torch.randn(128, generator=g).cuda()
    gamma = (1 + 0.1 * torch.randn(128, generator=g)).cuda()
    beta = (0.1 * torch.randn(128, generator=g)).cuda()
    res_row = torch.randperm(rows, generator=g)[:m].to(torch.int32).cuda()     # the residual reads x itself (a block input)
    dy = torch.randn(m, 128, generator=g).cuda()
    return x, src, w, bias, gamma, beta, res_row, dy


@pytest.mark.parametrize("m,rows,taps", [(1, 7, 3), (127, 300, 1), (129, 200, 2), (385, 1000, 3), (5000, 9000, 8),
                                         (148 * 128 + 77, 40000, 3)])
def test_conv_train_forward_and_backward_against_fp64(m, rows, taps):
    x, src, w, bias, gamma, beta, res_row, dy = _case(m, rows, taps, m * 7 + taps)
    y, z, st, live = ops.tcn_conv_train(x, src, w, bias, gamma, beta, 1e-5, res=x, res_row=res_row)
    # drop_p = 0: the forward is the inference kernel's, bit for bit
    assert torch.equal(y, ops.tcn_conv(x, src, w, bias, gamma, beta, 1e-5, True, res=x, res_row=res_row))
    # fp64 truth with the kernel's live bits as the ReLU gate
    xd = x.double().requires_grad_()
    wd, bd, gd, ed = (t.double().requires_grad_() for t in (w, bias, gamma, beta))
    pad = torch.cat([xd, xd.new_zeros(1, 128)])
    idx = torch.where(src < 0, torch.full_like(src, rows), src).long()
    zd = bd.unsqueeze(0) + sum(pad[idx[t]] @ wd[t].t() for t in range(taps))
    yd = xd[res_row.long()] + torch.nn.functional.layer_norm(zd, (128,), gd, ed, 1e-5) * _unpack(live)
    (yd * dy.double()).sum().backward()
    assert rel_err(z, zd) <= TOL and rel_err(y, yd) <= TOL
    assert (st[:, 0].double() - zd.mean(1)).abs().max().item() <= TOL * zd.abs().max().item()   # relative to the row values
    # backward: epilogue, weight gradient, input gradient (+ the residual pass-through folded into the same launch)
    dz, dg, de, db = ops.tcn_ln_bwd(dy, live, z, st, gamma, 1.0)
    dw = ops.tcn_wgrad(dz, x, src)
    zero = torch.zeros(128, device="cuda")
    dx = ops.tcn_conv(dz, _invert(src, rows), w.transpose(1, 2).contiguous(), zero, relu=False, res=dy,
                      res_row=_invert(res_row.view(1, -1), rows)[0])
    errs = {"dX": rel_err(dx, xd.grad), "dW": max(rel_err(dw[t], wd.grad[t]) for t in range(taps)),
            "dbias": rel_err(db, bd.grad), "dgamma": rel_err(dg, gd.grad), "dbeta": rel_err(de, ed.grad), "tol": TOL}
    parity_log(f"tcn train conv M={m} taps={taps}", errs)
    assert all(v <= TOL for k, v in errs.items() if k != "tol"), errs
    # fixed order: bitwise equal run to run
    dz2, dg2, de2, db2 = ops.tcn_ln_bwd(dy, live, z, st, gamma, 1.0)
    assert torch.equal(dz, dz2) and torch.equal(dg, dg2) and torch.equal(de, de2) and torch.equal(db, db2)
    assert torch.equal(dw, ops.tcn_wgrad(dz, x, src))


def test_long_reductions_at_residual_builder_size():
    """9 216 windows x 36 positions = 331 776 rows at the first convolution: where a truncating tensor-memory accumulator
    would show (DESIGN section 2)."""
    m, taps = 9216 * 36, 3
    g = torch.Generator().manual_seed(5)
    x = torch.randn(m, 128, generator=g).cuda()
    src = _injective_src(g, taps, m, m).cuda()
    dy = torch.randn(m, 128, generator=g).cuda()
    gamma = (1 + 0.1 * torch.randn(128, generator=g)).cuda()
    z = torch.randn(m, 128, generator=g).cuda()
    st = torch.stack([z.mean(1), torch.rsqrt(z.var(1, unbiased=False) + 1e-5)], 1).contiguous()
    live = torch.randint(-2**31, 2**31 - 1, (m, 4), generator=g, dtype=torch.int64).to(torch.int32).cuda()
    dz, dg, de, db = ops.tcn_ln_bwd(dy, live, z, st, gamma, 1.0 / 0.9)
    dw = ops.tcn_wgrad(dz, x, src)
    gg = dy.double() * _unpack(live) / 0.9
    xh = (z.double() - st[:, :1].double()) * st[:, 1:].double()
    dxh = gg * gamma.double()
    dzd = st[:, 1:].double() * (dxh - dxh.mean(1, keepdim=True) - xh * (dxh * xh).mean(1, keepdim=True))
    pad = torch.cat([x.double(), x.new_zeros(1, 128).double()])
    idx = torch.where(src < 0, torch.full_like(src, m), src).long()
    errs = {"dz": rel_err(dz, dzd), "dgamma": rel_err(dg, (gg * xh).sum(0)), "dbeta": rel_err(de, gg.sum(0)),
            "dbias": rel_err(db, dzd.sum(0)),
            "dW": max(rel_err(dw[t], dz.double().t() @ pad[idx[t]]) for t in range(taps)), "tol": TOL}
    parity_log("tcn train long reductions M=331776", errs)
    assert all(v <= TOL for k, v in errs.items() if k != "tol"), errs


def _model(seed, p=0.1):
    torch.manual_seed(seed)
    m = NormalPredictorTCN(29, 9, dropout=p)
    with torch.no_grad():
        for blk in m.tcn:                                   # LayerNorm parameters off their (1, 0) initialisation
            for nm in (blk.norm1, blk.norm2):
                nm.weight.add_(0.1 * torch.randn_like(nm.weight))
                nm.bias.add_(0.1 * torch.randn_like(nm.bias))
    return m


def _batch(b, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, 36, 29, generator=g), torch.randn(b, 36, 9, generator=g), torch.randn(b, 29, generator=g)


def _dense_gated64(model, x, xt, lives):
    """The reference's dense forward (every position of every convolution) in fp64, with the ReLU decisions at the cone
    positions taken from the kernels' live bits: a pre-activation within fp32 rounding of zero may land on the other side
    in fp64, and each such flip moves a gradient row by O(1 / B) -- that says nothing about the kernels."""
    b, length, _ = x.shape
    plan = cone_positions(length, model.tcn[0].conv1.conv.kernel_size[0], [blk.conv1.conv.dilation[0] for blk in model.tcn])
    h = model.input_proj(torch.cat([x, xt], -1).transpose(1, 2))
    k, flips = 0, 0
    for blk, (p1, p2) in zip(model.tcn, plan):
        y = h
        for conv, norm, pos in ((blk.conv1, blk.norm1, p1), (blk.conv2, blk.norm2, p2)):
            v = norm(conv(y).transpose(1, 2))                          # (B, L, C)
            gate = (v > 0).double()
            bits = _unpack(lives[k].cpu()).view(b, len(pos), -1)
            flips += int((gate[:, pos, :] != bits).sum())
            gate[:, pos, :] = bits
            y = (v * gate).transpose(1, 2)
            k += 1
        h = h + y
    return model.head(h[:, :, -1]), flips


def test_model_gradients_against_dense_fp64():
    m = _model(1).cuda().eval()                                  # dropout off
    x, xt, y = (t.cuda() for t in _batch(256, 2))
    ref = _model(1).double().eval()
    ops.DEBUG_CAPTURE = {}
    try:
        loss = torch.nn.functional.mse_loss(m.forward_cone(x, xt), y)
        lives = ops.DEBUG_CAPTURE["tcn_lives"]
    finally:
        ops.DEBUG_CAPTURE = None
    loss.backward()
    pd, flips = _dense_gated64(ref, x.double().cpu(), xt.double().cpu(), lives)
    loss_d = torch.nn.functional.mse_loss(pd, y.double().cpu())
    loss_d.backward()
    assert torch.allclose(pd, ref(x.double().cpu(), xt.double().cpu()), rtol=0, atol=1e-4)   # the gate changed ~nothing
    errs = {n: rel_err(p.grad, q.grad) for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters())}
    errs["loss"] = rel_err(loss, loss_d)
    units = 256 * 99 * 128
    parity_log("TCN forward_cone + backward (native) vs dense fp64, B=256", {**errs, "relu_flips": flips, "tol": TOL})
    assert flips <= units * 1e-5, flips
    assert len(errs) == 37 and all(p.grad is not None for p in m.parameters())
    assert all(v <= TOL for v in errs.values()), {k: v for k, v in errs.items() if v > TOL}


def _cone_replay64(model, x, xt, lives, scale):
    """fp64 cone of ``model`` with every ReLU + dropout replaced by the kernels' live bits times the dropout scale."""
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
            gate = _unpack(lives[k]).to(x.device).view(b, rows.shape[1], -1) * scale
            yv = norm(torch.nn.functional.linear(rows, w, conv.conv.bias)) * gate
            k += 1
        h = h.index_select(1, keep) + yv
    return model.head(h[:, 0, :])


def test_dropout_replays_fp64_and_draws_fresh_masks():
    m = _model(3, p=0.1).cuda().train()
    x, xt, y = (t.cuda() for t in _batch(64, 4))
    ops.DEBUG_CAPTURE = {}
    try:
        torch.manual_seed(11)
        pred = m.forward_cone(x, xt)
        torch.nn.functional.mse_loss(pred, y).backward()
        lives = [l.clone() for l in ops.DEBUG_CAPTURE["tcn_lives"]]
    finally:
        ops.DEBUG_CAPTURE = None
    ref = _model(3, p=0.1).double()
    pd = _cone_replay64(ref, x.double().cpu(), xt.double().cpu(), [l.cpu() for l in lives], 1.0 / 0.9)
    torch.nn.functional.mse_loss(pd, y.double().cpu()).backward()
    errs = {n: rel_err(p.grad, q.grad) for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters())}
    errs["pred"] = rel_err(pred, pd)
    parity_log("TCN forward_cone dropout 0.1 vs fp64 replay of the live bits", {**errs, "tol": TOL})
    assert all(v <= TOL for v in errs.values()), {k: v for k, v in errs.items() if v > TOL}
    with torch.no_grad():
        torch.manual_seed(11)
        assert torch.equal(m.forward_cone(x, xt), pred)           # same seed: same masks
        torch.manual_seed(12)
        assert not torch.equal(m.forward_cone(x, xt), pred)       # new seed: new masks


def test_dropout_fraction():
    m, p = 200000, 0.1
    g = torch.Generator().manual_seed(9)
    x = torch.randn(m, 128, generator=g).cuda()
    src = torch.arange(m, dtype=torch.int32).view(1, -1).cuda()
    w = torch.eye(128).view(1, 128, 128).cuda()
    beta = torch.full((128,), 10.0, device="cuda")             # every unit positive after the ReLU: live = kept
    _, _, _, live = ops.tcn_conv_train(x, src, w, torch.zeros(128, device="cuda"), torch.ones(128, device="cuda"), beta,
                                       1e-5, drop_p=p, drop_seed=1234)
    kept = _unpack(live).mean().item()
    sigma = (p * (1 - p) / (m * 128)) ** 0.5
    assert abs((1 - kept) - p) < 6 * sigma, (1 - kept, p)


def test_graphed_step_equals_eager():
    """Dropout off: the replayed training step (forward_cone, MSE, backward, clip, AdamW) equals the eager one bit for bit."""
    from leak_det_gnn_b200.parallel import FlatGradBucket
    from leak_det_gnn_b200.train_predictor_dp import PredictorStep

    def run(graph):
        m = _model(5, p=0.0).cuda()
        opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)
        step = PredictorStep(m, opt, FlatGradBucket(m.parameters()), 32, 1.0, graph)
        losses = [step(*(t.cuda() for t in _batch(32, 100 + i))).clone() for i in range(3)]
        return m, losses

    me, le = run(False)
    mg, lg = run(True)
    assert all(torch.equal(a, b) for a, b in zip(le, lg))
    assert all(torch.equal(a, b) for a, b in zip(me.parameters(), mg.parameters()))


def test_graphed_step_draws_fresh_dropout_masks():
    """Dropout 0.1 and no optimiser (the weights never change): replays on the same batch draw new live bits and give
    different losses, and the same torch seed reproduces the sequence."""
    from leak_det_gnn_b200.parallel import FlatGradBucket
    from leak_det_gnn_b200.train_predictor_dp import PredictorStep

    batch = [t.cuda() for t in _batch(32, 100)]

    def replays(n=4):
        m = _model(5, p=0.1).cuda()
        keep = [p.detach().clone() for p in m.parameters()]
        torch.manual_seed(6)
        ops.DEBUG_CAPTURE = {}
        try:
            step = PredictorStep(m, None, FlatGradBucket(m.parameters()), 32, 0.0, True)
            lives = ops.DEBUG_CAPTURE["tcn_lives"]          # the graph's own live-bit tensors, rewritten by every replay
        finally:
            ops.DEBUG_CAPTURE = None
        losses, bits = [], []
        for _ in range(n):
            losses.append(step(*batch).item())
            bits.append(torch.cat([l.flatten() for l in lives]).clone())
        assert all(torch.equal(a, b) for a, b in zip(keep, m.parameters()))
        return losses, bits

    la, ba = replays()
    lb, bb = replays()
    assert len(set(la)) == len(la), la
    assert all(not torch.equal(ba[i], ba[i + 1]) for i in range(len(ba) - 1))
    assert la == lb and all(torch.equal(a, b) for a, b in zip(ba, bb))


def test_conv_train_and_ln_bwd_reject_bad_arguments():
    """The C entry points return LTGNN_E_ARG / LTGNN_E_ALIGN instead of reading through bad pointers."""
    from leak_det_gnn_b200 import lib as _lib

    L = _lib.load()
    m, c = 256, 128
    x = torch.randn(m, c, device="cuda")
    src = torch.arange(m, dtype=torch.int32, device="cuda").view(1, -1)
    w = torch.randn(1, c, c, device="cuda")
    v = torch.ones(c, device="cuda")
    out = [torch.empty(m, c, device="cuda") for _ in range(2)]
    stats = torch.empty(m, 2, device="cuda")
    live = torch.empty(m, 4, dtype=torch.int32, device="cuda")
    ws = torch.empty(int(L.ltgnn_tcn_ws_floats(1)), device="cuda")
    rows = torch.zeros(m, dtype=torch.int32, device="cuda")
    buf = torch.empty(m * c + 4, device="cuda")
    stream = ops._stream(x)

    def conv_train(res, res_row, y):
        return L.ltgnn_tcn_conv_train(0, m, c, 1, x.data_ptr(), src.data_ptr(), w.data_ptr(), v.data_ptr(), v.data_ptr(),
                                      v.data_ptr(), 1e-5, res, res_row, 0.0, 0, y, out[1].data_ptr(), stats.data_ptr(),
                                      live.data_ptr(), ws.data_ptr(), stream)

    assert conv_train(x.data_ptr(), None, out[0].data_ptr()) == -1                  # res without res_row
    assert conv_train(None, rows.data_ptr(), out[0].data_ptr()) == -1               # res_row without res
    assert conv_train(None, None, buf.data_ptr() + 4) == -3                         # Y not 16-byte aligned
    assert conv_train(buf.data_ptr() + 4, rows.data_ptr(), out[0].data_ptr()) == -3  # res not 16-byte aligned
    assert conv_train(x.data_ptr(), rows.data_ptr(), out[0].data_ptr()) == 0
    lnws = torch.empty(int(L.ltgnn_tcn_ln_bwd_ws_floats(0)), device="cuda")
    dprm = torch.empty(3, c, device="cuda")
    rc = L.ltgnn_tcn_ln_bwd(0, m, c, x.data_ptr(), live.data_ptr(), out[1].data_ptr(), buf.data_ptr() + 4, v.data_ptr(), 1.0,
                            out[0].data_ptr(), dprm.data_ptr(), lnws.data_ptr(), stream)
    assert rc == -3                                                                  # stats not 8-byte aligned
    torch.cuda.synchronize()
