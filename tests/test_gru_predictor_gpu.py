"""The GRU normal-state predictor on sm_100a (reference models/predictor.py:84-111): one hidden-128 layer of
csrc/gru_pred.cu (ltgnn_gru_layer_fwd after the ltgnn_linear input projection) against an fp64 nn.GRU, the whole
NormalPredictorGRU.forward_last against the fp64 dense forward, the residual builder, the graphed detector step and the
detector launcher with a GRU checkpoint.  Tolerance: rel <= 1e-5 (2e-5 at L = 288, as the sensor GRU), 3xTF32 products."""
import copy
import ctypes

import pytest
import torch

from conftest import TOPO, parity_log, rel_err
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.models import NormalPredictorGRU, build_residual_sequence_from_segment

pytestmark = pytest.mark.gpu


def _layer(n_in, scale, seed):
    torch.manual_seed(seed)
    gru = torch.nn.GRU(n_in, 128, num_layers=1, batch_first=True)
    with torch.no_grad():
        for p in gru.parameters():
            p.mul_(scale)
    return gru.cuda()


@pytest.mark.parametrize("scale", [1.0, 3.0])
@pytest.mark.parametrize("l", [1, 36, 288])
@pytest.mark.parametrize("q", [1, 127, 128, 129, 9216])
def test_layer_matches_fp64(q, l, scale):
    """h_last and the state sequence of one layer, at nn.GRU's init scale and at 3x (saturated gates); ragged Q."""
    gru = _layer(38, scale, q + l)
    g = torch.Generator(device="cpu").manual_seed(7 * q + l)
    x = torch.randn(q, l, 38, generator=g).cuda()
    inp = torch.zeros(q, l, 64, device="cuda")
    inp[:, :, :38] = x
    layer = ops.gru_predictor_weights([(gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0)])[0]
    h_last, hseq = ops.gru_layer_fwd(inp.view(q * l, 64), q, l, layer, seq=True)
    with torch.no_grad():
        ref, _ = copy.deepcopy(gru).double()(x.double())
        ref32, _ = gru(x)
    tol = 1e-5 if l <= 36 else 2e-5
    err_last, err_seq = rel_err(h_last, ref[:, -1]), rel_err(hseq.view(q, l, 128), ref)
    parity_log(f"gru_pred_layer Q={q} L={l} scale={scale}",
               {"h_last": err_last, "hseq": err_seq, "torch_fp32_h_last": rel_err(ref32[:, -1], ref[:, -1]),
                "torch_fp32_hseq": rel_err(ref32, ref), "tol": tol})
    assert err_last <= tol and err_seq <= tol
    assert torch.equal(hseq[(l - 1)::l], h_last)
    h2, s2 = ops.gru_layer_fwd(inp.view(q * l, 64), q, l, layer, seq=True)
    assert torch.equal(h2, h_last) and torch.equal(s2, hseq)          # no atomics, fixed order
    h3, none = ops.gru_layer_fwd(inp.view(q * l, 64), q, l, layer)
    assert none is None and torch.equal(h3, h_last)                   # the state sequence is optional


def _predictor(seed=11):
    torch.manual_seed(seed)
    return NormalPredictorGRU(29, 9).cuda().eval()


def test_forward_last_matches_fp64_dense_forward():
    m = _predictor()
    g = torch.Generator(device="cpu").manual_seed(3)
    x, tf = torch.randn(256, 36, 29, generator=g).cuda(), torch.randn(256, 36, 9, generator=g).cuda()
    y = m.forward_last(x, tf)
    with torch.no_grad():
        y32 = m(x, tf)
        m64 = NormalPredictorGRU(29, 9).cuda().double().eval()
        m64.load_state_dict(m.state_dict())
        ref = m64(x.double(), tf.double())
    err = rel_err(y, ref)
    parity_log("gru_predictor forward_last B=256 L=36", {"y": err, "torch_fp32": rel_err(y32, ref), "tol": 1e-5})
    assert y.shape == (256, 29) and err <= 1e-5
    assert torch.equal(m.forward_last(x, tf), y)
    m.use_native = False
    assert torch.equal(m.forward_last(x, tf), y32)                    # the cuDNN cross-check is the dense forward
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.forward_last(x, tf)


def test_forward_last_other_layer_counts():
    """num_layers = 1 and 3 go through the same kernels (no inter-layer dropout in eval)."""
    g = torch.Generator(device="cpu").manual_seed(5)
    x, tf = torch.randn(130, 20, 29, generator=g).cuda(), torch.randn(130, 20, 9, generator=g).cuda()
    for layers in (1, 3):
        torch.manual_seed(layers)
        m = NormalPredictorGRU(29, 9, num_layers=layers).cuda().eval()
        y = m.forward_last(x, tf)
        with torch.no_grad():
            m64 = NormalPredictorGRU(29, 9, num_layers=layers).cuda().double().eval()
            m64.load_state_dict(m.state_dict())
            err = rel_err(y, m64(x.double(), tf.double()))
        parity_log(f"gru_predictor forward_last layers={layers}", {"y": err, "tol": 1e-5})
        assert err <= 1e-5


def test_residual_builder_with_gru_predictor():
    """9 216 windows (B = 256, l_pred = l_det = 36): against the fp64 builder, and bit for bit what forward_last gives on
    the explicitly materialised windows (reference models/utils.py:169-216)."""
    m = _predictor(13)
    b, l_pred, l_det = 256, 36, 36
    g = torch.Generator(device="cpu").manual_seed(9)
    noisy = torch.randn(b, l_pred + l_det, 29, generator=g).cuda()
    tf = torch.randn(b, l_pred + l_det, 9, generator=g).cuda()
    with torch.no_grad():
        res = build_residual_sequence_from_segment(m, noisy, tf, l_pred, l_det)
        m64 = NormalPredictorGRU(29, 9).cuda().double().eval()
        m64.load_state_dict(m.state_dict())
        ref = build_residual_sequence_from_segment(m64, noisy.double(), tf.double(), l_pred, l_det)
        xw = torch.cat([noisy[:, kk:kk + l_pred] for kk in range(l_det)], dim=0)
        tw = torch.cat([tf[:, kk:kk + l_pred] for kk in range(l_det)], dim=0)
        y = m.forward_last(xw, tw)
        target = torch.cat([noisy[:, l_pred + kk] for kk in range(l_det)], dim=0)
        manual = (target - y).view(l_det, b, 29).transpose(0, 1)
    err = rel_err(res, ref)
    parity_log("gru_predictor residual B=256 l_pred=l_det=36", {"residual": err, "tol": 1e-5})
    assert res.shape == (b, l_det, 29) and err <= 1e-5
    assert torch.equal(res, manual)


def test_graphed_step_with_gru_predictor_equals_eager_step(graph_golden):
    """Three replays of the captured detector step (the predictor's cluster launches inside the graph) against three
    eager steps from the same start, dropout off: identical losses and parameters, bit for bit."""
    from test_graphed_gpu import _batches, _model
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.parallel import FlatGradBucket

    g = graph_golden("LTA")
    bsz, l_pred, l_det, n_pipes = 16, 36, 12, 24
    data = _batches(3, bsz, l_pred + l_det, 29, n_pipes + 1)
    predictor = _predictor(3)

    def fresh():
        m = _model(g, n_pipes, 0.0)
        return m, FlatGradBucket(m.parameters()), torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)

    m_e, bucket_e, opt_e = fresh()
    losses_e = []
    for noisy, tf, label in data:
        noisy, tf, label = noisy.cuda(), tf.cuda(), label.cuda()
        with torch.no_grad():
            residual = build_residual_sequence_from_segment(predictor, noisy, tf, l_pred, l_det)
        bucket_e.zero()
        loss = torch.nn.functional.cross_entropy(m_e(residual, tf[:, l_pred:, :].contiguous()), label)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m_e.parameters(), 1.0)
        opt_e.step()
        losses_e.append(loss.item())

    m_g, bucket_g, opt_g = fresh()
    step = GraphedTrainStep(m_g, opt_g, bucket_g, bsz, l_det, predictor=predictor, l_pred=l_pred, grad_clip=1.0)
    losses_g = [step(*b).item() for b in data]
    assert losses_g == losses_e, (losses_g, losses_e)
    for (n, a), b in zip(m_e.named_parameters(), m_g.parameters()):
        assert torch.equal(a, b), n


def test_detector_launcher_with_gru_checkpoint(tmp_path, graph_golden):
    from leak_det_gnn_b200.train_detector_dp import load_predictor, main

    sensors = [str(s) for s in graph_golden("LTA")["sensor_node_ids"]]
    torch.manual_seed(1)
    pred = NormalPredictorGRU(len(sensors), 9)
    ckpt = tmp_path / "predictor_best.ckpt"
    torch.save({"epoch": 1, "arch": "gru", "model_state": pred.state_dict(), "standardizer_mean": [0.0] * len(sensors),
                "standardizer_std": [1.0] * len(sensors), "sensor_ids": sensors, "args": {}}, ckpt)
    model, _ = load_predictor(ckpt, torch.device("cuda"))
    assert isinstance(model, NormalPredictorGRU) and model._native_ok(torch.zeros(1, device="cuda"))
    main(["--inp_path", str(TOPO["LTA"]), "--out_dir", str(tmp_path / "det"), "--synthetic", "32", "--predictor_ckpt",
          str(ckpt), "--synthetic_pipes", "40", "--batch_size", "32", "--epochs", "1", "--val_steps", "32"])
    for name in ("detector_best.ckpt", "detector_last.ckpt"):
        assert (tmp_path / "det" / name).exists(), name


def test_layer_rejects_bad_arguments():
    lib = _lib.load()
    q, l = 4, 3
    gx = torch.zeros(3, q * l, 128, device="cuda")
    w = torch.zeros(384, 128, device="cuda")
    b = torch.zeros(128, device="cuda")
    h = torch.zeros(q, 128, device="cuda")
    s = torch.zeros(q * l, 128, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(q_=q, l_=l, hd=128, gx_=gx.data_ptr(), w_=w.data_ptr(), b_=b.data_ptr(), s_=s.data_ptr(), h_=h.data_ptr()):
        return lib.ltgnn_gru_layer_fwd(0, q_, l_, hd, gx_, w_, b_, s_, h_, stream)

    assert call() == 0
    assert call(hd=64) == -2                                           # LTGNN_E_SHAPE
    assert call(q_=0) == -1 and call(l_=0) == -1 and call(q_=-1) == -1  # LTGNN_E_ARG
    assert call(gx_=None) == -1 and call(w_=None) == -1 and call(b_=None) == -1 and call(h_=None) == -1
    assert call(s_=None) == 0                                          # the state sequence is optional
    assert call(gx_=gx.data_ptr() + 4) == -3 and call(h_=h.data_ptr() + 4) == -3   # LTGNN_E_ALIGN
    assert call(s_=s.data_ptr() + 4) == -3 and call(w_=w.data_ptr() + 4) == -3
    with pytest.raises(_lib.LtgnnError) as e:
        _lib.check(call(hd=64))
    assert e.value.code == -2 and "128" in str(e.value)
    torch.cuda.synchronize()
    layer = (torch.zeros(3, 128, 64, device="cuda"), torch.zeros(3, 128, device="cuda"), w, b)
    with pytest.raises(ValueError):
        ops.gru_layer_fwd(torch.zeros(q * l, 32, device="cuda"), q, l, layer)       # K does not match the weights
    with pytest.raises(ValueError):
        ops.gru_layer_fwd(torch.zeros(q * l, 64, device="cuda", dtype=torch.float64), q, l, layer)
    with pytest.raises(ValueError):
        ops.gru_predictor_fwd(torch.zeros(q, l, 60, device="cuda"), torch.zeros(q, l, 9, device="cuda"), [layer])
