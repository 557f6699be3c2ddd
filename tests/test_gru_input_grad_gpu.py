"""Gradients of the shared sensor GRU encoder and of the whole LeakDetector with respect to their inputs (residual and
time features) on the native kernels, at sensor hidden 64 (csrc/gru.cu) and 128 (csrc/gru_pred.cu): against fp64
torch.nn.GRU autograd, in frozen and trainable modes, across slab splits, at the lta4096 shape, against the fp64 oracle
detector and the cuDNN route, and the C argument checks of ltgnn_gru_bwd_dx / ltgnn_gru_sensor_bwd_dx."""
import copy
import ctypes

import pytest
import torch

from conftest import TOPO, parity_log, rel_err
from leak_det_gnn_b200 import instrument
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops

pytestmark = pytest.mark.gpu
NAMES = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")
WEIGHT_KERNELS = {"gru_bwd_w", "wgrad", "wgrad_tc"}


def _ref(r, tf, gru):
    b, l, s = r.shape
    seq = r.transpose(1, 2).reshape(b * s, l, 1)
    if tf is not None:
        seq = torch.cat([seq, tf.unsqueeze(1).expand(b, s, l, tf.shape[-1]).reshape(b * s, l, -1)], dim=-1)
    out, _ = gru(seq)
    return out  # (B*S, L, H)


def _case(hd, b, l, s, f, seed):
    torch.manual_seed(seed)
    gru = torch.nn.GRU(input_size=1 + f, hidden_size=hd, num_layers=1, batch_first=True).double()
    r = torch.randn(b, l, s)
    tf = torch.randn(b, l, f) if f else None
    dh = torch.randn(b * s, hd)
    return gru, r, tf, dh


def _native(gru, r, tf, dh, params_grad=False):
    """(dr, dtf, parameter gradients or None) of sum(h_last * dh) through ops.gru_encode."""
    w = [getattr(gru, n).detach().float().cuda().contiguous().requires_grad_(params_grad) for n in NAMES]
    rc = r.cuda().requires_grad_(True)
    tfc = None if tf is None else tf.cuda().requires_grad_(True)
    h = ops.gru_encode(rc, tfc, *w)
    (h.reshape(dh.shape) * dh.cuda()).sum().backward()
    return rc.grad, None if tfc is None else tfc.grad, [p.grad for p in w] if params_grad else None


@pytest.mark.parametrize("hd", [64, 128])
@pytest.mark.parametrize("b,l,s,f", [(1, 1, 1, 0), (3, 36, 29, 9), (5, 7, 29, 9)])
def test_input_grad_matches_fp64(hd, b, l, s, f):
    """d residual and d tfeat within 1e-5 of fp64 nn.GRU autograd (max|a - b| / max|b| per tensor); B S = 145 at
    (5, 7, 29) leaves a ragged last tile of 17 sequences."""
    gru, r, tf, dh = _case(hd, b, l, s, f, 13 * b + l + hd)
    r64 = r.double().requires_grad_(True)
    tf64 = None if tf is None else tf.double().requires_grad_(True)
    (_ref(r64, tf64, gru)[:, -1, :] * dh.double()).sum().backward()
    dr, dtf, _ = _native(gru, r, tf, dh)
    rep = {"d_residual": rel_err(dr, r64.grad)}
    if tf is not None:
        rep["d_tfeat"] = rel_err(dtf, tf64.grad)
    parity_log(f"gru input grad H={hd} B={b} L={l} S={s} F={f}", rep)
    assert all(e <= 1e-5 for e in rep.values()), rep


@pytest.mark.parametrize("hd", [64, 128])
def test_frozen_and_trainable_modes(hd, monkeypatch):
    """Frozen parameters and trainable ones give the same input gradients bit for bit; frozen, every parameter's .grad
    stays None and no weight-gradient kernel runs; the parameter gradients with input gradients asked for are those of
    the parameter-only backward bit for bit; a repeated run gives the same bits."""
    from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder

    b, l, s = 5, 36, 29
    torch.manual_seed(hd)
    enc = SharedSensorGRUEncoder(hidden_size=hd).cuda()
    r, tf = torch.randn(b, l, s, device="cuda"), torch.randn(b, l, 9, device="cuda")
    dh = torch.randn(b, s, hd, device="cuda")
    launched = []
    monkeypatch.setattr(instrument, "begin", lambda name: launched.append(name))

    def run(params_grad, inputs_grad):
        enc.zero_grad(set_to_none=True)
        for p in enc.parameters():
            p.requires_grad_(params_grad)
        rc, tfc = r.clone().requires_grad_(inputs_grad), tf.clone().requires_grad_(inputs_grad)
        launched.clear()
        (enc(rc, tfc) * dh).sum().backward()
        return rc.grad, tfc.grad, [None if p.grad is None else p.grad.clone() for p in enc.parameters()], set(launched)

    dr_f, dtf_f, g_f, names_f = run(False, True)
    dr_t, dtf_t, g_t, names_t = run(True, True)
    _, _, g_p, names_p = run(True, False)
    dr_f2, dtf_f2, _, _ = run(False, True)
    dx_kernel = "gru_bwd_dx" if hd == 64 else "gru_sensor_bwd_dx"
    assert all(g is None for g in g_f)
    assert dx_kernel in names_f and not names_f & WEIGHT_KERNELS, names_f
    assert dx_kernel in names_t and names_t & WEIGHT_KERNELS, names_t
    assert dx_kernel not in names_p
    assert torch.equal(dr_f, dr_t) and torch.equal(dtf_f, dtf_t)
    assert torch.equal(dr_f, dr_f2) and torch.equal(dtf_f, dtf_f2)
    for a, c in zip(g_t, g_p):
        assert torch.equal(a, c)


def test_input_grad_in_several_slabs(monkeypatch):
    """Hidden 128 with one wave per slab (three slabs, boundaries inside windows): d residual and d tfeat equal the
    one-slab backward's bit for bit."""
    dev = torch.cuda.current_device()
    wave = 128 * ops.gru_resident_tiles(dev)
    s, l = 29, 6
    b = (5 * wave // 2 + s - 1) // s
    gru, r, tf, dh = _case(128, b, l, s, 9, 3)
    one = _native(gru, r, tf, dh)
    assert len(ops.gru_sensor_slabs(b * s, l, dev)) == 1
    monkeypatch.setattr(ops, "_SLAB_BYTES", 1)
    slabs = ops.gru_sensor_slabs(b * s, l, dev)
    assert len(slabs) == 3 and any(q0 % s for q0, _ in slabs[1:])
    several = _native(gru, r, tf, dh)
    assert torch.equal(one[0], several[0]) and torch.equal(one[1], several[1])


@pytest.mark.parametrize("hd", [64, 128])
def test_input_grad_at_lta4096_shape(hd):
    """Frozen encoder, all 118 784 sequences of lta4096 (L = 288): d residual and d tfeat within 5e-5 of fp64 cuDNN (run
    in slabs of 256 windows, as test_encoder_at_lta4096_shape does), and the peak allocation printed."""
    import bench
    from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder

    b, l, s = 4096, 288, 29
    residual, tfeat, _ = bench.synthetic_batch(b, l, s, 765, 198)
    r, tf = residual.cuda().requires_grad_(True), tfeat.cuda().requires_grad_(True)
    torch.manual_seed(42)
    enc = SharedSensorGRUEncoder(hidden_size=hd).cuda().requires_grad_(False)
    ref64, ref32 = copy.deepcopy(enc).double(), copy.deepcopy(enc)
    dh = torch.randn(b, s, hd, device="cuda", generator=torch.Generator(device="cuda").manual_seed(23))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    (enc(r, tf) * dh).sum().backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    print(f"gru input grad H={hd} B={b} L={l} S={s}: peak allocated {peak / 2**30:.1f} GiB")
    refs = {}
    for m, dt in ((ref64, torch.float64), (ref32, torch.float32)):
        m.use_native = False
        dr, dtf = torch.empty(b, l, s, device="cuda", dtype=dt), torch.empty(b, l, 9, device="cuda", dtype=dt)
        for i in range(0, b, 256):
            sl = slice(i, i + 256)
            ri, ti = r[sl].detach().to(dt).requires_grad_(True), tf[sl].detach().to(dt).requires_grad_(True)
            dr[sl], dtf[sl] = torch.autograd.grad((m(ri, ti) * dh[sl].to(dt)).sum(), (ri, ti))
        refs[dt] = (dr, dtf)
    rep = {n: {"ours": rel_err(a, refs[torch.float64][i]), "torch_fp32": rel_err(refs[torch.float32][i],
                                                                                 refs[torch.float64][i])}
           for i, (n, a) in enumerate((("d_residual", r.grad), ("d_tfeat", tf.grad)))}
    rep["peak_allocated_gib"] = peak / 2**30
    parity_log(f"gru input grad H={hd} B={b} L={l} S={s}", rep)
    for n in ("d_residual", "d_tfeat"):
        assert rep[n]["ours"] <= 5e-5, (n, rep[n])


def _pipes(n):
    from leak_det_gnn_b200.graph import parse_epanet_inp
    return [ln.split()[0] for ln in parse_epanet_inp(TOPO["LTA"])["PIPES"]][:n]


@pytest.mark.parametrize("sensor_hidden,node_hidden", [(64, 64), (128, 128)])
def test_detector_input_grad_matches_oracle(graph_golden, sensor_hidden, node_hidden):
    """Frozen LeakDetector on L-TOWN-A, B = 8, L = 36, eval mode: the gradient of each window's own target logit with
    respect to residual and tfeat, from one backward of logits.gather(1, target).sum(), within 1e-5 of the fp64 oracle
    per tensor or no further than 3x the fp32 oracle's own distance; the cuDNN route (use_native = False) meets the
    same bound."""
    from leak_det_gnn_b200.models import LeakDetector
    from oracle.detector_oracle import OracleLeakDetector

    g = graph_golden("LTA")
    pipes = _pipes(40)
    torch.manual_seed(19)
    ours = LeakDetector(TOPO["LTA"], [str(x) for x in g["sensor_node_ids"]], pipes, sensor_hidden=sensor_hidden,
                        node_hidden=node_hidden)
    state = {k: v.clone() for k, v in ours.state_dict().items()}
    ours = ours.cuda().eval().requires_grad_(False)
    gen = torch.Generator().manual_seed(6)
    b, l, s = 8, 36, len(ours.sensor_node_ids)
    residual, tfeat = torch.randn(b, l, s, generator=gen), torch.randn(b, l, 9, generator=gen)
    # targets whose logit depends on the inputs: the no-leak class (mean pool) and pipes with a sensor at one end; after
    # two GCN layers the logits of pipes far from every sensor are constant
    near = [p for p, (u, v) in enumerate(ours.pipe_ends.tolist())
            if u in ours.sensor_node_idx.tolist() or v in ours.sensor_node_idx.tolist()]
    classes = torch.tensor(near + [len(pipes)])
    assert len(classes) >= 2
    target = classes[torch.randint(0, len(classes), (b,), generator=gen)]

    def input_grads(model, dtype, device):
        x, t = residual.to(device, dtype).requires_grad_(True), tfeat.to(device, dtype).requires_grad_(True)
        logits = model(x, t)
        return torch.autograd.grad(logits.gather(1, target.to(device)[:, None]).sum(), (x, t))

    def oracle(dtype):
        m = OracleLeakDetector(len(ours.node_names), ours.edge_index_single, ours.pipe_ends, ours.sensor_node_idx.tolist(),
                               sensor_hidden, node_hidden, 2, 0.1, True).to(dtype)
        m.load_state_dict({k: v.to(dtype) for k, v in state.items()}, strict=True)
        return input_grads(m.eval(), dtype, "cpu")

    o64, o32 = oracle(torch.float64), oracle(torch.float32)
    native = input_grads(ours, torch.float32, "cuda")
    # cuDNN's RNN backward runs only in training mode; a one-layer GRU has no dropout, so it computes the same function
    ours.sensor_encoder.use_native = False
    ours.sensor_encoder.train()
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        cudnn = input_grads(ours, torch.float32, "cuda")
    finally:
        torch.backends.cudnn.allow_tf32 = old
    rep = {n: {"ours": rel_err(native[i], o64[i]), "oracle_fp32": rel_err(o32[i], o64[i]),
               "cudnn_route": rel_err(cudnn[i], o64[i])} for i, n in enumerate(("d_residual", "d_tfeat"))}
    parity_log(f"detector input grad sensor_hidden={sensor_hidden} node_hidden={node_hidden}", rep)
    assert all(t.abs().max() > 0 for t in o64)
    for n, e in rep.items():
        assert e["ours"] <= max(1e-5, 3.0 * e["oracle_fp32"]), (n, e)
        assert e["cudnn_route"] <= max(1e-5, 3.0 * e["oracle_fp32"]), (n, e)


def test_dx_entry_points_reject_bad_arguments():
    lib = _lib.load()
    b, l, s, f = 2, 3, 5, 4
    q = b * s
    qp = (q + 127) // 128 * 128
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    dr = torch.zeros(b, l, s, device="cuda")
    dxt = torch.zeros(b, l, s, f, device="cuda")

    w64 = torch.zeros(192, 1 + f, device="cuda")
    dg64 = torch.zeros(l * qp, 256, device="cuda")

    def call64(b_=b, l_=l, s_=s, f_=f, hd=64, w_=w64.data_ptr(), g_=dg64.data_ptr(), dr_=dr.data_ptr(),
               dxt_=dxt.data_ptr()):
        return lib.ltgnn_gru_bwd_dx(0, b_, l_, s_, f_, hd, w_, g_, dr_, dxt_, stream)

    assert call64() == 0 and call64(dr_=None) == 0 and call64(dxt_=None) == 0 and call64(b_=0) == 0
    assert call64(f_=0, dxt_=None) == 0
    assert call64(hd=128) == -2 and call64(f_=31) == -2 and call64(b_=1 << 30, s_=4) == -2    # LTGNN_E_SHAPE
    assert call64(b_=-1) == -1 and call64(l_=0) == -1 and call64(s_=0) == -1 and call64(f_=-1) == -1  # LTGNN_E_ARG
    assert call64(w_=None) == -1 and call64(g_=None) == -1 and call64(dr_=None, dxt_=None) == -1
    assert call64(f_=0) == -1                                                                  # dxt needs F > 0
    assert call64(g_=dg64.data_ptr() + 4) == -3 and call64(dr_=dr.data_ptr() + 2) == -3       # LTGNN_E_ALIGN
    assert call64(w_=w64.data_ptr() + 2) == -3 and call64(dxt_=dxt.data_ptr() + 2) == -3

    w128 = torch.zeros(384, 1 + f, device="cuda")
    dg128 = torch.zeros(4, q * l, 128, device="cuda")

    def call128(b_=b, l_=l, s_=s, f_=f, q0=0, n=q, hd=128, w_=w128.data_ptr(), g_=dg128.data_ptr(), dr_=dr.data_ptr(),
                dxt_=dxt.data_ptr()):
        return lib.ltgnn_gru_sensor_bwd_dx(0, b_, l_, s_, f_, q0, n, hd, w_, g_, dr_, dxt_, stream)

    assert call128() == 0 and call128(dr_=None) == 0 and call128(dxt_=None) == 0 and call128(q0=3, n=q - 3) == 0
    assert call128(hd=64) == -2 and call128(f_=31) == -2 and call128(b_=1 << 30, s_=4, n=1) == -2  # LTGNN_E_SHAPE
    assert call128(b_=0) == -1 and call128(l_=0) == -1 and call128(s_=0) == -1 and call128(f_=-1) == -1
    assert call128(q0=-1) == -1 and call128(q0=1) == -1 and call128(n=0) == -1 and call128(n=q + 1) == -1
    assert call128(w_=None) == -1 and call128(g_=None) == -1 and call128(dr_=None, dxt_=None) == -1
    assert call128(f_=0) == -1
    assert call128(g_=dg128.data_ptr() + 4) == -3 and call128(dr_=dr.data_ptr() + 2) == -3
    assert call128(w_=w128.data_ptr() + 2) == -3 and call128(dxt_=dxt.data_ptr() + 2) == -3
    with pytest.raises(_lib.LtgnnError) as e:
        _lib.check(call128(hd=64))
    assert e.value.code == -2 and "128" in str(e.value)
    torch.cuda.synchronize()
