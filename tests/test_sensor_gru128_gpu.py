"""The shared sensor GRU encoder at hidden 128 (reference detector.py:28-73 with sensor_hidden = 128) on the cluster
recurrence of csrc/gru_pred.cu: the sensor input form of the forward against fp64 torch.nn.GRU, the slabbed BPTT's
parameter gradients, the module against cuDNN, the whole detector against the fp64 oracle, the graphed step, the
lta4096 shape and the C argument checks."""
import copy
import ctypes

import pytest
import torch

from conftest import TOPO, parity_log, rel_err
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops

pytestmark = pytest.mark.gpu
NAMES = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")
FWD_TOL, BPTT_TOL = 2e-5, 5e-5     # test_gru_forward / test_gru_backward's bounds at hidden 64


def _ref(r, tf, gru):
    b, l, s = r.shape
    seq = r.transpose(1, 2).reshape(b * s, l, 1)
    if tf is not None:
        seq = torch.cat([seq, tf.unsqueeze(1).expand(b, s, l, tf.shape[-1]).reshape(b * s, l, -1)], dim=-1)
    out, _ = gru(seq)
    return out  # (B*S, L, H)


def _case(b, l, s, f, seed):
    torch.manual_seed(seed)
    gru = torch.nn.GRU(input_size=1 + f, hidden_size=128, num_layers=1, batch_first=True).double()
    r = torch.randn(b, l, s)
    tf = torch.randn(b, l, f) if f else None
    return gru, r, tf


def _weights(gru):
    return [getattr(gru, n).detach().float().cuda().contiguous() for n in NAMES]


@pytest.mark.parametrize("b,l,s,f", [(1, 1, 1, 0), (3, 36, 29, 9), (10, 36, 29, 9), (2, 288, 29, 9), (5, 12, 7, 3),
                                     (32, 6, 4, 9), (40, 5, 29, 0)])
def test_sensor_forward(b, l, s, f):
    """h_last and every state within 2e-5 of fp64 nn.GRU; the inference and training forwards give the same h_last bit
    for bit, and so does a repeated run.  Q = B S covers below, at and across multiples of the 128-sequence tile, with
    tiles that span window boundaries."""
    gru, r, tf = _case(b, l, s, f, b * 100 + l)
    out = _ref(r.double(), None if tf is None else tf.double(), gru)
    w_ih, w_hh, b_ih, b_hh = _weights(gru)
    rc, tfc = r.cuda(), None if tf is None else tf.cuda()
    q = b * s
    tproj = ops.gru_sensor_tproj(tfc, w_ih, b_ih, b_hh, b, l)
    args = (rc, tproj, w_ih[:, 0].contiguous(), w_hh, b_hh[256:].contiguous())
    h_inf = torch.empty(q, 128, device="cuda")
    ops.gru_sensor_fwd(*args, 0, q, h_inf)
    h_tr = torch.empty(q, 128, device="cuda")
    hseq = torch.empty(q * l, 128, device="cuda")
    gates = torch.empty(4, q * l, 128, device="cuda")
    ops.gru_sensor_fwd(*args, 0, q, h_tr, hseq, gates)
    e_last, e_seq = rel_err(h_inf, out[:, -1, :]), rel_err(hseq.view(q, l, 128), out)
    parity_log(f"sensor_gru128 forward B={b} L={l} S={s} F={f}", {"h_last": e_last, "hseq": e_seq})
    assert e_last <= FWD_TOL and e_seq <= FWD_TOL
    assert torch.equal(h_inf, h_tr)
    h_again = torch.empty_like(h_inf)
    ops.gru_sensor_fwd(*args, 0, q, h_again)
    assert torch.equal(h_again, h_inf)
    assert torch.equal(ops.gru_encode(rc, tfc, w_ih, w_hh, b_ih, b_hh).view(q, 128), h_inf)


def test_no_grad_saves_nothing():
    """In grad mode off (eval, event evaluation) with parameters that require gradients, the encoder makes one launch and
    keeps nothing: its allocations stay at T and h_last (the saved gates alone would be 137 MB here)."""
    from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder
    b, l, s = 64, 36, 29
    torch.manual_seed(4)
    enc = SharedSensorGRUEncoder(hidden_size=128).cuda()
    r, tf = torch.randn(b, l, s, device="cuda"), torch.randn(b, l, 9, device="cuda")
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with torch.no_grad():
        h = enc(r, tf)
    torch.cuda.synchronize()
    assert h.grad_fn is None and torch.cuda.max_memory_allocated() - base < 16 << 20
    assert torch.equal(h, enc(r, tf).detach())


def test_sensor_forward_sequence_range():
    """A launch over sequences q0 .. q0 + n - 1 gives exactly those rows of the whole launch, including ranges that
    start inside a window."""
    b, l, s, f = 12, 20, 29, 9
    gru, r, tf = _case(b, l, s, f, 11)
    w_ih, w_hh, b_ih, b_hh = _weights(gru)
    rc, tfc = r.cuda(), tf.cuda()
    q = b * s
    args = (rc, ops.gru_sensor_tproj(tfc, w_ih, b_ih, b_hh, b, l), w_ih[:, 0].contiguous(), w_hh,
            b_hh[256:].contiguous())
    h_all, hs_all, g_all = torch.empty(q, 128, device="cuda"), torch.empty(q * l, 128, device="cuda"), \
        torch.empty(4, q * l, 128, device="cuda")
    ops.gru_sensor_fwd(*args, 0, q, h_all, hs_all, g_all)
    for q0, n in ((0, 128), (128, 129), (257, q - 257), (31, 1)):
        h, hs, g = torch.empty(n, 128, device="cuda"), torch.empty(n * l, 128, device="cuda"), \
            torch.empty(4, n * l, 128, device="cuda")
        ops.gru_sensor_fwd(*args, q0, n, h, hs, g)
        assert torch.equal(h, h_all[q0:q0 + n])
        assert torch.equal(hs, hs_all[q0 * l:(q0 + n) * l])
        assert torch.equal(g, g_all[:, q0 * l:(q0 + n) * l])


def _grad_case(b, l, s, f, seed):
    gru, r, tf = _case(b, l, s, f, seed)
    dh = torch.randn(b * s, 128)
    out = _ref(r.double(), None if tf is None else tf.double(), gru)
    (out[:, -1, :] * dh.double()).sum().backward()
    w = [t.requires_grad_(True) for t in _weights(gru)]
    h = ops.gru_encode(r.cuda(), None if tf is None else tf.cuda(), *w)
    (h.reshape(b * s, 128) * dh.cuda()).sum().backward()
    return {n: rel_err(p.grad, getattr(gru, n).grad) for n, p in zip(NAMES, w)}


@pytest.mark.parametrize("b,l,s,f", [(2, 5, 3, 2), (3, 36, 29, 9), (7, 20, 29, 9), (2, 100, 29, 9), (9, 8, 11, 0),
                                     (32, 6, 4, 9)])
def test_sensor_backward(b, l, s, f):
    """The four parameter gradients (BPTT of ltgnn_gru_layer_bwd, weight gradients against [r | tf | 1]) within 5e-5 of
    fp64 nn.GRU autograd."""
    rep = _grad_case(b, l, s, f, 7 * b + l)
    parity_log(f"sensor_gru128 backward B={b} L={l} S={s} F={f}", rep)
    assert all(e <= BPTT_TOL for e in rep.values()), rep


def test_sensor_backward_in_several_slabs(monkeypatch):
    """One wave of resident tiles per slab and 2.5 waves of sequences: three slabs, the last one partial and starting
    inside a window; the slabs' gradients are added in order."""
    monkeypatch.setattr(ops, "_SLAB_BYTES", 1)
    wave = 128 * ops.gru_resident_tiles(torch.cuda.current_device())
    s, l = 29, 6
    b = (5 * wave // 2 + s - 1) // s
    assert len(ops.gru_sensor_slabs(b * s, l, torch.cuda.current_device())) == 3
    rep = _grad_case(b, l, s, 9, 5)
    parity_log(f"sensor_gru128 backward 3 slabs B={b} L={l} S={s} F=9", rep)
    assert all(e <= BPTT_TOL for e in rep.values()), rep


def test_encoder_module_native_matches_cudnn():
    from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder
    torch.manual_seed(3)
    enc = SharedSensorGRUEncoder(hidden_size=128).cuda().train()
    r = torch.randn(6, 36, 29, device="cuda")
    tf = torch.randn(6, 36, 9, device="cuda")
    dh = torch.randn(6, 29, 128, device="cuda")
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


def _pipes(n):
    from leak_det_gnn_b200.graph import parse_epanet_inp
    return [ln.split()[0] for ln in parse_epanet_inp(TOPO["LTA"])["PIPES"]][:n]


@pytest.mark.parametrize("node_hidden", [64, 128])
def test_detector_sensor_hidden_128_matches_oracle(graph_golden, node_hidden):
    """LeakDetector(sensor_hidden=128) on L-TOWN-A, B = 8, L = 36, from a seeded state_dict: logits, the loss and all 18
    gradients within 1e-5 of the fp64 oracle per tensor, or no further than 3x the fp32 oracle's own distance."""
    from leak_det_gnn_b200.models import LeakDetector
    from oracle.detector_oracle import OracleLeakDetector

    g = graph_golden("LTA")
    pipes = _pipes(40)
    torch.manual_seed(17)
    ours = LeakDetector(TOPO["LTA"], [str(x) for x in g["sensor_node_ids"]], pipes, sensor_hidden=128,
                        node_hidden=node_hidden)
    state = {k: v.clone() for k, v in ours.state_dict().items()}
    assert len(state) == 18
    ours = ours.cuda().eval()
    gen = torch.Generator().manual_seed(2)
    b, l, s = 8, 36, len(ours.sensor_node_ids)
    residual, tfeat = torch.randn(b, l, s, generator=gen), torch.randn(b, l, 9, generator=gen)
    label = torch.randint(0, len(pipes) + 1, (b,), generator=gen)

    def oracle(dtype):
        m = OracleLeakDetector(len(ours.node_names), ours.edge_index_single, ours.pipe_ends, ours.sensor_node_idx.tolist(),
                               128, node_hidden, 2, 0.1, True).to(dtype)
        m.load_state_dict({k: v.to(dtype) for k, v in state.items()}, strict=True)
        m.eval()
        logits = m(residual.to(dtype), tfeat.to(dtype))
        loss = torch.nn.functional.cross_entropy(logits, label)
        loss.backward()
        return logits, loss, {n: p.grad for n, p in m.named_parameters()}

    l64, loss64, g64 = oracle(torch.float64)
    l32, loss32, g32 = oracle(torch.float32)
    logits = ours(residual.cuda(), tfeat.cuda())
    loss = torch.nn.functional.cross_entropy(logits, label.cuda())
    loss.backward()
    rep = {"logits": (rel_err(logits, l64), rel_err(l32, l64)),
           "loss": (rel_err(loss.reshape(1), loss64.reshape(1)), rel_err(loss32.reshape(1), loss64.reshape(1)))}
    for n, p in ours.named_parameters():
        rep[n] = (rel_err(p.grad, g64[n]), rel_err(g32[n], g64[n]))
    assert len(rep) == 2 + 18
    parity_log(f"sensor_gru128 detector node_hidden={node_hidden}",
               {k: {"ours": a, "oracle_fp32": r} for k, (a, r) in rep.items()})
    for k, (a, r) in rep.items():
        assert a <= max(1e-5, 3.0 * r), (k, a, r)


def test_graphed_step_equals_eager_step_sensor_hidden_128(graph_golden):
    """GraphedTrainStep at sensor_hidden = 128, dropout off: three replays equal three eager steps bit for bit."""
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.models import LeakDetector
    from leak_det_gnn_b200.parallel import FlatGradBucket

    g = graph_golden("LTA")
    bsz, l_det, n_pipes = 16, 12, 24
    gen = torch.Generator().manual_seed(5)
    data = [(torch.randn(bsz, l_det, 29, generator=gen), torch.randn(bsz, l_det, 9, generator=gen),
             torch.randint(0, n_pipes + 1, (bsz,), generator=gen)) for _ in range(3)]

    def fresh():
        torch.manual_seed(42)
        m = LeakDetector(TOPO["LTA"], [str(x) for x in g["sensor_node_ids"]], _pipes(n_pipes), sensor_hidden=128,
                         dropout=0.0).cuda().train()
        return m, FlatGradBucket(m.parameters()), torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4,
                                                                     capturable=True)

    m_e, bucket_e, opt_e = fresh()
    losses_e = []
    for noisy, tf, label in data:
        bucket_e.zero()
        loss = torch.nn.functional.cross_entropy(m_e(noisy.cuda(), tf.cuda()), label.cuda())
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m_e.parameters(), 1.0)
        opt_e.step()
        losses_e.append(loss.item())
    m_g, bucket_g, opt_g = fresh()
    step = GraphedTrainStep(m_g, opt_g, bucket_g, bsz, l_det, grad_clip=1.0)
    losses_g = [step(*b).item() for b in data]
    assert losses_g == losses_e, (losses_g, losses_e)
    for (n, a), b in zip(m_e.named_parameters(), m_g.parameters()):
        assert torch.equal(a, b), n


def test_encoder_at_lta4096_shape():
    """One encoder forward + backward on all 118 784 sequences of lta4096 (L = 288), in slabs: the weight gradients
    within 5e-5 of fp64 cuDNN (run in slabs of 256 windows, as test_gru_bptt_at_bench_size does at hidden 64), and the
    peak allocation printed."""
    import bench
    from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder

    b, l, s = 4096, 288, 29
    residual, tfeat, _ = bench.synthetic_batch(b, l, s, 765, 198)
    r, tf = residual.cuda(), tfeat.cuda()
    torch.manual_seed(42)
    enc = SharedSensorGRUEncoder(hidden_size=128).cuda().train()
    ref64, ref32 = copy.deepcopy(enc).double(), copy.deepcopy(enc)
    dh = torch.randn(b, s, 128, device="cuda", generator=torch.Generator(device="cuda").manual_seed(23))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    (enc(r, tf) * dh).sum().backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    print(f"sensor_gru128 B={b} L={l} S={s}: peak allocated {peak / 2**30:.1f} GiB ({(peak - base) / 2**30:.1f} GiB "
          f"above the inputs), {len(ops.gru_sensor_slabs(b * s, l, torch.cuda.current_device()))} slabs")
    assert peak < torch.cuda.get_device_properties(0).total_memory
    for m, dt in ((ref64, torch.float64), (ref32, torch.float32)):
        m.use_native = False
        for i in range(0, b, 256):
            sl = slice(i, i + 256)
            (m(r[sl].to(dt), tf[sl].to(dt)) * dh[sl].to(dt)).sum().backward()
    rep = {n: {"ours": rel_err(getattr(enc.gru, n).grad, getattr(ref64.gru, n).grad),
               "torch_fp32": rel_err(getattr(ref32.gru, n).grad, getattr(ref64.gru, n).grad)} for n in NAMES}
    rep["peak_allocated_gib"] = peak / 2**30
    parity_log(f"sensor_gru128 bptt B={b} L={l} S={s}", rep)
    for n in NAMES:
        assert rep[n]["ours"] <= BPTT_TOL, (n, rep[n])


def test_sensor_fwd_rejects_bad_arguments():
    lib = _lib.load()
    b, l, s = 2, 3, 5
    q = b * s
    r = torch.zeros(b, l, s, device="cuda")
    t = torch.zeros(3, b * l, 128, device="cuda")
    wr = torch.zeros(3, 128, device="cuda")
    w = torch.zeros(384, 128, device="cuda")
    bh = torch.zeros(128, device="cuda")
    h = torch.zeros(q, 128, device="cuda")
    hs = torch.zeros(q * l, 128, device="cuda")
    gt = torch.zeros(4, q * l, 128, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(b_=b, l_=l, s_=s, q0=0, n=q, hd=128, r_=r.data_ptr(), t_=t.data_ptr(), wr_=wr.data_ptr(), w_=w.data_ptr(),
             bh_=bh.data_ptr(), hs_=hs.data_ptr(), h_=h.data_ptr(), g_=gt.data_ptr()):
        return lib.ltgnn_gru_sensor_fwd(0, b_, l_, s_, q0, n, hd, r_, t_, wr_, w_, bh_, hs_, h_, g_, stream)

    assert call() == 0 and call(g_=None) == 0 and call(g_=None, hs_=None) == 0 and call(q0=3, n=q - 3) == 0
    assert call(hd=64) == -2 and call(b_=1 << 30, s_=4) == -2                                   # LTGNN_E_SHAPE
    assert call(b_=0) == -1 and call(l_=0) == -1 and call(s_=0) == -1 and call(n=0) == -1       # LTGNN_E_ARG
    assert call(q0=-1) == -1 and call(q0=1) == -1 and call(n=q + 1) == -1
    for k in ("r_", "t_", "wr_", "w_", "bh_", "h_"):
        assert call(**{k: None}) == -1, k
    assert call(hs_=None) == -1                                                                 # gates need hseq
    for k, p in (("t_", t), ("wr_", wr), ("w_", w), ("hs_", hs), ("h_", h), ("g_", gt)):       # LTGNN_E_ALIGN
        assert call(**{k: p.data_ptr() + 4}) == -3, k
    with pytest.raises(_lib.LtgnnError) as e:
        _lib.check(call(hd=64))
    assert e.value.code == -2 and "128" in str(e.value)
    n = ctypes.c_int32(0)
    assert lib.ltgnn_gru_resident_tiles(0, ctypes.byref(n)) == 0 and n.value > 0
    assert lib.ltgnn_gru_resident_tiles(0, None) == -1
    torch.cuda.synchronize()
