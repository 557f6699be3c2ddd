"""Explainer edge masks on the GPU: the masked detector and GCNConv against the fp64 oracle (oracle/pyg_explain.py),
the pruned frozen backward, the fused explainer update against torch.optim.Adam in fp64, and explain_edges against the
fp64 restatement of PyG's GNNExplainer loop -- batched, graphed and at the lta4096 shape.  Tolerance as everywhere here:
max|a - b| <= max(1e-5, 3x the fp32 oracle's own distance) max|b| against fp64."""
import numpy as np
import pytest
import torch

from conftest import TOPO, parity_log, rel_err
from leak_det_gnn_b200 import explain, instrument, ops
from leak_det_gnn_b200.graph import parse_epanet_inp
from oracle.pyg_explain import GCNConv as OracleConv
from oracle.pyg_explain import MaskedOracleLeakDetector, explain_batched, initial_logits

pytestmark = pytest.mark.gpu
TOL = 1e-5
WEIGHT_KERNELS = ("wgrad", "wgrad_tc", "pipe_head_bwd_w", "head_wide_finish", "node_init_bwd")


def _pipes(n):
    return [ln.split()[0] for ln in parse_epanet_inp(TOPO["LTA"])["PIPES"]][:n]


def _detector(sensor_hidden, node_hidden, n_pipes=40, seed=19):
    from leak_det_gnn_b200.models import LeakDetector

    z = np.load(TOPO["LTA"].parent / "graph_LTA.npz")
    torch.manual_seed(seed)
    return LeakDetector(TOPO["LTA"], [str(x) for x in z["sensor_node_ids"]], _pipes(n_pipes), sensor_hidden=sensor_hidden,
                        node_hidden=node_hidden)


def _oracle(ours, state, dtype):
    m = MaskedOracleLeakDetector(len(ours.node_names), ours.edge_index_single, ours.pipe_ends,
                                 ours.sensor_node_idx.tolist(), ours.sensor_encoder.hidden_size,
                                 ours.sensor_to_node.out_features, 2, 0.0, True).to(dtype)
    m.load_state_dict({k: v.to(dtype) for k, v in state.items()}, strict=True)
    return m.eval()


def _cuda_eval(ours):
    return ours.cuda().eval()


# ------------------------------------------------------------------------------------------------ masked detector
@pytest.mark.parametrize("sensor_hidden,node_hidden", [(64, 64), (128, 128)])
@pytest.mark.parametrize("shape", ["shared", "per_window"])
@pytest.mark.parametrize("weights", [False, True])
def test_masked_detector_matches_oracle(sensor_hidden, node_hidden, shape, weights):
    """Logits and d mask (and the joint d edge_weight with weights) against fp64, eval mode."""
    ours = _detector(sensor_hidden, node_hidden)
    state = {k: v.clone() for k, v in ours.state_dict().items()}
    ours = _cuda_eval(ours)
    gen = torch.Generator().manual_seed(8)
    b, l, s, e = 6, 36, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen), torch.randn(b, l, 9, generator=gen)
    rows = (e,) if shape == "shared" else (b, e)
    mask = torch.rand(*rows, generator=gen)
    w = torch.rand(*rows, generator=gen) + 0.2 if weights else None
    label = torch.randint(0, 41, (b,), generator=gen)

    def run(model, dtype, device):
        mk = mask.to(device, dtype, copy=True).requires_grad_(True)
        ew = None if w is None else w.to(device, dtype, copy=True).requires_grad_(True)
        logits = model(residual.to(device, dtype), tfeat.to(device, dtype), edge_weight=ew, edge_mask=mk)
        loss = torch.nn.functional.cross_entropy(logits, label.to(device))
        grads = torch.autograd.grad(loss, [mk] + ([] if ew is None else [ew]))
        return [logits] + list(grads)

    o64 = run(_oracle(ours, state, torch.float64), torch.float64, "cpu")
    o32 = run(_oracle(ours, state, torch.float32), torch.float32, "cpu")
    got = run(ours, torch.float32, "cuda")
    assert got[1].shape == mask.shape
    names = ["logits", "d_mask", "d_edge_weight"][:len(got)]
    rep = {k: {"ours": rel_err(a, c), "oracle_fp32": rel_err(o, c)} for k, a, o, c in zip(names, got, o32, o64)}
    parity_log(f"masked detector {shape} weights={weights} sensor={sensor_hidden} node={node_hidden}", rep)
    for k, r in rep.items():
        assert r["ours"] <= max(TOL, 3.0 * r["oracle_fp32"]), (k, r)


def test_all_ones_mask_is_the_unmasked_detector():
    ours = _cuda_eval(_detector(64, 64)).requires_grad_(False)
    gen = torch.Generator().manual_seed(3)
    b, s, e = 5, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    h_s = torch.randn(b, s, 64, generator=gen).cuda()
    plain = ours.gnn_stack(h_s)
    for ones in (torch.ones(e, device="cuda"), torch.ones(b, e, device="cuda")):
        assert rel_err(ours.gnn_stack(h_s, edge_mask=ones), plain) <= 1e-6
    ew = (torch.rand(b, e, generator=gen) + 0.5).cuda()
    assert rel_err(ours.gnn_stack(h_s, ew, torch.ones(e, device="cuda")), ours.gnn_stack(h_s, ew)) <= 1e-6
    assert torch.equal(ours.gnn_stack(h_s), plain)  # the unmasked path is untouched


def test_input_self_loop_mask_has_no_effect_and_no_gradient():
    from leak_det_gnn_b200.nn import GCNConv

    ei = torch.tensor([[0, 1, 1, 2, 2, 2, 3, 3, 4], [1, 0, 2, 1, 2, 3, 2, 4, 3]])  # edge 4: node 2's input self loop
    torch.manual_seed(5)
    conv = GCNConv(32, 32).cuda()
    with torch.no_grad():
        conv.bias.normal_()
    gen = torch.Generator().manual_seed(6)
    x = torch.randn(5, 32, generator=gen)
    m = torch.rand(9, generator=gen)
    r = torch.randn(5, 32, generator=gen)
    mc = m.cuda().requires_grad_(True)
    y = conv(x.cuda(), ei.cuda(), edge_mask=mc)
    (dm,) = torch.autograd.grad((y * r.cuda()).sum(), mc)
    assert dm[4].item() == 0.0 and (dm[[0, 1, 2, 3, 5, 6, 7, 8]] != 0).all()
    m2 = m.clone()
    m2[4] = 123.0
    assert torch.equal(conv(x.cuda(), ei.cuda(), edge_mask=m2.cuda()), y.detach())
    ref = OracleConv(32, 32).double()
    ref.load_state_dict({k: v.double().cpu() for k, v in conv.state_dict().items()})
    m64 = m.double().requires_grad_(True)
    y64 = ref(x.double(), ei, None, m64)
    (y64 * r.double()).sum().backward()
    rep = {"y": rel_err(y, y64), "d_mask": rel_err(dm, m64.grad)}
    parity_log("GCNConv input self loop mask", rep)
    assert all(v <= TOL for v in rep.values()), rep


# ------------------------------------------------------------------------------------------------ frozen pruning
@pytest.mark.parametrize("node_hidden", [64, 128])
def test_frozen_backward_keeps_bits_and_skips_weight_kernels(node_hidden):
    ours = _cuda_eval(_detector(node_hidden, node_hidden))
    gen = torch.Generator().manual_seed(10)
    b, l, s, e = 6, 36, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen).cuda(), torch.randn(b, l, 9, generator=gen).cuda()
    ew0 = (torch.rand(b, e, generator=gen) + 0.5).cuda()
    mk0 = torch.rand(b, e, generator=gen).cuda()
    target = torch.randint(0, 41, (b,), generator=gen).cuda()

    def grads():
        x, t = residual.clone().requires_grad_(True), tfeat.clone().requires_grad_(True)
        ew, mk = ew0.clone().requires_grad_(True), mk0.clone().requires_grad_(True)
        logits = ours(x, t, edge_weight=ew, edge_mask=mk)
        return torch.autograd.grad(logits.gather(1, target[:, None]).sum(), [x, t, ew, mk])

    ours.requires_grad_(True)
    trainable = grads()
    ours.requires_grad_(False)
    frozen = grads()
    for name, a, c in zip(("d_residual", "d_tfeat", "d_edge_weight", "d_mask"), trainable, frozen):
        assert torch.equal(a, c), name

    # the explainer's call: sensor embeddings without gradient, mask (and weights) with
    with torch.no_grad():
        h_s = ours.sensor_encoder(residual, tfeat)
    mk = mk0.clone().requires_grad_(True)
    ew = ew0.clone().requires_grad_(True)
    torch.cuda.synchronize()
    instrument.reset(timing=True)
    logits = ours.gnn_stack(h_s, ew, mk)
    torch.autograd.grad(logits.gather(1, target[:, None]).sum(), [ew, mk])
    torch.cuda.synchronize()
    launched = set(instrument.summary())
    instrument.reset()
    assert {"gcn_adj_grad", "edge_mask_bwd", "edge_norm_bwd"} <= launched, launched
    assert not launched & set(WEIGHT_KERNELS), launched & set(WEIGHT_KERNELS)


# ------------------------------------------------------------------------------------------------ explain step
def _adam64(m, g, state, step, hard, edge_size, edge_ent):
    """One fp64 step of the restated loss (sum(g * sigmoid(m)) standing in for the prediction loss) with Adam."""
    p = torch.nn.Parameter(m.double().clone())
    opt = torch.optim.Adam([p], lr=0.01)
    if step:
        opt.state[p] = {"step": torch.tensor(float(step)), "exp_avg": state[0].double().clone(),
                        "exp_avg_sq": state[1].double().clone()}
    loss = (g.double() * p.sigmoid()).sum()
    if hard is not None:
        for b in range(m.shape[0]):
            if hard[b].any():
                sm = p[b][hard[b]].sigmoid()
                ent = -sm * torch.log(sm + 1e-15) - (1 - sm) * torch.log(1 - sm + 1e-15)
                loss = loss + edge_size * sm.sum() + edge_ent * ent.mean()
    loss.backward()
    grad = p.grad.clone()
    opt.step()
    st = opt.state[p]
    return p.detach(), st["exp_avg"], st["exp_avg_sq"], grad


def test_explain_step_matches_fp64_adam():
    gen = torch.Generator().manual_seed(4)
    b, e = 4, 300
    m = torch.randn(b, e, generator=gen)
    g = torch.randn(b, e, generator=gen)
    g[:, ::7] = 0.0           # entries the prediction does not depend on
    g[3] = 0.0                # a window with no hard entry
    m_d, s_d = m.cuda(), torch.sigmoid(m).cuda()
    ea, eas = torch.zeros(b, e, device="cuda"), torch.zeros(b, e, device="cuda")
    hard = torch.zeros(b, e, device="cuda", dtype=torch.bool)
    n_hard = torch.zeros(b, device="cuda", dtype=torch.int32)
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    ops.explain_step(g.cuda(), m_d, s_d, ea, eas, hard, n_hard, step, True)
    want = _adam64(m, g, None, 0, None, 0.005, 1.0)
    assert torch.equal(hard.cpu(), want[3] != 0) and torch.equal(n_hard.cpu(), (want[3] != 0).sum(1).int())
    assert n_hard[3].item() == 0 and step.item() == 1
    rep = {"epoch0 m": rel_err(m_d, want[0]), "epoch0 s": rel_err(s_d, want[0].sigmoid()),
           "epoch0 exp_avg": rel_err(ea, want[1]), "epoch0 exp_avg_sq": rel_err(eas, want[2])}
    # a later epoch (step 5): regularisers on the hard mask, the empty window's entropy term 0 (no NaN)
    g2 = torch.randn(b, e, generator=gen)
    step.fill_(4)
    before = (m_d.cpu(), (ea.cpu(), eas.cpu()))
    ops.explain_step(g2.cuda(), m_d, s_d, ea, eas, hard, n_hard, step, False)
    want = _adam64(before[0], g2, before[1], 4, hard.cpu(), 0.005, 1.0)
    assert step.item() == 5 and torch.isfinite(m_d).all()
    rep.update({"epoch4 m": rel_err(m_d, want[0]), "epoch4 s": rel_err(s_d, want[0].sigmoid()),
                "epoch4 exp_avg": rel_err(ea, want[1]), "epoch4 exp_avg_sq": rel_err(eas, want[2])})
    parity_log("explain_step vs fp64 Adam", rep)
    assert all(v <= TOL for v in rep.values()), rep


# ------------------------------------------------------------------------------------------------ explain_edges
def _oracle_explain(ours, state, residual, tfeat, target, m0, epochs):
    model = _oracle(ours, state, torch.float64)
    with torch.no_grad():
        h_s = model.sensor_encoder(residual.double(), tfeat.double())
    return explain_batched(model, h_s, target, m0.double(), epochs=epochs)


def _compare_masks(tag, got, want, want_hard):
    err = (got.cpu().double() - want).abs().max().item()
    got_hard = got.cpu() != 0
    top_ok = [set(got[i].cpu().topk(10).indices.tolist()) == set(want[i].topk(10).indices.tolist())
              for i in range(got.shape[0])]
    parity_log(tag, {"max_abs": err, "hard_equal": bool(torch.equal(got_hard, want_hard)), "top10_equal": top_ok})
    assert torch.equal(got_hard, want_hard)
    assert err <= 1e-4, err
    assert all(top_ok), top_ok


def test_explain_edges_matches_fp64_loop():
    ours = _detector(64, 64, seed=29)
    state = {k: v.clone() for k, v in ours.state_dict().items()}
    ours = ours.cuda().train()
    gen = torch.Generator().manual_seed(30)
    b, l, s, e = 4, 36, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen), torch.randn(b, l, 9, generator=gen)
    got = explain.explain_edges(ours, residual.cuda(), tfeat.cuda(), generator=torch.Generator().manual_seed(31))
    assert ours.training and all(p.requires_grad for p in ours.parameters())  # restored
    assert got.shape == (b, e)
    model = _oracle(ours, state, torch.float64)
    with torch.no_grad():
        target = model(residual.double(), tfeat.double()).argmax(-1)
        assert torch.equal(target, ours.eval()(residual.cuda(), tfeat.cuda()).argmax(-1).cpu())
    m0 = initial_logits(b, e, len(ours.node_names), torch.Generator().manual_seed(31))
    want, want_hard, _ = _oracle_explain(ours, state, residual, tfeat, target, m0, 100)
    _compare_masks("explain_edges B=4 vs fp64", got, want, want_hard)
    # the phenomenon explanation of the no-leak class
    t_noleak = torch.full((b,), len(ours.pipe_ids), dtype=torch.long)
    got = explain.explain_edges(ours, residual.cuda(), tfeat.cuda(), t_noleak.cuda(), epochs=30,
                                generator=torch.Generator().manual_seed(31))
    want, want_hard, _ = _oracle_explain(ours, state, residual, tfeat, t_noleak, m0, 30)
    _compare_masks("explain_edges no-leak target vs fp64", got, want, want_hard)


def test_explain_edges_batched_equals_single_windows_and_repeats(monkeypatch):
    ours = _cuda_eval(_detector(64, 64))
    gen = torch.Generator().manual_seed(40)
    b, l, s, e = 5, 36, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen).cuda(), torch.randn(b, l, 9, generator=gen).cuda()
    target = torch.randint(0, 41, (b,), generator=gen).cuda()
    m0 = initial_logits(b, e, len(ours.node_names), torch.Generator().manual_seed(41))
    rows = {"m0": m0}
    monkeypatch.setattr(explain, "initial_mask_logits", lambda *a, **k: rows["m0"].clone())
    full = explain.explain_edges(ours, residual, tfeat, target, epochs=40)
    again = explain.explain_edges(ours, residual, tfeat, target, epochs=40)
    assert torch.equal(full, again)
    worst = 0.0
    for i in range(b):
        rows["m0"] = m0[i:i + 1]
        one = explain.explain_edges(ours, residual[i:i + 1], tfeat[i:i + 1], target[i:i + 1], epochs=40)
        worst = max(worst, (one[0] - full[i]).abs().max().item())
        assert torch.equal(one[0] != 0, full[i] != 0), i
    parity_log("explain_edges B=5 vs B=1", {"max_abs": worst})
    assert worst <= 1e-6, worst


def test_graphed_explainer_equals_eager_loop():
    ours = _cuda_eval(_detector(128, 128))
    gen = torch.Generator().manual_seed(50)
    b, l, s, e = 3, 36, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen).cuda(), torch.randn(b, l, 9, generator=gen).cuda()
    target = torch.tensor([1, 7, 40]).cuda()
    epochs = 12
    got = explain.explain_edges(ours, residual, tfeat, target, epochs=epochs, generator=torch.Generator().manual_seed(51))

    ours.requires_grad_(False)
    with torch.no_grad():
        h_s = ours.sensor_encoder(residual, tfeat)
    m = explain.initial_mask_logits(b, e, len(ours.node_names), torch.Generator().manual_seed(51)).cuda()
    s_ = torch.sigmoid(m).requires_grad_(True)
    ea, eas = torch.zeros_like(m), torch.zeros_like(m)
    hard = torch.zeros(b, e, device="cuda", dtype=torch.bool)
    n_hard = torch.zeros(b, device="cuda", dtype=torch.int32)
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    for ep in range(epochs):
        loss = torch.nn.functional.cross_entropy(ours.gnn_stack(h_s, edge_mask=s_), target, reduction="sum")
        (g,) = torch.autograd.grad(loss, s_)
        ops.explain_step(g, m, s_.detach(), ea, eas, hard, n_hard, step, ep == 0)
    ours.requires_grad_(True)
    assert torch.equal(got, torch.where(hard, s_.detach(), torch.zeros((), device="cuda")))


def test_lta4096_explainer_matches_fp64_on_sampled_windows():
    ours = _detector(64, 64, n_pipes=764, seed=23)
    state = {k: v.clone() for k, v in ours.state_dict().items()}
    ours = _cuda_eval(ours)
    gen = torch.Generator().manual_seed(9)
    b, l, s, e = 4096, 288, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    residual, tfeat = torch.randn(b, l, s, generator=gen), torch.randn(b, l, 9, generator=gen)
    target = torch.randint(0, 765, (b,), generator=gen)
    got = explain.explain_edges(ours, residual.cuda(), tfeat.cuda(), target.cuda(),
                                generator=torch.Generator().manual_seed(60))
    sample = [0, 1, 2047, 4095]
    m0 = initial_logits(b, e, len(ours.node_names), torch.Generator().manual_seed(60))[sample]
    want, want_hard, _ = _oracle_explain(ours, state, residual[sample], tfeat[sample], target[sample], m0, 100)
    _compare_masks("explain_edges lta4096 sampled windows vs fp64", got[sample], want, want_hard)


def test_bad_masks_raise_before_any_launch():
    ours = _cuda_eval(_detector(64, 64)).requires_grad_(False)
    b, s, e = 2, len(ours.sensor_node_ids), ours.edge_index_single.shape[1]
    h_s = torch.randn(b, s, 64, device="cuda")
    bad = [torch.ones(e + 1, device="cuda"), torch.ones(b + 1, e, device="cuda"),
           torch.ones(e, device="cuda", dtype=torch.float64), torch.ones(e), torch.ones(e, 2, device="cuda").t()[0],
           torch.ones(e, b, device="cuda").t()]
    torch.cuda.synchronize()
    instrument.reset()
    for m in bad:
        with pytest.raises(ValueError, match="edge_mask"):
            ours.gnn_stack(h_s, edge_mask=m)
    assert instrument.launches == 0
