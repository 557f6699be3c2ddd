"""PGExplainer on the GPU: the edge network's kernels (ltgnn_pg_edge_fwd / _bwd + the [P | Q] GEMM and its weight
gradient) against fp64, a whole training step, 30 steps and ``explain`` against the fp64 restatement of PyG's
PGExplainer (oracle/pyg_pg_explainer.py), the graphed step against the eager one, and what the frozen detector launches.
Tolerance as everywhere here: max|a - b| <= max(1e-5, 3x the fp32 oracle's own distance) max|b| against fp64."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN, TOPO, parity_log, rel_err
from leak_det_gnn_b200 import explain, instrument, ops
from leak_det_gnn_b200.graph import parse_epanet_inp
from oracle.pyg_explain import MaskedOracleLeakDetector
from oracle.pyg_pg_explainer import PGExplainerOracle

pytestmark = pytest.mark.gpu
TOL = 1e-5
TRAJ_TOL = 5e-5   # 30 Adam steps: see test_thirty_steps_and_explain_match_fp64_oracle
DETECTOR_WEIGHT_KERNELS = ("wgrad", "pipe_head_bwd_w", "head_wide_finish", "node_init_bwd")


def _check(tag, got, o32, o64, tol=TOL):
    rep = {k: {"ours": rel_err(got[k], o64[k]), "oracle_fp32": rel_err(o32[k], o64[k])} for k in o64}
    parity_log(tag, rep)
    for k, r in rep.items():
        assert r["ours"] <= max(tol, 3.0 * r["oracle_fp32"]), (tag, k, r)


# ------------------------------------------------------------------------------------------------ kernels
def _graph(name):
    if name == "random":
        gen = torch.Generator().manual_seed(11)
        ei = torch.randint(0, 37, (2, 150), generator=gen)
        ei[:, 7] = torch.tensor([4, 4])
        return ei, 37
    z = np.load(GOLDEN / f"graph_{name}.npz")
    return torch.from_numpy(z["edge_index"]).long(), len(z["node_names"])


def _mlp_params(d, seed, device, dtype=torch.float32):
    torch.manual_seed(seed)
    mlp = torch.nn.Sequential(torch.nn.Linear(2 * d, 64), torch.nn.ReLU(), torch.nn.Linear(64, 1))
    return [p.detach().to(device, dtype).contiguous() for p in mlp.parameters()]


def _gate_bits(gate):
    """(B, E, 2) int32 gate words -> (B, E, 64) bool: bit l of word j is unit 2l + j."""
    unit = torch.arange(64, device=gate.device)
    return ((gate[..., unit % 2] >> (unit // 2)) & 1).bool()


def _reference(z, ei, params, u, inv_t, bias, tie_gate=None):
    """The factorised edge network (equal to PyG's concatenated form, test_pg_explain_cpu.py) in torch, any dtype.
    ``tie_gate``: the device's ReLU decisions, used where the pre-activation lies within fp32 rounding of 0 (there
    either decision is right, but it moves d W1 by a whole d logit w2 z term)."""
    w1, b1, w2, b2 = params
    d = z.shape[-1]
    pq = z @ torch.cat([w1[:, :d], w1[:, d:]], 0).t()
    pre = (pq[:, ei[0], :64] + pq[:, ei[1], 64:]) + b1
    on = pre > 0
    if tie_gate is not None:
        mag = pre.detach().abs()
        on = torch.where(mag <= 1e-5 * mag.max(), tie_gate, on)
    logit = (pre * on) @ w2[0] + b2
    if u is None:
        return {"mask": logit.sigmoid()}, pre
    eps = (1 - 2 * bias) * u.to(z.dtype) + bias
    s = (eps.log() - (1 - eps).log() + logit) * inv_t
    return {"s": s, "mask": s.sigmoid()}, pre


@pytest.mark.parametrize("graph", ["LTA", "LT", "random"])
@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("b", [1, 3, 257])
def test_edge_fwd_matches_fp64(graph, d, b):
    ei, n = _graph(graph)
    dev = torch.device("cuda")
    idx = ops.pg_edge_index(ei, n, dev)
    eic = ei.to(dev)
    gen = torch.Generator().manual_seed(b + d)
    z = torch.randn(b, n, d, generator=gen).to(dev)
    p32 = _mlp_params(d, 3, dev)
    p64 = [p.double() for p in p32]
    # explaining: sigmoid(logit)
    got = {"mask": ops.pg_edge_mask(z, idx, *p32)}
    o64, _ = _reference(z.double(), eic, p64, None, 1.0, 0.0)
    o32, _ = _reference(z, eic, p32, None, 1.0, 0.0)
    _check(f"pg_edge_fwd explain {graph} D={d} B={b}", got, o32, o64)
    # the logits: bias 0.5 (no noise) and 1 / T = 1 give s = logit exactly
    one = torch.ones(1, device=dev)
    mask, s = ops.pg_edge_mask(z, idx, *p32, inv_t=one, bias=0.5, seed=5)
    o64, pre64 = _reference(z.double(), eic, p64, torch.zeros(b, ei.shape[1], device=dev), 1.0, 0.5)
    o32, _ = _reference(z, eic, p32, torch.zeros(b, ei.shape[1], device=dev), 1.0, 0.5)
    _check(f"pg_edge_fwd logits {graph} D={d} B={b}", {"s": s, "mask": mask}, o32, o64)
    # training: the concrete sample with the drawn uniforms replayed in fp64, and the gate bits
    inv_t = torch.full((1,), 1.0 / 3.7, device=dev)
    u = torch.empty(b, ei.shape[1], device=dev)
    pq = ops._PgProject.apply(z, p32[0])
    mask, s, gate = ops.pg_edge_fwd(pq, idx, *p32[1:], inv_t=inv_t, bias=0.01, seed=99, uniform=u)
    assert 0.0 <= u.min().item() and u.max().item() < 1.0 and u.std().item() > 0.25
    o64, pre64 = _reference(z.double(), eic, p64, u, inv_t.double(), 0.01)
    o32, _ = _reference(z, eic, p32, u, inv_t, 0.01)
    _check(f"pg_edge_fwd train {graph} D={d} B={b}", {"s": s, "mask": mask}, o32, o64)
    bits = _gate_bits(gate)
    clear = pre64.abs() > 1e-4 * pre64.abs().max()
    assert torch.equal(bits[clear], (pre64 > 0)[clear])


def _edge_grads(z, ei, idx, params, dmask, inv_t, bias, seed):
    """(ours, fp32, fp64) d W1, d b1, d w2, d b2 of sum(mask * dmask) through the training-mode edge network."""
    names = ("dW1", "db1", "dw2", "db2")
    ps = [p.clone().requires_grad_(True) for p in params]
    debug = {}
    old, ops.DEBUG_CAPTURE = ops.DEBUG_CAPTURE, debug
    try:
        mask, _ = ops.pg_edge_mask(z, idx, *ps, inv_t=inv_t, bias=bias, seed=seed)
    finally:
        ops.DEBUG_CAPTURE = old
    ours = dict(zip(names, torch.autograd.grad((mask * dmask).sum(), ps)))
    u, tie = debug["pg_uniform"], _gate_bits(debug["pg_gate"])
    out = [ours]
    for dt in (torch.float32, torch.float64):
        pr = [p.to(dt).clone().requires_grad_(True) for p in params]
        ref, _ = _reference(z.to(dt), ei, pr, u, inv_t.to(dt), bias, tie if dt == torch.float64 else None)
        out.append(dict(zip(names, torch.autograd.grad((ref["mask"] * dmask.to(dt)).sum(), pr))))
    return out


@pytest.mark.parametrize("graph", ["LTA", "LT", "random"])
@pytest.mark.parametrize("d", [64, 128])
def test_edge_bwd_and_wgrad_match_fp64(graph, d):
    ei, n = _graph(graph)
    dev = torch.device("cuda")
    b = 257
    gen = torch.Generator().manual_seed(d)
    z = torch.randn(b, n, d, generator=gen).to(dev)
    dmask = torch.randn(b, ei.shape[1], generator=gen).to(dev)
    got, o32, o64 = _edge_grads(z, ei.to(dev), ops.pg_edge_index(ei, n, dev), _mlp_params(d, 4, dev), dmask,
                                torch.full((1,), 0.31, device=dev), 0.01, 7)
    _check(f"pg_edge_bwd {graph} D={d} B={b}", got, o32, o64)


def test_edge_bwd_and_wgrad_match_fp64_at_lta4096():
    ei, n = _graph("LTA")
    dev = torch.device("cuda")
    b = 4096
    gen = torch.Generator().manual_seed(12)
    z = torch.randn(b, n, 64, generator=gen).to(dev)
    dmask = torch.randn(b, ei.shape[1], generator=gen).to(dev)
    got, o32, o64 = _edge_grads(z, ei.to(dev), ops.pg_edge_index(ei, n, dev), _mlp_params(64, 5, dev), dmask,
                                torch.full((1,), 0.2, device=dev), 0.01, 8)
    _check(f"pg_edge_bwd lta4096 B*E={b * ei.shape[1]}", got, o32, o64)


# ------------------------------------------------------------------------------------------------ the explainer
def _pipes(n):
    return [ln.split()[0] for ln in parse_epanet_inp(TOPO["LTA"])["PIPES"]][:n]


def _detector(d, n_pipes=40, seed=19):
    from leak_det_gnn_b200.models import LeakDetector

    z = np.load(TOPO["LTA"].parent / "graph_LTA.npz")
    torch.manual_seed(seed)
    det = LeakDetector(TOPO["LTA"], [str(x) for x in z["sensor_node_ids"]], _pipes(n_pipes), sensor_hidden=d,
                       node_hidden=d)
    return det, {k: v.clone() for k, v in det.state_dict().items()}


def _oracle(ours, state, dtype):
    m = MaskedOracleLeakDetector(len(ours.node_names), ours.edge_index_single, ours.pipe_ends,
                                 ours.sensor_node_idx.tolist(), ours.sensor_encoder.hidden_size,
                                 ours.sensor_to_node.out_features, 2, 0.0, True).to(dtype)
    m.load_state_dict({k: v.to(dtype) for k, v in state.items()}, strict=True)
    return m.eval()


def _batches(det, n_batches, b, seed):
    gen = torch.Generator().manual_seed(seed)
    s = len(det.sensor_node_ids)
    return [(torch.randn(b, 36, s, generator=gen), torch.randn(b, 36, 9, generator=gen),
             torch.randint(0, len(det.pipe_ids) + 1, (b,), generator=gen)) for _ in range(n_batches)]


class _TieReLU(torch.nn.Module):
    """ReLU that takes the device's decision where the pre-activation lies within fp32 rounding of 0 (either decision
    is right there, but over many Adam steps a different one moves the parameters far beyond rounding)."""

    gate = None

    def forward(self, x):
        on = x > 0
        if self.gate is not None:
            mag = x.detach().abs()
            on = torch.where(mag <= 1e-5 * mag.max(), self.gate.reshape(on.shape), on)
        return x * on


class _Oracles:
    """The fp64 and fp32 restatements of one explainer, driven with the device's uniforms (and, in fp64, its ReLU
    decisions at ties)."""

    def __init__(self, ours, state, ex, epochs):
        d = ex.mlp[0].weight.shape[1] // 2
        self.runs = []
        for dt in (torch.float32, torch.float64):
            o = PGExplainerOracle(d, epochs, lr=ex.lr).to(dt)
            o.mlp.load_state_dict({k: v.detach().cpu().to(dt) for k, v in ex.mlp.state_dict().items()})
            if dt == torch.float64:
                o.mlp[1] = _TieReLU()
            self.runs.append((_oracle(ours, state, dt), o, dt))

    def train(self, epoch, r, t, target, u, h_s=None, gate=None):
        """``h_s``: the device's sensor embeddings, fed to both restatements instead of their own sensor encoders;
        ``gate``: the device's (B, E, 2) ReLU words of this step."""
        out = []
        for model, o, dt in self.runs:
            with torch.no_grad():
                hs = model.sensor_encoder(r.to(dt), t.to(dt)) if h_s is None else h_s.cpu().to(dt)
            if isinstance(o.mlp[1], _TieReLU):
                o.mlp[1].gate = None if gate is None else _gate_bits(gate).cpu()
            out.append(o.train(epoch, model, hs, target, u.cpu().to(dt)))
            if isinstance(o.mlp[1], _TieReLU):
                o.mlp[1].gate = None
        return out

    def explain(self, r, t, h_s=None):
        out = []
        for model, o, dt in self.runs:
            with torch.no_grad():
                hs = model.sensor_encoder(r.to(dt), t.to(dt)) if h_s is None else h_s.cpu().to(dt)
                out.append(o(model, hs))
        return out


@pytest.mark.parametrize("d", [64, 128])
def test_training_step_matches_fp64_oracle(d, monkeypatch):
    det, state = _detector(d)
    det = det.cuda().train()
    ex = explain.PGExplainer(det, epochs=5)
    oracles = _Oracles(det, state, ex, 5)
    ((r, t, target),) = _batches(det, 1, 4, 20 + d)
    debug = {}
    monkeypatch.setattr(ops, "DEBUG_CAPTURE", debug)
    loss = ex.train(2, r.cuda(), t.cuda(), target.cuda())
    assert loss.is_cuda and loss.dim() == 0
    l32, l64 = oracles.train(2, r, t, target, debug["pg_uniform"])
    names = ("loss", "dW1", "db1", "dw2", "db2")
    got = dict(zip(names, [loss] + [p.grad for p in ex.mlp.parameters()]))
    o32 = dict(zip(names, [l32] + [p.grad for p in oracles.runs[0][1].mlp.parameters()]))
    o64 = dict(zip(names, [l64] + [p.grad for p in oracles.runs[1][1].mlp.parameters()]))
    _check(f"PGExplainer step D={d}", got, o32, o64)
    # the detector: parameters bit for bit, flags restored
    assert det.training and all(p.requires_grad for p in det.parameters())
    for k, v in det.state_dict().items():
        assert torch.equal(v.cpu(), state[k]), k


def test_thirty_steps_and_explain_match_fp64_oracle(monkeypatch):
    """30 Adam steps over three batches.  Both restatements read the device's sensor embeddings (the sensor GRU is
    checked on its own elsewhere), and the fp64 one takes the device's ReLU decisions at ties: a unit whose
    pre-activation rounds to either side of 0 changes d W1 by a whole term, which Adam's normalised update then carries
    into the parameters.  Each step's gradients meet the project's 1e-5 bound (test_training_step_matches_fp64_oracle),
    but Adam divides by the running gradient scale, so a relative difference of ~1e-6 in a gradient that nearly cancels
    (d b2 sums d logit over all B E edges, of both signs) moves a parameter by up to ~1e-5 of its size over 30 steps;
    measured on one B200: W1 8.3e-6, b1 3.9e-6, w2 3.3e-6, b2 1.0e-5, the explained masks 1.6e-5.  The trajectory is
    held to TRAJ_TOL, 3x above that."""
    det, state = _detector(64, seed=23)
    det = det.cuda().eval()
    epochs = 10
    ex = explain.PGExplainer(det, epochs=epochs)
    oracles = _Oracles(det, state, ex, epochs)
    batches = _batches(det, 3, 4, 31)
    debug = {}
    monkeypatch.setattr(ops, "DEBUG_CAPTURE", debug)
    for ep in range(epochs):
        for r, t, target in batches:
            r, t = r.cuda(), t.cuda()
            ex.train(ep, r, t, target.cuda())
            with torch.no_grad():
                h_s = det.sensor_encoder(r, t)
            oracles.train(ep, r, t, target, debug["pg_uniform"], h_s, debug["pg_gate"])
    names = ("W1", "b1", "w2", "b2")
    params = (dict(zip(names, ex.mlp.parameters())), dict(zip(names, oracles.runs[0][1].mlp.parameters())),
              dict(zip(names, oracles.runs[1][1].mlp.parameters())))
    r, t, _ = (x.cuda() for x in _batches(det, 1, 6, 32)[0])
    with torch.no_grad():
        h_s = det.sensor_encoder(r, t)
    m32, m64 = oracles.explain(r, t, h_s)
    got = ex.explain(r, t)
    assert got.shape == (6, det.edge_index_single.shape[1])
    _check("PGExplainer 30 steps: MLP parameters", *params, tol=TRAJ_TOL)
    _check("PGExplainer 30 steps: explain", {"mask": got}, {"mask": m32}, {"mask": m64}, tol=TRAJ_TOL)


def _run(det, k, graphed, bias, seed, batch):
    torch.manual_seed(seed)
    ex = explain.PGExplainer(det, epochs=k, graphed=graphed, bias=bias)
    r, t, target = (x.cuda() for x in batch)
    losses = [ex.train(ep, r, t, target) for ep in range(k)]
    return ex, torch.stack(losses), [p.detach().clone() for p in ex.mlp.parameters()]


def test_graphed_steps_equal_eager_and_repeat():
    det, _ = _detector(64)
    det = det.cuda()
    batch = _batches(det, 1, 5, 40)[0]
    k = 6
    ex_e, loss_e, par_e = _run(det, k, False, 0.5, 1, batch)
    ex_g, loss_g, par_g = _run(det, k, True, 0.5, 1, batch)
    assert ex_g._step is not None and ex_e._step is None
    assert torch.equal(loss_e, loss_g)
    for a, c in zip(par_e, par_g):
        assert torch.equal(a, c)
    r, t = batch[0].cuda(), batch[1].cuda()
    assert torch.equal(ex_e.explain(r, t), ex_g.explain(r, t))
    # default bias: reproducible under torch.manual_seed, and each replay draws new noise
    _, loss_a, par_a = _run(det, k, True, 0.01, 2, batch)
    _, loss_b, par_b = _run(det, k, True, 0.01, 2, batch)
    assert torch.equal(loss_a, loss_b) and all(torch.equal(a, c) for a, c in zip(par_a, par_b))
    _, loss_c, _ = _run(det, k, True, 0.01, 3, batch)
    assert not torch.equal(loss_a, loss_c)
    debug = {}
    old, ops.DEBUG_CAPTURE = ops.DEBUG_CAPTURE, debug
    try:
        torch.manual_seed(4)
        ex = explain.PGExplainer(det, epochs=3, graphed=True)
        draws = []
        for ep in range(3):
            ex.train(ep, r, t, batch[2].cuda())
            draws.append(debug["pg_uniform"].clone())   # the captured step's buffer, rewritten by every replay
    finally:
        ops.DEBUG_CAPTURE = old
    assert not torch.equal(draws[1], draws[2])
    # a second batch size runs eagerly next to the graph
    ex.train(2, r[:3], t[:3], batch[2][:3].cuda())


def test_frozen_detector_launches_no_weight_gradient_and_explain_no_backward():
    det, state = _detector(64)
    det = det.cuda().train()
    ex = explain.PGExplainer(det, epochs=1)
    r, t, target = (x.cuda() for x in _batches(det, 1, 4, 50)[0])
    ex.train(0, r, t, target)  # builds the index tensors
    torch.cuda.synchronize()
    instrument.reset(timing=True)
    ex.train(0, r, t, target)
    torch.cuda.synchronize()
    launched = instrument.summary()
    instrument.reset()
    assert {"pg_edge_fwd", "pg_edge_bwd", "edge_mask_bwd", "gcn_adj_grad"} <= set(launched), launched
    assert launched["wgrad_tc"]["count"] == 1, launched        # the explainer's own d W1
    assert not set(launched) & set(DETECTOR_WEIGHT_KERNELS), launched
    torch.cuda.synchronize()
    instrument.reset(timing=True)
    mask = ex.explain(r, t)
    torch.cuda.synchronize()
    launched = instrument.summary()
    instrument.reset()
    assert "pg_edge_fwd" in launched and mask.shape == (4, det.edge_index_single.shape[1])
    assert not [k for k in launched if "bwd" in k or "grad" in k], launched
    assert det.training and all(p.requires_grad for p in det.parameters())
    for k, v in det.state_dict().items():
        assert torch.equal(v.cpu(), state[k]), k


def test_pyg_state_dict_round_trips():
    det, _ = _detector(128)
    det = det.cuda()
    torch.manual_seed(6)
    ex = explain.PGExplainer(det, epochs=2)
    r, t, target = (x.cuda() for x in _batches(det, 1, 3, 60)[0])
    for ep in range(2):
        ex.train(ep, r, t, target)
    sd = ex.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {"mlp.0.weight": (64, 256), "mlp.0.bias": (64,),
                                                          "mlp.2.weight": (1, 64), "mlp.2.bias": (1,)}
    other = explain.PGExplainer(det, epochs=50)
    other.load_state_dict({k: v.cpu() for k, v in sd.items()})
    assert torch.equal(other.explain(r, t), ex.explain(r, t))
