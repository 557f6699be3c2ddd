"""The fused pipe head at node width 64 (csrc/heads.cu, csrc/tgrad.cu) at every plan its three kernels take, on the
class-pipe sets of tests/head_plans.py, against fp64 elementwise: logits, pooled output, dx, dW1, db1, dw2 and db2 in
eval and train mode, the captured gate against the fp64 pre-activation, NaN-poisoned workspaces and outputs with the
index tables read back, window independence, bitwise repeatability, and the composed D = 128 head and a whole
detector on the same kind of incidence.  Margins go to conftest.parity_log."""
import functools

import numpy as np
import pytest
import torch

import head_plans as H
from conftest import parity_log, rel_err
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops

pytestmark = pytest.mark.gpu
CASES = H.cases()
SETS = H.pipe_sets()
P_DROP = 0.1


@functools.lru_cache(maxsize=None)
def _set(name):
    s = SETS[name]
    ends = H.pipe_ends(s)
    ends32 = ends.to(torch.int32).cuda()
    return s, ends, ends32, ops.pipe_incidence(ends32, s.n)


def _cuda(inp):
    return H.Inputs(*(t.cuda() for t in inp))


def _run(inp, ends32, inc, train, frozen=False, seed=11):
    """ops.heads forward + backward; -> outputs, gradients and the captured gate words."""
    leaves = [inp.x.clone().requires_grad_(True)] + [t.clone().requires_grad_(not frozen)
                                                     for t in (inp.w1, inp.b1, inp.w2, inp.b2)]
    ops.DEBUG_CAPTURE = cap = {}
    try:
        torch.manual_seed(seed)
        part, pooled = ops.heads(leaves[0], ends32, *leaves[1:4], P_DROP, train, inc)
    finally:
        ops.DEBUG_CAPTURE = None
    logits = part.sum(0) + leaves[4]
    ((logits * inp.dlogit).sum() + (pooled * inp.dpool).sum()).backward()
    out = {"logits": logits.detach(), "pooled": pooled.detach(), "dx": leaves[0].grad}
    if not frozen:
        out.update(dW1=leaves[1].grad, db1=leaves[2].grad, dw2=leaves[3].grad, db2=leaves[4].grad)
    return out, cap["head_mask_words"].clone()


def _compare(tag, got, want, scale):
    rep = {k: {"bound": H.bound_ratio(got[k], want[k], scale[k], k), "rel": rel_err(got[k], want[k].reshape(got[k].shape))}
           for k in got}
    parity_log(tag, rep)
    for k, v in rep.items():
        assert v["bound"] <= 1.0 and v["rel"] <= 1e-5, (k, rep)
    return rep


@pytest.mark.parametrize("train", [False, True], ids=["eval", "train"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_head_vs_fp64(case, train):
    s, ends, ends32, inc = _set(case.set)
    inp = _cuda(H.inputs(s, case.B))
    got, words = _run(inp, ends32, inc, train)
    live = H.unpack_gate(words).view(case.B, s.p, H.H)
    keep = H.keep_scale(P_DROP) if train else 1.0
    want, scale, (pre, s_pre) = H.reference(inp, ends, live, keep)
    _compare(f"head_plans {case.name} {'train' if train else 'eval'}", got, want, scale)

    # the gate: the kernel's ReLU decision may differ from fp64's only within the forward bound of zero
    near = pre.abs() <= H.TAU["logits"] * s_pre
    pos = pre > 0
    clear = pos & ~near
    dropped = (clear & ~live).sum().item() / max(clear.sum().item(), 1)
    if not train:
        assert bool((live == pos)[~near].all())
    else:
        assert not bool((live & ~pos & ~near).any())
        if clear.sum().item() >= 2000:
            assert 0.06 < dropped < 0.14, dropped
    parity_log(f"head_plans gate {case.name} {'train' if train else 'eval'}",
               {"near_zero": int(near.sum().item()), "near_zero_disagree": int(((live != pos) & near).sum().item()),
                "dropped": dropped})


def _direct(inp, s, ends32, inc, poison=float("nan"), dpooled=True):
    """The three kernels called through the C ABI with every output and workspace filled with ``poison`` first (the
    gate words' padding rows with all-ones: a live unit past M would show)."""
    L = _lib.load()
    x = inp.x
    b, dev, st = x.shape[0], ops._dev_index(x), ops._stream(x)
    m = b * s.p
    mp = (m + 127) // 128 * 128
    w2v = inp.w2.reshape(-1).contiguous()
    part = torch.full((m,), poison, device="cuda")
    hmask = torch.full((mp, 4), -1, dtype=torch.int32, device="cuda")
    hsign = torch.full((mp, 4), -1, dtype=torch.int32, device="cuda")
    _lib.check(L.ltgnn_pipe_head_fwd(dev, b, s.n, s.p, H.D, H.H, x.data_ptr(), ends32.data_ptr(), inp.w1.data_ptr(),
                                     inp.b1.data_ptr(), w2v.data_ptr(), 0.0, 0, part.data_ptr(), None, hmask.data_ptr(),
                                     hsign.data_ptr(), st))
    ws = torch.full((int(L.ltgnn_pipe_head_dx_ws_floats(dev, s.n, s.p)),), poison, device="cuda")
    dx = torch.full_like(x, poison)
    dl = inp.dlogit.reshape(-1).contiguous()
    _lib.check(L.ltgnn_pipe_head_bwd_dx(dev, b, s.n, s.p, H.D, H.H, inc[0].data_ptr(), inc[1].data_ptr(),
                                        inp.w1.data_ptr(), w2v.data_ptr(), hmask.data_ptr(), hsign.data_ptr(),
                                        dl.data_ptr(), 1.0, inp.dpool.data_ptr() if dpooled else None, ws.data_ptr(),
                                        dx.data_ptr(), st))
    wsw = torch.full((int(L.ltgnn_pipe_head_ws_floats(dev)),), poison, device="cuda")
    dw1, db1, dw2 = (torch.full(t, poison, device="cuda") for t in ((H.H, 3 * H.D), (H.H,), (1, H.H)))
    _lib.check(L.ltgnn_pipe_head_bwd_w(dev, b, s.n, s.p, H.D, H.H, x.data_ptr(), ends32.data_ptr(), inp.w1.data_ptr(),
                                       inp.b1.data_ptr(), w2v.data_ptr(), hmask.data_ptr(), dl.data_ptr(), 1.0,
                                       dw1.data_ptr(), db1.data_ptr(), dw2.data_ptr(), wsw.data_ptr(), st))
    torch.cuda.synchronize()
    return {"logits": part.view(b, s.p) + inp.b2, "dx": dx, "dW1": dw1, "db1": db1, "dw2": dw2}, ws


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_poisoned_workspace_and_tables(case):
    """NaN in every output and workspace: every logit and every dx row (nodes with no pipe end included) is written and
    no unwritten scratch row is read; the results equal the autograd path's bit for bit; end_pos and the chunk table
    in the workspace equal the restatement, so the case reaches the branch it was built for."""
    s, ends, ends32, inc = _set(case.set)
    inp = _cuda(H.inputs(s, case.B))
    got, ws = _direct(inp, s, ends32, inc)
    for k, v in got.items():
        assert not bool(v.isnan().any()), k
    want, _ = _run(inp, ends32, inc, False)
    for k, v in got.items():
        assert torch.equal(v, want[k].reshape(v.shape)), k
    ptr, inc_h = H.incidence(ends, s.n)
    words = ws.view(torch.int32).cpu().numpy()
    assert np.array_equal(words[:2 * s.p], H.end_positions(inc_h))
    plan = H.dx_plan(case.B, ptr)
    c = plan.n_chunks
    assert np.array_equal(words[2 * s.p:2 * s.p + c + 2], np.array([c, *plan.first], dtype=np.int32))
    # dpooled = nullptr (the pooled output unused) equals dpooled = 0, bit for bit
    zero = inp._replace(dpool=torch.zeros_like(inp.dpool))
    a, _ = _direct(zero, s, ends32, inc)
    b, _ = _direct(zero, s, ends32, inc, dpooled=False)
    assert torch.equal(a["dx"], b["dx"]) and not bool(b["dx"].isnan().any())


@pytest.mark.parametrize("name", list(SETS))
def test_windows_are_independent(name):
    """B = 3 (SMs / 2) + 5 windows (a bwd_dx CTA runs three or four, the scratch parities alternate): sampled windows'
    logits and dx equal the same window run alone, bit for bit."""
    s, ends, ends32, inc = _set(name)
    half = torch.cuda.get_device_properties(0).multi_processor_count // 2
    bsz = 3 * half + 5
    inp = _cuda(H.inputs(s, bsz, seed=3))
    got, _ = _run(inp, ends32, inc, False)
    for i in (0, 1, 2, 3, half - 1, half, 2 * half + 1, 3 * half, bsz - 2, bsz - 1):
        one = H.Inputs(inp.x[i:i + 1].contiguous(), *inp[1:5], inp.dlogit[i:i + 1].contiguous(),
                       inp.dpool[i:i + 1].contiguous())
        alone, _ = _run(one, ends32, inc, False)
        assert torch.equal(got["logits"][i:i + 1], alone["logits"]), i
        assert torch.equal(got["dx"][i:i + 1], alone["dx"]), i


@pytest.mark.parametrize("case", CASES[::3], ids=lambda c: c.name)
def test_bitwise_repeatable_and_frozen(case):
    """Repeated runs give the same bits (train mode, same seed); a frozen head's dx equals a trainable head's."""
    s, ends, ends32, inc = _set(case.set)
    inp = _cuda(H.inputs(s, case.B, seed=5))
    a, wa = _run(inp, ends32, inc, True)
    b, wb = _run(inp, ends32, inc, True)
    assert torch.equal(wa, wb)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    frozen, _ = _run(inp, ends32, inc, True, frozen=True)
    assert torch.equal(frozen["dx"], a["dx"]) and torch.equal(frozen["logits"], a["logits"])


# ------------------------------------------------------------------------------------------------ D = 128
def _wide_cases():
    seen, out = set(), []
    for c in CASES:
        if c.set not in seen:
            seen.add(c.set)
            out.append(c)
    return out


@pytest.mark.parametrize("case", _wide_cases(), ids=lambda c: c.name)
def test_wide_head_vs_fp64(case):
    """The composed D = 128 head (_HeadsWide) on the same incidence, eval mode: its feature gradient is a separate
    gather over the same pipe_incidence."""
    s, ends, ends32, inc = _set(case.set)
    inp = _cuda(H.inputs(s, case.B, d=128))
    leaves = [t.clone().requires_grad_(True) for t in inp[:5]]
    ops.DEBUG_CAPTURE = cap = {}
    try:
        part, pooled = ops.heads(leaves[0], ends32, *leaves[1:4], P_DROP, False, inc)
    finally:
        ops.DEBUG_CAPTURE = None
    logits = part.sum(0) + leaves[4]
    ((logits * inp.dlogit).sum() + (pooled * inp.dpool).sum()).backward()
    got = {"logits": logits.detach(), "pooled": pooled.detach(), "dx": leaves[0].grad, "dW1": leaves[1].grad,
           "db1": leaves[2].grad, "dw2": leaves[3].grad, "db2": leaves[4].grad}
    live = cap["head_live"].view(case.B, s.p, H.H)
    want, _, _ = H.reference(inp, ends, live, 1.0)
    rep = {k: rel_err(got[k], want[k].reshape(got[k].shape)) for k in got}
    parity_log(f"head_plans wide {case.name}", rep)
    assert all(v <= 1e-5 for v in rep.values()), rep


# ------------------------------------------------------------------------------------------------ whole detector
def _hub_network(tmp_path, n=2500, hub_deg=60, seed=12):
    """A pipe network of ``n`` junctions: a chain, random chords, and a hub joined to ``hub_deg`` junctions.  The class
    pipes are the hub's pipes and every seventh other pipe, so the hub has ``hub_deg`` class-pipe ends."""
    from bench import write_inp
    rng = np.random.default_rng(seed)
    names = [f"J{i}" for i in range(n)]
    links = [(i, i + 1) for i in range(n - 1)]
    links += [tuple(sorted(int(v) for v in rng.choice(n, 2, replace=False))) for _ in range(n // 10)]
    hub = n // 2
    others = [int(v) for v in rng.choice([v for v in range(n) if abs(v - hub) > 1], hub_deg, replace=False)]
    hub_links = [(hub, v) for v in others]
    links += hub_links
    pipe_ids = [f"P{k}" for k in range(len(links))]
    inp = tmp_path / "hub.inp"
    write_inp(inp, names, links, pipe_ids)
    classes = [pipe_ids[k] for k in range(len(links)) if links[k] in hub_links or k % 7 == 0]
    sensors = [names[int(v)] for v in rng.choice(n, 29, replace=False)]
    return inp, sensors, classes


def test_detector_with_a_hub_vs_fp64(tmp_path):
    """LeakDetector(node_hidden=64) on a 2 500-junction network (chunk tables past shared memory) with a class-pipe hub
    of 60 ends (the unstaged gather), eval mode: logits, loss and all 18 gradients against OracleLeakDetector in fp64,
    within 1e-5 norm-relative -- or 3 x the fp32 oracle's own error where the fp32 arithmetic cannot do better: the
    pipe-logit bias gradient is the sum of the pipe classes' cross-entropy gradients, terms of size ~1 that cancel to
    -p(no leak) ~ -2e-3, and the fp32 oracle misses it by ~5e-5."""
    from leak_det_gnn_b200.models import LeakDetector
    from oracle.detector_oracle import OracleLeakDetector
    inp_path, sensors, classes = _hub_network(tmp_path)
    torch.manual_seed(42)
    ours = LeakDetector(inp_path, sensors, classes, sensor_hidden=64, node_hidden=64, gnn_layers=2, dropout=0.1,
                        use_time=True).cuda().eval()
    n, p = len(ours.node_names), len(ours.pipe_ids)
    cnt = np.bincount(ours.pipe_ends.reshape(-1).numpy(), minlength=n)
    ptr = np.concatenate([[0], np.cumsum(cnt)])
    plan = H.dx_plan(4, ptr)
    assert cnt.max() > H.CAP_ROWS and not plan.tbl_fits, (cnt.max(), plan.n_chunks)
    state = {k: v.detach().clone() for k, v in ours.state_dict().items()}
    gen = torch.Generator().manual_seed(8)
    b, l = 4, 12
    residual, tfeat = torch.randn(b, l, len(sensors), generator=gen), torch.randn(b, l, 9, generator=gen)
    label = torch.randint(0, p + 1, (b,), generator=gen)

    logits = ours(residual.cuda(), tfeat.cuda())
    loss = torch.nn.functional.cross_entropy(logits, label.cuda())
    loss.backward()
    ref = {}
    for dt in (torch.float64, torch.float32):
        orc = OracleLeakDetector(n, ours.edge_index_single, ours.pipe_ends, ours.sensor_node_idx.tolist(), 64, 64, 2,
                                 0.1, True).to(dt)
        orc.load_state_dict({k: v.to(dt) for k, v in state.items()}, strict=True)
        orc.eval()
        lo = orc(residual.to(dt), tfeat.to(dt))
        lf = torch.nn.functional.cross_entropy(lo, label)
        lf.backward()
        ref[dt] = {"logits": lo.detach(), "loss": lf.detach().reshape(1),
                   **{k: v.grad for k, v in orc.named_parameters()}}
    grads = dict(ours.named_parameters())
    assert len(grads) == 18 and set(grads) | {"logits", "loss"} == set(ref[torch.float64])
    got = {"logits": logits, "loss": loss.reshape(1), **{k: v.grad for k, v in grads.items()}}
    rep = {k: {"ours": rel_err(got[k], ref[torch.float64][k]),
               "oracle_fp32": rel_err(ref[torch.float32][k], ref[torch.float64][k])} for k in got}
    parity_log(f"head_plans detector hub n={n} P={p} hub={int(cnt.max())}", rep)
    for k, e in rep.items():
        assert e["ours"] <= max(1e-5, 3.0 * e["oracle_fp32"]), (k, e)
