"""Training of the GRU normal-state predictor on sm_100a (csrc/gru_pred.cu): the saved-gates forward against the inference
kernel and fp64, one layer's backward through time against fp64 nn.GRU autograd, NormalPredictorGRU.forward_cone against
the dense fp64 model (eval, and train mode through an fp64 replay of the dropout's live bits), the weight-gradient
reductions at batch 4096, the graphed PredictorStep, two NCCL ranks, and the C argument checks.  Gradient tolerance
5e-5 (the sensor GRU BPTT's), 3xTF32 products."""
import copy
import ctypes
import os
import socket
import subprocess
import sys

import pytest
import torch

from conftest import REPO, parity_log, rel_err
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.models import NormalPredictorGRU

pytestmark = pytest.mark.gpu
TOL = 5e-5
N_IN = 38          # 29 sensors + 9 time features
NAMES = ["weight_ih", "weight_hh", "bias_ih", "bias_hh"]


def _layer(scale, seed):
    torch.manual_seed(seed)
    gru = torch.nn.GRU(N_IN, 128, num_layers=1, batch_first=True)
    with torch.no_grad():
        for p in gru.parameters():
            p.mul_(scale)
    return gru.cuda()


def _inp(x):
    """(q, l, 38) -> (q * l, 64): zero-padded, ones column at 38 (what ops.gru_predictor_cone builds)."""
    q, l, _ = x.shape
    inp = torch.zeros(q, l, 64, device="cuda")
    inp[:, :, :N_IN] = x
    inp[:, :, N_IN] = 1.0
    return inp.view(q * l, 64)


def _native_layer(gru, x, dh_last=None, dh_seq=None):
    """One layer, forward with saved gates + BPTT + weight gradients, as _GruPredictor runs it."""
    q, l, _ = x.shape
    inp = _inp(x)
    w_x, b_x, w_hh, b_hn = ops.gru_predictor_weights([(gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0,
                                                        gru.bias_hh_l0)])[0]
    gx = torch.empty(3, q * l, 128, device="cuda")
    for g in range(3):
        ops.linear_tc(inp, w_x[g], b_x[g], out=gx[g])
    h_last, hseq, gates = ops.gru_layer_fwd_train(gx, q, l, w_hh, b_hn)
    dg = ops.gru_layer_bwd(q, l, w_hh, gates, hseq, dh_last=dh_last, dh_seq=dh_seq)
    return (h_last, hseq, gates, dg), ops.gru_layer_param_grads(dg, hseq, inp, N_IN, q, l)


def _autograd(gru, x, dh_last, dh_seq):
    gru.zero_grad()
    out, _ = gru(x)
    loss = (out * dh_seq).sum() if dh_seq is not None else (out[:, -1] * dh_last).sum()
    loss.backward()
    return [getattr(gru, f"{n}_l0").grad.clone() for n in NAMES]


def test_training_forward_equals_inference_and_fp64_gates():
    """h_last and hseq are the inference kernel's bit for bit; r, z, n, hn match fp64 recomputed from the saved states."""
    for q, l in ((129, 36), (1, 1), (9216, 36)):
        gru = _layer(1.0, q + l)
        x = torch.randn(q, l, N_IN, generator=torch.Generator().manual_seed(q)).cuda()
        layer = ops.gru_predictor_weights([(gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0)])[0]
        inp = _inp(x)
        h_ref, s_ref = ops.gru_layer_fwd(inp, q, l, layer, seq=True)
        (h_last, hseq, gates, _), _ = _native_layer(gru, x, dh_last=torch.zeros(q, 128, device="cuda"))
        assert torch.equal(h_last, h_ref) and torch.equal(hseq, s_ref)
        hp = torch.zeros(q, l, 128, device="cuda", dtype=torch.float64)
        hp[:, 1:] = hseq.view(q, l, 128)[:, :-1].double()
        w_ih, w_hh = gru.weight_ih_l0.double(), gru.weight_hh_l0.double()
        b_ih, b_hh = gru.bias_ih_l0.double(), gru.bias_hh_l0.double()
        gi = (x.double() @ w_ih.t() + b_ih).view(q, l, 3, 128)
        gh = (hp @ w_hh.t() + b_hh).view(q, l, 3, 128)
        r = torch.sigmoid(gi[..., 0, :] + gh[..., 0, :])
        z = torch.sigmoid(gi[..., 1, :] + gh[..., 1, :])
        n = torch.tanh(gi[..., 2, :] + r * gh[..., 2, :])
        errs = {nm: rel_err(gates[k].view(q, l, 128), ref) for k, (nm, ref) in enumerate(
            (("r", r), ("z", z), ("n", n), ("hn", gh[..., 2, :])))}
        parity_log(f"gru_pred train forward gates Q={q} L={l}", {**errs, "tol": 1e-5})
        assert all(v <= 1e-5 for v in errs.values()), errs


@pytest.mark.parametrize("mode", ["last", "seq"])
@pytest.mark.parametrize("scale", [1.0, 3.0])
@pytest.mark.parametrize("l", [1, 36, 288])
@pytest.mark.parametrize("q", [1, 127, 128, 129, 9216])
def test_layer_bptt_matches_fp64(q, l, scale, mode):
    """Every parameter gradient of one layer against fp64 nn.GRU autograd, from dh_last only or from a random dh_seq;
    repeated runs are bitwise equal."""
    gru = _layer(scale, 3 * q + l)
    g = torch.Generator().manual_seed(5 * q + l)
    x = torch.randn(q, l, N_IN, generator=g).cuda()
    dh_last = torch.randn(q, 128, generator=g).cuda() if mode == "last" else None
    dh_seq = torch.randn(q * l, 128, generator=g).cuda() if mode == "seq" else None
    (_, _, _, dg), grads = _native_layer(gru, x, dh_last, dh_seq)
    dseq3 = None if dh_seq is None else dh_seq.view(q, l, 128)
    g64 = copy.deepcopy(gru).double()
    ref = _autograd(g64, x.double(), None if dh_last is None else dh_last.double(),
                    None if dseq3 is None else dseq3.double())
    ref32 = _autograd(gru, x, dh_last, dseq3)
    errs = {nm: rel_err(a, b) for nm, a, b in zip(NAMES, grads, ref)}
    rep = {**errs, **{f"torch_fp32_{nm}": rel_err(a, b) for nm, a, b in zip(NAMES, ref32, ref)}, "tol": TOL}
    parity_log(f"gru_pred layer bptt Q={q} L={l} scale={scale} {mode}", rep)
    assert all(v <= TOL for v in errs.values()), errs
    (_, _, _, dg2), grads2 = _native_layer(gru, x, dh_last, dh_seq)
    assert torch.equal(dg2, dg) and all(torch.equal(a, b) for a, b in zip(grads2, grads))


def _predictor(layers, seed, p=0.1):
    torch.manual_seed(seed)
    return NormalPredictorGRU(29, 9, num_layers=layers, dropout=p)


def _batch(b, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(b, 36, 29, generator=g), torch.randn(b, 36, 9, generator=g), torch.randn(b, 29, generator=g)


def _dense(m, dtype):
    """A copy of ``m`` whose cuDNN forward can be differentiated: train mode (cuDNN has no eval-mode RNN backward) with
    the inter-layer dropout off, i.e. the eval-mode function."""
    d = copy.deepcopy(m).to(dtype).train()
    d.gru.dropout = 0.0
    d.zero_grad()
    return d


def _grads_vs_fp64(m, x, xt, y, ref_pred_fn):
    loss = torch.nn.functional.mse_loss(m.forward_cone(x, xt), y)
    loss.backward()
    m64 = _dense(m, torch.float64)
    loss64 = torch.nn.functional.mse_loss(ref_pred_fn(m64, x.double(), xt.double()), y.double())
    loss64.backward()
    errs = {n: rel_err(p.grad, q.grad) for (n, p), (_, q) in zip(m.named_parameters(), m64.named_parameters())}
    errs["loss"] = rel_err(loss, loss64)
    return errs


@pytest.mark.parametrize("layers", [1, 2, 3])
def test_forward_cone_matches_dense_fp64(layers):
    m = _predictor(layers, layers).cuda().eval()
    x, xt, y = (t.cuda() for t in _batch(256, layers))
    with torch.no_grad():
        assert torch.equal(m.forward_cone(x, xt), m.forward_last(x, xt))    # same kernels, same bits
    errs = _grads_vs_fp64(m, x, xt, y, lambda mm, a, b: mm(a, b))
    parity_log(f"gru_predictor forward_cone + backward vs dense fp64 B=256 layers={layers}", {**errs, "tol": TOL})
    assert len(errs) == 4 * layers + 3 and all(p.grad is not None for p in m.parameters())
    assert all(v <= TOL for v in errs.values()), {k: v for k, v in errs.items() if v > TOL}


def _gru64(h, w_ih, w_hh, b_ih, b_hh):
    """One torch.nn.GRU layer written out step by step (autograd reaches the parameters): (B, L, K) -> (B, L, H)."""
    gi = (h @ w_ih.t() + b_ih).chunk(3, -1)
    s = h.new_zeros(h.shape[0], w_hh.shape[1])
    out = []
    for t in range(h.shape[1]):
        gh = (s @ w_hh.t() + b_hh).chunk(3, -1)
        r = torch.sigmoid(gi[0][:, t] + gh[0])
        z = torch.sigmoid(gi[1][:, t] + gh[1])
        n = torch.tanh(gi[2][:, t] + r * gh[2])
        s = (1 - z) * n + z * s
        out.append(s)
    return torch.stack(out, 1)


def _replay64(m, x, xt, lives, p):
    """fp64 stacked GRU with the kernels' kept units (times 1 / (1 - p)) between the layers."""
    g = m.gru
    h = torch.cat([x, xt], -1)
    b, l, _ = h.shape
    for i in range(g.num_layers):
        h = _gru64(h, *(getattr(g, f"{n}_l{i}") for n in NAMES))
        if i + 1 < g.num_layers:
            h = h * ops.unpack_gru_live(lives[i]).view(b, l, -1).double() / (1.0 - p)
    return m.head(h[:, -1])


def test_forward_cone_dropout_replays_fp64_and_draws_fresh_masks():
    m = _predictor(2, 3).cuda().train()
    x, xt, y = (t.cuda() for t in _batch(256, 4))
    ops.DEBUG_CAPTURE = {}
    try:
        torch.manual_seed(11)
        pred = m.forward_cone(x, xt)
        loss = torch.nn.functional.mse_loss(pred, y)
        loss.backward()
        lives = [lv.clone() for lv in ops.DEBUG_CAPTURE["gru_lives"]]
    finally:
        ops.DEBUG_CAPTURE = None
    m64 = _dense(m, torch.float64)
    pred64 = _replay64(m64, x.double(), xt.double(), lives, 0.1)
    loss64 = torch.nn.functional.mse_loss(pred64, y.double())
    loss64.backward()
    errs = {n: rel_err(p.grad, q.grad) for (n, p), (_, q) in zip(m.named_parameters(), m64.named_parameters())}
    errs["pred"], errs["loss"] = rel_err(pred, pred64), rel_err(loss, loss64)
    assert len(lives) == 1
    kept = ops.unpack_gru_live(lives[0]).double().mean().item()
    parity_log("gru_predictor forward_cone dropout 0.1 vs fp64 replay of the live bits", {**errs, "kept": kept, "tol": TOL})
    assert all(v <= TOL for v in errs.values()), {k: v for k, v in errs.items() if v > TOL}
    assert abs(kept - 0.9) < 0.01
    with torch.no_grad():
        torch.manual_seed(11)
        assert torch.equal(m.forward_cone(x, xt), pred)           # same seed: same masks
        torch.manual_seed(12)
        assert not torch.equal(m.forward_cone(x, xt), pred)       # new seed: new masks


def test_dropout_kernel_p0_is_a_copy_and_backward_sums_in_order():
    g = torch.Generator().manual_seed(2)
    x = torch.randn(1000, 128, generator=g).cuda()
    y, live = ops.gru_dropout(x, 0.0, 123)
    assert torch.equal(y, x) and bool((live == -1).all())
    y, live = ops.gru_dropout(x, 0.25, 123)
    keep = ops.unpack_gru_live(live)
    assert torch.equal(y, torch.where(keep, x * (1.0 / 0.75), torch.zeros_like(x)))
    parts = torch.randn(3, 1000, 128, generator=g).cuda()
    dx = ops.gru_dropout_bwd(parts, live, 0.25)
    assert torch.equal(dx, torch.where(keep, (parts[0] + parts[1] + parts[2]) * (1.0 / 0.75), torch.zeros_like(x)))
    assert torch.equal(ops.gru_dropout_bwd(parts, None, 0.0), parts[0] + parts[1] + parts[2])


def test_weight_gradient_reductions_at_batch_4096():
    """B = 4096, L = 36: every weight gradient sums 147 456 rows.  The whole model against fp64 (torch fp32 beside it),
    then the three weight-gradient shapes of the step (128 x 160 for W_hh and layer >= 1's W_ih, 128 x 64 for layer 0's,
    64 x 160 for the head) at that row count with test_bench_sizes_gpu's operands and rules: ReLU-like and same-sign
    operands, the mean signed deviation of a same-sign sum held to the tensor-core accumulator's bias bound."""
    from test_bench_sizes_gpu import _assert_report, _wgrad_entry

    m = _predictor(2, 21, p=0.0).cuda().eval()
    x, xt, y = (t.cuda() for t in _batch(4096, 22))
    errs = _grads_vs_fp64(m, x, xt, y, lambda mm, a, b: mm(a, b))
    m32, m64 = _dense(m, torch.float32), _dense(m, torch.float64)
    torch.nn.functional.mse_loss(m32(x, xt), y).backward()
    torch.nn.functional.mse_loss(m64(x.double(), xt.double()), y.double()).backward()
    fp32 = {n: rel_err(p.grad, q.grad) for (n, p), (_, q) in zip(m32.named_parameters(), m64.named_parameters())}
    parity_log("gru_predictor forward_cone grads B=4096 vs fp64",
               {**errs, **{f"torch_fp32_{k}": v for k, v in fp32.items()}, "tol": TOL})
    assert all(v <= TOL for v in errs.values()), {k: v for k, v in errs.items() if v > TOL}
    rows = 4096 * 36
    for do, di in ((128, 160), (128, 64), (64, 160)):
        for kind in ("relu", "same"):
            _assert_report(f"gru_predictor wgrad {kind} M={rows} {do}x{di}", {"dW": _wgrad_entry(kind, rows, do, di)})


def _step(m, graph, batch=32, clip=1.0, opt=True):
    from leak_det_gnn_b200.parallel import FlatGradBucket
    from leak_det_gnn_b200.train_predictor_dp import PredictorStep

    o = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True) if opt else None
    return PredictorStep(m, o, FlatGradBucket(m.parameters()), batch, clip, graph)


def test_graphed_step_equals_eager():
    """Dropout off: the replayed training step (forward_cone, MSE, backward, clip, AdamW) equals the eager one bit for bit."""
    def run(graph):
        m = _predictor(2, 5, p=0.0).cuda()
        step = _step(m, graph)
        return m, [step(*(t.cuda() for t in _batch(32, 100 + i))).clone() for i in range(3)]

    me, le = run(False)
    mg, lg = run(True)
    assert all(torch.equal(a, b) for a, b in zip(le, lg))
    assert all(torch.equal(a, b) for a, b in zip(me.parameters(), mg.parameters()))


def test_graphed_step_draws_fresh_dropout_masks():
    """Dropout 0.1 and no optimiser: replays on the same batch draw new live bits and give different losses, and the same
    torch seed reproduces the sequence."""
    batch = [t.cuda() for t in _batch(32, 100)]

    def replays(n=4):
        m = _predictor(2, 5, p=0.1).cuda()
        keep = [p.detach().clone() for p in m.parameters()]
        torch.manual_seed(6)
        ops.DEBUG_CAPTURE = {}
        try:
            step = _step(m, True, clip=0.0, opt=False)
            lives = ops.DEBUG_CAPTURE["gru_lives"]          # the graph's own live-bit tensors, rewritten by every replay
        finally:
            ops.DEBUG_CAPTURE = None
        losses, bits = [], []
        for _ in range(n):
            losses.append(step(*batch).item())
            bits.append(torch.cat([lv.flatten() for lv in lives]).clone())
        assert all(torch.equal(a, b) for a, b in zip(keep, m.parameters()))
        return losses, bits

    la, ba = replays()
    lb, bb = replays()
    assert len(set(la)) == len(la), la
    assert all(not torch.equal(ba[i], ba[i + 1]) for i in range(len(ba) - 1))
    assert la == lb and all(torch.equal(a, b) for a, b in zip(ba, bb))


def test_fifty_adamw_steps_track_dense_fp64():
    """Dropout off, batch 256: 50 graphed native steps and 50 dense fp64 steps from the same weights on the same batches."""
    m = _predictor(2, 31, p=0.0).cuda()
    m64 = copy.deepcopy(m).double()
    step = _step(m, True, batch=256)
    opt64 = torch.optim.AdamW(m64.parameters(), lr=1e-3, weight_decay=1e-4)
    worst = 0.0
    for i in range(50):
        x, xt, y = (t.cuda() for t in _batch(256, 500 + i))
        loss = step(x, xt, y).item()
        opt64.zero_grad()
        loss64 = torch.nn.functional.mse_loss(m64(x.double(), xt.double()), y.double())
        loss64.backward()
        torch.nn.utils.clip_grad_norm_(m64.parameters(), 1.0)
        opt64.step()
        worst = max(worst, abs(loss - loss64.item()) / loss64.item())
    drift = max(rel_err(p, q) for p, q in zip(m.parameters(), m64.parameters()))
    parity_log("gru_predictor 50 AdamW steps native graphed vs dense fp64", {"loss": worst, "params": drift})
    # Adam normalises every step, so a parameter whose gradient is near zero may step either way in fp32 and fp64: the
    # parameters are held loosely, the losses closely
    assert worst <= 1e-3 and drift <= 1e-2, (worst, drift)


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {repo!r})
from leak_det_gnn_b200.models import NormalPredictorGRU
from leak_det_gnn_b200.parallel import FlatGradBucket
rank = int(os.environ["RANK"]); torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
blob = torch.load({blob!r})
m = NormalPredictorGRU(29, 9).cuda().eval()        # eval: no dropout, so the split is exact
m.load_state_dict(blob["state"])
bucket = FlatGradBucket(m.parameters())
lo, hi = (0, 128) if rank == 0 else (128, 256)
pred = m.forward_cone(blob["x"][lo:hi].cuda(), blob["xt"][lo:hi].cuda())
torch.nn.functional.mse_loss(pred, blob["y"][lo:hi].cuda()).backward()
bucket.allreduce()
if rank == 0:
    torch.save({{n: p.grad.cpu() for n, p in m.named_parameters()}}, {out!r})
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_gradients_equal_single_gpu_on_concatenated_batch(tmp_path):
    torch.manual_seed(7)
    m = NormalPredictorGRU(29, 9).cuda().eval()
    gen = torch.Generator().manual_seed(8)
    blob = {"state": {k: v.cpu() for k, v in m.state_dict().items()}, "x": torch.randn(256, 36, 29, generator=gen),
            "xt": torch.randn(256, 36, 9, generator=gen), "y": torch.randn(256, 29, generator=gen)}
    torch.save(blob, tmp_path / "blob.pt")
    torch.nn.functional.mse_loss(m.forward_cone(blob["x"].cuda(), blob["xt"].cuda()), blob["y"].cuda()).backward()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(repo=str(REPO), blob=str(tmp_path / "blob.pt"), out=str(tmp_path / "g.pt")))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=600,
                       env={**os.environ, "PYTHONPATH": str(REPO)})
    assert r.returncode == 0, r.stderr[-3000:]
    got = torch.load(tmp_path / "g.pt")
    errs = {n: rel_err(got[n], p.grad) for n, p in m.named_parameters()}
    assert all(e <= 3e-6 for e in errs.values()), {n: e for n, e in errs.items() if e > 3e-6}


def test_training_entry_points_reject_bad_arguments():
    lib = _lib.load()
    q, l = 4, 3
    gx = torch.zeros(3, q * l, 128, device="cuda")
    w = torch.zeros(384, 128, device="cuda")
    b = torch.zeros(128, device="cuda")
    h = torch.zeros(q, 128, device="cuda")
    s = torch.zeros(q * l, 128, device="cuda")
    gates = torch.zeros(4, q * l, 128, device="cuda")
    dg = torch.zeros(4, q * l, 128, device="cuda")
    live = torch.zeros(q * l, 4, device="cuda", dtype=torch.int32)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def fwd(q_=q, l_=l, hd=128, gx_=gx.data_ptr(), w_=w.data_ptr(), b_=b.data_ptr(), s_=s.data_ptr(), h_=h.data_ptr(),
            g_=gates.data_ptr()):
        return lib.ltgnn_gru_layer_fwd_train(0, q_, l_, hd, gx_, w_, b_, s_, h_, g_, stream)

    assert fwd() == 0
    assert fwd(hd=64) == -2
    assert fwd(q_=0) == -1 and fwd(l_=0) == -1 and fwd(q_=-1) == -1
    assert fwd(gx_=None) == -1 and fwd(w_=None) == -1 and fwd(b_=None) == -1 and fwd(h_=None) == -1
    assert fwd(s_=None) == -1 and fwd(g_=None) == -1                  # training needs the states and the gates
    assert fwd(gx_=gx.data_ptr() + 4) == -3 and fwd(g_=gates.data_ptr() + 4) == -3 and fwd(s_=s.data_ptr() + 4) == -3

    def bwd(q_=q, l_=l, hd=128, w_=w.data_ptr(), g_=gates.data_ptr(), s_=s.data_ptr(), dl=h.data_ptr(), ds=None,
            d_=dg.data_ptr()):
        return lib.ltgnn_gru_layer_bwd(0, q_, l_, hd, w_, g_, s_, dl, ds, d_, stream)

    assert bwd() == 0 and bwd(dl=None, ds=s.data_ptr()) == 0 and bwd(ds=s.data_ptr()) == 0
    assert bwd(hd=256) == -2
    assert bwd(q_=0) == -1 and bwd(l_=-1) == -1 and bwd(dl=None) == -1      # one of dh_last / dh_seq is required
    assert bwd(w_=None) == -1 and bwd(g_=None) == -1 and bwd(s_=None) == -1 and bwd(d_=None) == -1
    assert bwd(dl=h.data_ptr() + 4) == -3 and bwd(ds=s.data_ptr() + 8) == -3 and bwd(d_=dg.data_ptr() + 4) == -3

    def drop(m=q * l, hd=128, x_=s.data_ptr(), p=0.1, y_=gx.data_ptr(), lv=live.data_ptr()):
        return lib.ltgnn_gru_dropout(0, m, hd, x_, p, 7, y_, lv, stream)

    assert drop() == 0 and drop(p=0.0) == 0
    assert drop(hd=64) == -2
    assert drop(m=0) == -1 and drop(p=1.0) == -1 and drop(p=-0.1) == -1
    assert drop(x_=None) == -1 and drop(y_=None) == -1 and drop(lv=None) == -1
    assert drop(x_=s.data_ptr() + 4) == -3 and drop(y_=gx.data_ptr() + 4) == -3

    def dbwd(m=q * l, hd=128, dy=gx.data_ptr(), n=3, lv=live.data_ptr(), p=0.1, dx=s.data_ptr()):
        return lib.ltgnn_gru_dropout_bwd(0, m, hd, dy, n, lv, p, dx, stream)

    assert dbwd() == 0 and dbwd(lv=None, p=0.0) == 0
    assert dbwd(hd=96) == -2
    assert dbwd(m=-1) == -1 and dbwd(n=0) == -1 and dbwd(n=5) == -1 and dbwd(p=1.5) == -1
    assert dbwd(dy=None) == -1 and dbwd(dx=None) == -1
    assert dbwd(dy=gx.data_ptr() + 4) == -3 and dbwd(dx=s.data_ptr() + 4) == -3
    with pytest.raises(_lib.LtgnnError) as e:
        _lib.check(bwd(dl=None))
    assert e.value.code == -1 and "dh_seq" in str(e.value)
    torch.cuda.synchronize()
