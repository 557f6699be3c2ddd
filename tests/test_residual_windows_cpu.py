"""The host side of ``forward_windows`` on the TCN predictor: the shared cone plan's row pools (counts, which rows are
shared, what every row reads) and an fp64 torch evaluation of the plan against the per-window cone."""
import pytest
import torch
import torch.nn.functional as F

from leak_det_gnn_b200.models import NormalPredictorTCN
from leak_det_gnn_b200.models.predictor import cone_reach, shared_cone_plan, windows_of

DIL = [1, 2, 4, 8]
REACH = cone_reach(3, DIL)


def test_reach_and_row_counts_of_a_training_segment():
    assert REACH == [2, 4, 8, 12, 20, 28, 44, 60]
    plan, shared = shared_cone_plan(72, 36, 36, 1, 3, DIL)
    counts = [t.shape[1] for src1, src2, _ in plan for t in (src1, src2)]
    assert counts == [141, 138, 206, 164, 228, 180, 108, 36]
    assert shared[-1] == 0                       # at window 36 the head's row (p = 35 < 60) is windowed
    plan, shared = shared_cone_plan(72, 36, 36, 4, 3, DIL)
    assert [t.shape[1] for src1, src2, _ in plan for t in (src1, src2)] == [4 * c for c in counts]


def _readers(plan, batch, count, window, length):
    """Walk the plan back from each window's head row: per pool (-1 = input projection, then one per convolution) the
    (row, window, position) triples that window reads."""
    n_win = batch * count
    last = (torch.arange(n_win), torch.arange(n_win), torch.full((n_win,), window - 1))
    pools = {7: last}
    for i in range(len(plan) - 1, -1, -1):
        src1, src2, res = plan[i]
        d = DIL[i]
        rows, wins, ps = pools[2 * i + 1]
        mid, inp = [], [(res[rows], wins, ps)]
        for k in range(3):
            shift = (2 - k) * d
            mid.append((src2[k, rows], wins, ps - shift))
        m = tuple(torch.cat(c) for c in zip(*mid))
        keep = m[0] >= 0
        assert torch.equal(keep, m[2] >= 0)                  # -1 exactly where the tap is left padding
        m = torch.unique(torch.stack([t[keep] for t in m]), dim=1)
        pools[2 * i] = tuple(m)
        for k in range(3):
            inp.append((src1[k, m[0]], m[1], m[2] - (2 - k) * d))
        a = tuple(torch.cat(c) for c in zip(*inp))
        keep = a[0] >= 0
        assert torch.equal(keep, a[2] >= 0)
        pools[2 * i - 1] = tuple(torch.unique(torch.stack([t[keep] for t in a]), dim=1))
    return pools


@pytest.mark.parametrize("window,length,batch", [(36, 72, 2), (20, 41, 3), (64, 130, 2), (36, 300, 1)])
def test_every_shared_row_is_window_independent(window, length, batch):
    count = length - window + 1 if length != 72 else 36
    plan, shared = shared_cone_plan(length, window, count, batch, 3, DIL)
    pools = _readers(plan, batch, count, window, length)
    b_of, j_of = lambda w: w // count, lambda w: w % count
    rows, wins, ps = pools[-1]                                # input projection: series row b T + t
    assert torch.equal(rows, b_of(wins) * length + j_of(wins) + ps)
    for i in range(8):
        rows, wins, ps = pools[i]
        n_rows = plan[i // 2][i % 2].shape[1]
        assert torch.equal(torch.unique(rows), torch.arange(n_rows))      # every row is read, none is missing
        sh = rows < batch * shared[i]
        assert bool((ps[sh] >= REACH[i]).all()) and bool((ps[~sh] < REACH[i]).all())
        # a shared row is one (series, step): every reader agrees on both
        step = b_of(wins[sh]) * length + j_of(wins[sh]) + ps[sh]
        first = torch.full((n_rows,), -1, dtype=torch.int64).scatter_reduce(0, rows[sh], step, "amax")
        assert torch.equal(first[rows[sh]], step)
        # a windowed row has one reader window
        w = torch.full((n_rows,), -1, dtype=torch.int64).scatter_reduce(0, rows[~sh], wins[~sh], "amax")
        assert torch.equal(w[rows[~sh]], wins[~sh])


def _eval_plan(m, plan, x, x_time):
    """fp64 torch evaluation of the shared plan (the computation ``_native_stack`` runs on the kernels)."""
    b, length, _ = x.shape
    h = F.linear(torch.cat([x, x_time], -1).reshape(b * length, -1), m.input_proj.weight[:, :, 0], m.input_proj.bias)
    for blk, (src1, src2, res) in zip(m.tcn, plan):
        y = h
        for conv, norm, src in ((blk.conv1, blk.norm1, src1), (blk.conv2, blk.norm2, src2)):
            w = conv.conv.weight.permute(0, 2, 1).reshape(conv.conv.weight.shape[0], -1)
            padded = torch.cat([y, y.new_zeros(1, y.shape[1])])
            taps = torch.where(src < 0, torch.full_like(src, y.shape[0]), src)
            y = F.relu(norm(F.linear(padded[taps.t()].reshape(src.shape[1], -1), w, conv.conv.bias)))
        h = h[res] + y
    return m.head(h)


@pytest.mark.parametrize("window", [20, 36, 64])
@pytest.mark.parametrize("extra", [0, 1, "72", 300])
@pytest.mark.parametrize("batch", [1, 3])
def test_shared_plan_equals_per_window_cone_fp64(window, extra, batch):
    length = 72 if extra == "72" else (window + extra if extra in (0, 1) else extra)
    if length < window:
        pytest.skip("a 72-step series holds no 64 + 9 window")
    torch.manual_seed(window + length)
    m = NormalPredictorTCN(29, 9).double().eval()
    x, xt = torch.randn(batch, length, 29).double(), torch.randn(batch, length, 9).double()
    count = length - window + 1
    plan, _ = shared_cone_plan(length, window, count, batch, 3, DIL)
    with torch.no_grad():
        got = _eval_plan(m, plan, x, xt).view(batch, count, -1)
        ref = m._cone_torch(windows_of(x, window, count), windows_of(xt, window, count)).view(batch, count, -1)
    assert (got - ref).abs().max().item() <= 1e-12


def test_forward_windows_off_the_native_path_is_forward_last():
    torch.manual_seed(0)
    m = NormalPredictorTCN(29, 9).eval()
    x, xt = torch.randn(2, 50, 29), torch.randn(2, 50, 9)
    out = m.forward_windows(x, xt, 36, count=10)
    assert out.shape == (2, 10, 29)
    # the CPU cone's GEMMs depend on the batch size in the last bits; the native path is the bitwise one
    assert torch.allclose(out[1, 4], m.forward_last(x[1:2, 4:40], xt[1:2, 4:40])[0], rtol=1e-5, atol=1e-6)
    with pytest.raises(ValueError):
        m.forward_windows(x, xt, 36, count=16)
    with pytest.raises(RuntimeError):
        m.train().forward_windows(x, xt, 36)
