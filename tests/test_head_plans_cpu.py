"""The plan space of the fused pipe head at node width 64 (csrc/heads.cu, csrc/tgrad.cu on tgrad.cuh) without a GPU:
the Python restatement of its plans follows the source, the case list of test_head_plans_gpu.py reaches every branch
the three kernels take, the class-pipe sets have the incidence the cases rely on, and the GPU file's elementwise
bounds catch a kernel that lost the lo half of W1, a pipe end, the sign of the |.| block or the mean-pool term."""
import re

import numpy as np
import pytest
import torch

import head_plans as H
from conftest import REPO

CSRC = REPO / "leak_det_gnn_b200" / "csrc"
HEADS, TGRAD, TGRAD_H = ((CSRC / f).read_text() for f in ("heads.cu", "tgrad.cu", "tgrad.cuh"))
CASES = H.cases()
SETS = H.pipe_sets()


def _consts(src):
    return {k: int(v) for k, v in re.findall(r"\b(k[A-Z]\w*) = (\d+)", src)}


def test_restatement_constants_follow_the_source():
    hb = _consts(HEADS[HEADS.index("namespace hb {"):])
    assert (hb["kCapRows"], hb["kGaWarps"], hb["kTblWords"]) == (H.CAP_ROWS, H.GATHER_WARPS, H.TBL_WORDS)
    assert hb["kHalf"] == H.D // 2 and "constexpr int kD = 64;" in HEADS
    tg = _consts(TGRAD_H)
    assert (tg["kChunk"], tg["kGroups"]) == (H.CHUNK, H.GROUPS)
    assert _consts(TGRAD)["kHeadSlices"] == H.SLICES
    # the pipe head's weight gradient: register-total form, main flushed every 4th chunk
    assert "tgrad::launch<1, 4, 2, -4>(device, g, x, ws, M, No, &grid, stream, \"pipe_head_bwd_w\")" in TGRAD
    assert "return seg < 0 ? static_cast<uint32_t>(-(seg + 1)) + 1u : 1u;" in TGRAD_H
    # forward: tiles of 128 rows, grid = min(tiles, SMs), contiguous tile ranges
    assert "const int64_t tiles = (M + 127) / 128;" in HEADS
    assert "tiles < di->sm_count ? tiles : di->sm_count" in HEADS
    assert "const uint32_t per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;" in HEADS
    # bwd_dx: T tiles per window, min(B, SMs / 2) window ranges of two CTAs, the chunk table, tbl_fits, chunks per warp
    assert "const uint32_t T = (P + 127) / 128;" in HEADS
    assert "const int64_t ranges = B < di->sm_count / 2 ? B : di->sm_count / 2;" in HEADS
    assert "const uint32_t per_cta = (B + n_ranges - 1) / n_ranges;" in HEADS
    assert "__popc(__ballot_sync(0xffffffffu, i <= N && re - r0 <= kCapRows))" in HEADS
    assert "n0 += cnt ? cnt : 1;" in HEADS
    assert "const bool tbl_fits = n_chunks + 2 + N + 1 <= kTblWords;" in HEADS
    assert "n_chunks > j ? (n_chunks - j + kGaWarps - 1) / kGaWarps : 0" in HEADS
    assert "if (r1 > r0 && r1 - r0 <= kCapRows)" in HEADS
    # bwd_w: SMs / 3 * 3 CTAs, three per row range, contiguous chunk ranges
    assert "const int grid = di->sm_count / kSl * kSl;" in TGRAD_H
    assert "const uint32_t n_chunks = (M + kChunk - 1) / kChunk;" in TGRAD_H
    assert "const uint32_t per = (n_chunks + n_ranges - 1) / n_ranges;" in TGRAD_H
    assert "constexpr uint32_t kStep = tgrad::kGroups * tgrad::kChunk;" in TGRAD


def _plans(c):
    s = SETS[c.set]
    ptr, _ = H.incidence(H.pipe_ends(s), s.n)
    return s, H.fwd_plan(c.B, s.p), H.dx_plan(c.B, ptr), H.w_plan(c.B, s.p)


def test_case_list_covers_the_plan_space():
    rows, table = [], []
    for c in CASES:
        s, f, d, w = _plans(c)
        rows.append((c, s, f, d, w))
        table.append(f"{c.name:18s} N={s.n:4d} P={s.p:3d} | fwd tiles={f.tiles:4d} per_cta={f.per_cta} "
                     f"straddle={f.straddle:3d} | dx T={d.T} wins/cta={d.per} idle={d.idle:2d} chunks={d.n_chunks:3d} "
                     f"N+C+3={s.n + d.n_chunks + 3:4d} fits={int(d.tbl_fits)} max_rows={max(d.rows):3d} "
                     f"own={d.own} | w chunks={w.chunks:4d} per={w.per:2d} per%4={w.per % 4} idle={w.idle:2d} "
                     f"M%32={w.m_mod:2d}")
    table = "\n".join(table)
    print(table)
    # bwd_dx
    assert any(max(d.rows) > H.CAP_ROWS for *_, d, _ in rows), table                 # unstaged gather
    assert any(H.CAP_ROWS in d.rows for *_, d, _ in rows), table                      # the exact-fit chunk
    assert any(0 in d.rows for *_, d, _ in rows), table                               # a chunk with no pipe end
    assert any(np.diff(d.first).max() == H.CAP_NODES for *_, d, _ in rows), table     # a chunk of 32 nodes
    assert {d.tbl_fits for *_, d, _ in rows} == {True, False}, table
    assert {s.n + d.n_chunks + 3 for _, s, _, d, _ in rows} >= {2048, 2049}, table
    for _, s, _, d, _ in rows:
        assert d.tbl_fits == (s.n + d.n_chunks + 3 <= H.TBL_WORDS)
    assert any(d.T == 1 and d.per >= 3 for *_, d, _ in rows), table                   # scratch reused (bar_wfree)
    assert {min(d.per, 3) for *_, d, _ in rows} == {1, 2, 3}, table
    assert any(d.idle for *_, d, _ in rows), table
    assert any(s.p % 128 == 0 for _, s, *_ in rows) and any(s.p < 32 for _, s, *_ in rows), table
    assert any(0 in d.own for *_, d, _ in rows), table
    # forward
    assert any(f.per_cta > 2 for _, _, f, _, _ in rows), table
    assert any(f.straddle for _, _, f, _, _ in rows), table
    assert any(s.p == 1 for _, s, *_ in rows), table                                  # magic == 0 (fwd and bwd_w)
    # bwd_w
    assert {w.per % 4 for *_, w in rows} == {0, 1, 2, 3}, table
    assert any(w.idle for *_, w in rows), table
    assert {w.m_mod == 0 for *_, w in rows} == {True, False}, table
    assert len({c.B for c, s, *_ in rows if s.p < H.GROUPS * H.CHUNK}) >= 3, table   # advance() over several windows
    # the restated chunk table is a partition of the nodes that keeps every rule
    for *_, d, _ in rows:
        for k in range(d.n_chunks):
            nodes = d.first[k + 1] - d.first[k]
            assert 1 <= nodes <= H.CAP_NODES and (d.rows[k] <= H.CAP_ROWS or nodes == 1)


@pytest.mark.parametrize("name", list(SETS))
def test_pipe_sets(name):
    """Exact node and pipe counts, hubs with exactly the asked end counts, the run of nodes with no end, a degenerate,
    a duplicated and a reversed pipe where P allows; deterministic."""
    s = SETS[name]
    ends = H.pipe_ends(s)
    assert ends.shape == (s.p, 2) and int(ends.min()) >= 0 and int(ends.max()) < s.n
    assert torch.equal(ends, H.pipe_ends(s))
    cnt = np.bincount(ends.reshape(-1).numpy(), minlength=s.n)
    others = sorted(cnt.tolist(), reverse=True)
    for d in sorted(s.hubs, reverse=True):
        assert d in others
        others.remove(d)
    assert not others or max(others) < min(s.hubs + (H.CAP_ROWS,)), others[:5]
    z0 = s.n // 3
    assert not cnt[z0:z0 + s.zero_run].any()
    pairs = [tuple(e) for e in ends.tolist()]
    if s.p >= 2:
        assert any(u == v for u, v in pairs)
    if s.p >= 5:
        assert len(set(pairs)) < len(pairs) and any((v, u) in pairs for u, v in pairs if u != v)
    ptr, inc = H.incidence(ends, s.n)
    assert ptr[-1] == 2 * s.p and np.array_equal(np.diff(ptr), cnt)
    assert np.array_equal(np.sort(inc), np.arange(2 * s.p))
    assert np.array_equal(ends.reshape(-1).numpy()[inc], np.repeat(np.arange(s.n), cnt))   # grouped by node


def test_tf32_helpers_and_designed_w1():
    x = torch.tensor([1.0, -1.0, 1 + 2.0 ** -11, 1 + 3 * 2.0 ** -12, 3.0e38, 1e-30])
    assert H.tf32_round(x).tolist()[:4] == [1.0, -1.0, 1 + 2.0 ** -10, 1 + 2.0 ** -10]
    assert (H.tf32_trunc(x).view(torch.int32) & 0x1FFF == 0).all()
    gen = torch.Generator().manual_seed(0)
    w2 = torch.where(torch.rand(1, H.H, generator=gen) < 0.5, -0.25, 0.5)
    w1 = H.designed_w1(gen, w2)
    res = w1.double() - H.tf32_round(w1).double()
    assert (torch.sign(res) == torch.sign(w2.double()).reshape(-1, 1)).all()
    rel = res.abs() / w1.double().abs()
    assert rel.min() >= 2.0 ** -14 and rel.max() <= 2.0 ** -11


def _split_logits(inp, ends, live):
    """Logits from the kernel's 3xTF32 arithmetic with exact sums: the fp32 features and W1 split into TF32 hi + lo,
    lo truncated to TF32 by the tensor core, lo * lo dropped."""
    x = inp.x
    hu, hv = x[:, ends[:, 0]], x[:, ends[:, 1]]
    f = torch.cat([hu, hv, (hu - hv).abs()], dim=-1)
    fh, wh = H.tf32_round(f), H.tf32_round(inp.w1)
    fl, wl = H.tf32_trunc(f - fh).double(), H.tf32_trunc(inp.w1 - wh).double()
    fh, wh = fh.double(), wh.double()
    pre = fh @ wh.t() + fh @ wl.t() + fl @ wh.t() + inp.b1.double()
    return (live.double() * pre) @ inp.w2.double().reshape(-1) + inp.b2.double()


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_bounds_catch_the_mutants(case):
    """At every case shape, each mutant breaks its bound: plain TF32 on W1 (logits and dx), one pipe end lost at the
    node with the most ends and at a node with one end (dx), the sign of the |.| block ignored (logits and dx), the
    mean-pool term lost (dx).  The correct 3xTF32 arithmetic uses less than 1/16 of the logit and dx bounds."""
    s = SETS[case.set]
    ends = H.pipe_ends(s)
    inp = H.inputs(s, case.B)
    live = torch.ones(case.B, s.p, H.H, dtype=torch.bool)
    _, _, (pre, _) = H.reference(inp, ends, live, 1.0)
    live = pre > 0
    out, sc, _ = H.reference(inp, ends, live, 1.0)

    def ratio(mut, kind):
        return H.bound_ratio(mut[kind], out[kind], sc[kind], kind)

    rep = {}
    wb = (inp.w2.reshape(-1, 1) * inp.w1)                                       # fp32, exact: w2 is a power of two
    wh = H.tf32_round(wb)
    split_dx, _, _ = H.reference(inp, ends, live, 1.0, dx_w=wh.double() + H.tf32_trunc(wb - wh).double())
    rep["split logits"] = H.bound_ratio(_split_logits(inp, ends, live), out["logits"], sc["logits"], "logits")
    rep["split dx"] = ratio(split_dx, "dx")
    plain, _, _ = H.reference(inp, ends, live, 1.0, fwd_w1=H.tf32_round(inp.w1), dx_w=wh)
    rep["plain_tf32 logits"], rep["plain_tf32 dx"] = ratio(plain, "logits"), ratio(plain, "dx")
    cnt = np.bincount(ends.reshape(-1).numpy(), minlength=s.n)
    g0 = inp.dlogit[0].abs()
    for tag, node in (("hub", int(cnt.argmax())), ("single", int(np.flatnonzero(cnt == 1)[0]))):
        mine = [(p, e) for p in range(s.p) for e in (0, 1) if int(ends[p, e]) == node]
        p, e = max(mine, key=lambda pe: g0[pe[0]].item())
        lost, _, _ = H.reference(inp, ends, live, 1.0, drop_end=(0, p, e))
        rep[f"lost_end_{tag} dx"] = ratio(lost, "dx")
    sign, _, _ = H.reference(inp, ends, live, 1.0, abs_as_diff=True)
    rep["abs_sign logits"], rep["abs_sign dx"] = ratio(sign, "logits"), ratio(sign, "dx")
    rep["no_pool dx"] = ratio(H.reference(inp, ends, live, 1.0, no_pool=True)[0], "dx")
    print(case.name, {k: f"{v:.3g}" for k, v in rep.items()})
    assert rep.pop("split logits") < 1 / 16 and rep.pop("split dx") < 1 / 16, rep
    assert all(v > 1.0 for v in rep.values()), rep
