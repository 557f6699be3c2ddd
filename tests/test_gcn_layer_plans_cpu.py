"""The plan space of the one-kernel GCN layer (csrc/gcn_layer.cu) without a GPU: the Python restatement of its plan
follows the source, the case list of test_gcn_layer_plans_gpu.py reaches every plan the kernel can pick, the synthetic
networks have the features the cases rely on, and the GPU file's elementwise bound is tight enough to catch a kernel
that lost the lo half of its 3xTF32 split."""
import re

import pytest
import torch

import gcn_plans as G
from conftest import REPO
from leak_det_gnn_b200.graph import build_gcn_csr

SRC = (REPO / "leak_det_gnn_b200" / "csrc" / "gcn_layer.cu").read_text()


def test_restatement_constants_follow_the_source():
    consts = dict(re.findall(r"\b(k[A-Z]\w*) = (\d+)", SRC))
    assert (consts["kLdWarps"], consts["kMaxSlots"], consts["kSlotCols"], consts["kMaxTiles"]) == ("4", "4", "32", "7")
    patch = (REPO / "leak_det_gnn_b200" / "csrc" / "patch.cuh").read_text()
    assert re.search(r"kPatchBytes = (\d+)", patch).group(1) == str(G.PATCH)
    assert "K > 128" in SRC and "D > 256" in SRC and "T * D + 2 * gl::kSlotCols > 512" in SRC
    # the static bytes the launch leaves room for: 10 mbarriers and the TMEM address
    assert "__shared__ uint64_t bar_full[kMaxSlots], bar_empty[kMaxSlots], bar_acc_full, bar_acc_empty;" in SRC
    assert G.STATIC_SMEM == 8 * (2 * 4 + 2) + 4


def test_case_list_covers_the_plan_space():
    plans = [(c, G.plan(c.n, c.nnz, c.K, c.D)) for c in G.cases()]
    table = "\n".join(f"{c.name:26s} n={c.n:4d} nnz={c.nnz:5d} {c.K:3d}->{c.D:3d}  T={p.T} slots={p.n_slots} "
                      f"depth={p.depth} smem={p.smem}" for c, p in plans)
    print(table)
    assert all(p.supported for _, p in plans), table
    assert {p.T for _, p in plans} == set(range(1, 8)), table
    assert any(c.n % 128 == 0 for c, _ in plans) and any(c.n % 128 for c, _ in plans), table
    assert any(c.n < 96 for c, _ in plans), table                  # fewer rows than one dropout pass
    assert {c.K for c, _ in plans} == {32, 64, 96, 128}, table
    assert {p.n_slots for _, p in plans} == {2, 4} and {p.depth for _, p in plans} == {2, 4}, table
    assert {(p.n_slots, p.depth) for _, p in plans} == {(2, 2), (2, 4), (4, 2), (4, 4)}, table
    for d in range(32, 257, 32):   # every width at the largest tile count it is accepted at
        t_max = max(t for t in range(1, 8) if t * d + 64 <= 512)
        assert any(c.D == d and p.T == t_max for c, p in plans), (d, t_max, table)
    assert any(p.smem == G.SMEM_OPTIN - 1024 and p.depth == 2 for _, p in plans), table
    assert any(p.smem == G.SMEM_OPTIN - 1024 and p.depth == 4 for _, p in plans), table


def test_refused_cases_are_refused():
    for c in G.refused_cases():
        assert not G.plan(c.n, c.nnz, c.K, c.D).supported, c


def test_exact_limit_bands():
    """The graph sizes whose launch asks for exactly the opt-in bytes of dynamic shared memory (no room left for the
    kernel's static barriers): with the static bytes counted they are refused (depth 2) or run at depth 2 (depth 4)."""
    want = {(384, 128, 128): ((1983, 2110), None), (512, 128, 64): ((8063, 8190), (3967, 4094)),
            (768, 96, 64): ((5887, 6014), (1791, 1918)), (785, 64, 64): ((7655, 7782), (3559, 3686))}
    for (n, k, d), bands in want.items():
        for depth, band in zip((2, 4), bands):
            got = G.nnz_band(n, k, d, depth, G.SMEM_OPTIN)
            assert (got[0], got[-1]) == band if band else len(got) == 0, (n, k, d, depth)
            for nnz in got:
                blind = G.plan(n, nnz, k, d, static_smem=0)
                assert blind.supported and blind.depth == depth and blind.smem == G.SMEM_OPTIN
                p = G.plan(n, nnz, k, d)
                assert (p.supported, p.depth) == ((False, 2) if depth == 2 else (True, 2)), (n, nnz, k, d)
                assert not p.supported or p.smem < G.SMEM_OPTIN - G.STATIC_SMEM


@pytest.mark.parametrize("case", G.cases() + G.refused_cases(), ids=lambda c: c.name)
def test_pipe_networks(case):
    """Exactly the nnz the case asks for, with an isolated node, a duplicated edge, an input self loop, and a hub of
    degree >= 200 wherever the network has that many nodes."""
    ei = G.pipe_edges(case.n, case.nnz)
    csr = build_gcn_csr(ei, case.n)
    assert csr.nnz == case.nnz
    deg = csr.rowptr[1:] - csr.rowptr[:-1]            # entries per row, self loop included
    assert deg[case.n - 1] == 1                        # isolated: its self loop only
    assert (ei[0] == ei[1]).any()
    pairs = ei.t().tolist()
    assert len(pairs) - len(set(map(tuple, pairs))) >= 1
    if case.n > 203:
        assert deg.max() >= 201
    assert torch.equal(ei, G.pipe_edges(case.n, case.nnz))  # deterministic


def test_tf32_round_is_the_kernels_hi_half():
    x = torch.tensor([1.0, -1.0, 1 + 2.0 ** -11, 1 + 3 * 2.0 ** -12, -(1 + 2.0 ** -11), 3.0e38, 1e-30])
    hi = G.tf32_round(x)
    assert hi.tolist()[:5] == [1.0, -1.0, 1 + 2.0 ** -10, 1 + 2.0 ** -10, -(1 + 2.0 ** -10)]
    assert (hi.view(torch.int32) & 0x1FFF == 0).all()
    assert ((hi.double() - x.double()).abs() <= x.double().abs() * 2.0 ** -11).all()


@pytest.mark.parametrize("case", G.cases(), ids=lambda c: c.name)
def test_bound_catches_plain_tf32(case):
    """At every case shape, the product with both operands rounded to plain TF32 (the lo half dropped; exact fp64 sums)
    breaks the GPU file's bound, while the 3xTF32 split (lo truncated to TF32 by the tensor core, lo * lo dropped)
    uses less than a quarter of it."""
    x, w, b = G.inputs(case, 1)
    a = G.gcn_dense(G.pipe_edges(case.n, case.nnz), case.n)
    y64, scale = G.reference(a, x.double(), w.double(), b)

    def trunc(v):  # what the tensor core reads of an fp32 operand: the top 19 bits
        return (v.float().contiguous().view(torch.int32) & -8192).view(torch.float32)

    xh, wh = G.tf32_round(x), G.tf32_round(w)
    plain, _ = G.reference(a, xh.double(), wh.double(), b)
    xl, wl = trunc(x - xh).double(), trunc(w - wh).double()
    xw3 = xh.double() @ wh.double().t() + xh.double() @ wl.t() + xl @ wh.double().t()
    split = a @ xw3 + b.double()
    r_plain, r_split = G.bound_ratio(plain, y64, scale), G.bound_ratio(split, y64, scale)
    print(f"{case.name}: plain TF32 {r_plain:.2f}, 3xTF32 {r_split:.3f} of the bound")
    assert r_plain > 1.0, r_plain
    assert r_split < 0.25, r_split
