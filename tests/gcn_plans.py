"""The launch plan of the one-kernel GCN layer (csrc/gcn_layer.cu), restated in Python, and the synthetic pipe networks
the plan tests run it on.  Shared by test_gcn_layer_plans_cpu.py (which checks that the case list covers the plan space)
and test_gcn_layer_plans_gpu.py (which runs the kernel at every case)."""
from __future__ import annotations

from typing import NamedTuple

import numpy as np
import torch

SMEM_OPTIN = 232448     # sm_100: opt-in shared memory per block (227 KB), dynamic + static
STATIC_SMEM = 84        # the kernel's static barriers and TMEM address; any value in 1..1024 gives the same plans, since
                        # every plan's dynamic bytes are a multiple of 1024
PATCH = 4096            # patch::kPatchBytes
LOADERS = 4             # loader warps, one ring each


class Plan(NamedTuple):
    supported: bool
    T: int              # 128-node tiles per window
    n_slots: int        # A slots in tensor memory
    depth: int          # loader ring depth
    smem: int           # dynamic shared memory of the launch


def _up(x: int, a: int) -> int:
    return (x + a - 1) // a * a


def _fixed(n: int, K: int, D: int) -> int:
    """Bytes ahead of the entries: resident weight (TF32 hi + lo), stage, row pointers."""
    return 2 * D * K * 4 + _up(n * 128, 128) + _up(4 * (n + 1), 16)


def ring_offset(n: int, nnz: int, K: int, D: int) -> int:
    """Bytes before the loader rings, 1024-aligned: the fixed part and 8 bytes per entry."""
    return _up(_fixed(n, K, D) + 8 * nnz, 1024)


def plan(n: int, nnz: int, K: int, D: int, smem_optin: int = SMEM_OPTIN, static_smem: int = STATIC_SMEM) -> Plan:
    """ltgnn_gcn_layer_supported + the plan of ltgnn_gcn_layer_fwd.  ``supported`` False: the other fields are what the
    launch would have asked for, where defined."""
    T = (n + 127) // 128
    if K % 32 or not 0 < K <= 128 or D % 32 or not 0 < D <= 256 or T > 7 or T * D + 64 > 512:
        return Plan(False, T, 0, 0, 0)
    n_slots = 4 if (512 - T * D) // 32 >= 4 else 2
    off_ring = ring_offset(n, nnz, K, D)
    limit = smem_optin - static_smem
    ok = 1024 + off_ring + LOADERS * 2 * PATCH <= limit
    depth = 4 if limit - 1024 - off_ring >= LOADERS * 4 * PATCH else 2
    return Plan(ok, T, n_slots, depth, 1024 + off_ring + LOADERS * depth * PATCH)


def nnz_band(n: int, K: int, D: int, depth: int, smem: int) -> range:
    """The nnz for which a (n, K, D) launch at ring ``depth`` asks for exactly ``smem`` dynamic bytes (may be empty)."""
    target = smem - 1024 - LOADERS * depth * PATCH
    base = _fixed(n, K, D)
    lo, hi = max(0, -(-(target - 1023 - base) // 8)), (target - base) // 8
    return range(lo, hi + 1) if target % 1024 == 0 and hi >= lo else range(0)


def last_nnz(n: int, K: int, D: int, depth: int) -> int:
    """Largest nnz the kernel accepts at (n, K, D) with ring ``depth`` (2: the support limit; 4: the depth switch)."""
    lo, hi = 0, 1 << 16
    while lo < hi:
        mid = (lo + hi + 1) // 2
        p = plan(n, mid, K, D)
        if p.supported and p.depth >= depth:
            lo = mid
        else:
            hi = mid - 1
    return lo


def min_nnz(n: int) -> int:
    return _pipe_base(n)[1]


def _pipe_base(n: int):
    """Chain 0-1-...-(m-1) with node n-1 left isolated, a hub at node 0 (degree 201) when the network has room for one,
    one duplicated edge and one self loop in the input (which gcn_norm replaces)."""
    m = n - 1 if n >= 3 else n
    und = [(i, i + 1) for i in range(m - 1)]
    if m > 202:
        und += [(0, j) for j in range(2, 202)]
    directed = [(a, b) for a, b in und] + [(b, a) for a, b in und]
    if m >= 3:
        directed.append((1, 2))          # duplicated edge: two CSR entries, counted twice in the degree
    loops = [(min(2, n - 1), min(2, n - 1))]
    return (m, set(und), directed, loops), len(directed) + n


def pipe_edges(n: int, nnz: int | None = None) -> torch.Tensor:
    """(2, E) int64 ``edge_index`` of a deterministic pipe-like network with ``n`` nodes whose GCN CSR (self loops
    included) has exactly ``nnz`` entries; default: mean degree ~2.3, as water networks have.  Chords between random
    node pairs, both directions, pad the chain up to ``nnz``."""
    (m, und, directed, loops), base = _pipe_base(n)
    if nnz is None:
        nnz = max(base, round(3.3 * n))
    if nnz < base:
        raise ValueError(f"{n} nodes need at least {base} entries, asked for {nnz}")
    rng = np.random.default_rng(1_000_003 * n + nnz)
    need = nnz - base
    if need % 2:
        directed.append((directed[0][1], directed[0][0]) if directed else (0, 1))  # a second duplicate: +1 entry
        need -= 1
    while need:
        a, b = (int(v) for v in rng.integers(0, m, 2))
        a, b = min(a, b), max(a, b)
        if a == b or (a, b) in und:
            continue
        und.add((a, b))
        directed += [(a, b), (b, a)]
        need -= 2
    ei = torch.tensor(directed + loops, dtype=torch.long).t().contiguous()
    return ei


# ------------------------------------------------------------------------------------------------ the case list
class Case(NamedTuple):
    name: str
    n: int
    nnz: int
    K: int
    D: int


def _case(name, n, K, D, nnz=None):
    return Case(name, n, max(min_nnz(n), round(3.3 * n)) if nnz is None else nnz, K, D)


def cases() -> list:
    """Accepted plans the GPU file runs: every tile count with partial and full last tiles, every K, every D at its
    largest accepted T, both slot counts and both ring depths, and the last accepted graph at each shared-memory limit."""
    out = [_case(f"T{(n + 127) // 128}_n{n}", n, 64, 64) for n in (40, 95, 128, 129, 256, 300, 384, 450, 512, 600, 700,
                                                                   785, 896)]
    out += [_case(f"K{k}_n200", 200, k, 64) for k in (32, 96, 128)]
    # each width at its largest tile count (T * D + 64 <= 512) with a K that fits the resident weight
    out += [_case("D32_T7", 840, 32, 32), _case("D96_T4", 500, 64, 96), _case("D128_T3_K128", 384, 128, 128),
            _case("D160_T2", 250, 64, 160), _case("D192_T2", 256, 64, 192), _case("D224_T2_K96", 129, 96, 224),
            _case("D256_T1", 100, 64, 256)]
    # the last graph each shared-memory limit accepts (depth 2: support; depth 4: the ring-depth switch), and a graph
    # whose depth-4 launch would ask for exactly the opt-in bytes: it runs at depth 2
    for n, k, d in LIMIT_SHAPES:
        for depth in (2, 4):
            nnz = last_nnz(n, k, d, depth)
            if nnz >= min_nnz(n):
                out.append(Case(f"edge_d{depth}_n{n}_{k}to{d}", n, nnz, k, d))
        band = nnz_band(n, k, d, 4, SMEM_OPTIN)
        if len(band) and band[0] >= min_nnz(n):
            out.append(Case(f"exact_d4_n{n}_{k}to{d}", n, band[len(band) // 2], k, d))
    return out


# (n, K, D) with a graph size whose launch would ask for exactly the opt-in bytes of dynamic shared memory, which the
# kernel's static bytes do not fit next to: at ring depth 2 the shape is refused, at depth 4 it drops to depth 2
LIMIT_SHAPES = ((384, 128, 128), (512, 128, 64), (768, 96, 64), (785, 64, 64))


def refused_cases() -> list:
    """Shapes outside the plan space: too many nodes, accumulators + two A slots over 512 columns, K over 128, and one
    entry past each shared-memory limit (the first graph of each exact-limit band)."""
    out = [_case("n897", 897, 64, 64), _case("TD_over_512", 300, 64, 160), _case("K160", 200, 160, 64)]
    for n, k, d in LIMIT_SHAPES:
        out.append(Case(f"past_n{n}_{k}to{d}", n, last_nnz(n, k, d, 2) + 1, k, d))
    return out


# ------------------------------------------------------------------------------------------------ tolerance
# Elementwise bound of the GPU file: |y - y64| <= TAU * (|A_hat| (|X| |W|^T) + |b|).  TAU = 2^-17 is derived from the
# arithmetic, for unit roundoff u = 2^-24 and the error sizes that are met in practice (probabilistic, sqrt(n) u for an
# n-term fp32 sum -- Higham & Mary 2019 -- with a factor 2 on top):
#   3xTF32 product  hi = round-to-nearest to TF32 (error <= 2^-11 |a|), lo = a - hi exact; the tensor core truncates lo
#                   to TF32 (<= 2^-21 |a|) and lo*lo is dropped (<= 2^-22 |a||b|): <= 2^-20 per product, 1e-6
#   X W^T           3K products summed in fp32: sqrt(3 * 128) u = 1.2e-6
#   aggregation     (deg + 1) entries, a multiply and an add each, hub degree ~200: sqrt(2 * 202) u = 1.2e-6
#   bias            one rounding: 6e-8
# which totals 3.4e-6, against TAU = 7.6e-6.  Plain TF32 (lo half dropped) errs by up to 2^-11 per operand, 2^-12 on
# average: the CPU file shows that such a kernel breaks the bound at every case shape.
TAU = 2.0 ** -17


def tf32_round(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> TF32 as the kernels' split rounds the hi half (umma.cuh tf32_hi: add half an ulp, drop 13 bits)."""
    b = (x.float().contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF) + 0x1000
    b = b & 0xFFFFE000
    return torch.where(b >= 1 << 31, b - (1 << 32), b).to(torch.int32).view(torch.float32)


def reference(a_hat: torch.Tensor, x: torch.Tensor, w: torch.Tensor, b):
    """(relu-free) A_hat (X W^T) + b in the dtype of ``a_hat``, and the elementwise scale of the bound:
    |A_hat| (|X| |W|^T) + |b|."""
    dt = a_hat.dtype
    y = a_hat @ (x.to(dt) @ w.to(dt).t())
    s = a_hat.abs() @ (x.to(dt).abs() @ w.to(dt).abs().t())
    if b is not None:
        y, s = y + b.to(dt), s + b.to(dt).abs()
    return y, s


def bound_ratio(y: torch.Tensor, y64: torch.Tensor, scale: torch.Tensor) -> float:
    """max |y - y64| / (TAU * scale): the bound holds iff this is <= 1."""
    return ((y.to(y64.dtype) - y64).abs() / (TAU * scale).clamp_min(1e-300)).max().item()


def gcn_dense(edge_index: torch.Tensor, n: int, dtype=torch.float64, device="cpu") -> torch.Tensor:
    """Dense A_hat (target row, source column) from the PyG restatement's gcn_norm -- not from PipeGraph.csr."""
    from oracle import pyg_restatement as pyg
    ei, norm = pyg.gcn_norm(edge_index.to(device), n, dtype=dtype)
    a = torch.zeros(n, n, dtype=dtype, device=device)
    return a.index_put_((ei[1], ei[0]), norm, accumulate=True)


def inputs(case: Case, bsz: int, seed: int = 0, spread: int = 20):
    """X (bsz, n, K) with row magnitudes spread over 2^-spread .. 2^spread, W (D, K), b (D,): fp32 on the CPU."""
    gen = torch.Generator().manual_seed(seed * 7919 + case.n * 31 + case.K + case.D)
    x = torch.randn(bsz, case.n, case.K, generator=gen)
    if spread:
        x = x * torch.exp2(torch.randint(-spread, spread + 1, (bsz, case.n, 1), generator=gen).float())
    w = torch.randn(case.D, case.K, generator=gen) * (1.0 / case.K ** 0.5)
    b = torch.randn(case.D, generator=gen) * 0.1
    return x, w, b
