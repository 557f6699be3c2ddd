"""The C-ABI shared library: loads, exports exactly what include/ltgnn.h declares, and fails
loudly (never falls back) when there is no CUDA device.  No compute calls here."""
import ctypes
import re

import pytest
import torch

from conftest import REPO
from leak_det_gnn_b200 import lib as L


def _declared():
    text = (REPO / "include" / "ltgnn.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ltgnn_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    names = _declared()
    assert "ltgnn_spmm" in names and "ltgnn_graph_create" in names
    lib = L.load()
    for n in names:
        assert hasattr(lib, n), f"{n} declared in ltgnn.h but not exported"
    assert sorted(L.SIGNATURES) == names, "lib.SIGNATURES must mirror ltgnn.h"
    assert lib.ltgnn_version() == 200


def test_no_cpu_fallback_in_product():
    """The product package never imports the oracle."""
    for p in (REPO / "leak_det_gnn_b200").rglob("*.py"):
        src = p.read_text()
        assert "import oracle" not in src and "from oracle" not in src, p


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu(graph_golden):
    from leak_det_gnn_b200.ops import PipeGraph, spmm
    g0 = graph_golden("LTA")
    pg = PipeGraph(torch.from_numpy(g0["edge_index"]), 661)
    with pytest.raises(ValueError, match="CUDA"):
        spmm(pg, torch.zeros(1, 661, 64))
    import numpy as np
    c = pg.csr
    out = ctypes.c_void_p()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = L.load().ltgnn_graph_create(0, c.num_nodes, c.nnz, p(c.rowptr), p(c.col), p(c.val), p(c.t_rowptr),
                                     p(c.t_col), p(c.t_val), ctypes.byref(out))
    assert rc == -4 and not out.value
    assert "cuda" in L.last_error().lower()
    with pytest.raises(L.LtgnnError):
        L.check(rc)


def test_live_mask_and_blocked32_layouts_documented_in_the_header():
    """Host-side mirrors of the two device layouts the C ABI documents (include/ltgnn.h): the 1-bit gate word
    (bit 8c+q <-> element 4q+c of a 32-feature slice) and the blocked-32 row layout [rows/32][W/4][32][4]."""
    from leak_det_gnn_b200 import ops
    gen = torch.Generator().manual_seed(0)
    b, n, d = 2, 37, 64
    y = torch.randn(b, n, d, generator=gen).relu()
    words = torch.zeros(b, d // 32, n, dtype=torch.int64)
    for s in range(d // 32):
        for e in range(32):
            q, c = divmod(e, 4)
            words[:, s, :] |= (y[:, :, 32 * s + e] > 0).long() << (8 * c + q)
    words = torch.where(words >= 2**31, words - 2**32, words).to(torch.int32)  # bit 31 lives in the sign
    assert torch.equal(ops.unpack_live_mask(words), y > 0)

    l, q_, w = 3, 70, 64
    qp = (q_ + 127) // 128 * 128
    logical = torch.randn(l, qp, w, generator=gen)
    rows = logical.reshape(l * qp, w)
    blocked = rows.reshape(l * qp // 32, 32, w // 4, 4).permute(0, 2, 1, 3).contiguous()
    assert torch.equal(ops.unblock32(blocked, l, q_), logical[:, :q_])


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_graphed_step_and_device_seed_need_cuda():
    """The CUDA-graph training step and the device-resident dropout seed have no CPU form either."""
    from leak_det_gnn_b200 import ops
    from leak_det_gnn_b200.graphed import GraphedStep
    from leak_det_gnn_b200.parallel import FlatGradBucket

    with pytest.raises(ValueError, match="CUDA"):
        ops.device_seed(torch.zeros(1, dtype=torch.int64))
    m = torch.nn.Linear(4, 4)
    with pytest.raises(ValueError, match="CUDA"):
        GraphedStep(m, lambda: m(torch.zeros(1, 4)).sum(), None, FlatGradBucket(m.parameters()))
