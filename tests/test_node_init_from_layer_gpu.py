"""Node init's backward straight from the first GCN layer's aggregated gradient (ltgnn_node_init_bwd_from_layer): the
tensor-core GEMM dX0 = G1 W1 gates its rows, sums its columns and keeps its sensor rows in the epilogue, and dX0 is never
stored.  Checked against fp64 torch on the GPU (cuBLAS DGEMM for dX0, fp64 autograd of detector.py:178-189 gated by the
forward's own live bits), and against the two-launch path it replaces (ltgnn_linear + ltgnn_node_init_bwd): d h_s and
d sensor_to_node.weight in the same bits, d sensor_to_node.bias up to summation order.  Shapes: the lta4096 rows, node
width 128, row counts off the 128-row tile, sensors on tile and window edges, one sensor, fewer nodes than a tile."""
import ctypes

import numpy as np
import pytest
import torch

import bench
from conftest import parity_log, rel_err
from leak_det_gnn_b200 import lib as _lib
from leak_det_gnn_b200 import ops

pytestmark = pytest.mark.gpu
TOL = 1e-5
SCALE = float(np.float32(1.0) / (np.float32(1.0) - np.float32(round(0.1 * 65536) / 65536)))

# name: (B, N, sensor nodes or a count, ds, D, K)
CASES = {
    "lta4096": (4096, 661, "LTA", 64, 64, 64),
    "d128": (37, 661, 29, 64, 128, 64),
    "ragged_k128": (3, 785, 33, 32, 128, 128),           # B*N = 2355: the last tile is partial
    "one_sensor": (5, 203, 1, 64, 64, 32),
    "tile_edges": (3, 130, [0, 1, 126, 127, 128, 129], 64, 64, 64),  # rows 127 | 128 and windows 0 | 1 | 2 in tiles
    "small_n": (7, 40, 5, 32, 64, 64),                  # several windows per 128-row tile
}


def _operands(name, seed=5):
    bsz, n, sens, ds, d, k = CASES[name]
    gen = torch.Generator(device="cuda").manual_seed(seed)
    if sens == "LTA":
        idx = torch.from_numpy(bench.network("LTA", 764)["sensor_idx"]).cuda()
    elif isinstance(sens, list):
        idx = torch.tensor(sens, device="cuda")
    else:
        idx = torch.randperm(n, device="cuda", generator=gen)[:sens]
    s = idx.numel()
    slot = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    slot[idx] = torch.arange(s, dtype=torch.int32, device="cuda")
    h_s = torch.randn(bsz, s, ds, device="cuda", generator=gen)
    w0 = torch.randn(d, ds + 1, device="cuda", generator=gen) * 0.2
    b0 = torch.randn(d, device="cuda", generator=gen) * 0.5
    gz = torch.randn(bsz, n, k, device="cuda", generator=gen)
    gz *= torch.rand(bsz, n, k, device="cuda", generator=gen) > 0.3
    w1 = torch.randn(k, d, device="cuda", generator=gen) * k ** -0.5
    live = ops.new_live_mask(bsz, n, d, "cuda")
    x0 = ops.node_init_fwd(h_s, slot, n, w0, b0, 0.1, 21, live_out=live)
    return dict(idx=idx, slot=slot, h_s=h_s, w0=w0, b0=b0, gz=gz, w1=w1, live=live, x0=x0)


def _from_layer(o):
    return ops.node_init_bwd_from_layer(o["h_s"], o["slot"], o["w0"], o["gz"], o["w1"], o["live"], SCALE)


def _two_launch(o):
    dx0 = ops.linear_tc(o["gz"], o["w1"], transposed=True)
    return ops.node_init_bwd(o["h_s"], o["slot"], o["w0"], dx0, o["x0"], SCALE, live=o["live"])


def _truth(o):
    """fp64 gradients of detector.py:178-189 for dX0 = gz @ w1, gated by the live bits the forward wrote."""
    h_s, w, b = (o[k].double().requires_grad_(True) for k in ("h_s", "w0", "b0"))
    bsz, n = o["gz"].shape[:2]
    ds = h_s.shape[2]
    h0 = torch.zeros(bsz, n, ds, dtype=torch.float64, device="cuda").index_copy(1, o["idx"], h_s)
    mask = torch.zeros(n, 1, dtype=torch.float64, device="cuda")
    mask[o["idx"], 0] = 1.0
    pre = torch.nn.functional.linear(torch.cat([h0, mask.unsqueeze(0).expand(bsz, -1, -1)], dim=-1), w, b)
    dx0 = o["gz"].double() @ o["w1"].double()
    (pre * ops.unpack_live_mask(o["live"]).double()).backward(dx0 * SCALE)
    return h_s.grad, w.grad, b.grad


@pytest.mark.parametrize("name", list(CASES))
def test_against_fp64_and_the_two_launch_path(name):
    o = _operands(name)
    got = _from_layer(o)
    old = _two_launch(o)
    assert torch.equal(got[0], old[0]) and torch.equal(got[1], old[1])   # dz is bit-identical: so are d h_s and dW
    truth = _truth(o)
    rep = {nm: {"ours": rel_err(a, t), "two_launch": rel_err(c, t)}
           for nm, a, c, t in zip(("dh_s", "dW", "db"), got, old, truth)}
    rep["db"]["vs_two_launch"] = rel_err(got[2], old[2])
    parity_log(f"node_init_bwd_from_layer {name} {CASES[name]}", rep)
    for nm, r in rep.items():
        assert r["ours"] <= max(TOL, 3.0 * r["two_launch"]), (nm, r)
    again = _from_layer(o)
    assert all(torch.equal(a, c) for a, c in zip(got, again))   # deterministic: no atomics


def test_nan_poisoned_workspace_and_outputs():
    """Every workspace entry the call reads it writes first: a NaN-filled workspace and NaN-filled outputs give the
    bits of a fresh call."""
    o = _operands("ragged_k128")
    want = _from_layer(o)
    bsz, s, ds = o["h_s"].shape
    n, k = o["gz"].shape[1:]
    d = o["w1"].shape[1]
    L = _lib.load()
    dev = o["h_s"].device.index
    ws = torch.full((int(L.ltgnn_node_init_ws_floats(dev, bsz, s, ds, d)),), float("nan"), device="cuda")
    out = [torch.full_like(o["h_s"], float("nan")), torch.full_like(o["w0"], float("nan")),
           torch.full((d,), float("nan"), device="cuda")]
    _lib.check(L.ltgnn_node_init_bwd_from_layer(dev, bsz, n, s, ds, d, k, o["h_s"].data_ptr(), o["slot"].data_ptr(),
                                                o["w0"].data_ptr(), o["gz"].data_ptr(), o["w1"].data_ptr(),
                                                o["live"].data_ptr(), SCALE, out[0].data_ptr(), out[1].data_ptr(),
                                                out[2].data_ptr(), ws.data_ptr(),
                                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert all(torch.equal(a, c) for a, c in zip(out, want))


def test_under_graph_capture():
    o = _operands("d128")
    want = _from_layer(o)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        _from_layer(o)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        got = _from_layer(o)
    for v in got:
        v.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, c) for a, c in zip(got, want))


def test_refuses_unbuilt_widths():
    o = _operands("one_sensor")
    with pytest.raises(ValueError, match="not built"):
        ops.node_init_bwd_from_layer(o["h_s"], o["slot"], o["w0"], o["gz"][..., :16].contiguous(),
                                     o["w1"][:16].contiguous(), o["live"], SCALE)
    with pytest.raises(ValueError, match="live"):
        ops.node_init_bwd_from_layer(o["h_s"], o["slot"], o["w0"], o["gz"], o["w1"], None, SCALE)


@pytest.mark.parametrize("width", [64, 128])
def test_body_switch(width, monkeypatch):
    """gnn_body with FUSED_NODE_INIT_BWD on and off: every gradient in the same bits except d b0 (summation order), and
    one input-gradient GEMM fewer per step with it on."""
    from leak_det_gnn_b200 import instrument
    from test_gcn_layer_plans_gpu import _graph

    n, bsz, s, ds = 661, 6, 29, 64
    graph, _ = _graph(n, None)
    gen = torch.Generator().manual_seed(width)
    idx = torch.randperm(n, generator=gen)[:s]
    slot = torch.full((n,), -1, dtype=torch.int32)
    slot[idx] = torch.arange(s, dtype=torch.int32)
    h_s = torch.randn(bsz, s, ds, generator=gen)
    prm = [torch.randn(width, ds + 1, generator=gen) * 0.2, torch.randn(width, generator=gen) * 0.1]
    for _ in range(2):
        prm += [torch.randn(width, width, generator=gen) * width ** -0.5, torch.randn(width, generator=gen) * 0.1]
    dy = torch.randn(bsz, n, width, generator=gen).cuda()
    runs = []
    for on in (True, False):
        monkeypatch.setattr(ops, "FUSED_NODE_INIT_BWD", on)
        leaves = [t.cuda().requires_grad_(True) for t in [h_s] + prm]
        y = ops.gnn_body(leaves[0], slot.cuda(), graph, 0.1, False, leaves[1], leaves[2], leaves[3:])
        torch.cuda.synchronize()
        instrument.reset(timing=True)
        (y * dy).sum().backward()
        torch.cuda.synchronize()
        calls = instrument.summary()
        instrument.reset()
        runs.append(([t.grad for t in leaves], calls.get("linear_tc", {}).get("count", 0)))
    (on_g, on_lin), (off_g, off_lin) = runs
    assert on_lin == off_lin - 1, (on_lin, off_lin)
    names = ["h_s", "w0", "b0", "w1", "b1", "w2", "b2"]
    for nm, a, c in zip(names, on_g, off_g):
        if nm == "b0":
            assert rel_err(a, c) <= TOL, nm
        else:
            assert torch.equal(a, c), nm
