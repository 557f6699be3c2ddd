"""torch.autograd bindings of the libltgnn kernels.

Everything here runs on CUDA tensors only and calls straight into the C ABI with raw
device pointers and the current torch stream.  Non-CUDA / non-fp32 inputs are a
``ValueError``; a missing extension is a ``RuntimeError`` -- there is no fallback path.
"""
from __future__ import annotations

import contextlib
import ctypes
import gc
import threading
from typing import Dict, Optional

import numpy as np
import torch

from . import instrument as _inst
from . import lib as _lib
from .graph import GCNCsr, build_gcn_csr

__all__ = ["PipeGraph", "capture", "device_seed", "spmm", "spmm_fused", "aggregate", "linear_tc", "wgrad", "gcn_conv", "mean_pool", "gnn_body", "heads", "heads_supported", "heads_wide_supported", "pipe_incidence", "gru_encode", "gru_supported", "tcn_cone", "gru_predictor_fwd", "gru_predictor_cone", "row_gather_sum", "tcn_windows", "gru_windows", "edge_norm", "gcn_adj_grad", "edge_mask_fwd", "explain_step", "pg_edge_index", "pg_edge_mask"]


# Test hook: when set to a dict, the autograd nodes drop the masks they saved into it (``lives``: the 1-bit ReLU-and-
# dropout records of x_0..x_L; ``head_live``: the same for the pipe head's hidden layer), so that a test can replay a
# train-mode step with exactly these masks in the fp64 oracle.  Never set by the product.
DEBUG_CAPTURE: Optional[dict] = None


def _ptr(a: np.ndarray) -> ctypes.c_void_p:
    return a.ctypes.data_as(ctypes.c_void_p)


@contextlib.contextmanager
def capture(graph: torch.cuda.CUDAGraph, pool=None):
    """``torch.cuda.graph(graph, pool)`` with Python's cycle collector kept out of the capture.  A finaliser that frees
    device memory or destroys a CUDA graph -- a dead PipeGraph's handle, the graphs of a dead training step -- is not
    permitted while a capture is underway and invalidates it, and torch no longer collects before capturing.  So dead
    cycles are finalised first, and no collection runs until the capture has ended."""
    gc.collect()
    enabled = gc.isenabled()
    gc.disable()
    try:
        with torch.cuda.graph(graph, pool=pool):
            yield
    finally:
        if enabled:
            gc.enable()


# Graph handles of PipeGraphs finalised during a capture (by a caller's own torch.cuda.graph, or by reference count
# inside one), waiting for ltgnn_graph_destroy: its cudaFree is not permitted during a capture.  They are released at
# the next release point with no capture underway on this thread.
_RETIRED: list = []


def _release_retired() -> None:
    if not _RETIRED or torch.cuda.is_current_stream_capturing():
        return
    L = _lib.load()
    while _RETIRED:
        L.ltgnn_graph_destroy(_RETIRED.pop())


class PipeGraph:
    """The normalised adjacency of ONE pipe network, uploaded once per device.

    Stands in for what the reference rebuilds on every forward: the B-times replicated
    ``edge_index`` (models/detector.py:105-114,195-196) and PyG's ``gcn_norm`` inside each
    ``GCNConv`` call (models/detector.py:199).
    """

    def __init__(self, edge_index: torch.Tensor, num_nodes: int) -> None:
        self.num_nodes = int(num_nodes)
        self.csr: GCNCsr = build_gcn_csr(edge_index, self.num_nodes)
        self._handles: Dict[int, ctypes.c_void_p] = {}
        self._edge_maps: Dict[int, tuple] = {}
        self._lock = threading.Lock()

    @property
    def nnz(self) -> int:
        return self.csr.nnz

    def handle(self, device: torch.device) -> ctypes.c_void_p:
        if device.type != "cuda":
            raise ValueError(f"PipeGraph needs a CUDA device, got {device}")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        h = self._handles.get(idx)
        if h is None:
            _release_retired()
            with self._lock:
                h = self._handles.get(idx)
                if h is None:
                    c = self.csr
                    out = ctypes.c_void_p()
                    L = _lib.load()
                    _lib.check(L.ltgnn_graph_create(idx, c.num_nodes, c.nnz, _ptr(c.rowptr), _ptr(c.col), _ptr(c.val),
                                                    _ptr(c.t_rowptr), _ptr(c.t_col), _ptr(c.t_val), ctypes.byref(out)))
                    self._handles[idx] = h = out
        return h

    @property
    def num_edges(self) -> int:
        """Edges of the ``edge_index`` the graph was built from: the length of an ``edge_weight`` row."""
        return self.csr.num_edges

    def edge_maps(self, device: torch.device):
        """(edge, t_edge, t_perm) of :class:`~leak_det_gnn_b200.graph.GCNCsr` as int32 tensors on ``device``, uploaded
        once: what the device normalisation of per-call edge weights reads."""
        self.handle(device)
        idx = device.index if device.index is not None else torch.cuda.current_device()
        hit = self._edge_maps.get(idx)
        if hit is None:
            c = self.csr
            hit = tuple(torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda", idx))
                        for a in (c.edge, c.t_edge, c.t_perm))
            self._edge_maps[idx] = hit
        return hit

    def __del__(self) -> None:  # best effort; the handle only owns ~40 KB of device memory
        try:
            _RETIRED.extend(self._handles.values())
            self._handles.clear()
            _release_retired()
        except Exception:
            pass


def _check_act(x: torch.Tensor, name: str) -> None:
    if not x.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (libltgnn has no CPU path), got {x.device}")
    if x.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, got {x.dtype}")
    if not x.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def _stream(x: torch.Tensor) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)


def spmm(graph: PipeGraph, x: torch.Tensor, transpose: bool = False, algo: int = _lib.SPMM_AUTO,
         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw (non-differentiable) batched aggregation.  x: (B, N, D) or (B*N, D) fp32 CUDA."""
    _check_act(x, "x")
    n = graph.num_nodes
    d = x.shape[-1]
    if x.numel() % (n * d) != 0:
        raise ValueError(f"x with shape {tuple(x.shape)} is not a whole number of {n}-node graphs")
    b = x.numel() // (n * d)
    y = torch.empty_like(x) if out is None else out
    if out is not None:
        _check_act(out, "out")
        if out.shape != x.shape:
            raise ValueError("out shape mismatch")
    L = _lib.load()
    h = graph.handle(x.device)
    tok = _inst.begin("spmm_bwd" if transpose else "spmm_fwd")
    _lib.check(L.ltgnn_spmm(h, int(bool(transpose)), b, d, x.data_ptr(), y.data_ptr(), int(algo), _stream(x)))
    _inst.end(tok)
    return y


class _Aggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: torch.Tensor, graph: PipeGraph) -> torch.Tensor:
        ctx.graph = graph
        return spmm(graph, x.contiguous(), transpose=False)

    @staticmethod
    def backward(ctx, dy: torch.Tensor):
        return spmm(ctx.graph, dy.contiguous(), transpose=True), None


def aggregate(x: torch.Tensor, graph: PipeGraph) -> torch.Tensor:
    """Differentiable ``A_hat @ x`` per window; backward is the CSC-transpose gather."""
    return _Aggregate.apply(x, graph)


def _dev_index(x: torch.Tensor) -> int:
    return x.device.index if x.device.index is not None else torch.cuda.current_device()


def linear_tc(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, relu: bool = False,
              transposed: bool = False, gate: Optional[torch.Tensor] = None, gate_scale: float = 1.0,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw (non-differentiable) tensor-core dense layer (tcgen05, 3xTF32):
    ``gate(act(x @ weight.T + bias))``, or ``x @ weight`` when ``transposed``; see ltgnn_linear."""
    _check_act(x, "x")
    _check_act(weight, "weight")
    k = x.shape[-1]
    n = weight.shape[1] if transposed else weight.shape[0]
    if (weight.shape[0] if transposed else weight.shape[1]) != k:
        raise ValueError(f"weight {tuple(weight.shape)} does not match x[..., {k}] (transposed={transposed})")
    m = x.numel() // k
    if out is None:
        y = torch.empty(*x.shape[:-1], n, device=x.device, dtype=torch.float32)
    else:
        _check_act(out, "out")
        if out.numel() != m * n:
            raise ValueError(f"out must hold {m} x {n} values")
        y = out
    if gate is not None:
        _check_act(gate, "gate")
        if gate.numel() != y.numel():
            raise ValueError("gate must have the shape of the output")
    L = _lib.load()
    tok = _inst.begin("linear_tc")
    _lib.check(L.ltgnn_linear(_dev_index(x), m, k, n, x.data_ptr(), weight.data_ptr(), int(transposed),
                              None if bias is None else bias.data_ptr(), int(relu),
                              None if gate is None else gate.data_ptr(), float(gate_scale), y.data_ptr(), _stream(x)))
    _inst.end(tok)
    return y


def new_dropout_seed() -> int:
    """A fresh 63-bit key for one in-kernel dropout stream, drawn from torch's CPU generator so that
    ``torch.manual_seed`` makes training runs reproducible."""
    return int(torch.randint(0, 2**62, (1,), dtype=torch.int64).item())


class device_seed:
    """``with device_seed(word): ...`` -- every dropout-bearing kernel launched from this thread inside the block keys
    its random stream with ``drop_seed + word[0]``, the int64 CUDA tensor ``word`` being read when the kernel RUNS
    (``ltgnn_seed_source``).  This is what lets a captured CUDA graph of a training step draw fresh masks on every
    replay (graphed.GraphedTrainStep bumps the word inside the graph)."""

    def __init__(self, word: torch.Tensor) -> None:
        if not word.is_cuda or word.dtype != torch.int64 or word.numel() != 1:
            raise ValueError("device_seed needs a one-element int64 CUDA tensor")
        self.word = word

    def __enter__(self):
        _lib.load().ltgnn_seed_source(ctypes.c_void_p(self.word.data_ptr()))
        return self

    def __exit__(self, *exc) -> None:
        _lib.load().ltgnn_seed_source(None)


def new_live_mask(b: int, n: int, d: int, device) -> torch.Tensor:
    """Storage for the 1-bit-per-element record of ``activation > 0`` the fused kernels write in the forward and
    gate with in the backward: word (b, s, i), bit 8 c + q <-> element (b, i, 32 s + 4 q + c)."""
    return torch.empty(b, d // 32, n, device=device, dtype=torch.int32)


def unpack_live_mask(live: torch.Tensor) -> torch.Tensor:
    """(B, D/32, N) int32 -> bool (B, N, D); for tests and debugging."""
    e = torch.arange(32, device=live.device, dtype=torch.int32)
    bits = (live.unsqueeze(-1) >> (8 * (e % 4) + e // 4)) & 1  # (B, S, N, 32): element e of a slice is bit 8 (e % 4) + e // 4
    return bits.permute(0, 2, 1, 3).reshape(live.shape[0], live.shape[2], -1).bool()


def spmm_fused(graph: PipeGraph, x: torch.Tensor, transpose: bool = False, bias: Optional[torch.Tensor] = None,
               relu: bool = False, drop_p: float = 0.0, drop_seed: int = 0, gate: Optional[torch.Tensor] = None,
               gate_scale: float = 1.0, want_colsum: bool = False, live_out: Optional[torch.Tensor] = None,
               live_in: Optional[torch.Tensor] = None, vals: Optional[torch.Tensor] = None, algo: int = _lib.SPMM_AUTO):
    """Raw fused aggregation (see ltgnn_spmm_fused): ``dropout(relu(A (x * gatemask) + bias))``.
    Returns ``y`` or ``(y, colsum)`` when ``want_colsum`` (column sums of the gated input).
    ``live_out`` / ``live_in``: int32 (B, D/32, N) tensors holding ``y > 0`` / the gate as one bit per element
    (see :func:`new_live_mask`).  ``vals``: per-call entry values (1 or B, nnz) in the order of the chosen orientation
    (:func:`edge_norm`) instead of the graph's own (ltgnn_spmm_fused_vals; ``algo`` forces a kernel there)."""
    _check_act(x, "x")
    n, d = graph.num_nodes, x.shape[-1]
    if x.numel() % (n * d) != 0:
        raise ValueError(f"x with shape {tuple(x.shape)} is not a whole number of {n}-node graphs")
    b = x.numel() // (n * d)
    if gate is not None:
        _check_act(gate, "gate")
        if gate.shape != x.shape:
            raise ValueError("gate must have the shape of x")
    if bias is not None:
        _check_act(bias, "bias")
    for lv, nm in ((live_out, "live_out"), (live_in, "live_in")):
        if lv is not None and (lv.dtype != torch.int32 or not lv.is_cuda or not lv.is_contiguous()
                               or tuple(lv.shape) != (b, d // 32, n)):
            raise ValueError(f"{nm} must be a contiguous int32 CUDA tensor of shape {(b, d // 32, n)}")
    if vals is not None:
        _check_act(vals, "vals")
        if vals.dim() != 2 or vals.shape[1] != graph.nnz or vals.shape[0] not in (1, b):
            raise ValueError(f"vals must be (1, {graph.nnz}) or ({b}, {graph.nnz}), got {tuple(vals.shape)}")
        if vals.device != x.device:
            raise ValueError("vals must be on the device of x")
    y = torch.empty_like(x)
    L = _lib.load()
    h = graph.handle(x.device)
    colsum = ws = None
    if want_colsum:
        if gate is None and live_in is None:
            raise ValueError("want_colsum needs a gate")
        colsum = torch.empty(d, device=x.device, dtype=torch.float32)
        ws = torch.empty(int(L.ltgnn_spmm_ws_floats(h)), device=x.device, dtype=torch.float32)
    if vals is not None:
        tok = _inst.begin("spmm_vals_bwd" if transpose else "spmm_vals_fwd")
        _lib.check(L.ltgnn_spmm_fused_vals(h, int(bool(transpose)), b, d, x.data_ptr(), y.data_ptr(), vals.data_ptr(),
                                           0 if vals.shape[0] == 1 else graph.nnz, int(algo),
                                           None if bias is None else bias.data_ptr(), int(relu), float(drop_p),
                                           int(drop_seed) & (2**64 - 1), None if gate is None else gate.data_ptr(),
                                           float(gate_scale), None if colsum is None else colsum.data_ptr(),
                                           None if ws is None else ws.data_ptr(),
                                           None if live_out is None else live_out.data_ptr(),
                                           None if live_in is None else live_in.data_ptr(), _stream(x)))
        _inst.end(tok)
        return (y, colsum) if want_colsum else y
    tok = _inst.begin("spmm_fused_bwd" if transpose else "spmm_fused_fwd")
    _lib.check(L.ltgnn_spmm_fused(h, int(bool(transpose)), b, d, x.data_ptr(), y.data_ptr(),
                                  None if bias is None else bias.data_ptr(), int(relu), float(drop_p),
                                  int(drop_seed) & (2**64 - 1), None if gate is None else gate.data_ptr(),
                                  float(gate_scale), None if colsum is None else colsum.data_ptr(),
                                  None if ws is None else ws.data_ptr(),
                                  None if live_out is None else live_out.data_ptr(),
                                  None if live_in is None else live_in.data_ptr(), _stream(x)))
    _inst.end(tok)
    return (y, colsum) if want_colsum else y


# ----------------------------------------------------------------------------------------------
# shape support predicates (mirrors of the checks in csrc/).  Channel counts off the kernels' granularity are zero-padded
# to it (operator-level GCNConv); anything larger raises -- no cuBLAS / eager-torch path anywhere
# ----------------------------------------------------------------------------------------------
_SMEM_LIMIT = 232448  # sm_100: 227 KB opt-in dynamic shared memory per block


def _linear_tc_ok(k: int, n: int) -> bool:
    if k % 32 or n % 16 or not (0 < k <= 256) or not (0 < n <= 256):
        return False
    # >= 2 ring stages and the 4 epilogue transposition patches next to the resident weight
    return 1024 + 2 * 32768 + 4 * 4096 + 2 * n * k * 4 <= _SMEM_LIMIT


def _wgrad_ok(do: int, di: int) -> bool:
    if do % 8 or di % 8:
        return False
    tpg = (do // 8) * (di // 8)
    return tpg <= 256 and 256 % tpg == 0


def _staged_ok(graph: PipeGraph, d: int) -> bool:
    if d % 32:
        return False
    n = graph.num_nodes
    boxes = (n + 255) // 256
    rows = (n + boxes - 1) // boxes
    stage = boxes * rows * 128
    off = ((128 + 4 * (n + 1) + 15) // 16 * 16 + 8 * graph.nnz + 127) // 128 * 128
    return _SMEM_LIMIT - 128 - off >= stage


def _pad_cols(t: torch.Tensor, cols: int) -> torch.Tensor:
    """Zero-pad the last dimension to ``cols`` (a copy; no arithmetic)."""
    if t.shape[-1] == cols:
        return t
    out = torch.zeros(*t.shape[:-1], cols, device=t.device, dtype=t.dtype)
    out[..., : t.shape[-1]] = t
    return out


def _linear_any(x, weight, transposed=False):
    """``x @ weight.T`` (or ``x @ weight``) for any channel counts up to 256: shapes off the tensor-core kernel's
    granularity (K % 32, N % 16) are zero-padded to it -- the operator-level ``GCNConv`` drop-in takes the channel counts PyG
    takes, and there is no library GEMM behind it."""
    k = x.shape[-1]
    n = weight.shape[1] if transposed else weight.shape[0]
    if _linear_tc_ok(k, n):
        return linear_tc(x, weight, transposed=transposed)
    kp, np_ = (k + 31) // 32 * 32, (n + 15) // 16 * 16
    if not _linear_tc_ok(kp, np_):
        raise ValueError(f"linear: {k} -> {n} channels exceed what the sm_100a kernel holds resident (<= 256, K*N*8 bytes of "
                         "shared memory); there is no library fallback")
    w = weight.detach()
    wp = torch.zeros((kp, np_) if transposed else (np_, kp), device=w.device, dtype=w.dtype)
    wp[: w.shape[0], : w.shape[1]] = w
    return linear_tc(_pad_cols(x, kp), wp, transposed=transposed)[..., :n].contiguous()


def wgrad(g: torch.Tensor, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dW[Do, Di] = sum_rows g[row, :]^T x[row, :]; g: (..., Do), x: (..., Di), same leading shape.
    ``out``: a contiguous (Do, Di) fp32 CUDA tensor to write into."""
    _check_act(g, "g")
    _check_act(x, "x")
    do, di = g.shape[-1], x.shape[-1]
    m = g.numel() // do
    if x.numel() // di != m:
        raise ValueError("wgrad: row counts differ")
    L = _lib.load()
    dev = _dev_index(g)
    if out is not None:
        _check_act(out, "out")
        if tuple(out.shape) != (do, di):
            raise ValueError(f"out must be {(do, di)}")
    dw = torch.empty(do, di, device=g.device, dtype=torch.float32) if out is None else out
    if do in (64, 128) and di % 32 == 0 and 0 < di <= 192 and m > 0:
        ws = torch.empty(int(L.ltgnn_tgrad_ws_floats(dev, di)), device=g.device, dtype=torch.float32)
        tok = _inst.begin("wgrad_tc")
        _lib.check(L.ltgnn_wgrad_tc(dev, m, do, di, g.data_ptr(), x.data_ptr(), dw.data_ptr(), 0, ws.data_ptr(),
                                    _stream(g)))
        _inst.end(tok)
        return dw
    if not _wgrad_ok(do, di):
        # off-granularity channel counts (operator-level GCNConv only): zero-pad to the tensor-core kernel's shapes
        dop, dip = (64 if do <= 64 else 128), (di + 31) // 32 * 32
        if do > 128 or dip > 192 or m == 0:
            raise ValueError(f"wgrad: ({do}, {di}) not built (<= 128 x 192 channels); there is no library fallback")
        res = wgrad(_pad_cols(g.reshape(m, do), dop), _pad_cols(x.reshape(m, di), dip))[:do, :di].contiguous()
        return res if out is None else out.copy_(res)
    ws = torch.empty(int(L.ltgnn_wgrad_ws_floats(dev, do, di)), device=g.device, dtype=torch.float32)
    tok = _inst.begin("wgrad")
    _lib.check(L.ltgnn_wgrad(dev, m, do, di, g.data_ptr(), x.data_ptr(), dw.data_ptr(), 0, ws.data_ptr(), _stream(g)))
    _inst.end(tok)
    return dw


# One kernel per GCN layer forward (csrc/gcn_layer.cu) where the shape allows; False = the two-launch path
# (ltgnn_linear + ltgnn_spmm_fused), which computes the same bits and stays as the cross-check.
FUSED_LAYER = True

# Node init's backward straight from the first layer's aggregated gradient (ltgnn_node_init_bwd_from_layer: the input
# gradient of that layer is never stored) where the shapes allow; False = ltgnn_linear + ltgnn_node_init_bwd, which give
# d h_s and d sensor_to_node.weight in the same bits and d sensor_to_node.bias up to summation order -- the cross-check.
FUSED_NODE_INIT_BWD = True


def gcn_layer_supported(graph: PipeGraph, x: torch.Tensor, weight: torch.Tensor) -> bool:
    return bool(_lib.load().ltgnn_gcn_layer_supported(graph.handle(x.device), int(weight.shape[1]), int(weight.shape[0])))


def gcn_layer_fwd(graph: PipeGraph, x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
                  relu: bool = False, drop_p: float = 0.0, drop_seed: int = 0,
                  live_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw fused layer forward (see ltgnn_gcn_layer_fwd): ``dropout(relu(A_hat (x W^T) + bias))`` in one kernel.
    x (B, N, K) fp32 CUDA, weight (D, K); returns (B, N, D)."""
    _check_act(x, "x")
    _check_act(weight, "weight")
    n, k, d = graph.num_nodes, x.shape[-1], weight.shape[0]
    if weight.shape[1] != k or x.numel() % (n * k) != 0:
        raise ValueError(f"x {tuple(x.shape)} / weight {tuple(weight.shape)} do not fit a {n}-node graph")
    b = x.numel() // (n * k)
    if live_out is not None and (live_out.dtype != torch.int32 or tuple(live_out.shape) != (b, d // 32, n)):
        raise ValueError(f"live_out must be int32 of shape {(b, d // 32, n)}")
    y = torch.empty(b, n, d, device=x.device, dtype=torch.float32)
    L = _lib.load()
    tok = _inst.begin("gcn_layer_fwd")
    _lib.check(L.ltgnn_gcn_layer_fwd(graph.handle(x.device), b, k, d, x.data_ptr(), weight.data_ptr(),
                                     None if bias is None else bias.data_ptr(), int(relu), float(drop_p),
                                     int(drop_seed) & (2**64 - 1), y.data_ptr(),
                                     None if live_out is None else live_out.data_ptr(), _stream(x)))
    _inst.end(tok)
    return y


def node_init_fwd(h_s, slot, num_nodes, weight, bias, drop_p=0.0, drop_seed=0, live_out=None):
    """Raw node-feature initialisation (see ltgnn_node_init_fwd).  h_s (B,S,ds) -> (B,N,D).
    ``live_out``: optional int32 (B, D/32, N) tensor that receives ``x0 > 0`` as one bit per element."""
    _check_act(h_s, "h_s")
    _check_act(weight, "weight")
    _check_act(bias, "bias")
    b, s, ds = h_s.shape
    d = weight.shape[0]
    x0 = torch.empty(b, num_nodes, d, device=h_s.device, dtype=torch.float32)
    L = _lib.load()
    tok = _inst.begin("node_init_fwd")
    _lib.check(L.ltgnn_node_init_fwd(_dev_index(h_s), b, num_nodes, s, ds, d, h_s.data_ptr(), slot.data_ptr(),
                                     weight.data_ptr(), bias.data_ptr(), float(drop_p), int(drop_seed) & (2**64 - 1),
                                     x0.data_ptr(), None if live_out is None else live_out.data_ptr(), _stream(h_s)))
    _inst.end(tok)
    return x0


def node_init_bwd(h_s, slot, weight, dx0, x0, gate_scale, live=None):
    """Raw backward of node_init: returns (dh_s, dW, dbias); dx0 is gated by (x0 > 0) * gate_scale.
    ``live``: the gate as one bit per element (from node_init_fwd's ``live_out``); x0 is then not read."""
    for t, nm in ((h_s, "h_s"), (weight, "weight"), (dx0, "dx0"), (x0, "x0")):
        _check_act(t, nm)
    b, s, ds = h_s.shape
    n, d = x0.shape[1], x0.shape[2]
    if d not in (64, 128) or ds % 32:
        raise ValueError(f"node_init_bwd: node width {d} / sensor width {ds} not built (64 or 128 / a multiple of 32); the "
                         "sm_100a kernels have no library fallback")
    L = _lib.load()
    dev = _dev_index(h_s)
    dhs = torch.empty_like(h_s)
    dw = torch.empty_like(weight)
    db = torch.empty(d, device=h_s.device, dtype=torch.float32)
    ws = torch.empty(int(L.ltgnn_node_init_ws_floats(dev, b, s, ds, d)), device=h_s.device, dtype=torch.float32)
    tok = _inst.begin("node_init_bwd")
    _lib.check(L.ltgnn_node_init_bwd(dev, b, n, s, ds, d, h_s.data_ptr(), slot.data_ptr(), weight.data_ptr(),
                                     dx0.data_ptr(), x0.data_ptr(), None if live is None else live.data_ptr(),
                                     float(gate_scale), dhs.data_ptr(), dw.data_ptr(), db.data_ptr(), ws.data_ptr(),
                                     _stream(h_s)))
    _inst.end(tok)
    return dhs, dw, db


def node_init_bwd_from_layer(h_s, slot, weight, gz, w1, live, gate_scale):
    """node_init_bwd for dx0 = gz @ w1, the input gradient of the first GCN layer, without forming dx0 (see
    ltgnn_node_init_bwd_from_layer): gz (B, N, K) the layer's aggregated output gradient, w1 (K, D) its weight,
    ``live`` node_init_fwd's ``live_out`` (required).  Returns (dh_s, dW, dbias); dh_s and dW carry the bits of
    ``node_init_bwd(h_s, slot, weight, gz @ w1, x0, gate_scale, live=live)``, dbias differs by summation order."""
    for t, nm in ((h_s, "h_s"), (weight, "weight"), (gz, "gz"), (w1, "w1")):
        _check_act(t, nm)
    b, s, ds = h_s.shape
    n, k = gz.shape[1], gz.shape[2]
    d = w1.shape[1]
    if d not in (64, 128) or ds % 32 or k % 32 or k > 128:
        raise ValueError(f"node_init_bwd_from_layer: node width {d} / sensor width {ds} / layer width {k} not built (64 or "
                         "128 / a multiple of 32 / a multiple of 32 up to 128); the sm_100a kernels have no library fallback")
    if tuple(gz.shape) != (b, n, k) or tuple(w1.shape) != (k, d) or tuple(weight.shape) != (d, ds + 1):
        raise ValueError(f"gz {tuple(gz.shape)} / w1 {tuple(w1.shape)} / weight {tuple(weight.shape)} do not fit h_s "
                         f"{tuple(h_s.shape)}")
    if live is None or live.dtype != torch.int32 or tuple(live.shape) != (b, d // 32, n):
        raise ValueError(f"live must be int32 of shape {(b, d // 32, n)}")
    L = _lib.load()
    dev = _dev_index(h_s)
    dhs = torch.empty_like(h_s)
    dw = torch.empty_like(weight)
    db = torch.empty(d, device=h_s.device, dtype=torch.float32)
    ws = torch.empty(int(L.ltgnn_node_init_ws_floats(dev, b, s, ds, d)), device=h_s.device, dtype=torch.float32)
    tok = _inst.begin("node_init_bwd")
    _lib.check(L.ltgnn_node_init_bwd_from_layer(dev, b, n, s, ds, d, k, h_s.data_ptr(), slot.data_ptr(),
                                                weight.data_ptr(), gz.data_ptr(), w1.data_ptr(), live.data_ptr(),
                                                float(gate_scale), dhs.data_ptr(), dw.data_ptr(), db.data_ptr(),
                                                ws.data_ptr(), _stream(h_s)))
    _inst.end(tok)
    return dhs, dw, db


# ----------------------------------------------------------------------------------------------
# per-call edge weights: PyG's gcn_norm on the device and the gradient with respect to the adjacency values
# ----------------------------------------------------------------------------------------------
def _check_edge_weight(graph: PipeGraph, w: torch.Tensor, b: int, name: str = "edge_weight") -> None:
    if not isinstance(w, torch.Tensor):
        raise ValueError(f"{name} must be a tensor")
    e = graph.num_edges
    if not (tuple(w.shape) == (e,) or (w.dim() == 2 and tuple(w.shape) == (b, e))):
        raise ValueError(f"{name} must be ({e},) (shared by every window) or ({b}, {e}) (one row per window), "
                         f"got {tuple(w.shape)}")
    if not w.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (libltgnn has no CPU path)")
    if w.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, got {w.dtype}")


def _check_edge_mask(graph: PipeGraph, m: torch.Tensor, b: int) -> None:
    _check_edge_weight(graph, m, b, "edge_mask")
    if not m.is_contiguous():
        raise ValueError("edge_mask must be contiguous")


def edge_norm(graph: PipeGraph, w: torch.Tensor):
    """Raw device normalisation (see ltgnn_edge_norm_fwd): edge weights (E,) or (Bw, E) in ``edge_index`` order ->
    ``(vals, t_vals, dis)``: the entry values of A_hat and of A_hat^T, (1 or Bw, nnz) each, and deg^-1/2 (1 or Bw, N)."""
    _check_act(w, "edge_weight")
    w2 = w.view(1, -1) if w.dim() == 1 else w
    if w2.dim() != 2 or w2.shape[1] != graph.num_edges:
        raise ValueError(f"edge_weight rows must hold {graph.num_edges} values, got {tuple(w.shape)}")
    bw = w2.shape[0]
    ent, t_ent, _ = graph.edge_maps(w.device)
    vals = torch.empty(bw, graph.nnz, device=w.device, dtype=torch.float32)
    t_vals = torch.empty_like(vals)
    dis = torch.empty(bw, graph.num_nodes, device=w.device, dtype=torch.float32)
    tok = _inst.begin("edge_norm_fwd")
    _lib.check(_lib.load().ltgnn_edge_norm_fwd(graph.handle(w.device), bw, graph.num_edges, w2.data_ptr(), graph.num_edges,
                                               ent.data_ptr(), t_ent.data_ptr(), dis.data_ptr(), vals.data_ptr(),
                                               t_vals.data_ptr(), _stream(w)))
    _inst.end(tok)
    return vals, t_vals, dis


def edge_norm_bwd(graph: PipeGraph, w: torch.Tensor, dis: torch.Tensor, dvals: torch.Tensor) -> torch.Tensor:
    """Raw backward of :func:`edge_norm`: d vals (Bw, nnz) in A_hat order -> d edge_weight of ``w``'s shape."""
    w2 = w.view(1, -1) if w.dim() == 1 else w
    dvals = dvals.contiguous()
    ent, t_ent, t_perm = graph.edge_maps(w.device)
    bw = w2.shape[0]
    ddeg = torch.empty(bw, graph.num_nodes, device=w.device, dtype=torch.float32)
    dw = torch.empty(bw, graph.num_edges, device=w.device, dtype=torch.float32)
    tok = _inst.begin("edge_norm_bwd")
    _lib.check(_lib.load().ltgnn_edge_norm_bwd(graph.handle(w.device), bw, graph.num_edges, w2.data_ptr(), graph.num_edges,
                                               ent.data_ptr(), t_ent.data_ptr(), t_perm.data_ptr(), dis.data_ptr(),
                                               dvals.data_ptr(), ddeg.data_ptr(), dw.data_ptr(), _stream(w)))
    _inst.end(tok)
    return dw.view(w.shape)


def gcn_adj_grad(graph: PipeGraph, g: torch.Tensor, xw: torch.Tensor, gate: Optional[torch.Tensor] = None,
                 live_in: Optional[torch.Tensor] = None, gate_scale: float = 1.0, out: Optional[torch.Tensor] = None,
                 shared: bool = False, accumulate: bool = False) -> torch.Tensor:
    """Raw adjacency-value gradient (see ltgnn_gcn_adj_grad): ``dA[b, k] = <Gg[b, row_k], xw[b, col_k]>`` over A_hat's
    entries, Gg = g gated by ``gate`` / ``live_in`` times ``gate_scale``.  Returns (B, nnz), or with ``shared`` the sum
    over windows (1, nnz); ``accumulate`` adds into ``out``."""
    _check_act(g, "g")
    _check_act(xw, "xw")
    n, d = graph.num_nodes, g.shape[-1]
    if xw.shape != g.shape or g.numel() % (n * d) != 0:
        raise ValueError(f"g {tuple(g.shape)} and xw {tuple(xw.shape)} must be the same whole number of {n}-node graphs")
    b = g.numel() // (n * d)
    if gate is not None:
        _check_act(gate, "gate")
    rows = 1 if shared else b
    if out is None:
        out = torch.empty(rows, graph.nnz, device=g.device, dtype=torch.float32)
    elif tuple(out.shape) != (rows, graph.nnz):
        raise ValueError(f"out must be {(rows, graph.nnz)}")
    scratch = torch.empty(b, graph.nnz, device=g.device, dtype=torch.float32) if shared else out
    tok = _inst.begin("gcn_adj_grad")
    _lib.check(_lib.load().ltgnn_gcn_adj_grad(graph.handle(g.device), b, d, g.data_ptr(),
                                              None if gate is None else gate.data_ptr(),
                                              None if live_in is None else live_in.data_ptr(), float(gate_scale),
                                              xw.data_ptr(), scratch.data_ptr(), int(bool(accumulate)),
                                              out.data_ptr() if shared else None, _stream(g)))
    _inst.end(tok)
    return out


class _EdgeNorm(torch.autograd.Function):
    """edge_weight -> (vals, t_vals): the normalised entry values in both orders.  The layers report the gradient of
    the adjacency through ``vals`` (A_hat order); ``t_vals`` is the same matrix transposed, for their backward."""

    @staticmethod
    def forward(ctx, w, graph):
        w = w.contiguous()
        vals, t_vals, dis = edge_norm(graph, w)
        ctx.mark_non_differentiable(t_vals)
        ctx.save_for_backward(w, dis)
        ctx.graph = graph
        return vals, t_vals

    @staticmethod
    def backward(ctx, dvals, _dt_vals):
        w, dis = ctx.saved_tensors
        if dvals is None:
            return None, None
        return edge_norm_bwd(ctx.graph, w, dis, dvals), None


def edge_mask_fwd(graph: PipeGraph, mask: torch.Tensor, base: Optional[torch.Tensor] = None,
                  t_base: Optional[torch.Tensor] = None):
    """Raw message mask (see ltgnn_edge_mask_fwd): mask (E,) or (Bm, E) in ``edge_index`` order on the entry values
    ``base`` / ``t_base`` ((1 or Bv, nnz) in A_hat / A_hat^T order, e.g. :func:`edge_norm`'s) or on the graph's own
    (both ``None``) -> masked ``(vals, t_vals)``, (max(Bm, Bv), nnz) each; gcn_norm's self loops keep factor 1."""
    _check_act(mask, "edge_mask")
    m2 = mask.view(1, -1) if mask.dim() == 1 else mask
    if m2.dim() != 2 or m2.shape[1] != graph.num_edges:
        raise ValueError(f"edge_mask rows must hold {graph.num_edges} values, got {tuple(mask.shape)}")
    rows = m2.shape[0]
    if base is not None:
        _check_act(base, "base")
        _check_act(t_base, "t_base")
        if base.shape != t_base.shape or base.dim() != 2 or base.shape[1] != graph.nnz:
            raise ValueError(f"base and t_base must both be (rows, {graph.nnz})")
        if 1 not in (rows, base.shape[0]) and rows != base.shape[0]:
            raise ValueError(f"edge_mask rows ({rows}) and base rows ({base.shape[0]}) do not broadcast")
        rows = max(rows, base.shape[0])
    ent, t_ent, _ = graph.edge_maps(mask.device)
    vals = torch.empty(rows, graph.nnz, device=mask.device, dtype=torch.float32)
    t_vals = torch.empty_like(vals)
    tok = _inst.begin("edge_mask_fwd")
    _lib.check(_lib.load().ltgnn_edge_mask_fwd(graph.handle(mask.device), rows, graph.num_edges, m2.data_ptr(),
                                               0 if m2.shape[0] == 1 else graph.num_edges,
                                               None if base is None else base.data_ptr(),
                                               None if t_base is None else t_base.data_ptr(),
                                               0 if base is None or base.shape[0] == 1 else graph.nnz, ent.data_ptr(),
                                               t_ent.data_ptr(), vals.data_ptr(), t_vals.data_ptr(), _stream(mask)))
    _inst.end(tok)
    return vals, t_vals


def edge_mask_bwd(graph: PipeGraph, mask: torch.Tensor, dvals: torch.Tensor, base: Optional[torch.Tensor] = None,
                  want_base: bool = False):
    """Raw backward of :func:`edge_mask_fwd`: d vals (rows, nnz) in A_hat order -> ``(d mask, d base)`` of the shapes of
    ``mask`` and ``base`` (``d base`` only with ``want_base``, else ``None``); an operand with one row shared by
    several output rows gets the sum over them."""
    m2 = mask.view(1, -1) if mask.dim() == 1 else mask
    dvals = dvals.contiguous()
    rows, e, nnz = dvals.shape[0], graph.num_edges, graph.nnz
    dev = mask.device
    dmask = torch.empty(rows, e, device=dev, dtype=torch.float32)
    dmask_sum = torch.empty(1, e, device=dev, dtype=torch.float32) if m2.shape[0] < rows else None
    dbase = dbase_sum = None
    if want_base:
        dbase = torch.empty(rows, nnz, device=dev, dtype=torch.float32)
        dbase_sum = torch.empty(1, nnz, device=dev, dtype=torch.float32) if base.shape[0] < rows else None
    ent, _, _ = graph.edge_maps(dev)
    tok = _inst.begin("edge_mask_bwd")
    _lib.check(_lib.load().ltgnn_edge_mask_bwd(graph.handle(dev), rows, e, m2.data_ptr(), 0 if m2.shape[0] == 1 else e,
                                               None if base is None else base.data_ptr(),
                                               0 if base is None or base.shape[0] == 1 else nnz, ent.data_ptr(),
                                               dvals.data_ptr(), dmask.data_ptr(),
                                               None if dmask_sum is None else dmask_sum.data_ptr(),
                                               None if dbase is None else dbase.data_ptr(),
                                               None if dbase_sum is None else dbase_sum.data_ptr(), _stream(dvals)))
    _inst.end(tok)
    dmask = (dmask if dmask_sum is None else dmask_sum).view(mask.shape)
    if want_base:
        dbase = (dbase if dbase_sum is None else dbase_sum).view(base.shape)
    return dmask, dbase


class _EdgeMask(torch.autograd.Function):
    """(edge_mask, vals, t_vals) -> masked (vals, t_vals): PyG's explainer mask on each message after the normalisation.
    ``vals`` / ``t_vals`` ``None``: the graph's own values.  Differentiable in the mask and in ``vals`` (and so, through
    :class:`_EdgeNorm`, in ``edge_weight``)."""

    @staticmethod
    def forward(ctx, mask, vals, t_vals, graph):
        mvals, mt_vals = edge_mask_fwd(graph, mask, vals, t_vals)
        ctx.mark_non_differentiable(mt_vals)
        ctx.save_for_backward(mask, vals)
        ctx.graph = graph
        return mvals, mt_vals

    @staticmethod
    def backward(ctx, dvals, _dt_vals):
        mask, vals = ctx.saved_tensors
        if dvals is None:
            return None, None, None, None
        dmask, dbase = edge_mask_bwd(ctx.graph, mask, dvals, vals, want_base=ctx.needs_input_grad[1])
        return dmask, dbase, None, None


def normalized_edge_values(graph: PipeGraph, edge_weight: Optional[torch.Tensor], b: int,
                           edge_mask: Optional[torch.Tensor] = None):
    """Differentiable ``(vals, t_vals)`` of ``edge_weight`` ((E,) or (b, E); ``None``: the graph's own normalisation)
    for the weighted layers, each message scaled by ``edge_mask`` ((E,) or (b, E)) when one is given.  Both are
    validated before anything is launched."""
    if edge_weight is not None:
        _check_edge_weight(graph, edge_weight, b)
    if edge_mask is not None:
        _check_edge_mask(graph, edge_mask, b)
    vals = t_vals = None
    if edge_weight is not None:
        vals, t_vals = _EdgeNorm.apply(edge_weight, graph)
    if edge_mask is not None:
        vals, t_vals = _EdgeMask.apply(edge_mask, vals, t_vals, graph)
    return vals, t_vals


def explain_step(g: torch.Tensor, m: torch.Tensor, s: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
                 hard: torch.Tensor, n_hard: torch.Tensor, step: torch.Tensor, record: bool, lr: float = 0.01,
                 edge_size: float = 0.005, edge_ent: float = 1.0, betas=(0.9, 0.999), eps: float = 1e-8) -> None:
    """One GNNExplainer epoch on (B, E) mask logits, in place (see ltgnn_explain_step): ``g`` = d loss / d ``s``,
    ``s`` = sigmoid(``m``); Adam state ``exp_avg`` / ``exp_avg_sq`` and the int32 step count ``step`` (1,) on the device;
    ``record`` (epoch 0): no regulariser, writes the hard mask ``hard`` (bool (B, E)) and its counts ``n_hard``
    (int32 (B,)); later epochs regularise on them."""
    for t, nm in ((g, "g"), (m, "m"), (s, "s"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _check_act(t, nm)
        if t.dim() != 2 or t.shape != m.shape:
            raise ValueError(f"explain_step: {nm} must be (B, E) like m {tuple(m.shape)}")
    b, e = m.shape
    if hard.dtype != torch.bool or hard.shape != m.shape or not hard.is_contiguous():
        raise ValueError("explain_step: hard must be a contiguous bool tensor shaped like m")
    for t, nm, shape in ((n_hard, "n_hard", (b,)), (step, "step", (1,))):
        if t.dtype != torch.int32 or tuple(t.shape) != shape or not t.is_cuda:
            raise ValueError(f"explain_step: {nm} must be an int32 CUDA tensor of shape {shape}")
    tok = _inst.begin("explain_step")
    _lib.check(_lib.load().ltgnn_explain_step(_dev_index(m), b, e, g.data_ptr(), m.data_ptr(), s.data_ptr(),
                                              exp_avg.data_ptr(), exp_avg_sq.data_ptr(), hard.data_ptr(), n_hard.data_ptr(),
                                              step.data_ptr(), float(lr), float(betas[0]), float(betas[1]), float(eps),
                                              float(edge_size), float(edge_ent), int(bool(record)), _stream(m)))
    _inst.end(tok)


# ----------------------------------------------------------------------------------------------
# PGExplainer's edge network (csrc/pg_explain.cu): [P | Q] = z [W1a; W1b]^T on the tensor cores, then per edge
# sigmoid(w2 . relu(P[src] + Q[dst] + b1) + b2), with PyG's concrete sample in training
# ----------------------------------------------------------------------------------------------
PG_HIDDEN = 64  # PyG's PGExplainer MLP: Linear(2D, 64) -> ReLU -> Linear(64, 1)


def pg_edge_index(edge_index: torch.Tensor, num_nodes: int, device: torch.device) -> tuple:
    """``(src, dst, out_ptr, out_edge, in_ptr, in_edge)`` int32 on ``device``: each edge's end nodes, and the edges
    grouped by source and by target, ascending within a node -- what ltgnn_pg_edge_fwd / _bwd read.  Host work, once
    per graph."""
    ei = edge_index.detach().cpu().numpy().astype(np.int64)
    if ei.ndim != 2 or ei.shape[0] != 2 or (ei.size and (ei.min() < 0 or ei.max() >= num_nodes)):
        raise ValueError(f"edge_index must be (2, E) with node indices in [0, {num_nodes})")
    out = [ei[0], ei[1]]
    for row in (ei[0], ei[1]):
        ptr = np.zeros(num_nodes + 1, dtype=np.int64)
        np.cumsum(np.bincount(row, minlength=num_nodes), out=ptr[1:])
        out += [ptr, np.argsort(row, kind="stable")]
    return tuple(torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(device) for a in out)


def _check_pg_mlp(d: int, w1, b1, w2, b2) -> None:
    want = ((w1, (PG_HIDDEN, 2 * d), "mlp.0.weight"), (b1, (PG_HIDDEN,), "mlp.0.bias"), (w2, (1, PG_HIDDEN), "mlp.2.weight"),
            (b2, (1,), "mlp.2.bias"))
    for t, shape, nm in want:
        _check_act(t, nm)
        if tuple(t.shape) != shape:
            raise ValueError(f"{nm} must be {shape} for node width {d}, got {tuple(t.shape)}")


def pg_edge_fwd(pq: torch.Tensor, idx: tuple, b1: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor,
                inv_t: Optional[torch.Tensor] = None, bias: float = 0.01, seed: int = 0,
                uniform: Optional[torch.Tensor] = None):
    """Raw edge network (see ltgnn_pg_edge_fwd) on ``pq`` (B, N, 128) = [P | Q] with ``idx`` from
    :func:`pg_edge_index`.  ``inv_t`` ``None``: returns the mask sigmoid(logit) (B, E).  ``inv_t`` (a one-element
    device tensor 1 / T): returns ``(mask, s, gate)`` of the concrete sample, ``uniform`` (B, E) receiving the draws."""
    b, n = pq.shape[0], pq.shape[1]
    e = idx[0].numel()
    mask = torch.empty(b, e, device=pq.device, dtype=torch.float32)
    s = gate = None
    if inv_t is not None:
        s = torch.empty_like(mask)
        gate = torch.empty(b, e, 2, device=pq.device, dtype=torch.int32)
    tok = _inst.begin("pg_edge_fwd")
    _lib.check(_lib.load().ltgnn_pg_edge_fwd(_dev_index(pq), b, n, e, idx[0].data_ptr(), idx[1].data_ptr(), pq.data_ptr(),
                                             b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                                             None if inv_t is None else inv_t.data_ptr(), float(bias),
                                             int(seed) & (2**64 - 1), mask.data_ptr(), None if s is None else s.data_ptr(),
                                             None if gate is None else gate.data_ptr(),
                                             None if uniform is None else uniform.data_ptr(), _stream(pq)))
    _inst.end(tok)
    return mask if inv_t is None else (mask, s, gate)


def pg_edge_bwd(pq: torch.Tensor, idx: tuple, b1: torch.Tensor, w2: torch.Tensor, inv_t: torch.Tensor,
                mask: torch.Tensor, dmask: torch.Tensor, gate: torch.Tensor):
    """Raw backward of :func:`pg_edge_fwd` in training (see ltgnn_pg_edge_bwd): d mask (B, E) -> ``(R, dparams)``,
    R = d[P | Q] (B, N, 128) and dparams (129,) = d b1 | d w2 | d b2."""
    b, n = pq.shape[0], pq.shape[1]
    e = idx[0].numel()
    dev = _dev_index(pq)
    L = _lib.load()
    r = torch.empty_like(pq)
    dparams = torch.empty(2 * PG_HIDDEN + 1, device=pq.device, dtype=torch.float32)
    ws = torch.empty(int(L.ltgnn_pg_edge_bwd_ws_floats(dev)), device=pq.device, dtype=torch.float32)
    tok = _inst.begin("pg_edge_bwd")
    _lib.check(L.ltgnn_pg_edge_bwd(dev, b, n, e, idx[2].data_ptr(), idx[3].data_ptr(), idx[4].data_ptr(),
                                   idx[5].data_ptr(), idx[1].data_ptr(), pq.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                                   inv_t.data_ptr(), mask.data_ptr(), dmask.data_ptr(), gate.data_ptr(), r.data_ptr(),
                                   dparams.data_ptr(), ws.data_ptr(), _stream(pq)))
    _inst.end(tok)
    return r, dparams


class _PgProject(torch.autograd.Function):
    """(z, W1) -> [P | Q] = z [W1a; W1b]^T, (B, N, 128): PyG's first MLP layer on [z[src] | z[dst]] without its bias,
    factored per node (W1a acts on the source half).  Backward: d W1 only (z is the frozen detector's embedding), from
    R^T z on the tensor cores, re-laid out as PyG's (64, 2D)."""

    @staticmethod
    def forward(ctx, z, w1):
        d = z.shape[-1]
        w_stack = torch.cat([w1[:, :d], w1[:, d:]], 0).contiguous()
        ctx.save_for_backward(z)
        return linear_tc(z, w_stack)

    @staticmethod
    def backward(ctx, dpq):
        (z,) = ctx.saved_tensors
        dw = wgrad(dpq.contiguous(), z)
        return None, torch.cat([dw[:PG_HIDDEN], dw[PG_HIDDEN:]], 1)


class _PgEdge(torch.autograd.Function):
    """([P | Q], b1, w2, b2) -> (mask, s) of the concrete sample; differentiable in the mask (s is returned for
    inspection).  Backward: ltgnn_pg_edge_bwd -> d[P | Q], d b1, d w2, d b2."""

    @staticmethod
    def forward(ctx, pq, b1, w2, b2, idx, inv_t, bias, seed):
        uniform = None
        if DEBUG_CAPTURE is not None:
            uniform = torch.empty(pq.shape[0], idx[0].numel(), device=pq.device, dtype=torch.float32)
            DEBUG_CAPTURE["pg_uniform"] = uniform
        mask, s, gate = pg_edge_fwd(pq, idx, b1, w2, b2, inv_t, bias, seed, uniform)
        if DEBUG_CAPTURE is not None:
            DEBUG_CAPTURE["pg_gate"] = gate
        ctx.mark_non_differentiable(s)
        ctx.save_for_backward(pq, b1, w2, inv_t, mask, gate)
        ctx.idx = idx
        return mask, s

    @staticmethod
    def backward(ctx, dmask, _ds):
        pq, b1, w2, inv_t, mask, gate = ctx.saved_tensors
        if dmask is None:
            return (None,) * 8
        r, dp = pg_edge_bwd(pq, ctx.idx, b1, w2, inv_t, mask, dmask.contiguous(), gate)
        return r, dp[:PG_HIDDEN], dp[PG_HIDDEN:2 * PG_HIDDEN].view(1, PG_HIDDEN), dp[2 * PG_HIDDEN:], None, None, None, None


def pg_edge_mask(z: torch.Tensor, idx: tuple, w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor,
                 inv_t: Optional[torch.Tensor] = None, bias: float = 0.01, seed: int = 0):
    """PGExplainer's edge mask from node embeddings ``z`` (B, N, D) over the edges of ``idx`` (:func:`pg_edge_index`)
    with the MLP ``Linear(2D, 64) -> ReLU -> Linear(64, 1)`` (``w1`` (64, 2D), ``b1`` (64,), ``w2`` (1, 64), ``b2``
    (1,)).  ``inv_t`` ``None``: explaining, returns sigmoid(logit) (B, E).  ``inv_t`` (one-element CUDA tensor, 1 / T):
    training, returns ``(mask, s)`` with s = (log eps - log(1 - eps) + logit) / T, eps = (1 - 2 bias) U + bias, mask =
    sigmoid(s), differentiable in the MLP's parameters.  Every input is checked before anything is launched."""
    _check_act(z, "z")
    if z.dim() != 3 or z.shape[-1] % 32 or not 0 < z.shape[-1] <= 192:
        raise ValueError(f"z must be (B, N, D) with D a multiple of 32 up to 192, got {tuple(z.shape)}")
    _check_pg_mlp(z.shape[-1], w1, b1, w2, b2)
    if len(idx) != 6 or any(t.dtype != torch.int32 or t.device != z.device for t in idx):
        raise ValueError("idx must be pg_edge_index(...) on the device of z")
    if idx[2].numel() != z.shape[1] + 1:
        raise ValueError(f"idx is for a {idx[2].numel() - 1}-node graph, z has {z.shape[1]} nodes")
    if inv_t is not None:
        _check_act(inv_t, "inv_t")
        if inv_t.numel() != 1:
            raise ValueError("inv_t must be a one-element tensor")
    if not 0.0 <= float(bias) <= 0.5:
        raise ValueError(f"bias must lie in [0, 0.5], got {bias}")
    pq = _PgProject.apply(z, w1)
    if inv_t is None:
        return pg_edge_fwd(pq, idx, b1, w2, b2)
    return _PgEdge.apply(pq, b1, w2, b2, idx, inv_t, float(bias), int(seed))


# ----------------------------------------------------------------------------------------------
# operator-level autograd: GCNConv  (reference call site models/detector.py:199)
# ----------------------------------------------------------------------------------------------
class _GcnConv(torch.autograd.Function):
    """out = A_hat (x W^T) + b, PyG's operation order; backward: G = A_hat^T dout (CSC gather),
    dW = G^T x, dx = G W, db = column sums of dout."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph, vals=None, t_vals=None):
        x = x.contiguous()
        n = graph.num_nodes
        xw = _linear_any(x, weight)
        xw3 = xw.view(-1, n, xw.shape[-1])
        if vals is not None:  # weighted adjacency: the per-call values (bias fused where the STAGED kernel takes it)
            fuse = bias is not None and _staged_ok(graph, xw.shape[-1])
            y = spmm_fused(graph, xw3, bias=bias if fuse else None, vals=vals)
            if bias is not None and not fuse:
                y += bias
        elif bias is not None and _staged_ok(graph, xw.shape[-1]):
            y = spmm_fused(graph, xw3, bias=bias)
        else:
            y = spmm(graph, xw3)
            if bias is not None:
                y += bias
        keep_xw = vals is not None and ctx.needs_input_grad[4]
        ctx.save_for_backward(x, weight, t_vals, xw3 if keep_xw else None)
        ctx.graph, ctx.has_bias, ctx.shared = graph, bias is not None, vals is not None and vals.shape[0] == 1
        return y.view(*x.shape[:-1], xw.shape[-1])

    @staticmethod
    def backward(ctx, dy):
        x, weight, t_vals, xw3 = ctx.saved_tensors
        dy = dy.contiguous()
        dy3 = dy.view(-1, ctx.graph.num_nodes, dy.shape[-1])
        if t_vals is None:
            g = spmm(ctx.graph, dy3, transpose=True).view(dy.shape)
        else:
            g = spmm_fused(ctx.graph, dy3, transpose=True, vals=t_vals).view(dy.shape)
        dw = wgrad(g, x) if ctx.needs_input_grad[1] else None
        dx = _linear_any(g, weight, transposed=True) if ctx.needs_input_grad[0] else None
        db = dy.reshape(-1, dy.shape[-1]).sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        dvals = gcn_adj_grad(ctx.graph, dy3, xw3, shared=ctx.shared) if xw3 is not None else None
        return dx, dw, db, None, dvals, None


def gcn_conv(x: torch.Tensor, graph: PipeGraph, weight: torch.Tensor, bias: Optional[torch.Tensor],
             edge_weight: Optional[torch.Tensor] = None, edge_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``A_hat (x W^T) + b`` -- the operator ``torch_geometric.nn.GCNConv.forward`` computes
    (reference call site models/detector.py:199).  x: (B, N, Din) or (B*N, Din), fp32 CUDA.  ``edge_weight``: PyG's
    per-edge weights in ``edge_index`` order, (E,) shared by every window or (B, E), normalised on the device
    (gcn_norm with self loops) on each call and differentiable; ``None`` runs the graph's own normalised adjacency.
    ``edge_mask``: PyG's explainer mask, same shapes, scaling each edge's message after the normalisation (the self
    loops gcn_norm adds are not masked; an input self loop's value has no effect); differentiable."""
    _check_act(x.contiguous(), "x")
    if edge_weight is None and edge_mask is None:
        return _GcnConv.apply(x, weight, bias, graph)
    b = x.numel() // (graph.num_nodes * x.shape[-1])
    vals, t_vals = normalized_edge_values(graph, edge_weight, b, edge_mask)
    return _GcnConv.apply(x, weight, bias, graph, vals, t_vals)


class _MeanPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = x.contiguous()
        b, n, d = x.shape
        pooled = torch.empty(b, d, device=x.device, dtype=torch.float32)
        L = _lib.load()
        tok = _inst.begin("mean_pool_fwd")
        _lib.check(L.ltgnn_mean_pool_fwd(_dev_index(x), b, n, d, x.data_ptr(), pooled.data_ptr(), _stream(x)))
        _inst.end(tok)
        ctx.shape = (b, n, d)
        return pooled

    @staticmethod
    def backward(ctx, dpooled):
        b, n, d = ctx.shape
        dpooled = dpooled.contiguous()
        dx = torch.empty(b, n, d, device=dpooled.device, dtype=torch.float32)
        L = _lib.load()
        tok = _inst.begin("mean_pool_bwd")
        _lib.check(L.ltgnn_mean_pool_bwd_fill(_dev_index(dpooled), b, n, d, dpooled.data_ptr(), dx.data_ptr(),
                                              _stream(dpooled)))
        _inst.end(tok)
        return dx


def mean_pool(x: torch.Tensor) -> torch.Tensor:
    """(B, N, D) -> (B, D): ``global_mean_pool`` for equal-sized graphs (detector.py:214-215)."""
    _check_act(x.contiguous(), "x")
    if x.shape[-1] % 4 or 256 % (x.shape[-1] // 4):
        raise ValueError(f"mean_pool: width {x.shape[-1]} not built (D / 4 must divide 256); no library fallback")
    return _MeanPool.apply(x)


def heads_supported(d: int, h: int) -> bool:
    return d == 64 and h == 128


def pipe_incidence(ends: torch.Tensor, num_nodes: int):
    """Node -> incident pipe-end lists of the class pipes, for the gather form of the pipe head's input gradient:
    ``(inc_ptr int32 [N+1], inc int32 [2P])`` on the device of ``ends``, entry = pipe << 1 | end, grouped by node in
    (pipe, end) order.  Host work, once per model (the detector caches it next to its other index tensors)."""
    e = ends.detach().cpu().numpy().astype(np.int64).reshape(-1)           # element 2 p + end = node of that pipe end
    order = np.argsort(e, kind="stable").astype(np.int32)
    cnt = np.bincount(e, minlength=num_nodes)
    ptr = np.zeros(num_nodes + 1, dtype=np.int32)
    np.cumsum(cnt, out=ptr[1:])
    return torch.from_numpy(ptr).to(ends.device), torch.from_numpy(order).to(ends.device)


class _Heads(torch.autograd.Function):
    """Pipe head partial logits + mean pool of the last node states as one autograd node, so that the backward
    writes d loss / d x exactly once: every node gathers the pool gradient and its incident pipe ends in a fixed order."""

    @staticmethod
    def forward(ctx, x, ends, inc_ptr, inc, w1, b1, w2, drop_p, training):
        x = x.contiguous()
        b, n, d = x.shape
        p_cnt, h = ends.shape[0], w1.shape[0]
        dev = _dev_index(x)
        L = _lib.load()
        p = float(drop_p) if training else 0.0
        need_grad = any(ctx.needs_input_grad)
        part = torch.empty(1, b, p_cnt, device=x.device, dtype=torch.float32)
        # saved for the backward: ONE BIT per hidden unit, the ReLU-and-dropout gate [Mp, H/32] (rows padded to Mp = B*P
        # rounded up to 128), and TWO BITS per feature, sign(x_u - x_v) [Mp, 4].  The hidden activations themselves
        # (1.6 GB at B = 4096) are not needed: they are linear in W1, b1 under the gate, and d w2 follows from the
        # accumulators of the d W1 GEMM (csrc/tgrad.cu).  The test hook still asks for them.
        mp = (b * p_cnt + 127) // 128 * 128
        hpost = (torch.empty(mp // 32, h // 4, 32, 4, device=x.device, dtype=torch.float32)
                 if DEBUG_CAPTURE is not None else None)
        hmask = torch.empty(mp, h // 32, device=x.device, dtype=torch.int32) if need_grad else None
        hsign = torch.empty(mp, 4, device=x.device, dtype=torch.int32) if need_grad else None
        w2v = w2.reshape(-1).contiguous()
        tok = _inst.begin("pipe_head_fwd")
        _lib.check(L.ltgnn_pipe_head_fwd(dev, b, n, p_cnt, d, h, x.data_ptr(), ends.data_ptr(), w1.data_ptr(),
                                         b1.data_ptr(), w2v.data_ptr(), p, new_dropout_seed() if p > 0 else 0,
                                         part.data_ptr(), None if hpost is None else hpost.data_ptr(),
                                         None if hmask is None else hmask.data_ptr(),
                                         None if hsign is None else hsign.data_ptr(), _stream(x)))
        _inst.end(tok)
        pooled = torch.empty(b, d, device=x.device, dtype=torch.float32)
        tok = _inst.begin("mean_pool_fwd")
        _lib.check(L.ltgnn_mean_pool_fwd(dev, b, n, d, x.data_ptr(), pooled.data_ptr(), _stream(x)))
        _inst.end(tok)
        if DEBUG_CAPTURE is not None and hpost is not None:
            DEBUG_CAPTURE["head_live"] = unblock32(hpost, 1, b * p_cnt)[0] != 0   # (B*P, H) bool
            DEBUG_CAPTURE["head_mask_words"] = hmask[: b * p_cnt]
        if need_grad:
            ctx.save_for_backward(x, ends, inc_ptr, inc, w1, b1, w2v, hmask, hsign)
        # the kernel draws 16 random bits per hidden unit: its keep probability is 1 - round(p * 2^16) / 2^16
        ctx.scale = 1.0 / (1.0 - int(p * 65536.0 + 0.5) / 65536.0)
        return part, pooled

    @staticmethod
    def backward(ctx, dpart, dpooled):
        x, ends, inc_ptr, inc, w1, b1, w2v, hmask, hsign = ctx.saved_tensors
        b, n, d = x.shape
        p_cnt, h = ends.shape[0], w1.shape[0]
        dev = _dev_index(x)
        L = _lib.load()
        dlogit = dpart[0].contiguous().view(-1)
        dx = torch.empty_like(x)
        dpooled = None if dpooled is None else dpooled.contiguous()
        ws = torch.empty(int(L.ltgnn_pipe_head_dx_ws_floats(dev, n, p_cnt)), device=x.device, dtype=torch.float32)
        tok = _inst.begin("pipe_head_bwd_dx")
        _lib.check(L.ltgnn_pipe_head_bwd_dx(dev, b, n, p_cnt, d, h, inc_ptr.data_ptr(), inc.data_ptr(), w1.data_ptr(),
                                            w2v.data_ptr(), hmask.data_ptr(), hsign.data_ptr(), dlogit.data_ptr(), ctx.scale,
                                            None if dpooled is None else dpooled.data_ptr(), ws.data_ptr(), dx.data_ptr(),
                                            _stream(x)))
        _inst.end(tok)
        del ws
        if not any(ctx.needs_input_grad[4:7]):  # frozen head
            return dx, None, None, None, None, None, None, None, None
        # parameter gradients: dW1 on tensor cores with operands formed on the fly; db1 and dw2 from the same accumulators
        dw1 = torch.empty_like(w1)
        db1 = torch.empty(h, device=x.device, dtype=torch.float32)
        dw2 = torch.empty(1, h, device=x.device, dtype=torch.float32)
        ws = torch.empty(int(L.ltgnn_pipe_head_ws_floats(dev)), device=x.device, dtype=torch.float32)
        tok = _inst.begin("pipe_head_bwd_w")
        _lib.check(L.ltgnn_pipe_head_bwd_w(dev, b, n, p_cnt, d, h, x.data_ptr(), ends.data_ptr(), w1.data_ptr(),
                                           b1.data_ptr(), w2v.data_ptr(), hmask.data_ptr(), dlogit.data_ptr(), ctx.scale,
                                           dw1.data_ptr(), db1.data_ptr(), dw2.data_ptr(), ws.data_ptr(), _stream(x)))
        _inst.end(tok)
        return dx, None, None, None, dw1, db1, dw2, None, None


def heads_wide_supported(d: int, h: int) -> bool:
    """Shapes of the composed pipe head (csrc/heads_wide.cu + the gathered-row GEMM of csrc/tcn.cu, 128 channels)."""
    return d == 128 and h == 128


_ROWS3_CACHE: Dict = {}


def _rows3(m: int, device) -> torch.Tensor:
    """src of the three-tap GEMM over F [3][M][D]: tap t of output row r reads row t * M + r."""
    key = (m, str(device))
    hit = _ROWS3_CACHE.get(key)
    if hit is None:
        if len(_ROWS3_CACHE) > 8:
            _ROWS3_CACHE.clear()
        hit = (torch.arange(m, dtype=torch.int32).unsqueeze(0) + torch.arange(3, dtype=torch.int32).unsqueeze(1) * m
               ).contiguous().to(device)
        _ROWS3_CACHE[key] = hit
    return hit


class _HeadsWide(torch.autograd.Function):
    """The pipe head + mean pool for D = H = 128 (BASELINE configs[4]): features materialised once, the 3D -> H product
    as a three-tap gathered-row GEMM on the tensor cores, the H -> 1 layer / dropout / feature gradient as streaming
    kernels (csrc/heads_wide.cu).  Same contract as :class:`_Heads`; gradients are gathers and fixed-order sums."""

    @staticmethod
    def forward(ctx, x, ends, inc_ptr, inc, w1, b1, w2, drop_p, training):
        x = x.contiguous()
        b, n, d = x.shape
        p_cnt, h = ends.shape[0], w1.shape[0]
        m = b * p_cnt
        if 3 * m >= 2**31:
            raise ValueError("heads: B * P too large for int32 row indices")
        dev = _dev_index(x)
        L = _lib.load()
        p = float(drop_p) if training else 0.0
        feat = torch.empty(3, m, d, device=x.device, dtype=torch.float32)
        tok = _inst.begin("pipe_feat_fwd")
        _lib.check(L.ltgnn_pipe_feat_fwd(dev, b, n, p_cnt, d, x.data_ptr(), ends.data_ptr(), feat.data_ptr(), _stream(x)))
        _inst.end(tok)
        w3 = w1.detach().view(h, 3, d).permute(1, 0, 2).contiguous()          # [tap][H][D]: W1[:, tD:(t+1)D]
        hid = tcn_conv(feat.view(3 * m, d), _rows3(m, x.device), w3, b1.detach().contiguous(), relu=True)   # relu(pre), (M, H)
        part = torch.empty(1, b, p_cnt, device=x.device, dtype=torch.float32)
        w2v = w2.detach().reshape(-1).contiguous()
        tok = _inst.begin("head_out_fwd")
        _lib.check(L.ltgnn_head_out_fwd(dev, m, h, hid.data_ptr(), w2v.data_ptr(), p, new_dropout_seed() if p > 0 else 0,
                                        part.data_ptr(), _stream(x)))
        _inst.end(tok)
        pooled = torch.empty(b, d, device=x.device, dtype=torch.float32)
        tok = _inst.begin("mean_pool_fwd")
        _lib.check(L.ltgnn_mean_pool_fwd(dev, b, n, d, x.data_ptr(), pooled.data_ptr(), _stream(x)))
        _inst.end(tok)
        if DEBUG_CAPTURE is not None:
            DEBUG_CAPTURE["head_live"] = hid > 0
        ctx.save_for_backward(x, ends, inc_ptr, inc, w3, w2v, feat, hid, w1, b1)
        ctx.scale = 1.0 / (1.0 - int(p * 65536.0 + 0.5) / 65536.0)
        return part, pooled

    @staticmethod
    def backward(ctx, dpart, dpooled):
        x, ends, inc_ptr, inc, w3, w2v, feat, hid, w1, b1 = ctx.saved_tensors
        b, n, d = x.shape
        p_cnt, h = ends.shape[0], w3.shape[1]
        m = b * p_cnt
        dev = _dev_index(x)
        L = _lib.load()
        dlogit = dpart[0].contiguous().view(-1)
        dh = torch.empty(m, h, device=x.device, dtype=torch.float32)
        gq = torch.empty(m, h, device=x.device, dtype=torch.float32)
        cs = torch.empty(h, device=x.device, dtype=torch.float32)
        ws = torch.empty(int(L.ltgnn_head_out_ws_floats(dev, h)), device=x.device, dtype=torch.float32)
        tok = _inst.begin("head_out_bwd")
        _lib.check(L.ltgnn_head_out_bwd(dev, m, h, hid.data_ptr(), w2v.data_ptr(), dlogit.data_ptr(), ctx.scale, dh.data_ptr(),
                                        gq.data_ptr(), cs.data_ptr(), ws.data_ptr(), _stream(x)))
        _inst.end(tok)
        # parameter gradients: T[t] = gq^T F[t] on the tensor cores; dW1, db1, dw2 follow from T and cs (the hidden layer is
        # linear in W1, b1 under the gate -- no second pass over the hidden activations).  Skipped for a frozen head.
        dw1 = db1 = dw2 = None
        if any(ctx.needs_input_grad[4:7]):
            t3 = torch.empty(3, h, d, device=x.device, dtype=torch.float32)
            for t in range(3):
                wgrad(gq, feat[t], out=t3[t])
            dw1 = torch.empty_like(w1)
            db1 = torch.empty(h, device=x.device, dtype=torch.float32)
            dw2 = torch.empty(1, h, device=x.device, dtype=torch.float32)
            w1c, b1c = w1.detach().contiguous(), b1.detach().contiguous()
            tok = _inst.begin("head_wide_finish")
            _lib.check(L.ltgnn_head_wide_finish(dev, h, d, t3.data_ptr(), w1c.data_ptr(), b1c.data_ptr(), w2v.data_ptr(),
                                                cs.data_ptr(), dw1.data_ptr(), db1.data_ptr(), dw2.data_ptr(), _stream(x)))
            _inst.end(tok)
        dfeat = torch.empty_like(feat)
        for t in range(3):
            linear_tc(dh, w3[t], transposed=True, out=dfeat[t])                        # dF_t = dh W1[:, tD:(t+1)D]
        dx = torch.empty_like(x)
        dpooled = None if dpooled is None else dpooled.contiguous()
        tok = _inst.begin("pipe_feat_bwd")
        _lib.check(L.ltgnn_pipe_feat_bwd(dev, b, n, p_cnt, d, x.data_ptr(), ends.data_ptr(), inc_ptr.data_ptr(), inc.data_ptr(),
                                         dfeat.data_ptr(), None if dpooled is None else dpooled.data_ptr(), dx.data_ptr(),
                                         _stream(x)))
        _inst.end(tok)
        return dx, None, None, None, dw1, db1, dw2, None, None


def heads(x: torch.Tensor, ends: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, drop_p: float,
          training: bool, incidence=None):
    """x (B,N,D), ends int32 (P,2) -> (part (1,B,P), pooled (B,D)); pipe_logits = part.sum(0) + b2.
    D = 64: the fused tensor-memory kernels (csrc/heads.cu); D = 128: the composed form (csrc/heads_wide.cu); the hidden
    width is the reference's 128.  Other widths raise -- there is no library fallback.
    ``incidence``: the result of :func:`pipe_incidence` for these ends (built on the fly, with a host round trip, when
    omitted)."""
    _check_act(x.contiguous(), "x")
    d, h = x.shape[-1], w1.shape[0]
    if incidence is None:
        incidence = pipe_incidence(ends, x.shape[1])
    if heads_supported(d, h):
        return _Heads.apply(x, ends, incidence[0], incidence[1], w1, b1, w2, drop_p, training)
    if heads_wide_supported(d, h):
        return _HeadsWide.apply(x, ends, incidence[0], incidence[1], w1, b1, w2, drop_p, training)
    raise ValueError(f"heads: node width {d} / hidden width {h} not built (64 or 128 / 128); the sm_100a kernels have no "
                     "library fallback")


# ----------------------------------------------------------------------------------------------
# the message-passing body of the detector as ONE autograd node
#   h_s -> node init -> L x [GCNConv -> ReLU -> Dropout] -> x_L        (detector.py:178-201)
# ----------------------------------------------------------------------------------------------
class _GnnBody(torch.autograd.Function):
    """Forward keeps only the layer outputs x_0..x_L (each doubles as the ReLU/dropout mask of its own
    layer: x > 0 <=> unit was active and kept).  Backward per layer: gate + CSC-transpose aggregation +
    bias gradient in one staged kernel, weight gradient, input gradient on tensor cores."""

    @staticmethod
    def forward(ctx, h_s, slot, graph, drop_p, training, vals, t_vals, w0, b0, *conv_params):
        h_s = h_s.contiguous()
        n = graph.num_nodes
        p = float(drop_p) if training else 0.0
        n_layers = len(conv_params) // 2
        need_grad = any(ctx.needs_input_grad)
        bsz = h_s.shape[0]

        def live_for(d):  # 1-bit record of (x > 0) for the backward gates: 1/32 of the bytes of x
            return new_live_mask(bsz, n, d, h_s.device) if need_grad and d % 32 == 0 and n <= 1024 else None

        lives = [live_for(w0.shape[0])]
        x = node_init_fwd(h_s, slot, n, w0, b0, p, new_dropout_seed() if p > 0 else 0, live_out=lives[0])
        xs = [x]
        # weighted adjacency: every layer runs ltgnn_linear + the weighted aggregation; XW of each layer is kept for the
        # adjacency-value gradient when one is asked for
        keep_xw = vals is not None and ctx.needs_input_grad[5]
        xws = []
        for l in range(n_layers):
            w, b = conv_params[2 * l], conv_params[2 * l + 1]
            if vals is None and FUSED_LAYER and w.is_contiguous() and gcn_layer_supported(graph, x, w):
                lives.append(live_for(w.shape[0]))
                x = gcn_layer_fwd(graph, x, w, bias=b, relu=True, drop_p=p, drop_seed=new_dropout_seed() if p > 0 else 0,
                                  live_out=lives[-1])
                xs.append(x)
                continue
            xw = _linear_any(x, w)
            # graphs that fit shared memory: STAGED kernel; larger ones: the L2-gather kernel with the same fused epilogue.
            # Both write the 1-bit live mask the backward gates with (D % 32 == 0; else the float activations gate)
            d_out = xw.shape[-1]
            lives.append(live_for(d_out) if _staged_ok(graph, d_out)
                         else (new_live_mask(bsz, n, d_out, h_s.device) if need_grad and d_out % 32 == 0 else None))
            x = spmm_fused(graph, xw.view(bsz, n, -1), bias=b, relu=True, drop_p=p,
                           drop_seed=new_dropout_seed() if p > 0 else 0, live_out=lives[-1], vals=vals)
            if keep_xw:
                xws.append(xw.view(bsz, n, -1))
            del xw
            xs.append(x)
        ctx.lives = lives
        if DEBUG_CAPTURE is not None:
            DEBUG_CAPTURE["lives"] = lives
            DEBUG_CAPTURE["xs"] = xs   # the gates of the layers without a live mask (None in `lives`)
        ctx.save_for_backward(h_s, slot, w0, *conv_params[0::2], *xs, t_vals, *xws)
        ctx.shared = vals is not None and vals.shape[0] == 1
        # the kernels draw 16 random bits per element: keep probability 1 - round(p * 2^16) / 2^16
        ctx.graph, ctx.n_layers, ctx.scale = graph, n_layers, 1.0 / (1.0 - int(p * 65536.0 + 0.5) / 65536.0)
        return xs[-1]

    @staticmethod
    def backward(ctx, dx):
        saved = ctx.saved_tensors
        L_ = ctx.n_layers
        h_s, slot, w0 = saved[0], saved[1], saved[2]
        ws_ = saved[3:3 + L_]
        xs = saved[3 + L_:3 + 2 * L_ + 1]
        t_vals, xws = saved[3 + 2 * L_ + 1], saved[3 + 2 * L_ + 2:]
        graph, scale = ctx.graph, ctx.scale
        need = ctx.needs_input_grad
        # below[l]: the gradient at layer l's input is needed -- by node init (h_s, w0, b0), by a lower layer's
        # parameters, or by a lower layer's d A_hat (which reads it at that layer's output).  A frozen stack skips the rest.
        below = [need[0] or need[7] or need[8]]
        for l in range(1, L_):
            below.append(below[-1] or need[7 + 2 * l] or need[8 + 2 * l] or bool(xws))
        g = dx.contiguous()
        grads = [None] * (2 * L_)
        dvals = None
        for l in range(L_ - 1, -1, -1):
            x_out, x_in, w = xs[l + 1], xs[l], ws_[l]
            live = ctx.lives[l + 1]
            if xws:  # d A_hat of this layer, gated exactly as the aggregation below gates g; layers add up
                dvals = gcn_adj_grad(graph, g, xws[l], gate=x_out if live is None else None, live_in=live,
                                     gate_scale=scale, out=dvals, shared=ctx.shared, accumulate=dvals is not None)
            want_w, want_b = need[9 + 2 * l], need[10 + 2 * l]
            if not (want_w or want_b or below[l]):
                break
            gz = spmm_fused(graph, g, transpose=True, gate=x_out if live is None else None, live_in=live,
                            gate_scale=scale, want_colsum=want_b, vals=t_vals)
            if want_b:
                gz, grads[2 * l + 1] = gz
            if want_w:
                grads[2 * l] = wgrad(gz, x_in)
            if not below[l]:
                break
            if l == 0 and FUSED_NODE_INIT_BWD and ctx.lives[0] is not None and w0.shape[0] in (64, 128) \
                    and h_s.shape[2] % 32 == 0 and w.shape[0] % 32 == 0 and w.shape[0] <= 128:
                # node init reads only the gated column sums and sensor rows of this layer's input gradient
                dhs, dw0, db0 = node_init_bwd_from_layer(h_s, slot, w0, gz, w.contiguous(), ctx.lives[0], scale)
                return (dhs, None, None, None, None, dvals, None, dw0, db0, *grads)
            g = _linear_any(gz, w, transposed=True)
            del gz
        dhs = dw0 = db0 = None
        if below[0]:
            dhs, dw0, db0 = node_init_bwd(h_s, slot, w0, g, xs[0], scale, live=ctx.lives[0])
        return (dhs, None, None, None, None, dvals, None, dw0, db0, *grads)


def gnn_body(h_s: torch.Tensor, slot: torch.Tensor, graph: PipeGraph, drop_p: float, training: bool,
             w0: torch.Tensor, b0: torch.Tensor, conv_params, edge_weight: Optional[torch.Tensor] = None,
             edge_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Sensor embeddings (B,S,ds) -> node states after the last GCN layer (B,N,D).  ``edge_weight``: (E,) or (B, E)
    weights of the graph's edges, normalised once on the device and used by every layer (as PyG passes one
    ``edge_weight`` to every conv); differentiable.  ``edge_mask``: (E,) or (B, E) explainer mask on every layer's
    messages after the normalisation (as PyG's ``set_masks`` puts one mask on every conv); differentiable.  Both
    ``None``: the graph's own adjacency, on the one-kernel layers."""
    _check_act(h_s.contiguous(), "h_s")
    vals = t_vals = None
    if edge_weight is not None or edge_mask is not None:
        vals, t_vals = normalized_edge_values(graph, edge_weight, h_s.shape[0], edge_mask)
    return _GnnBody.apply(h_s, slot, graph, drop_p, training, vals, t_vals, w0, b0, *conv_params)


# ----------------------------------------------------------------------------------------------
# shared per-sensor GRU encoder (reference models/detector.py:28-73)
# ----------------------------------------------------------------------------------------------
def gru_supported(hidden: int, n_time: int) -> bool:
    """Hidden 64: csrc/gru.cu; hidden 128: the cluster recurrence of csrc/gru_pred.cu (``_SensorGru128``)."""
    return hidden in (64, 128) and 0 <= n_time <= 30


def gru_fwd(r: torch.Tensor, tf: Optional[torch.Tensor], w_ih, w_hh, b_ih, b_hh, save: bool = False):
    """Raw forward: r (B,L,S), tf (B,L,F) or None -> h_last (B,S,H) [, hseq, gates r | z | n in blocked-32 layout].
    The BPTT rebuilds the fourth pre-activation group W_hn h + b_hn instead of reading it."""
    _check_act(r, "r")
    b, l, s = r.shape
    f = 0 if tf is None else tf.shape[-1]
    if tf is not None:
        _check_act(tf, "tf")
    hdim = w_hh.shape[1]
    h_last = torch.empty(b, s, hdim, device=r.device, dtype=torch.float32)
    # saved tensors use the kernels' "blocked-32" layout: logical [L * Qp, W] with Qp = B*S rounded up to 128,
    # stored as [L * Qp / 32, W / 4, 32, 4] (see csrc/gru.cu)
    qp = (b * s + 127) // 128 * 128
    hseq = torch.empty(l * qp // 32, hdim // 4, 32, 4, device=r.device, dtype=torch.float32) if save else None
    gates = torch.empty(l * qp // 32, 3 * hdim // 4, 32, 4, device=r.device, dtype=torch.float32) if save else None
    L = _lib.load()
    tok = _inst.begin("gru_fwd")
    _lib.check(L.ltgnn_gru_fwd(_dev_index(r), b, l, s, f, hdim, r.data_ptr(), None if tf is None else tf.data_ptr(),
                               w_ih.data_ptr(), w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(), h_last.data_ptr(),
                               None if hseq is None else hseq.data_ptr(), None if gates is None else gates.data_ptr(),
                               _stream(r)))
    _inst.end(tok)
    return (h_last, hseq, gates) if save else h_last


def _dx_outputs(r: torch.Tensor, f: int, want_r: bool, want_tf: bool):
    """(dr (B, L, S), dxt (B, L, S, F)) for ``gru_bwd_dx`` / ``gru_sensor_bwd_dx``, each only where it is asked for."""
    dr = torch.empty_like(r) if want_r else None
    dxt = torch.empty(*r.shape, f, device=r.device, dtype=torch.float32) if want_tf and f else None
    return dr, dxt


def gru_bwd_dx(dg: torch.Tensor, w_ih: torch.Tensor, r: torch.Tensor, dr: Optional[torch.Tensor],
               dxt: Optional[torch.Tensor]) -> None:
    """Raw input gradient at hidden 64 (see ltgnn_gru_bwd_dx) from ``ltgnn_gru_bwd_dg_hn``'s blocked-32 dG: writes
    dr (B, L, S) and the per-sequence time-feature rows dxt (B, L, S, F) (``dxt.sum(2)`` is d tf)."""
    b, l, s = r.shape
    f = w_ih.shape[1] - 1
    L = _lib.load()
    tok = _inst.begin("gru_bwd_dx")
    _lib.check(L.ltgnn_gru_bwd_dx(_dev_index(dg), b, l, s, f, w_ih.shape[0] // 3, w_ih.data_ptr(), dg.data_ptr(),
                                  None if dr is None else dr.data_ptr(), None if dxt is None else dxt.data_ptr(),
                                  _stream(dg)))
    _inst.end(tok)


class _GruEncoder(torch.autograd.Function):
    """h_last = GRU(cat([r_s, tf]))[:, -1] for every (window, sensor) sequence, with back-propagation through time
    to the four GRU parameters and to the inputs r and tf, each only where a gradient is asked for.  The backward runs
    the BPTT (``ltgnn_gru_bwd_dg_hn``), then the input gradient (``ltgnn_gru_bwd_dx``) if r or tf wants one, then the
    weight gradients (``ltgnn_gru_bwd_w``) if a parameter does: a frozen encoder pays nothing for the latter."""

    @staticmethod
    def forward(ctx, r, tf, w_ih, w_hh, b_ih, b_hh):
        r = r.contiguous()
        tf = None if tf is None else tf.contiguous()
        params = [t.contiguous() for t in (w_ih, w_hh, b_ih, b_hh)]
        if any(ctx.needs_input_grad):
            h_last, hseq, gates = gru_fwd(r, tf, *params, save=True)
            ctx.save_for_backward(r, tf, params[0], params[1], params[3], hseq, gates)
        else:  # nothing requires a gradient: backward is never reached
            h_last = gru_fwd(r, tf, *params)
        return h_last

    @staticmethod
    def backward(ctx, dh):
        r, tf, w_ih, w_hh, b_hh, hseq, gates = ctx.saved_tensors
        b, l, s = r.shape
        f = 0 if tf is None else tf.shape[-1]
        hd = w_hh.shape[1]
        q = b * s
        dev = _dev_index(r)
        L = _lib.load()
        dh = dh.contiguous()
        dg = torch.empty(hseq.shape[0], hd, 32, 4, device=r.device, dtype=torch.float32)  # blocked-32 [L*Qp, 4H]
        tok = _inst.begin("gru_bwd_dg")
        _lib.check(L.ltgnn_gru_bwd_dg_hn(dev, q, l, hd, w_hh.data_ptr(), b_hh.data_ptr(), gates.data_ptr(),
                                         hseq.data_ptr(), dh.data_ptr(), dg.data_ptr(), _stream(r)))
        _inst.end(tok)
        del gates
        dr, dxt = _dx_outputs(r, f, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        if dr is not None or dxt is not None:
            gru_bwd_dx(dg, w_ih, r, dr, dxt)
        dtf = None if dxt is None else dxt.sum(2)
        if not any(ctx.needs_input_grad[2:]):
            return dr, dtf, None, None, None, None
        fused = torch.empty(4 * hd, 96, device=r.device, dtype=torch.float32)
        ws = torch.empty(int(L.ltgnn_gru_ws_floats(dev)), device=r.device, dtype=torch.float32)
        tok = _inst.begin("gru_bwd_w")
        _lib.check(L.ltgnn_gru_bwd_w(dev, b, l, s, f, hd, r.data_ptr(), None if tf is None else tf.data_ptr(),
                                     hseq.data_ptr(), dg.data_ptr(), fused.data_ptr(), ws.data_ptr(), _stream(r)))
        _inst.end(tok)
        # rows of `fused`: r | z | (W_hn h + b_hn) | (W_in x + b_in); columns: h (hd) | x, tf (1 + f) | 1
        rr, zz, hn, inn = fused[0:hd], fused[hd:2 * hd], fused[2 * hd:3 * hd], fused[3 * hd:4 * hd]
        kb = hd + 1 + f
        dw_hh = torch.cat([rr[:, :hd], zz[:, :hd], hn[:, :hd]], dim=0)
        dw_ih = torch.cat([rr[:, hd:kb], zz[:, hd:kb], inn[:, hd:kb]], dim=0)
        db_ih = torch.cat([rr[:, kb], zz[:, kb], inn[:, kb]], dim=0)
        db_hh = torch.cat([rr[:, kb], zz[:, kb], hn[:, kb]], dim=0)
        return dr, dtf, dw_ih, dw_hh, db_ih, db_hh


def gru_encode(r: torch.Tensor, tf: Optional[torch.Tensor], w_ih, w_hh, b_ih, b_hh) -> torch.Tensor:
    """Differentiable shared sensor GRU: (B,L,S) [+ (B,L,F)] -> (B,S,H), H = 64 or 128.  Gradients flow to the four
    parameters and to r and tf, each only where one is asked for.  d tf is the sum over the sensors of the per-sequence
    input gradients, taken in a fixed order once every sequence is done, so it does not depend on how the hidden-128
    backward splits the sequences into slabs."""
    _check_act(r.contiguous(), "r")
    if w_hh.shape[1] == 128:
        if not torch.is_grad_enabled():   # eval, event evaluation: one launch, nothing saved
            return _SensorGru128.infer(r.contiguous(), None if tf is None else tf.contiguous(), w_ih, w_hh, b_ih, b_hh)
        return _SensorGru128.apply(r, tf, w_ih, w_hh, b_ih, b_hh)
    return _GruEncoder.apply(r, tf, w_ih, w_hh, b_ih, b_hh)


# ----------------------------------------------------------------------------------------------
# GRU normal-state predictor at hidden 128 (reference models/predictor.py:84-111), inference only (csrc/gru_pred.cu)
# ----------------------------------------------------------------------------------------------
def gru_predictor_weights(layers, k0: int = 64) -> list:
    """torch.nn.GRU parameters [(w_ih, w_hh, b_ih, b_hh) per layer] -> per layer (w_x [3, H, K], b_x [3, H], w_hh [3H, H],
    b_hn [H]): the input projection per gate group with layer 0's input columns zero-padded to K = k0 (the projection
    kernel's K granularity), b_hh of the r and z gates folded into b_x; b_hn = b_hh of the n gate stays inside r * (.)."""
    out = []
    for i, (w_ih, w_hh, b_ih, b_hh) in enumerate(layers):
        h = w_hh.shape[1]
        k = k0 if i == 0 else h
        if w_ih.shape[1] > k:
            raise ValueError(f"gru_predictor_weights: layer {i} has {w_ih.shape[1]} inputs, the projection takes <= {k}")
        w_x = w_ih.new_zeros(3, h, k)
        w_x[:, :, : w_ih.shape[1]] = w_ih.detach().view(3, h, -1)
        b_x = b_ih.detach().view(3, h).clone()
        b_x[:2] += b_hh.detach().view(3, h)[:2]
        out.append((w_x, b_x, w_hh.detach().contiguous(), b_hh.detach()[2 * h:].contiguous()))
    return out


def gru_layer_fwd(inp: torch.Tensor, q: int, l: int, layer, seq: bool = False):
    """Raw (non-differentiable) forward of one GRU layer over q sequences of l steps.  inp (q * l, K) fp32 CUDA, row
    q_i * l + t = the input of sequence q_i at step t; ``layer`` = one entry of ``gru_predictor_weights``.
    Returns (h_last (q, H), hseq (q * l, H) or None): gx = inp W_x[g]^T + b_x[g] by ``linear_tc`` (one N = H launch per
    gate group), then the recurrence ``ltgnn_gru_layer_fwd``."""
    _check_act(inp, "inp")
    w_x, b_x, w_hh, b_hn = layer
    hdim = w_hh.shape[1]
    if inp.shape != (q * l, w_x.shape[2]):
        raise ValueError(f"inp must be ({q * l}, {w_x.shape[2]}), got {tuple(inp.shape)}")
    gx = torch.empty(3, q * l, hdim, device=inp.device, dtype=torch.float32)
    for g in range(3):
        linear_tc(inp, w_x[g], b_x[g], out=gx[g])
    h_last = torch.empty(q, hdim, device=inp.device, dtype=torch.float32)
    hseq = torch.empty(q * l, hdim, device=inp.device, dtype=torch.float32) if seq else None
    L = _lib.load()
    tok = _inst.begin("gru_pred_layer")
    _lib.check(L.ltgnn_gru_layer_fwd(_dev_index(inp), q, l, hdim, gx.data_ptr(), w_hh.data_ptr(), b_hn.data_ptr(),
                                     None if hseq is None else hseq.data_ptr(), h_last.data_ptr(), _stream(inp)))
    _inst.end(tok)
    return h_last, hseq


def gru_predictor_fwd(x: torch.Tensor, x_time: torch.Tensor, layers) -> torch.Tensor:
    """Raw (non-differentiable) stacked GRU: x (Q, L, S), x_time (Q, L, F) -> the last layer's state after step L-1, (Q, H).
    Layer i's input is cat([x, x_time]) (zero-padded to K) for i = 0 and layer i-1's state sequence otherwise (no
    inter-layer dropout: inference).  ``layers``: ``gru_predictor_weights(...)``."""
    q, l, s = x.shape
    f = x_time.shape[-1]
    k0 = layers[0][0].shape[2]
    if s + f > k0:
        raise ValueError(f"gru_predictor_fwd: {s} + {f} inputs exceed K = {k0}")
    inp = torch.zeros(q, l, k0, device=x.device, dtype=torch.float32)
    inp[:, :, :s] = x
    inp[:, :, s:s + f] = x_time
    inp = inp.view(q * l, k0)
    for i, layer in enumerate(layers):
        h_last, inp = gru_layer_fwd(inp, q, l, layer, seq=i + 1 < len(layers))
    return h_last


def gru_layer_fwd_windows(gx: torch.Tensor, row_base: torch.Tensor, l: int, layer, seq: bool = False):
    """Raw forward of one GRU layer over windows that share one input projection (see ltgnn_gru_layer_fwd_windows):
    gx [3, rows, H] holds the projection of every series row once, row_base int32 (Q,) the gx row of each window's step 0.
    The caller guarantees 0 <= row_base[q] and row_base[q] + l <= rows (the entry point cannot check device data).
    Returns (h_last (Q, H), hseq (Q * l, H) or None): ``gru_layer_fwd``'s on the materialised windows, bit for bit."""
    _check_act(gx, "gx")
    _w_x, _b_x, w_hh, b_hn = layer
    hdim = w_hh.shape[1]
    if gx.dim() != 3 or gx.shape[0] != 3 or gx.shape[2] != hdim:
        raise ValueError(f"gx must be (3, rows, {hdim}), got {tuple(gx.shape)}")
    if row_base.dtype != torch.int32 or not row_base.is_cuda or not row_base.is_contiguous() or row_base.dim() != 1:
        raise ValueError("row_base must be a contiguous 1-D int32 CUDA tensor")
    q = row_base.numel()
    h_last = torch.empty(q, hdim, device=gx.device, dtype=torch.float32)
    hseq = torch.empty(q * l, hdim, device=gx.device, dtype=torch.float32) if seq else None
    L = _lib.load()
    tok = _inst.begin("gru_pred_layer_windows")
    _lib.check(L.ltgnn_gru_layer_fwd_windows(_dev_index(gx), q, l, hdim, gx.data_ptr(), gx.shape[1], row_base.data_ptr(),
                                             w_hh.data_ptr(), b_hn.data_ptr(), None if hseq is None else hseq.data_ptr(),
                                             h_last.data_ptr(), _stream(gx)))
    _inst.end(tok)
    return h_last, hseq


def gru_predictor_windows(x: torch.Tensor, x_time: torch.Tensor, window: int, count: int, layers) -> torch.Tensor:
    """Raw stacked GRU on the ``count`` windows of ``window`` steps that start at steps 0 .. count-1 of every series:
    x (B, T, S), x_time (B, T, F) -> the last layer's state after each window's last step, (B * count, H), window
    (b, j) at row b * count + j.  Layer 0 projects the B * T series rows once and every window reads its rows from that
    plane (``gru_layer_fwd_windows``); layers >= 1 run planar as in ``gru_predictor_fwd``, whose result this is bit for
    bit on the materialised windows."""
    b, t, s = x.shape
    f = x_time.shape[-1]
    k0 = layers[0][0].shape[2]
    if s + f > k0:
        raise ValueError(f"gru_predictor_windows: {s} + {f} inputs exceed K = {k0}")
    if window < 1 or count < 1 or count + window - 1 > t:
        raise ValueError(f"gru_predictor_windows: {count} windows of {window} steps do not fit {t} steps")
    w_x, b_x, w_hh, _ = layers[0]
    inp = torch.zeros(b * t, k0, device=x.device, dtype=torch.float32)
    inp.view(b, t, k0)[:, :, :s] = x
    inp.view(b, t, k0)[:, :, s:s + f] = x_time
    gx = torch.empty(3, b * t, w_hh.shape[1], device=x.device, dtype=torch.float32)
    for g in range(3):
        linear_tc(inp, w_x[g], b_x[g], out=gx[g])
    # window (b, j) starts at series row b t + j; j + window <= count - 1 + window <= t keeps every read inside the plane
    row_base = ((torch.arange(b, device=x.device, dtype=torch.int32) * t).unsqueeze(1)
                + torch.arange(count, device=x.device, dtype=torch.int32)).reshape(-1)
    h_last, seq = gru_layer_fwd_windows(gx, row_base, window, layers[0], seq=len(layers) > 1)
    for i, layer in enumerate(layers[1:], start=1):
        h_last, seq = gru_layer_fwd(seq, b * count, window, layer, seq=i + 1 < len(layers))
    return h_last



# ----------------------------------------------------------------------------------------------
# training of the GRU normal-state predictor (csrc/gru_pred.cu): saved-gates forward, BPTT, inter-layer dropout
# ----------------------------------------------------------------------------------------------
def gru_layer_fwd_train(gx: torch.Tensor, q: int, l: int, w_hh: torch.Tensor, b_hn: torch.Tensor):
    """Raw training forward of one layer's recurrence (see ltgnn_gru_layer_fwd_train) on a precomputed input projection
    gx [3, q * l, H].  Returns (h_last (q, H), hseq (q * l, H), gates [4, q * l, H] = r | z | n | hn)."""
    _check_act(gx, "gx")
    hdim = w_hh.shape[1]
    h_last = torch.empty(q, hdim, device=gx.device, dtype=torch.float32)
    hseq = torch.empty(q * l, hdim, device=gx.device, dtype=torch.float32)
    gates = torch.empty(4, q * l, hdim, device=gx.device, dtype=torch.float32)
    L = _lib.load()
    tok = _inst.begin("gru_pred_layer_train")
    _lib.check(L.ltgnn_gru_layer_fwd_train(_dev_index(gx), q, l, hdim, gx.data_ptr(), w_hh.data_ptr(), b_hn.data_ptr(),
                                           hseq.data_ptr(), h_last.data_ptr(), gates.data_ptr(), _stream(gx)))
    _inst.end(tok)
    return h_last, hseq, gates


def gru_layer_bwd(q: int, l: int, w_hh: torch.Tensor, gates: torch.Tensor, hseq: torch.Tensor,
                  dh_last: Optional[torch.Tensor] = None, dh_seq: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw backward through time of one layer (see ltgnn_gru_layer_bwd): dG [4, q * l, H] = dr_pre | dz_pre | dn_pre | dhn
    from the gradient of h_last (q, H) and / or of every state (q * l, H)."""
    for t, nm in ((w_hh, "w_hh"), (gates, "gates"), (hseq, "hseq")):
        _check_act(t, nm)
    for t, nm in ((dh_last, "dh_last"), (dh_seq, "dh_seq")):
        if t is not None:
            _check_act(t, nm)
    hdim = w_hh.shape[1]
    dg = torch.empty(4, q * l, hdim, device=gates.device, dtype=torch.float32)
    L = _lib.load()
    tok = _inst.begin("gru_pred_layer_bwd")
    _lib.check(L.ltgnn_gru_layer_bwd(_dev_index(gates), q, l, hdim, w_hh.data_ptr(), gates.data_ptr(), hseq.data_ptr(),
                                     None if dh_last is None else dh_last.data_ptr(),
                                     None if dh_seq is None else dh_seq.data_ptr(), dg.data_ptr(), _stream(gates)))
    _inst.end(tok)
    return dg


def gru_dropout(x: torch.Tensor, drop_p: float, drop_seed: int):
    """Raw inter-layer dropout (see ltgnn_gru_dropout): (y, live) with live int32 (M, H / 32), bit b of word w = unit
    32 w + b kept."""
    _check_act(x, "x")
    m, hdim = x.shape
    y = torch.empty_like(x)
    live = torch.empty(m, hdim // 32, device=x.device, dtype=torch.int32)
    L = _lib.load()
    tok = _inst.begin("gru_dropout")
    _lib.check(L.ltgnn_gru_dropout(_dev_index(x), m, hdim, x.data_ptr(), float(drop_p), int(drop_seed) & (2**64 - 1),
                                   y.data_ptr(), live.data_ptr(), _stream(x)))
    _inst.end(tok)
    return y, live


def gru_dropout_bwd(parts: torch.Tensor, live: Optional[torch.Tensor], drop_p: float) -> torch.Tensor:
    """Raw backward of the inter-layer dropout (see ltgnn_gru_dropout_bwd): parts [n, M, H] added in order, times the
    kept mask / (1 - p) (``live = None``: no dropout)."""
    _check_act(parts, "parts")
    n, m, hdim = parts.shape
    dx = torch.empty(m, hdim, device=parts.device, dtype=torch.float32)
    L = _lib.load()
    tok = _inst.begin("gru_dropout_bwd")
    _lib.check(L.ltgnn_gru_dropout_bwd(_dev_index(parts), m, hdim, parts.data_ptr(), n,
                                       None if live is None else live.data_ptr(), float(drop_p), dx.data_ptr(),
                                       _stream(parts)))
    _inst.end(tok)
    return dx


def gru_input_grad(dg: torch.Tensor, w_x: torch.Tensor) -> torch.Tensor:
    """``sum_g dG[g] @ W_x[g]`` over the input planes r, z, n: dG (>= 3, M, H), W_x (3, H, K) (layer 0's
    ``gru_predictor_weights`` entry, K zero-padded) -> (M, K).  One ``linear_tc`` per plane; the planes are added in
    index order by ``gru_dropout_bwd`` over a 128-wide view of the K-wide parts (the tail past M K is zero)."""
    m, k = dg.shape[1], w_x.shape[2]
    n = m * k
    flat = torch.empty(3, (n + 127) // 128 * 128, device=dg.device, dtype=torch.float32)
    flat[:, n:] = 0.0
    for g in range(3):
        linear_tc(dg[g], w_x[g], transposed=True, out=flat[g, :n])
    return gru_dropout_bwd(flat.view(3, -1, 128), None, 0.0).view(-1)[:n].view(m, k)


def unpack_gru_live(live: torch.Tensor) -> torch.Tensor:
    """int32 (M, H / 32) -> bool (M, H): the units ``gru_dropout`` kept (tests and debugging)."""
    bits = (live.unsqueeze(-1) >> torch.arange(32, device=live.device, dtype=torch.int32)) & 1
    return bits.reshape(live.shape[0], -1).bool()


def _ones_aug(x: torch.Tensor, width: int) -> torch.Tensor:
    """[x | 1 | 0 ...] with ``width`` columns: the operand whose ones column turns a weight gradient into the bias's."""
    out = torch.zeros(x.shape[0], width, device=x.device, dtype=torch.float32)
    out[:, :x.shape[1]] = x
    out[:, x.shape[1]] = 1.0
    return out


def gru_layer_param_grads(dg: torch.Tensor, hseq: torch.Tensor, x_aug: torch.Tensor, n_in: int, q: int, l: int):
    """(d weight_ih, d weight_hh, d bias_ih, d bias_hh) of one torch.nn.GRU layer from its dG [4, q * l, H]
    (``gru_layer_bwd``), its states hseq (q * l, H) and its input with a ones column at ``n_in``, x_aug (q * l, K), K a
    multiple of 32: six ``wgrad`` products, dG planes r, z, hn against [h_{t-1} | 1 | 0] and r, z, n against x_aug."""
    hdim = hseq.shape[1]
    hprev = torch.zeros(q, l, hdim + 32, device=dg.device, dtype=torch.float32)
    hprev[:, 1:, :hdim] = hseq.view(q, l, hdim)[:, :-1]
    hprev[:, :, hdim] = 1.0
    hprev = hprev.view(q * l, hdim + 32)
    t_r, t_z, t_hn = (wgrad(dg[g], hprev) for g in (0, 1, 3))
    del hprev
    u_r, u_z, u_n = (wgrad(dg[g], x_aug) for g in (0, 1, 2))
    d_w_ih = torch.cat([u_r[:, :n_in], u_z[:, :n_in], u_n[:, :n_in]], dim=0)
    d_w_hh = torch.cat([t_r[:, :hdim], t_z[:, :hdim], t_hn[:, :hdim]], dim=0)
    d_b_ih = torch.cat([t_r[:, hdim], t_z[:, hdim], u_n[:, n_in]], dim=0)   # b_hr, b_hz are folded into gx: same sums
    d_b_hh = torch.cat([t_r[:, hdim], t_z[:, hdim], t_hn[:, hdim]], dim=0)
    return [d_w_ih, d_w_hh, d_b_ih, d_b_hh]


class _GruPredictor(torch.autograd.Function):
    """The GRU predictor -- every layer and the head on the last step -- as ONE autograd node: gradients for all GRU and
    head parameters, and for the input rows when they require grad (``gru_input_grad`` of layer 0's dG).

    Forward per layer: input projection (``linear_tc``, b_hr and b_hz folded), the recurrence saving its gates, and for
    every layer but the last the inter-layer dropout.  Backward per layer, top down: BPTT -> dG; dW_hh and d b_hh from
    planes r, z, hn against [h_{t-1} | 1 | 0]; dW_ih and d b_ih (n) from planes r, z, n against [input | 1 | 0]; for a
    lower layer, its state gradient sum_g dG[g] W_ih[g] through the dropout's mask."""

    @staticmethod
    def forward(ctx, inp, q, l, c_in, n_sensors, drop_p, *params):
        n_layers = (len(params) - 2) // 4
        raw = [params[4 * i:4 * i + 4] for i in range(n_layers)]
        w_head, b_head = params[-2], params[-1]
        hdim = raw[0][1].shape[1]
        p = float(drop_p)
        layers = gru_predictor_weights(raw, k0=inp.shape[1])
        x, saved, lives = inp, [], []
        for i, (w_x, b_x, w_hh, b_hn) in enumerate(layers):
            gx = torch.empty(3, q * l, hdim, device=inp.device, dtype=torch.float32)
            for g in range(3):
                linear_tc(x, w_x[g], b_x[g], out=gx[g])
            h_last, hseq, gates = gru_layer_fwd_train(gx, q, l, w_hh, b_hn)
            del gx
            saved.append((x, hseq, gates, w_hh, raw[i][0].detach().view(3, hdim, -1)))
            if i + 1 < n_layers:
                live = None
                if p > 0:
                    x, live = gru_dropout(hseq, p, new_dropout_seed())
                else:
                    x = hseq
                lives.append(live)
        if DEBUG_CAPTURE is not None:
            DEBUG_CAPTURE["gru_lives"] = lives
        n_pad = (n_sensors + 31) // 32 * 32
        w_out = torch.zeros(n_pad, hdim, device=inp.device, dtype=torch.float32)
        w_out[:n_sensors] = w_head
        b_out = torch.zeros(n_pad, device=inp.device, dtype=torch.float32)
        b_out[:n_sensors] = b_head
        pred = linear_tc(h_last, w_out, b_out)[:, :n_sensors]
        ctx.save_for_backward(h_last, w_out, *[t for layer in saved for t in layer],
                              *[lv for lv in lives if lv is not None])
        ctx.q, ctx.l, ctx.c_in, ctx.n_sensors, ctx.n_layers, ctx.p = q, l, c_in, n_sensors, n_layers, p
        ctx.has_live = [lv is not None for lv in lives]
        ctx.w_x0 = layers[0][0]                     # layer 0's W_ih per gate group, zero-padded to the input's width
        return pred

    @staticmethod
    def backward(ctx, dpred):
        h_last, w_out, *rest = ctx.saved_tensors
        n, q, l, s = ctx.n_layers, ctx.q, ctx.l, ctx.n_sensors
        saved = [rest[5 * i:5 * i + 5] for i in range(n)]
        it = iter(rest[5 * n:])
        lives = [next(it) if has else None for has in ctx.has_live]
        hdim = h_last.shape[1]
        bsz = h_last.shape[0]
        dp = torch.zeros(bsz, 64 if s <= 64 else 128, device=dpred.device, dtype=torch.float32)
        dp[:, :s] = dpred
        t_head = wgrad(dp, _ones_aug(h_last, hdim + 32))
        dh_last = linear_tc(dp[:, :w_out.shape[0]].contiguous(), w_out, transposed=True)
        dh_seq = d_inp = None
        grads = [None] * (4 * n)
        for i in range(n - 1, -1, -1):
            x, hseq, gates, w_hh, w_ih3 = saved[i]
            dg = gru_layer_bwd(q, l, w_hh, gates, hseq, dh_last=dh_last, dh_seq=dh_seq)
            if i == 0:
                grads[0:4] = gru_layer_param_grads(dg, hseq, x, ctx.c_in, q, l)   # layer 0's input carries the ones
                if ctx.needs_input_grad[0]:
                    d_inp = gru_input_grad(dg, ctx.w_x0)
            else:
                grads[4 * i:4 * i + 4] = gru_layer_param_grads(dg, hseq, _ones_aug(x, hdim + 32), hdim, q, l)
            if i > 0:
                parts = torch.empty(3, q * l, hdim, device=dg.device, dtype=torch.float32)
                for g in range(3):
                    linear_tc(dg[g], w_ih3[g], transposed=True, out=parts[g])
                dh_seq = gru_dropout_bwd(parts, lives[i - 1], ctx.p)
                dh_last = None
            del dg
        return (d_inp, None, None, None, None, None, *grads, t_head[:s, :hdim].contiguous(),
                t_head[:s, hdim].contiguous())


def gru_predictor_cone(x: torch.Tensor, x_time: torch.Tensor, drop_p: float, params) -> torch.Tensor:
    """Differentiable prediction (B, S) of the GRU predictor's last step on the sm_100a kernels.  ``params``: per layer
    weight_ih, weight_hh, bias_ih, bias_hh (torch.nn.GRU), then head.{weight, bias}; ``drop_p``: the inter-layer dropout
    (0 in eval mode)."""
    _check_act(x.contiguous(), "x")
    b, length, s = x.shape
    c_in = s + x_time.shape[-1]
    kp = 64 if c_in < 64 else 96           # one zero-weight column for the ones that turn the weight gradient into d bias
    inp = torch.zeros(b * length, kp, device=x.device, dtype=torch.float32)
    inp.view(b, length, kp)[:, :, :s] = x
    inp.view(b, length, kp)[:, :, s:c_in] = x_time
    inp[:, c_in] = 1.0
    return _GruPredictor.apply(inp, b, length, c_in, s, float(drop_p), *params)


# ----------------------------------------------------------------------------------------------
# shared sensor GRU encoder at hidden 128 (reference models/detector.py:28-73, sensor_hidden = 128): the predictor's
# cluster recurrence and BPTT (csrc/gru_pred.cu) with the encoder's input formed in the kernel
# ----------------------------------------------------------------------------------------------
_SLAB_BYTES = 8 << 30     # backward temporaries of one slab: dG, [h_{t-1} | 1 | 0], [r | tf | 1 | 0] = 2 816 B per row
_RESIDENT_TILES: Dict[int, int] = {}


def gru_resident_tiles(dev: int) -> int:
    """128-sequence tiles the cluster recurrence runs at once on device ``dev`` (one wave); cached per device."""
    if dev not in _RESIDENT_TILES:
        n = ctypes.c_int32(0)
        _lib.check(_lib.load().ltgnn_gru_resident_tiles(dev, ctypes.byref(n)))
        if n.value <= 0:
            raise RuntimeError(f"gru_resident_tiles: the device runs no 4-CTA cluster of the GRU recurrence ({n.value})")
        _RESIDENT_TILES[dev] = n.value
    return _RESIDENT_TILES[dev]


def gru_sensor_slabs(q: int, l: int, dev: int) -> list:
    """[(q0, n)]: the training slabs of q sequences of l steps, each a whole number of waves of resident tiles (the last
    one what is left), as many waves per slab as keep its backward temporaries within _SLAB_BYTES (at least one)."""
    wave = 128 * gru_resident_tiles(dev)
    n = max(1, _SLAB_BYTES // (wave * l * 2816)) * wave
    return [(q0, min(n, q - q0)) for q0 in range(0, q, n)]


def gru_sensor_tproj(tf: Optional[torch.Tensor], w_ih: torch.Tensor, b_ih: torch.Tensor, b_hh: torch.Tensor,
                     b: int, l: int) -> torch.Tensor:
    """T [3, b * l, H] = tf W_ih[:, 1:]^T + b_ih, plus b_hh for r and z (folded as ``gru_predictor_weights`` folds them):
    ``linear_tc`` at K = 32 on the zero-padded time features, one launch per gate group; without time features every
    row is the folded bias."""
    h = w_ih.shape[0] // 3
    f = w_ih.shape[1] - 1
    b_x = b_ih.detach().view(3, h).clone()
    b_x[:2] += b_hh.detach().view(3, h)[:2]
    if f == 0:
        return b_x.unsqueeze(1).expand(3, b * l, h).contiguous()
    x = torch.zeros(b * l, 32, device=w_ih.device, dtype=torch.float32)
    x[:, :f] = tf.reshape(b * l, f)
    w_t = torch.zeros(3, h, 32, device=w_ih.device, dtype=torch.float32)
    w_t[:, :, :f] = w_ih.detach()[:, 1:].reshape(3, h, f)
    t = torch.empty(3, b * l, h, device=w_ih.device, dtype=torch.float32)
    for g in range(3):
        linear_tc(x, w_t[g], b_x[g], out=t[g])
    return t


def gru_sensor_fwd(r: torch.Tensor, tproj: torch.Tensor, w_r: torch.Tensor, w_hh: torch.Tensor, b_hn: torch.Tensor,
                   q0: int, n: int, h_last: torch.Tensor, hseq: Optional[torch.Tensor] = None,
                   gates: Optional[torch.Tensor] = None) -> None:
    """Raw forward of sequences q0 .. q0 + n - 1 of the encoder (see ltgnn_gru_sensor_fwd): r (B, L, S), tproj
    [3, B * L, H] (``gru_sensor_tproj``), w_r [3, H] = W_ih[:, 0]; writes h_last (n, H) and, for training, hseq
    (n * L, H) and gates [4, n * L, H] in the planar layout ``gru_layer_bwd`` reads."""
    for t, nm in ((r, "r"), (tproj, "tproj"), (w_r, "w_r"), (w_hh, "w_hh"), (b_hn, "b_hn"), (h_last, "h_last")):
        _check_act(t, nm)
    b, l, s = r.shape
    L = _lib.load()
    tok = _inst.begin("gru_sensor_train" if gates is not None else "gru_sensor")
    _lib.check(L.ltgnn_gru_sensor_fwd(_dev_index(r), b, l, s, q0, n, w_hh.shape[1], r.data_ptr(), tproj.data_ptr(),
                                      w_r.data_ptr(), w_hh.data_ptr(), b_hn.data_ptr(),
                                      None if hseq is None else hseq.data_ptr(), h_last.data_ptr(),
                                      None if gates is None else gates.data_ptr(), _stream(r)))
    _inst.end(tok)


def gru_sensor_bwd_dx(dg: torch.Tensor, w_ih: torch.Tensor, r: torch.Tensor, q0: int, n: int, dr: Optional[torch.Tensor],
                      dxt: Optional[torch.Tensor]) -> None:
    """Raw input gradient at hidden 128 of sequences q0 .. q0 + n - 1 (see ltgnn_gru_sensor_bwd_dx) from their
    ``gru_layer_bwd`` dG [4, n * L, H]: writes their elements of dr (B, L, S) and dxt (B, L, S, F)."""
    b, l, s = r.shape
    f = w_ih.shape[1] - 1
    L = _lib.load()
    tok = _inst.begin("gru_sensor_bwd_dx")
    _lib.check(L.ltgnn_gru_sensor_bwd_dx(_dev_index(dg), b, l, s, f, q0, n, w_ih.shape[0] // 3, w_ih.data_ptr(),
                                         dg.data_ptr(), None if dr is None else dr.data_ptr(),
                                         None if dxt is None else dxt.data_ptr(), _stream(dg)))
    _inst.end(tok)


def _sensor_x_aug(r: torch.Tensor, tf: Optional[torch.Tensor], q0: int, n: int) -> torch.Tensor:
    """[r | tf | 1 | 0 ...] (n * L, 32) for sequences q0 .. q0 + n - 1: the layer input with the ones column."""
    b, l, s = r.shape
    f = 0 if tf is None else tf.shape[-1]
    q = torch.arange(q0, q0 + n, device=r.device)
    bi, si = q // s, q % s
    x = torch.zeros(n, l, 32, device=r.device, dtype=torch.float32)
    x[:, :, 0] = r[bi, :, si]
    if f:
        x[:, :, 1:1 + f] = tf[bi]
    x[:, :, 1 + f] = 1.0
    return x.view(n * l, 32)


class _SensorGru128(torch.autograd.Function):
    """The shared sensor GRU at hidden 128: h_last (B, S, 128), with back-propagation through time to the four GRU
    parameters and to the inputs r and tf, each only where a gradient is asked for.

    Without gradients (grad mode off, or nothing requires one): T (``gru_sensor_tproj``) and one recurrence launch,
    nothing saved.  With gradients the sequences
    run in slabs (``gru_sensor_slabs``): each slab's training forward saves its gates and states; the backward runs per
    slab ``gru_layer_bwd`` from that slab's rows of dh, then ``gru_sensor_bwd_dx`` if r or tf wants a gradient and
    ``gru_layer_param_grads`` against [r | tf | 1] if a parameter does, and adds the slabs' parameter gradients in slab
    order.  At B = 4096, L = 288, S = 29 the saved state alone is 87.5 GB, so the backward's dG and operands (96 GB more
    in one piece) must be formed a slab at a time.  The per-sequence time-feature gradients (F x 4 B per row, 1.2 GB
    there) are kept for all sequences and summed over the sensors after the last slab, since a window's sensors can
    straddle a slab boundary; the slab sizes stay those of the parameter-only backward, so asking for input gradients
    does not change the parameter gradients' bits."""

    @staticmethod
    def _operands(r, tf, w_ih, w_hh, b_ih, b_hh):
        b, l, s = r.shape
        hd = w_hh.shape[1]
        return (gru_sensor_tproj(tf, w_ih, b_ih, b_hh, b, l), w_ih.detach()[:, 0].contiguous(), w_hh.detach().contiguous(),
                b_hh.detach()[2 * hd:].contiguous(), torch.empty(b, s, hd, device=r.device, dtype=torch.float32))

    @staticmethod
    def infer(r, tf, w_ih, w_hh, b_ih, b_hh):
        tproj, w_r, w_hh_c, b_hn, h_last = _SensorGru128._operands(r, tf, w_ih, w_hh, b_ih, b_hh)
        gru_sensor_fwd(r, tproj, w_r, w_hh_c, b_hn, 0, r.shape[0] * r.shape[2], h_last.view(-1, w_hh.shape[1]))
        return h_last

    @staticmethod
    def forward(ctx, r, tf, w_ih, w_hh, b_ih, b_hh):
        r = r.contiguous()
        tf = None if tf is None else tf.contiguous()
        if not any(ctx.needs_input_grad):   # nothing requires a gradient: backward is never reached
            return _SensorGru128.infer(r, tf, w_ih, w_hh, b_ih, b_hh)
        b, l, s = r.shape
        q, hd = b * s, w_hh.shape[1]
        tproj, w_r, w_hh_c, b_hn, h_last = _SensorGru128._operands(r, tf, w_ih, w_hh, b_ih, b_hh)
        flat = h_last.view(q, hd)
        slabs = gru_sensor_slabs(q, l, _dev_index(r))
        saved = []
        for q0, n in slabs:
            hseq = torch.empty(n * l, hd, device=r.device, dtype=torch.float32)
            gates = torch.empty(4, n * l, hd, device=r.device, dtype=torch.float32)
            gru_sensor_fwd(r, tproj, w_r, w_hh_c, b_hn, q0, n, flat[q0:q0 + n], hseq, gates)
            saved += [hseq, gates]
        ctx.save_for_backward(r, tf, w_ih.detach().contiguous(), w_hh_c, *saved)
        ctx.slabs = slabs
        return h_last

    @staticmethod
    def backward(ctx, dh):
        r, tf, w_ih, w_hh, *saved = ctx.saved_tensors
        l = r.shape[1]
        f = 0 if tf is None else tf.shape[-1]
        dh = dh.contiguous().view(-1, w_hh.shape[1])
        dr, dxt = _dx_outputs(r, f, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        want_w = any(ctx.needs_input_grad[2:])
        grads = [None] * 4
        for i, (q0, n) in enumerate(ctx.slabs):
            hseq, gates = saved[2 * i], saved[2 * i + 1]
            dg = gru_layer_bwd(n, l, w_hh, gates, hseq, dh_last=dh[q0:q0 + n])
            if dr is not None or dxt is not None:
                gru_sensor_bwd_dx(dg, w_ih, r, q0, n, dr, dxt)
            if want_w:
                part = gru_layer_param_grads(dg, hseq, _sensor_x_aug(r, tf, q0, n), 1 + f, n, l)
                grads = part if i == 0 else [a + p for a, p in zip(grads, part)]
            del dg
        return (dr, None if dxt is None else dxt.sum(2), *grads)


def tcn_conv(x: torch.Tensor, src: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor,
             gamma: Optional[torch.Tensor] = None, beta: Optional[torch.Tensor] = None, eps: float = 1e-5, relu: bool = True,
             res: Optional[torch.Tensor] = None, res_row: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw gathered-row convolution of the frozen TCN predictor (see ltgnn_tcn_conv):
    ``y[m] = [res[res_row[m]] +] relu(LayerNorm(bias + sum_tap x[src[tap, m]] @ weight[tap].T))``.
    x (rows, 128) fp32 CUDA, src int32 (taps, M) with -1 for the zero padding, weight (taps, 128, 128)."""
    _check_act(x, "x")
    _check_act(weight, "weight")
    taps, m = src.shape
    c = x.shape[-1]
    if src.dtype != torch.int32 or not src.is_cuda or not src.is_contiguous():
        raise ValueError("src must be a contiguous int32 CUDA tensor (taps, M)")
    if tuple(weight.shape) != (taps, c, c):
        raise ValueError(f"weight must be {(taps, c, c)}, got {tuple(weight.shape)}")
    if (res is None) != (res_row is None):
        raise ValueError("res and res_row come together")
    y = torch.empty(m, c, device=x.device, dtype=torch.float32)
    L = _lib.load()
    ws = torch.empty(int(L.ltgnn_tcn_ws_floats(taps)), device=x.device, dtype=torch.float32)   # the packed hi / lo weight
    tok = _inst.begin("tcn_conv")
    _lib.check(L.ltgnn_tcn_conv(_dev_index(x), m, c, taps, x.data_ptr(), src.data_ptr(), weight.data_ptr(), bias.data_ptr(),
                                None if gamma is None else gamma.data_ptr(), None if beta is None else beta.data_ptr(),
                                float(eps), int(relu), None if res is None else res.data_ptr(),
                                None if res_row is None else res_row.data_ptr(), y.data_ptr(), ws.data_ptr(), _stream(x)))
    _inst.end(tok)
    return y


def unblock32(t: torch.Tensor, l: int, q: int) -> torch.Tensor:
    """Blocked-32 saved tensor [L*Qp/32, W/4, 32, 4] -> logical (L, Q, W) (tests / debugging)."""
    w = t.shape[1] * 4
    qp = t.shape[0] * 32 // l
    return t.permute(0, 2, 1, 3).reshape(l, qp, w)[:, :q, :]


# ----------------------------------------------------------------------------------------------
# training of the TCN normal-state predictor on the dependency cone of the last time step (csrc/tcn_train.cu)
# ----------------------------------------------------------------------------------------------
def tcn_conv_train(x: torch.Tensor, src: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, gamma: torch.Tensor,
                   beta: torch.Tensor, eps: float, res: Optional[torch.Tensor] = None, res_row: Optional[torch.Tensor] = None,
                   drop_p: float = 0.0, drop_seed: int = 0):
    """Raw training forward of one gathered-row convolution (see ltgnn_tcn_conv_train):
    ``y[m] = [res[res_row[m]] +] dropout(relu(LayerNorm(z[m])))``, ``z = bias + sum_tap x[src[tap, m]] @ weight[tap].T``.
    Returns ``(y, z, stats, live)``: stats (M, 2) = (mean, rstd) per row, live int32 (M, 4) = the 1-bit record of
    ``dropout(relu(.)) > 0`` (bit b of word w <-> channel 32 w + b)."""
    _check_act(x, "x")
    _check_act(weight, "weight")
    taps, m = src.shape
    c = x.shape[-1]
    if src.dtype != torch.int32 or not src.is_cuda or not src.is_contiguous():
        raise ValueError("src must be a contiguous int32 CUDA tensor (taps, M)")
    if tuple(weight.shape) != (taps, c, c):
        raise ValueError(f"weight must be {(taps, c, c)}, got {tuple(weight.shape)}")
    if (res is None) != (res_row is None):
        raise ValueError("res and res_row come together")
    y = torch.empty(m, c, device=x.device, dtype=torch.float32)
    z = torch.empty(m, c, device=x.device, dtype=torch.float32)
    stats = torch.empty(m, 2, device=x.device, dtype=torch.float32)
    live = torch.empty(m, c // 32, device=x.device, dtype=torch.int32)
    L = _lib.load()
    ws = torch.empty(int(L.ltgnn_tcn_ws_floats(taps)), device=x.device, dtype=torch.float32)
    tok = _inst.begin("tcn_conv_train")
    _lib.check(L.ltgnn_tcn_conv_train(_dev_index(x), m, c, taps, x.data_ptr(), src.data_ptr(), weight.data_ptr(),
                                      bias.data_ptr(), gamma.data_ptr(), beta.data_ptr(), float(eps),
                                      None if res is None else res.data_ptr(), None if res_row is None else res_row.data_ptr(),
                                      float(drop_p), int(drop_seed) & (2**64 - 1), y.data_ptr(), z.data_ptr(),
                                      stats.data_ptr(), live.data_ptr(), ws.data_ptr(), _stream(x)))
    _inst.end(tok)
    return y, z, stats, live


def tcn_ln_bwd(dy: torch.Tensor, live: torch.Tensor, z: torch.Tensor, stats: torch.Tensor, gamma: torch.Tensor,
               scale: float):
    """Raw epilogue backward (see ltgnn_tcn_ln_bwd): ``dz = LayerNorm_bwd(dy * live * scale)`` and the column sums
    ``(d gamma, d beta, d bias)``.  Returns ``(dz, dgamma, dbeta, dbias)``."""
    _check_act(dy, "dy")
    m, c = dy.shape
    dz = torch.empty_like(dy)
    dprm = torch.empty(3, c, device=dy.device, dtype=torch.float32)
    L = _lib.load()
    dev = _dev_index(dy)
    ws = torch.empty(int(L.ltgnn_tcn_ln_bwd_ws_floats(dev)), device=dy.device, dtype=torch.float32)
    tok = _inst.begin("tcn_ln_bwd")
    _lib.check(L.ltgnn_tcn_ln_bwd(dev, m, c, dy.data_ptr(), live.data_ptr(), z.data_ptr(), stats.data_ptr(),
                                  gamma.data_ptr(), float(scale), dz.data_ptr(), dprm.data_ptr(), ws.data_ptr(), _stream(dy)))
    _inst.end(tok)
    return dz, dprm[0], dprm[1], dprm[2]


def tcn_wgrad(dz: torch.Tensor, x: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    """Raw weight gradient over gathered rows (see ltgnn_tcn_wgrad): ``dW[tap] = dz.T @ x[src[tap]]`` (row -1 = zeros),
    returned as (taps, C_out, C_in)."""
    _check_act(dz, "dz")
    _check_act(x, "x")
    taps, m = src.shape
    c = x.shape[-1]
    if dz.shape[0] != m or src.dtype != torch.int32 or not src.is_contiguous():
        raise ValueError("tcn_wgrad: dz (M, C) and a contiguous int32 src (taps, M)")
    dw = torch.empty(taps, c, c, device=dz.device, dtype=torch.float32)
    L = _lib.load()
    dev = _dev_index(dz)
    ws = torch.empty(int(L.ltgnn_tgrad_ws_floats(dev, c)), device=dz.device, dtype=torch.float32)
    tok = _inst.begin("tcn_wgrad")
    _lib.check(L.ltgnn_tcn_wgrad(dev, m, c, taps, dz.data_ptr(), x.data_ptr(), src.data_ptr(), dw.data_ptr(), ws.data_ptr(),
                                 _stream(dz)))
    _inst.end(tok)
    return dw


class _TcnCone(torch.autograd.Function):
    """The TCN predictor's cone as ONE autograd node: input projection -> per block two training convolutions (the
    second with the residual) -> head on the last position; gradients for all parameters, and for the input rows when
    they require grad (the input projection's ``dh`` times its padded weight).

    Backward per convolution: epilogue backward (dz and the LayerNorm / bias column sums), weight gradient over the
    gathered rows, input gradient as the forward's gathered GEMM with the inverse index and the per-tap transposed
    weight (the block input's also receives the block output's gradient on the rows it keeps)."""

    @staticmethod
    def forward(ctx, inp, rows, inv, n_sensors, drop_p, eps, w_in, b_in, *rest):
        n_blk = (len(rest) - 2) // 8
        blocks = [rest[8 * i:8 * i + 8] for i in range(n_blk)]     # conv1 w, b, norm1 w, b, conv2 w, b, norm2 w, b
        w_head, b_head = rest[-2], rest[-1]
        c_in, c = w_in.shape[1], w_in.shape[0]
        kp = inp.shape[1]
        p = float(drop_p)
        w_in_p = torch.zeros(c, kp, device=inp.device, dtype=torch.float32)
        w_in_p[:, :c_in] = w_in[:, :, 0]
        h = linear_tc(inp, w_in_p, b_in.contiguous())
        saved, lives = [], []
        for (w1, b1, g1, e1, w2, b2, g2, e2), (src1, src2, keep) in zip(blocks, rows):
            w1p, w2p = w1.permute(2, 0, 1).contiguous(), w2.permute(2, 0, 1).contiguous()   # (taps, C_out, C_in)
            y1, z1, s1, l1 = tcn_conv_train(h, src1, w1p, b1, g1, e1, eps, drop_p=p,
                                            drop_seed=new_dropout_seed() if p > 0 else 0)
            h2, z2, s2, l2 = tcn_conv_train(y1, src2, w2p, b2, g2, e2, eps, res=h, res_row=keep, drop_p=p,
                                            drop_seed=new_dropout_seed() if p > 0 else 0)
            saved += [h, y1, z1, s1, l1, z2, s2, l2, w1p, w2p, g1, g2]
            lives += [l1, l2]
            h = h2
        if DEBUG_CAPTURE is not None:
            DEBUG_CAPTURE["tcn_lives"] = lives
        n_pad = (n_sensors + 31) // 32 * 32
        w_out = torch.zeros(n_pad, c, device=inp.device, dtype=torch.float32)
        w_out[:n_sensors] = w_head
        b_out = torch.zeros(n_pad, device=inp.device, dtype=torch.float32)
        b_out[:n_sensors] = b_head
        pred = linear_tc(h, w_out, b_out)[:, :n_sensors]
        ctx.save_for_backward(inp, h, w_out, w_in_p, *saved)
        ctx.rows, ctx.inv, ctx.n_blk, ctx.c_in, ctx.n_sensors = rows, inv, n_blk, c_in, n_sensors
        ctx.scale = 1.0 / (1.0 - p)
        return pred

    @staticmethod
    def backward(ctx, dpred):
        inp, h_last, w_out, w_in_p, *saved = ctx.saved_tensors
        s, c = ctx.n_sensors, h_last.shape[1]
        bsz = h_last.shape[0]
        dp = torch.zeros(bsz, 64, device=dpred.device, dtype=torch.float32)   # wgrad_tc takes 64 or 128 output rows
        dp[:, :s] = dpred
        h_aug = torch.zeros(bsz, c + 32, device=dpred.device, dtype=torch.float32)
        h_aug[:, :c] = h_last
        h_aug[:, c] = 1.0                                           # the ones column: its product column is d bias
        t_head = wgrad(dp, h_aug)
        dh = linear_tc(dp[:, :w_out.shape[0]].contiguous(), w_out, transposed=True)
        zero_bias = torch.zeros(c, device=dpred.device, dtype=torch.float32)
        grads = [None] * (8 * ctx.n_blk)
        for i in range(ctx.n_blk - 1, -1, -1):
            h_in, y1, z1, s1, l1, z2, s2, l2, w1p, w2p, g1, g2 = saved[12 * i:12 * i + 12]
            src1, src2, _ = ctx.rows[i]
            inv1, inv2, keep_inv = ctx.inv[i]
            dz2, dg2, de2, db2 = tcn_ln_bwd(dh.contiguous(), l2, z2, s2, g2, ctx.scale)
            dw2 = tcn_wgrad(dz2, y1, src2)
            dy1 = tcn_conv(dz2, inv2, w2p.transpose(1, 2).contiguous(), zero_bias, relu=False)
            dz1, dg1, de1, db1 = tcn_ln_bwd(dy1, l1, z1, s1, g1, ctx.scale)
            dw1 = tcn_wgrad(dz1, h_in, src1)
            dh = tcn_conv(dz1, inv1, w1p.transpose(1, 2).contiguous(), zero_bias, relu=False, res=dh.contiguous(),
                          res_row=keep_inv)
            grads[8 * i:8 * i + 8] = [dw1.permute(1, 2, 0), db1, dg1, de1, dw2.permute(1, 2, 0), db2, dg2, de2]
        t_in = wgrad(dh, inp)
        d_w_in = t_in[:, :ctx.c_in].unsqueeze(-1)
        d_b_in = t_in[:, ctx.c_in].contiguous()
        d_inp = linear_tc(dh, w_in_p, transposed=True) if ctx.needs_input_grad[0] else None
        return (d_inp, None, None, None, None, None, d_w_in, d_b_in, *grads, t_head[:s, :c].contiguous(),
                t_head[:s, c].contiguous())


def tcn_cone(x: torch.Tensor, x_time: torch.Tensor, rows, inv, drop_p: float, eps: float, params) -> torch.Tensor:
    """Differentiable prediction (B, S) of the TCN predictor from its dependency cone on the sm_100a kernels.
    ``rows`` / ``inv``: per block the gather indices and their inverses (NormalPredictorTCN._native_rows /
    _native_inverse); ``params``: the 36 tensors in the order input_proj.{weight, bias}, per block conv1.{weight, bias},
    norm1.{weight, bias}, conv2.{weight, bias}, norm2.{weight, bias}, head.{weight, bias}."""
    _check_act(x.contiguous(), "x")
    b, length, s = x.shape
    c_in = s + x_time.shape[-1]
    kp = 64 if c_in < 64 else 96           # one zero-weight column for the ones that turn the weight gradient into d bias
    inp = torch.zeros(b * length, kp, device=x.device, dtype=torch.float32)
    inp.view(b, length, kp)[:, :, :s] = x
    inp.view(b, length, kp)[:, :, s:c_in] = x_time
    inp[:, c_in] = 1.0
    return _TcnCone.apply(inp, rows, inv, s, float(drop_p), float(eps), *params)


# ----------------------------------------------------------------------------------------------
# input gradients of the frozen predictor's shared windows (``forward_windows`` under autograd): the rows several windows
# read receive the sum of their readers' gradients (csrc/gather_sum.cu)
# ----------------------------------------------------------------------------------------------
def row_gather_sum(src: torch.Tensor, ptr: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """Raw deterministic sum of gathered rows (see ltgnn_row_gather_sum): src (R, C) or planes (P, R, C) fp32 CUDA, C % 4
    == 0; ptr int32 (rows + 1,), idx int32 a CSR whose every entry is a row of src (the host plans build them so) ->
    (rows, C) or (P, rows, C), ``out[.., r] = sum_{e = ptr[r]} ^ {ptr[r+1] - 1} src[.., idx[e]]`` in ascending e."""
    _check_act(src, "src")
    for t, nm in ((ptr, "ptr"), (idx, "idx")):
        if t.dtype != torch.int32 or not t.is_cuda or not t.is_contiguous() or t.dim() != 1:
            raise ValueError(f"{nm} must be a contiguous 1-D int32 CUDA tensor")
    if src.dim() not in (2, 3):
        raise ValueError(f"src must be (rows, C) or (planes, rows, C), got {tuple(src.shape)}")
    planes = src.shape[0] if src.dim() == 3 else 1
    r_in, c = src.shape[-2], src.shape[-1]
    rows = ptr.numel() - 1
    if idx.numel() == 0:                            # no row has a reader: the sums are zeros
        return torch.zeros(*src.shape[:-2], rows, c, device=src.device, dtype=torch.float32)
    out = torch.empty(*src.shape[:-2], rows, c, device=src.device, dtype=torch.float32)
    L = _lib.load()
    tok = _inst.begin("row_gather_sum")
    _lib.check(L.ltgnn_row_gather_sum(_dev_index(src), rows, c, planes, src.data_ptr(), r_in * c, ptr.data_ptr(),
                                      idx.data_ptr(), out.data_ptr(), rows * c, _stream(src)))
    _inst.end(tok)
    return out


class _TcnWindows(torch.autograd.Function):
    """Every window of the frozen TCN predictor from the shared plan (``NormalPredictorTCN.forward_windows``) as ONE
    autograd node, differentiable with respect to its input rows only.

    Forward: ``_native_stack`` with each convolution through ``tcn_conv_train`` at drop_p = 0 (the same values bit for
    bit), saving z, the row statistics and the live mask.  Backward per block, from the last: epilogue backward -> dz;
    per tap the gather-sum of dz into the rows of the convolution's input pool (the reader CSRs: a shared row is read
    through one tap by several windows); one ``tcn_conv`` over the stacked per-tap sums with an identity gather and the
    per-tap transposed weights; the block input also receives the gather-sum of the block output's gradient through the
    residual CSR.  Last, the input projection's transpose.  No weight gradient is computed."""

    @staticmethod
    def forward(ctx, inp, rows, readers, prep, norms, n_sensors):
        h = linear_tc(inp, prep["w_in"], prep["b_in"])
        saved, lives = [], []
        for (w1, w2), (src1, src2, keep), (b1, g1, e1, eps1, b2, g2, e2, eps2) in zip(prep["convs"], rows, norms):
            y1, z1, s1, l1 = tcn_conv_train(h, src1, w1, b1, g1, e1, eps1)
            h, z2, s2, l2 = tcn_conv_train(y1, src2, w2, b2, g2, e2, eps2, res=h, res_row=keep)
            saved += [z1, s1, l1, z2, s2, l2]
            lives += [l1, l2]
        if DEBUG_CAPTURE is not None:
            DEBUG_CAPTURE["tcn_lives"] = lives
        ctx.save_for_backward(*saved)
        ctx.readers, ctx.prep, ctx.norms, ctx.n_sensors = readers, prep, norms, n_sensors
        return linear_tc(h, prep["w_out"], prep["b_out"])[:, :n_sensors]

    @staticmethod
    def backward(ctx, dpred):
        saved, prep = ctx.saved_tensors, ctx.prep
        w_out = prep["w_out"]
        dp = torch.zeros(dpred.shape[0], w_out.shape[0], device=dpred.device, dtype=torch.float32)
        dp[:, :ctx.n_sensors] = dpred
        dh = linear_tc(dp, w_out, transposed=True)
        zero_bias = torch.zeros(dh.shape[1], device=dh.device, dtype=torch.float32)
        for i in range(len(prep["convs"]) - 1, -1, -1):
            z1, s1, l1, z2, s2, l2 = saved[6 * i:6 * i + 6]
            w1, w2 = prep["convs"][i]
            g1, g2 = ctx.norms[i][1], ctx.norms[i][5]
            ptr1, idx1, ptr2, idx2, ptr_r, idx_r, ident1, ident2, ident_r = ctx.readers[i]
            dz2 = tcn_ln_bwd(dh, l2, z2, s2, g2, 1.0)[0]
            dy1 = tcn_conv(row_gather_sum(dz2, ptr2, idx2), ident2, w2.transpose(1, 2).contiguous(), zero_bias,
                           relu=False)
            dz1 = tcn_ln_bwd(dy1, l1, z1, s1, g1, 1.0)[0]
            dh = tcn_conv(row_gather_sum(dz1, ptr1, idx1), ident1, w1.transpose(1, 2).contiguous(), zero_bias,
                          relu=False, res=row_gather_sum(dh, ptr_r, idx_r), res_row=ident_r)
        return linear_tc(dh, prep["w_in"], transposed=True), None, None, None, None, None


def tcn_windows(inp: torch.Tensor, rows, readers, prep, norms, n_sensors: int) -> torch.Tensor:
    """Differentiable ``forward_windows`` of a frozen TCN predictor: inp (B * T, 64) the zero-padded input rows ->
    (B * count, n_sensors).  ``rows`` / ``readers``: NormalPredictorTCN._shared_rows / _shared_readers; ``prep``: its
    _native_weights; ``norms``: per block (conv1 bias, norm1 weight, bias, eps, conv2 bias, norm2 weight, bias, eps)."""
    _check_act(inp.detach(), "inp")
    return _TcnWindows.apply(inp, rows, readers, prep, norms, n_sensors)


class _GruWindows(torch.autograd.Function):
    """Every window of the frozen GRU predictor (``NormalPredictorGRU.forward_windows``) as ONE autograd node,
    differentiable with respect to its input rows only.

    Forward: layer 0 projects the B * T series rows once (as ``gru_predictor_windows``), each window's rows of that
    projection are gathered into the planar form and every layer runs ``gru_layer_fwd_train`` (the inference recurrence's
    values bit for bit), saving its gates.  Backward: BPTT per layer, top down (upper layers take sum_g dG[g] W_ih[g]);
    layer 0's dG planes r, z, n are gather-summed over the windows into series rows (the window CSR), and one
    ``gru_input_grad`` on B * T rows instead of B * count * window gives the input rows' gradient."""

    @staticmethod
    def forward(ctx, inp, window, readers, prep, n_sensors):
        gather, ptr, idx = readers
        layers = prep["layers"]
        w_x, b_x, w_hh, b_hn = layers[0]
        hdim = w_hh.shape[1]
        q = gather.numel() // window
        gx = torch.empty(3, inp.shape[0], hdim, device=inp.device, dtype=torch.float32)
        for g in range(3):
            linear_tc(inp, w_x[g], b_x[g], out=gx[g])
        gx = gx.index_select(1, gather)                         # (3, Q * window, H): window (b, j) at rows of b T + j ..
        saved = []
        for i, (w_x, b_x, w_hh, b_hn) in enumerate(layers):
            if i > 0:
                gx = torch.empty(3, q * window, hdim, device=inp.device, dtype=torch.float32)
                for g in range(3):
                    linear_tc(hseq, w_x[g], b_x[g], out=gx[g])
            h_last, hseq, gates = gru_layer_fwd_train(gx, q, window, w_hh, b_hn)
            del gx
            saved += [hseq, gates]
        ctx.save_for_backward(*saved)
        ctx.window, ctx.readers, ctx.prep, ctx.n_sensors = window, readers, prep, n_sensors
        return linear_tc(h_last, prep["w_out"], prep["b_out"])[:, :n_sensors]

    @staticmethod
    def backward(ctx, dpred):
        saved, prep, l = ctx.saved_tensors, ctx.prep, ctx.window
        _, ptr, idx = ctx.readers
        layers = prep["layers"]
        w_out = prep["w_out"]
        q = dpred.shape[0]
        dp = torch.zeros(q, w_out.shape[0], device=dpred.device, dtype=torch.float32)
        dp[:, :ctx.n_sensors] = dpred
        dh_last, dh_seq = linear_tc(dp, w_out, transposed=True), None
        for i in range(len(layers) - 1, -1, -1):
            w_x, _, w_hh, _ = layers[i]
            hseq, gates = saved[2 * i], saved[2 * i + 1]
            dg = gru_layer_bwd(q, l, w_hh, gates, hseq, dh_last=dh_last, dh_seq=dh_seq)
            if i > 0:
                parts = torch.empty(3, q * l, w_hh.shape[1], device=dg.device, dtype=torch.float32)
                for g in range(3):
                    linear_tc(dg[g], w_x[g], transposed=True, out=parts[g])
                dh_seq, dh_last = gru_dropout_bwd(parts, None, 0.0), None
                del parts
            else:
                d_inp = gru_input_grad(row_gather_sum(dg[:3], ptr, idx), w_x)
            del dg
        return d_inp, None, None, None, None


def gru_windows(inp: torch.Tensor, window: int, readers, prep, n_sensors: int) -> torch.Tensor:
    """Differentiable ``forward_windows`` of a frozen GRU predictor: inp (B * T, 64) the zero-padded input rows ->
    (B * count, n_sensors).  ``readers``: NormalPredictorGRU._window_readers (the forward gather of the window rows and
    its transpose as a CSR); ``prep``: its _native_weights."""
    _check_act(inp.detach(), "inp")
    return _GruWindows.apply(inp, window, readers, prep, n_sensors)
