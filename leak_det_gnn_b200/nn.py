"""Operator-level drop-ins for the two torch_geometric names the reference imports
(models/detector.py:23): ``GCNConv`` and ``global_mean_pool``.

``GCNConv`` keeps PyG's constructor, parameter names (``lin.weight`` [out, in], ``bias``
[out] -> reference checkpoints load unchanged) and init stream (glorot drawn twice, bias
zero).  ``forward`` accepts

* ``conv(x, graph)`` with ``graph`` a :class:`~leak_det_gnn_b200.ops.PipeGraph` and ``x`` of
  shape (B, N, D) or (B*N, D): the fast path -- batch is a dense leading dimension;
* ``conv(x, edge_index)`` with a ``(2, E)`` int64 tensor, PyG's own signature: the graph over
  ``x.size(0)`` nodes is normalised on the host once per distinct ``edge_index`` content
  (the cache keeps its own copy and compares contents) and then runs the same kernels as one big window.

Both take PyG's third argument ``edge_weight``: one weight per edge of ``edge_index`` (the graph's, or the replicated
one's), or with a ``PipeGraph`` also (B, E), one row per window.  The weights are normalised on the device on every call
(``gcn_norm`` with self loops; a node's existing self loop keeps its weight, an added one weighs 1) and are
differentiable.  ``edge_mask`` (same shapes) is PyG's explainer mask: it scales each edge's message after the
normalisation, leaves the added self loops unmasked, and is differentiable (``explain_message`` of PyG 2.x).
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple, Union

import torch
import torch.nn as nn

from . import ops
from .ops import PipeGraph

__all__ = ["GCNConv", "global_mean_pool", "PipeGraph"]


class _GlorotLinear(nn.Module):
    """Bias-free linear whose only parameter is ``weight`` (PyG ``Linear`` naming)."""

    def __init__(self, in_channels: int, out_channels: int) -> None:
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))
        self.reset_parameters()

    def reset_parameters(self) -> None:
        bound = math.sqrt(6.0 / (self.in_channels + self.out_channels))
        with torch.no_grad():
            self.weight.uniform_(-bound, bound)


# PyG-signature path: one normalised graph per distinct ``edge_index`` CONTENT.  The entry keeps its own copy of the
# index tensor (the caller's may be freed and its storage recycled for a different graph of the same size), and a hit is
# confirmed by comparing contents, never by address.
_EDGE_CACHE: List[Tuple[torch.Tensor, int, PipeGraph]] = []


def _graph_from_edge_index(edge_index: torch.Tensor, num_nodes: int) -> PipeGraph:
    for kept, n, g in _EDGE_CACHE:
        if n == num_nodes and kept.shape == edge_index.shape and kept.device == edge_index.device \
                and torch.equal(kept, edge_index):
            return g
    if len(_EDGE_CACHE) >= 8:
        _EDGE_CACHE.pop(0)
    g = PipeGraph(edge_index, num_nodes)
    _EDGE_CACHE.append((edge_index.detach().clone(), num_nodes, g))
    return g


class GCNConv(nn.Module):
    def __init__(self, in_channels: int, out_channels: int, add_self_loops: bool = True, normalize: bool = True,
                 bias: bool = True) -> None:
        super().__init__()
        if not (add_self_loops and normalize):
            raise NotImplementedError("only the reference configuration add_self_loops=True, normalize=True "
                                      "(models/detector.py:162-164) is implemented")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin = _GlorotLinear(in_channels, out_channels)  # glorot draw #1, as PyG's Linear.__init__
        if bias:
            self.bias = nn.Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()  # glorot draw #2, as PyG's GCNConv.reset_parameters

    def reset_parameters(self) -> None:
        self.lin.reset_parameters()
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x: torch.Tensor, graph: Union[PipeGraph, torch.Tensor],
                edge_weight: Optional[torch.Tensor] = None, edge_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if isinstance(graph, torch.Tensor):
            graph = _graph_from_edge_index(graph, x.shape[0] if x.dim() == 2 else x.shape[-2])
        return ops.gcn_conv(x, graph, self.lin.weight, self.bias, edge_weight, edge_mask)

    def extra_repr(self) -> str:
        return f"{self.in_channels}, {self.out_channels}"


def global_mean_pool(x: torch.Tensor, batch: Optional[torch.Tensor], size: Optional[int] = None) -> torch.Tensor:
    """PyG signature.  ``batch`` must be the sorted, equal-sized assignment the reference builds
    (``arange(B).repeat_interleave(N)``, models/detector.py:214); pass ``size=B`` to avoid the
    device->host sync PyG's ``int(batch.max()) + 1`` costs."""
    if batch is None:
        return ops.mean_pool(x.unsqueeze(0))
    if size is None:
        size = int(batch[-1].item()) + 1
    if x.shape[0] % size != 0:
        raise ValueError("global_mean_pool: only equal-sized graphs are supported (fixed pipe network)")
    return ops.mean_pool(x.view(size, x.shape[0] // size, x.shape[1]))
