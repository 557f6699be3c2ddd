"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product package.

PyG's ``edge_weight`` on top of the restatement in ``oracle/pyg_restatement.py`` and ``oracle/detector_oracle.py``
(both used unchanged here; without weights everything below defers to them, so every unweighted output is theirs).
Restated from PyG 2.x's published source, unpinned like the rest of the restatement (see pyg_restatement.py):

* ``add_remaining_self_loops(edge_index, edge_weight, fill_value=1)`` (torch_geometric/utils/loop.py): existing self
  loops leave the edge list and one ``(i, i)`` per node is appended; its weight is the node's removed loop's (the last
  one if there were several) or 1.
* ``gcn_norm(edge_index, edge_weight, improved=False, add_self_loops=True)`` (torch_geometric/nn/conv/gcn_conv.py):
  ``deg = scatter_add(w, dst)``, ``dis = deg^-1/2`` with inf -> 0, ``norm = dis[src] * w * dis[dst]``.  Zero and
  negative weights are not rejected (PyG does not check).

Differentiable with respect to ``edge_weight`` (the fp64 truth of the weighted path's gradients): the appended loops'
weights are gathered, so a node's earlier duplicate loops, which the result does not depend on, get gradient 0.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import pyg_restatement as _pyg
from .detector_oracle import OracleLeakDetector


def add_remaining_self_loops(edge_index: torch.Tensor, num_nodes: int,
                             edge_weight: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    out = _pyg.add_remaining_self_loops(edge_index, num_nodes)
    keep = edge_index[0] != edge_index[1]
    last = torch.full((num_nodes,), -1, dtype=torch.long, device=edge_index.device)
    for e in torch.nonzero(~keep).flatten().tolist():  # edge order: the last loop of a node wins
        last[edge_index[0, e]] = e
    loop_w = torch.where(last >= 0, edge_weight[last.clamp(min=0)], torch.ones_like(last, dtype=edge_weight.dtype))
    return out, torch.cat([edge_weight[keep], loop_w])


def gcn_norm(edge_index: torch.Tensor, num_nodes: int, dtype=torch.float32,
             edge_weight: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """``pyg_restatement.gcn_norm`` when ``edge_weight`` is None; otherwise the weighted form (one weight per edge)."""
    if edge_weight is None:
        return _pyg.gcn_norm(edge_index, num_nodes, dtype=dtype)
    edge_index, w = add_remaining_self_loops(edge_index, num_nodes, edge_weight.to(dtype))
    row, col = edge_index[0], edge_index[1]
    deg = torch.zeros(num_nodes, dtype=dtype, device=edge_index.device).scatter_add(0, col, w)
    dis = deg.pow(-0.5)
    dis = dis.masked_fill(dis == float("inf"), 0)
    return edge_index, dis[row] * w * dis[col]


class GCNConv(_pyg.GCNConv):
    """``GCNConv.forward(x, edge_index, edge_weight=None)``; same parameters and ``state_dict`` as the unweighted
    restatement.  ``call_weight`` is the weight a caller without the third argument gets (``None``: unweighted) --
    :class:`WeightedOracleLeakDetector` sets it around the unchanged detector body, which calls ``conv(x, edge_index)``."""

    call_weight: Optional[torch.Tensor] = None

    def forward(self, x: torch.Tensor, edge_index: torch.Tensor, edge_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
        if edge_weight is None:
            edge_weight = self.call_weight
        if edge_weight is None:
            return super().forward(x, edge_index)
        ei, norm = gcn_norm(edge_index, x.size(0), dtype=x.dtype, edge_weight=edge_weight)
        return _pyg.propagate_add(ei, norm, self.lin(x)) + self.bias


class WeightedOracleLeakDetector(OracleLeakDetector):
    """``OracleLeakDetector`` whose GCN layers take one ``edge_weight`` per call, as PyG passes one ``edge_weight`` to
    every conv: (E,) weights of ``edge_index_single``'s edges shared by every window, or (B, E) one row per window,
    laid out over the B-times replicated graph.  Same ``state_dict``; load one (the convs are rebuilt here)."""

    def __init__(self, *args, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self.convs = torch.nn.ModuleList([GCNConv(c.in_channels, c.out_channels) for c in self.convs])

    def forward(self, residual: torch.Tensor, tfeat: Optional[torch.Tensor] = None,
                return_intermediates: bool = False, edge_weight: Optional[torch.Tensor] = None):
        return self.gnn_stack(self.sensor_encoder(residual, tfeat), return_intermediates, edge_weight)

    def gnn_stack(self, h_s: torch.Tensor, return_intermediates: bool = False,
                  edge_weight: Optional[torch.Tensor] = None):
        if edge_weight is not None:
            b = h_s.shape[0]
            edge_weight = edge_weight.reshape(-1) if edge_weight.dim() == 2 else edge_weight.repeat(b)
        for conv in self.convs:
            conv.call_weight = edge_weight
        try:
            return super().gnn_stack(h_s, return_intermediates)
        finally:
            for conv in self.convs:
                conv.call_weight = None
