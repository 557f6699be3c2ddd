"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product package.

PyG's explainer edge mask and ``GNNExplainer`` on top of ``oracle/pyg_weighted.py`` (used unchanged; without a mask
everything below defers to it).  Restated from PyG 2.x's published source, unpinned like the rest of the restatement:

* ``torch_geometric/explain/algorithm/utils.py`` ``set_masks(model, mask, edge_index, apply_sigmoid)``: every
  ``MessagePassing`` module gets ``explain = True``, ``_edge_mask = mask`` and ``_loop_mask = edge_index[0] !=
  edge_index[1]`` of the *input* ``edge_index``.  One mask serves every layer.
* ``torch_geometric/nn/conv/message_passing.py`` ``explain_message(inputs, dim_size)``: ``inputs`` are the messages
  (for ``GCNConv``, ``norm.view(-1, 1) * x_j`` after ``gcn_norm``).  When there are more messages than mask values
  (``gcn_norm`` appended self loops): ``edge_mask = cat([edge_mask[_loop_mask], ones(dim_size)])``; then
  ``inputs * edge_mask.view(-1, 1)``.  So the mask scales the normalised message, degrees do not see it, the appended
  loops carry 1 and an input self loop's mask value is never used.  The explainer below passes ``sigmoid(m)`` itself
  (``apply_sigmoid`` left to the caller).
* ``torch_geometric/explain/algorithm/gnn_explainer.py`` ``GNNExplainer`` with ``edge_mask_type='object'``, no node
  mask, multiclass classification, raw outputs, ``edge_reduction='sum'``, defaults ``edge_size=0.005``,
  ``edge_ent=1.0``, ``EPS=1e-15``:

      _initialize_masks:  edge_mask = Parameter(randn(E) * calculate_gain('relu') * sqrt(2 / (2 N)))
      _train:             optimizer = Adam([edge_mask], lr)
                          for i in range(epochs):
                              optimizer.zero_grad(); loss = _loss(model(x, edge_index), target); loss.backward()
                              optimizer.step()
                              if i == 0: hard_edge_mask = edge_mask.grad != 0
      _loss:              loss = cross_entropy(y_hat, y)
                          if hard_edge_mask is not None:
                              m = edge_mask[hard_edge_mask].sigmoid()
                              loss += edge_size * m.sum()
                              ent = -m * log(m + EPS) - (1 - m) * log(1 - m + EPS); loss += edge_ent * ent.mean()
      _post_process_mask: sigmoid(edge_mask), entries off hard_edge_mask set to 0

:func:`explain_single` restates that loop for one window; :func:`explain_batched` runs B windows at once with the
loss summed over windows, which is what the device explainer computes.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F

from . import pyg_restatement as _pyg
from . import pyg_weighted as _pw

EPS = 1e-15


def message_mask(edge_index: torch.Tensor, num_nodes: int, edge_mask: torch.Tensor) -> torch.Tensor:
    """explain_message's factor for every message after gcn_norm: the mask on the kept (non-loop) edges, 1 on the
    appended self loops."""
    keep = edge_index[0] != edge_index[1]
    return torch.cat([edge_mask[keep], torch.ones(num_nodes, dtype=edge_mask.dtype, device=edge_mask.device)])


class GCNConv(_pw.GCNConv):
    """``GCNConv`` with PyG's explainer mask; ``call_mask`` is set by :class:`MaskedOracleLeakDetector` around the
    unchanged detector body.  Same parameters and ``state_dict``."""

    call_mask: Optional[torch.Tensor] = None

    def forward(self, x: torch.Tensor, edge_index: torch.Tensor, edge_weight: Optional[torch.Tensor] = None,
                edge_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if edge_mask is None:
            edge_mask = self.call_mask
        if edge_mask is None:
            return super().forward(x, edge_index, edge_weight)
        if edge_weight is None:
            edge_weight = self.call_weight
        ei, norm = _pw.gcn_norm(edge_index, x.size(0), dtype=x.dtype, edge_weight=edge_weight)
        xl = self.lin(x)
        msg = norm.unsqueeze(-1) * xl.index_select(0, ei[0])                       # GCNConv.message
        msg = msg * message_mask(edge_index, x.size(0), edge_mask.to(x.dtype)).unsqueeze(-1)  # explain_message
        out = torch.zeros(x.size(0), xl.size(1), dtype=x.dtype, device=x.device)
        return out.index_add_(0, ei[1], msg) + self.bias


class MaskedOracleLeakDetector(_pw.WeightedOracleLeakDetector):
    """``WeightedOracleLeakDetector`` whose GCN layers all take one explainer mask per call: (E,) over
    ``edge_index_single``'s edges shared by every window, or (B, E), laid out over the replicated graph."""

    def __init__(self, *args, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self.convs = torch.nn.ModuleList([GCNConv(c.in_channels, c.out_channels) for c in self.convs])

    def forward(self, residual: torch.Tensor, tfeat: Optional[torch.Tensor] = None, return_intermediates: bool = False,
                edge_weight: Optional[torch.Tensor] = None, edge_mask: Optional[torch.Tensor] = None):
        return self.gnn_stack(self.sensor_encoder(residual, tfeat), return_intermediates, edge_weight, edge_mask)

    def gnn_stack(self, h_s: torch.Tensor, return_intermediates: bool = False,
                  edge_weight: Optional[torch.Tensor] = None, edge_mask: Optional[torch.Tensor] = None):
        if edge_mask is not None:
            b = h_s.shape[0]
            edge_mask = edge_mask.reshape(-1) if edge_mask.dim() == 2 else edge_mask.repeat(b)
        for conv in self.convs:
            conv.call_mask = edge_mask
        try:
            return super().gnn_stack(h_s, return_intermediates, edge_weight)
        finally:
            for conv in self.convs:
                conv.call_mask = None


def initial_logits(batch: int, num_edges: int, num_nodes: int, generator: torch.Generator) -> torch.Tensor:
    std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (2 * num_nodes))
    return torch.randn(batch, num_edges, generator=generator) * std


def _regulariser(m_hard: torch.Tensor, edge_size: float, edge_ent: float) -> torch.Tensor:
    m = m_hard.sigmoid()
    ent = -m * torch.log(m + EPS) - (1 - m) * torch.log(1 - m + EPS)
    return edge_size * m.sum() + edge_ent * ent.mean()


def explain_single(model, h_s: torch.Tensor, target: int, m0: torch.Tensor, epochs: int = 100, lr: float = 0.01,
                   edge_size: float = 0.005, edge_ent: float = 1.0):
    """PyG's loop, line by line, for ONE window: ``h_s`` (1, S, ds), ``m0`` (E,) initial logits.  Returns
    ``(post-processed mask, hard mask, final logits m)``."""
    edge_mask = torch.nn.Parameter(m0.clone().to(h_s.dtype))
    hard_edge_mask = None
    optimizer = torch.optim.Adam([edge_mask], lr=lr)
    y = torch.tensor([target])
    for i in range(epochs):
        optimizer.zero_grad()
        y_hat = model.gnn_stack(h_s, edge_mask=edge_mask.sigmoid())
        loss = F.cross_entropy(y_hat, y)
        if hard_edge_mask is not None:
            loss = loss + _regulariser(edge_mask[hard_edge_mask], edge_size, edge_ent)
        loss.backward()
        optimizer.step()
        if i == 0:
            hard_edge_mask = edge_mask.grad != 0.0
    out = edge_mask.detach().sigmoid()
    out[~hard_edge_mask] = 0.0
    return out, hard_edge_mask, edge_mask.detach()


def explain_batched(model, h_s: torch.Tensor, target: torch.Tensor, m0: torch.Tensor, epochs: int = 100,
                    lr: float = 0.01, edge_size: float = 0.005, edge_ent: float = 1.0):
    """All B windows at once: (B, E) logits, loss = sum over windows of each window's cross-entropy and regularisers
    (a window without hard entries contributes no regulariser).  Same returns as :func:`explain_single`, (B, E)."""
    edge_mask = torch.nn.Parameter(m0.clone().to(h_s.dtype))
    hard = None
    optimizer = torch.optim.Adam([edge_mask], lr=lr)
    for i in range(epochs):
        optimizer.zero_grad()
        y_hat = model.gnn_stack(h_s, edge_mask=edge_mask.sigmoid())
        loss = F.cross_entropy(y_hat, target, reduction="sum")
        if hard is not None:
            for b in range(h_s.shape[0]):
                if hard[b].any():
                    loss = loss + _regulariser(edge_mask[b][hard[b]], edge_size, edge_ent)
        loss.backward()
        optimizer.step()
        if i == 0:
            hard = edge_mask.grad != 0.0
    out = edge_mask.detach().sigmoid()
    out[~hard] = 0.0
    return out, hard, edge_mask.detach()
