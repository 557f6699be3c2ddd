"""Drop-in ``LeakDetector`` (reference models/detector.py:117-218).

Same constructor, same ``forward(residual[B,L,S], tfeat[B,L,9]) -> logits[B,P+1]``, same
public attributes, and the same 18-tensor ``state_dict`` (SURVEY.md section 8b), so
``ckpt["detector_state"]`` files written by reference ``train_detector.py:346-354`` load
unchanged and the callers (``train_detector.py:246-255,310``, ``window_evaluator.py:326``,
``event_evaluator.py:256,315``) need no edits.

What differs is below the module boundary: the pipe graph is normalised ONCE at construction
(CSR + CSC transpose on the device, :class:`~leak_det_gnn_b200.ops.PipeGraph`) and the batch
is a dense leading dimension, instead of re-materialising a B-times replicated ``edge_index``
and re-running ``gcn_norm`` inside every conv of every forward (detector.py:105-114,195-199).
CUDA only: running it on CPU tensors raises -- there is no fallback path.
"""
from __future__ import annotations

from pathlib import Path
from typing import Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from ..graph import WDNGraph, build_wdn_graph_from_inp
from ..nn import GCNConv
from ..ops import PipeGraph


class SharedSensorGRUEncoder(nn.Module):
    """One GRU shared by all sensors: (B, L, S) residuals [+ (B, L, 9) time features] -> (B, S, hidden)
    (reference detector.py:28-73).  It feeds the hot path (SURVEY.md section 8f, rank 2): hidden size 64 runs on
    the persistent tensor-memory GRU kernel (csrc/gru.cu), hidden size 128 on the 4-CTA cluster recurrence and BPTT
    of csrc/gru_pred.cu with the time-feature projection computed once per window and step (training runs it in
    slabs of sequences).  Both differentiate with respect to the parameters and to the inputs (residual and time
    features, e.g. for saliency), each only where a gradient is asked for.  Other sizes, more than one layer, or
    ``use_native = False`` take the reference's cuDNN route."""

    def __init__(self, time_dim: int = 9, hidden_size: int = 64, num_layers: int = 1, dropout: float = 0.0,
                 use_time: bool = True) -> None:
        super().__init__()
        self.use_time = bool(use_time)
        self.hidden_size = int(hidden_size)
        self.max_seqs_per_call = 8192
        self.use_native = True  # False: run the reference's cuDNN path (kept for comparison)
        self.gru = nn.GRU(input_size=1 + (time_dim if self.use_time else 0), hidden_size=self.hidden_size,
                          num_layers=num_layers, batch_first=True, dropout=dropout if num_layers > 1 else 0.0)

    def forward(self, r: torch.Tensor, tfeat: Optional[torch.Tensor] = None) -> torch.Tensor:
        if self.use_time and tfeat is None:
            raise ValueError("tfeat required when use_time=True")
        g = self.gru
        if (self.use_native and r.is_cuda and g.num_layers == 1 and
                ops.gru_supported(self.hidden_size, tfeat.shape[-1] if self.use_time else 0)):
            # persistent tcgen05 kernels: state in tensor memory, no per-timestep launches (csrc/gru.cu, gru_pred.cu)
            return ops.gru_encode(r, tfeat if self.use_time else None, g.weight_ih_l0, g.weight_hh_l0, g.bias_ih_l0,
                                  g.bias_hh_l0)
        b, l, s = r.shape
        seq = r.transpose(1, 2).reshape(b * s, l, 1)
        if self.use_time:
            if tfeat is None:
                raise ValueError("tfeat required when use_time=True")
            seq = torch.cat([seq, tfeat.unsqueeze(1).expand(b, s, l, tfeat.shape[-1]).reshape(b * s, l, -1)], dim=-1)
        # cuDNN's RNN workspace + reserve grow with (sequences x steps); at B*S ~ 1e5 sequences of 288
        # steps one call asks for > 150 GB.  Sequences are independent, so run them in slabs.
        if seq.shape[0] <= self.max_seqs_per_call:
            out, _ = self.gru(seq)
            return out[:, -1, :].view(b, s, -1)
        last = [self.gru(chunk)[0][:, -1, :] for chunk in seq.split(self.max_seqs_per_call, dim=0)]
        return torch.cat(last, dim=0).view(b, s, -1)


class EdgeHead(nn.Module):
    """Per-pipe logit from [h_u, h_v, |h_u - h_v|] (detector.py:76-88); ``mlp.0`` / ``mlp.3``."""

    def __init__(self, node_dim: int, hidden_dim: int = 128, dropout: float = 0.1) -> None:
        super().__init__()
        self.mlp = nn.Sequential(nn.Linear(node_dim * 3, hidden_dim), nn.ReLU(), nn.Dropout(dropout),
                                 nn.Linear(hidden_dim, 1))

    def forward(self, h_u: torch.Tensor, h_v: torch.Tensor) -> torch.Tensor:
        return self.mlp(torch.cat([h_u, h_v, (h_u - h_v).abs()], dim=-1)).squeeze(-1)


class NoLeakHead(nn.Module):
    """No-leak logit from the mean-pooled node state (detector.py:91-102)."""

    def __init__(self, node_dim: int, hidden_dim: int = 128, dropout: float = 0.1) -> None:
        super().__init__()
        self.mlp = nn.Sequential(nn.Linear(node_dim, hidden_dim), nn.ReLU(), nn.Dropout(dropout),
                                 nn.Linear(hidden_dim, 1))

    def forward(self, pooled: torch.Tensor) -> torch.Tensor:
        return self.mlp(pooled).squeeze(-1)


class LeakDetector(nn.Module):
    def __init__(self, inp_path: str | Path, sensor_node_ids: Sequence[str], pipe_ids_in_order: Sequence[str],
                 sensor_hidden: int = 64, node_hidden: int = 64, gnn_layers: int = 2, dropout: float = 0.1,
                 use_time: bool = True, include_links: Sequence[str] = ("PIPES", "PUMPS", "VALVES")) -> None:
        super().__init__()
        self.graph: WDNGraph = build_wdn_graph_from_inp(
            inp_path=inp_path, sensor_node_ids=sensor_node_ids, pipe_ids_in_order=pipe_ids_in_order,
            include_links=include_links, add_self_loops=False, make_undirected=True)
        # plain attributes, not buffers, exactly like the reference (detector.py:146-155)
        self.node_names = self.graph.node_names
        self.node_to_idx = self.graph.node_to_idx
        self.pipe_ids = self.graph.pipe_ids
        self.pipe_to_idx = self.graph.pipe_to_idx
        self.pipe_ends = torch.tensor(self.graph.pipe_ends, dtype=torch.long)
        self.edge_index_single = self.graph.edge_index
        self.sensor_node_ids = list(sensor_node_ids)
        self.sensor_node_idx = torch.tensor([self.node_to_idx[n] for n in self.sensor_node_ids], dtype=torch.long)

        # normalised CSR/CSC of the single graph: host once, device lazily per GPU
        self.pipe_graph = PipeGraph(self.edge_index_single, len(self.node_names))
        self._dev_cache: dict = {}

        # sub-module construction order == reference (detector.py:158-168): same seeded init stream
        self.sensor_encoder = SharedSensorGRUEncoder(hidden_size=sensor_hidden, use_time=use_time)
        self.sensor_to_node = nn.Linear(sensor_hidden + 1, node_hidden)
        self.convs = nn.ModuleList([GCNConv(node_hidden, node_hidden, add_self_loops=True, normalize=True)
                                    for _ in range(gnn_layers)])
        self.dropout = nn.Dropout(dropout)
        self.edge_head = EdgeHead(node_hidden, hidden_dim=128, dropout=dropout)
        self.noleak_head = NoLeakHead(node_hidden, hidden_dim=128, dropout=dropout)

    # ---- device-side copies of the small index tensors (not buffers: keep state_dict == reference)
    def _index_tensors(self, device: torch.device):
        key = (device.type, device.index)
        hit = self._dev_cache.get(key)
        if hit is None:
            slot = torch.full((len(self.node_names),), -1, dtype=torch.int32)
            slot[self.sensor_node_idx] = torch.arange(len(self.sensor_node_ids), dtype=torch.int32)
            ends32 = self.pipe_ends.to(device=device, dtype=torch.int32)
            hit = (slot.to(device), self.pipe_ends.to(device), ends32, ops.pipe_incidence(ends32, len(self.node_names)))
            self._dev_cache[key] = hit
        return hit

    def gnn_stack(self, h_s: torch.Tensor, edge_weight: Optional[torch.Tensor] = None,
                  edge_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Sensor embeddings (B, S, d_s) -> logits (B, P+1): reference detector.py:178-218, the
        message-passing hot path (SURVEY.md section 8a rows a4-a12).  ``edge_weight``: optional weights of the edges
        of ``edge_index_single`` -- (E,) shared by every window or (B, E) -- used by every GCN layer, as PyG's
        ``conv(x, edge_index, edge_weight)``; edges ``2p`` and ``2p + 1`` are the two directions of link ``p``.  Their
        gradient is the per-pipe attribution of a logit (INTEGRATION section 2).  ``edge_mask``: PyG's explainer
        edge mask, same shapes, on every GCN layer's messages after the normalisation (see :mod:`..explain`)."""
        if not h_s.is_cuda:
            raise ValueError("LeakDetector runs on CUDA only (sm_100a kernels; no CPU fallback)")
        slot, _, ends32, incidence = self._index_tensors(h_s.device)
        conv_params = [t for conv in self.convs for t in (conv.lin.weight, conv.bias)]
        x = ops.gnn_body(h_s, slot, self.pipe_graph, self.dropout.p, self.training, self.sensor_to_node.weight,
                         self.sensor_to_node.bias, conv_params, edge_weight=edge_weight, edge_mask=edge_mask)
        lin1, lin2 = self.edge_head.mlp[0], self.edge_head.mlp[3]
        # pipe head (features formed on the fly, tcgen05) + mean pool; the H -> 1 layer's bias and the tiny no-leak MLP
        # on the pooled (B, D) vector stay in torch.  Node widths other than 64 / 128 raise inside ops.heads.
        part, pooled = ops.heads(x, ends32, lin1.weight, lin1.bias, lin2.weight, self.dropout.p, self.training, incidence)
        pipe_logits = part.sum(0) + lin2.bias
        noleak_logit = self.noleak_head(pooled).unsqueeze(-1)
        return torch.cat([pipe_logits, noleak_logit], dim=-1)

    def embeddings(self, h_s: torch.Tensor) -> torch.Tensor:
        """Sensor embeddings (B, S, d_s) -> node embeddings (B, N, D): PyG's ``get_embeddings(model, ...)[-1]``, the
        last GCN layer's output ``A_hat (x W^T) + b`` before the ReLU and dropout that follow it, computed in eval mode
        without gradient and without a mask -- what PGExplainer's edge network reads (see :mod:`..explain`)."""
        if not h_s.is_cuda:
            raise ValueError("LeakDetector runs on CUDA only (sm_100a kernels; no CPU fallback)")
        slot = self._index_tensors(h_s.device)[0]
        conv_params = [t for conv in self.convs[:-1] for t in (conv.lin.weight, conv.bias)]
        last = self.convs[-1]
        with torch.no_grad():
            x = ops.gnn_body(h_s, slot, self.pipe_graph, 0.0, False, self.sensor_to_node.weight,
                             self.sensor_to_node.bias, conv_params)
            xw = ops._linear_any(x, last.lin.weight)
            return ops.spmm_fused(self.pipe_graph, xw.view(x.shape[0], x.shape[1], -1), bias=last.bias)

    def forward(self, residual: torch.Tensor, tfeat: Optional[torch.Tensor] = None,
                edge_weight: Optional[torch.Tensor] = None, edge_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        h_s = self.sensor_encoder(residual, tfeat)
        return self.gnn_stack(h_s, edge_weight, edge_mask)
