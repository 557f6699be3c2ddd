"""Learned edge masks for the leak detector: PyG's ``GNNExplainer`` on every window of a batch at once.

``explain_edges`` is ``GNNExplainer(epochs, lr)`` with ``edge_mask_type='object'``, no node mask, a multiclass model
with raw outputs and ``edge_reduction='sum'`` (PyG 2.x ``torch_geometric/explain/algorithm/gnn_explainer.py``): one
soft mask per edge, trained with Adam against the cross-entropy of the target class plus ``edge_size`` times the mask's
sum and ``edge_ent`` times its mean entropy, both over the edges the prediction depends on (the "hard" mask: the
entries with a nonzero gradient in the first epoch, which runs without regulariser).  The loss is the sum of every
window's own loss, and Adam is elementwise, so window ``b``'s mask is what PyG's single-window run on window ``b``
learns.

The sensor encoder runs once; only ``gnn_stack`` is inside the loop, with the detector frozen (eval mode, no parameter
requiring a gradient), so the backward launches no weight-gradient kernel.  Epoch 0 runs eagerly, epoch 1 -- masked
forward, cross-entropy, backward to the mask, the fused update ``ltgnn_explain_step`` -- is captured once as a CUDA
graph and replayed for the remaining epochs.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F

from . import ops

__all__ = ["explain_edges", "initial_mask_logits"]


def initial_mask_logits(batch: int, num_edges: int, num_nodes: int,
                        generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """PyG's ``_initialize_masks`` for an object-level edge mask, one row per window, drawn on the host:
    ``randn(B, E) * calculate_gain('relu') * sqrt(2 / (2 N))``."""
    std = torch.nn.init.calculate_gain("relu") * math.sqrt(2.0 / (2 * num_nodes))
    return torch.randn(batch, num_edges, generator=generator) * std


class _MaskState:
    """Device state of one explainer run: the logits ``m``, the mask ``s`` = sigmoid(m) the forward reads, Adam's
    moments and step count, and the hard mask with its per-window counts."""

    def __init__(self, m: torch.Tensor) -> None:
        self.m = m.contiguous()
        self.s = torch.sigmoid(self.m).requires_grad_(True)
        self.exp_avg = torch.zeros_like(self.m)
        self.exp_avg_sq = torch.zeros_like(self.m)
        self.hard = torch.zeros(self.m.shape, device=m.device, dtype=torch.bool)
        self.n_hard = torch.zeros(self.m.shape[0], device=m.device, dtype=torch.int32)
        self.step = torch.zeros(1, device=m.device, dtype=torch.int32)

    def epoch(self, detector, h_s: torch.Tensor, target: torch.Tensor, record: bool, lr: float, edge_size: float,
              edge_ent: float) -> None:
        logits = detector.gnn_stack(h_s, edge_mask=self.s)
        loss = F.cross_entropy(logits, target, reduction="sum")
        (g,) = torch.autograd.grad(loss, self.s)
        ops.explain_step(g, self.m, self.s.detach(), self.exp_avg, self.exp_avg_sq, self.hard, self.n_hard, self.step,
                         record, lr=lr, edge_size=edge_size, edge_ent=edge_ent)


def explain_edges(detector, residual: torch.Tensor, tfeat: Optional[torch.Tensor], target: Optional[torch.Tensor] = None,
                  *, epochs: int = 100, lr: float = 0.01, edge_size: float = 0.005, edge_ent: float = 1.0,
                  generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """Edge masks (B, E) explaining ``detector``'s output on each window of ``residual`` (B, L, S) / ``tfeat``.

    ``target``: ``None`` explains the model's own prediction (argmax of the unmasked logits, PyG's "model"
    explanation); a (B,) long tensor of classes the "phenomenon" explanation (the no-leak class P is allowed).
    Returns sigmoid(logits) with the entries off the hard mask set to 0 (PyG's ``_post_process_mask``).  Edge ``2p``
    and ``2p + 1`` are the two directions of link ``p``: ``mask.view(B, -1, 2)``.  ``generator`` draws the initial
    logits on the host.  The detector's ``training`` flag and its parameters' ``requires_grad`` are restored on return.
    """
    if int(epochs) < 1:
        raise ValueError(f"epochs must be at least 1, got {epochs}")
    params = list(detector.parameters())
    was_training, flags = detector.training, [p.requires_grad for p in params]
    try:
        detector.eval()
        detector.requires_grad_(False)
        with torch.no_grad():
            h_s = detector.sensor_encoder(residual, tfeat)
            if target is None:
                target = detector.gnn_stack(h_s).argmax(-1)
        b = h_s.shape[0]
        n_classes = len(detector.pipe_ids) + 1
        if (not isinstance(target, torch.Tensor) or target.dtype != torch.long or tuple(target.shape) != (b,)
                or target.device != h_s.device):
            raise ValueError(f"target must be a ({b},) long tensor on {h_s.device}")
        if b and (int(target.min()) < 0 or int(target.max()) >= n_classes):
            raise ValueError(f"target classes must lie in [0, {n_classes})")
        e = detector.edge_index_single.shape[1]
        st = _MaskState(initial_mask_logits(b, e, len(detector.node_names), generator).to(h_s.device))
        args = (detector, h_s, target)
        hyper = (lr, edge_size, edge_ent)
        # epoch 0 (no regulariser; records the hard mask) on a side stream doubles as the warm-up before capture
        side = torch.cuda.Stream(device=h_s.device)
        side.wait_stream(torch.cuda.current_stream(h_s.device))
        with torch.cuda.stream(side):
            st.epoch(*args, True, *hyper)
        torch.cuda.current_stream(h_s.device).wait_stream(side)
        if epochs > 1:
            graph = torch.cuda.CUDAGraph()
            with ops.capture(graph):
                st.epoch(*args, False, *hyper)
            for _ in range(int(epochs) - 1):
                graph.replay()
            del graph
        return torch.where(st.hard, st.s.detach(), torch.zeros((), device=h_s.device))
    finally:
        detector.train(was_training)
        for p, f in zip(params, flags):
            p.requires_grad_(f)
