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

``PGExplainer`` is PyG's ``PGExplainer`` (``torch_geometric/explain/algorithm/pg_explainer.py``, graph-level,
phenomenon explanations): one MLP, trained across windows, maps the frozen detector's last-layer node embeddings at the
two ends of an edge to that edge's mask logit, so that explaining a new window is one embedding pass and one MLP pass.
"""
from __future__ import annotations

import contextlib
import math
from typing import Optional

import torch
import torch.nn.functional as F

from . import ops
from .graphed import GraphedStep
from .parallel import FlatGradBucket

__all__ = ["PGExplainer", "explain_edges", "initial_mask_logits"]


def _check_target(target, b: int, n_classes: int, devices) -> None:
    if (not isinstance(target, torch.Tensor) or target.dtype != torch.long or tuple(target.shape) != (b,)
            or target.device not in devices):
        raise ValueError(f"target must be a ({b},) long tensor on {' or '.join(map(str, devices))}")
    if b and (int(target.min()) < 0 or int(target.max()) >= n_classes):
        raise ValueError(f"target classes must lie in [0, {n_classes})")


@contextlib.contextmanager
def _frozen(detector):
    """The detector in eval mode with no parameter requiring a gradient; its flags are restored on exit."""
    params = list(detector.parameters())
    was_training, flags = detector.training, [p.requires_grad for p in params]
    try:
        detector.eval()
        detector.requires_grad_(False)
        yield
    finally:
        detector.train(was_training)
        for p, f in zip(params, flags):
            p.requires_grad_(f)


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
    with _frozen(detector):
        with torch.no_grad():
            h_s = detector.sensor_encoder(residual, tfeat)
            if target is None:
                target = detector.gnn_stack(h_s).argmax(-1)
        b = h_s.shape[0]
        n_classes = len(detector.pipe_ids) + 1
        _check_target(target, b, n_classes, (h_s.device,))
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


class PGExplainer(torch.nn.Module):
    """PyG's ``PGExplainer(epochs, lr, **coeffs)`` for the leak detector, graph-level, with a required "phenomenon"
    target: an edge network ``mlp`` = ``Sequential(Linear(2D, 64), ReLU(), Linear(64, 1))`` (PyG's ``state_dict``
    keys) on ``[z[src] | z[dst]]``, z = ``detector.embeddings`` (the last GCN layer before its ReLU, eval mode, no
    mask).  ``train(epoch, ...)`` is PyG's step on the B windows' disjoint union: temperature ``temp[0] (temp[1] /
    temp[0]) ** (epoch / epochs)``, the concrete sample s, every GCN layer's messages scaled by sigmoid(s), loss =
    mean cross-entropy + ``edge_size`` sum(sigmoid(s)) + ``edge_ent`` mean(H(0.99 sigmoid(s) + 0.005)) over all B E
    edges, one Adam step on the MLP.  ``explain`` gives sigmoid(logit) per edge once training has reached its last
    epoch.  Edge ``2p`` and ``2p + 1`` are the two directions of link ``p``.

    The detector runs frozen (eval mode, no parameter requiring a gradient; restored on return), so its backward
    launches no weight-gradient kernel.  ``graphed=True`` captures the step (embedding, edge network, masked detector,
    loss, backward, Adam) as a CUDA graph at the first ``train`` call and replays it for every later call with the same
    batch size; ``1 / T`` is a device scalar written before each step, and the noise is keyed by a device word the
    graph bumps, so replays draw fresh noise, reproducibly under ``torch.manual_seed``.  Other batch sizes run eagerly."""

    coeffs = {"edge_size": 0.05, "edge_ent": 1.0, "temp": (5.0, 2.0), "bias": 0.01}

    def __init__(self, detector, epochs: int, lr: float = 0.003, graphed: bool = False, **coeffs) -> None:
        super().__init__()
        if int(epochs) < 1:
            raise ValueError(f"epochs must be at least 1, got {epochs}")
        unknown = set(coeffs) - set(PGExplainer.coeffs)
        if unknown:
            raise ValueError(f"unknown coefficients {sorted(unknown)}; PGExplainer takes {sorted(PGExplainer.coeffs)}")
        self.coeffs = {**PGExplainer.coeffs, **coeffs}
        if not 0.0 <= float(self.coeffs["bias"]) <= 0.5:
            raise ValueError(f"bias must lie in [0, 0.5], got {self.coeffs['bias']}")
        self.__dict__["detector"] = detector  # not a submodule: the state_dict is the MLP's alone, as in PyG
        self.epochs, self.lr, self.graphed = int(epochs), float(lr), bool(graphed)
        d = detector.convs[-1].lin.weight.shape[0]
        dev = detector.convs[-1].lin.weight.device
        self.mlp = torch.nn.Sequential(torch.nn.Linear(2 * d, ops.PG_HIDDEN), torch.nn.ReLU(),
                                       torch.nn.Linear(ops.PG_HIDDEN, 1)).to(dev)
        self.optimizer = torch.optim.Adam(self.mlp.parameters(), lr=self.lr, capturable=True)
        self._curr_epoch = -1
        self._dev: dict = {}
        self._step: Optional[GraphedStep] = None

    def train(self, epoch, residual: Optional[torch.Tensor] = None, tfeat: Optional[torch.Tensor] = None,
              target: Optional[torch.Tensor] = None):
        """One training step on the windows ``residual`` (B, L, S) / ``tfeat`` explaining classes ``target`` ((B,) long,
        the no-leak class P allowed; on the host, or on the device at the cost of one host synchronisation for its
        range check).  Returns the loss as a device tensor.  ``train(bool)`` is ``nn.Module.train``."""
        if isinstance(epoch, bool) and residual is None:  # nn.Module.train(mode), e.g. from .eval()
            return super().train(epoch)
        if isinstance(epoch, bool) or not isinstance(epoch, int) or not 0 <= epoch < self.epochs:
            raise ValueError(f"epoch must be an int in [0, {self.epochs}), got {epoch!r}")
        det = self.detector
        with _frozen(det):
            with torch.no_grad():
                h_s = det.sensor_encoder(residual, tfeat)
            dev = h_s.device
            _check_target(target, h_s.shape[0], len(det.pipe_ids) + 1, (dev, torch.device("cpu")))
            target = target.to(dev, non_blocking=True)
            st = self._state(dev)
            t0, t1 = self.coeffs["temp"]
            st["inv_t"].fill_(1.0 / (t0 * pow(t1 / t0, epoch / self.epochs)))
            if self.graphed and (self._step is not None or not self.optimizer.state):
                if self._step is None:
                    st["h_s"], st["target"] = torch.empty_like(h_s), torch.empty_like(target)
                    st["h_s"].copy_(h_s)
                    st["target"].copy_(target)
                    self._step = GraphedStep(self, lambda: self._forward_backward(st["h_s"], st["target"]),
                                             self.optimizer, st["bucket"])
                if st["h_s"].shape == h_s.shape:
                    st["h_s"].copy_(h_s)
                    st["target"].copy_(target)
                    loss = self._step.replay().clone()
                    self._curr_epoch = epoch
                    return loss
            loss = self._forward_backward(h_s, target)
            self.optimizer.step()
        self._curr_epoch = epoch
        return loss.detach()

    @torch.no_grad()
    def explain(self, residual: torch.Tensor, tfeat: Optional[torch.Tensor]) -> torch.Tensor:
        """Edge masks (B, E) = sigmoid(logit) of the trained edge network on each window (no noise, no temperature)."""
        if self._curr_epoch < self.epochs - 1:
            raise ValueError(f"PGExplainer is not yet fully trained (got {self._curr_epoch + 1} epochs from "
                             f"{self.epochs} epochs); run train(epoch, ...) for every epoch first")
        with _frozen(self.detector):
            h_s = self.detector.sensor_encoder(residual, tfeat)
            return self._edge_mask(h_s, None)

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """Load an MLP (PyG's keys ``mlp.0.weight``, ``mlp.0.bias``, ``mlp.2.weight``, ``mlp.2.bias``); the loaded
        network counts as trained, so ``explain`` runs on it."""
        out = super().load_state_dict(state_dict, strict=strict, assign=assign)
        self._curr_epoch = self.epochs - 1
        return out

    def _state(self, dev: torch.device) -> dict:
        st = self._dev.get(dev)
        if st is None:
            det = self.detector
            st = {"idx": ops.pg_edge_index(det.edge_index_single, len(det.node_names), dev),
                  "inv_t": torch.ones(1, device=dev), "bucket": FlatGradBucket(self.mlp.parameters())}
            self._dev[dev] = st
        return st

    def _edge_mask(self, h_s: torch.Tensor, inv_t: Optional[torch.Tensor], seed: int = 0):
        lin1, lin2 = self.mlp[0], self.mlp[2]
        return ops.pg_edge_mask(self.detector.embeddings(h_s), self._state(h_s.device)["idx"], lin1.weight, lin1.bias,
                                lin2.weight, lin2.bias, inv_t, self.coeffs["bias"], seed)

    def _forward_backward(self, h_s: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        st = self._state(h_s.device)
        st["bucket"].zero()
        mask, _ = self._edge_mask(h_s, st["inv_t"], ops.new_dropout_seed())
        logits = self.detector.gnn_stack(h_s, edge_mask=mask)
        m = 0.99 * mask + 0.005
        ent = -m * m.log() - (1 - m) * (1 - m).log()
        loss = F.cross_entropy(logits, target) + self.coeffs["edge_size"] * mask.sum() + self.coeffs["edge_ent"] * ent.mean()
        loss.backward()
        return loss
