"""A whole detector TRAINING step as CUDA graph replays (the small-batch path of SURVEY.md section 8d, configs 2 and 4).

The reference's step (models/train_detector.py:296-317) is: residual sequence from the frozen predictor under
``no_grad`` -> ``detector(residual, tfeat)`` -> cross-entropy -> ``backward`` -> ``clip_grad_norm_`` -> ``AdamW.step``.
At the reference's batch sizes (128 by default, 256 in ``cmd.sh``) the sm_100a kernels of that step add up to a
fraction of a millisecond, and what is left is the host: ~60 ctypes launches, the autograd graph, ~100 small torch
kernels for the loss, the gradient views, the clip and the optimiser.  For a FIXED batch shape all of it is the same
launch sequence every step, so it is captured once and replayed:

* world size 1: ONE graph = seed bump + residual builder + forward + loss + backward + clip + optimiser step;
* data parallel: graph A (... + backward into the flat gradient bucket), the eager NCCL all-reduce of the bucket
  (parallel.py), graph B (clip + optimiser step) -- the collective stays outside the capture.

Dropout: a captured launch would replay the ``drop_seed`` it was captured with.  The step owns a 64-bit device word
that the graph increments first thing and that every dropout-bearing kernel adds to its seed at run time
(``ltgnn_seed_source``, include/ltgnn.h), so every replay draws fresh masks, reproducibly under ``torch.manual_seed``.

The warm-up iterations torch needs before a capture run the real step (they initialise lazily built handles, index
tensors and the optimiser state); the parameters are put back and the optimiser state is zeroed afterwards, so the first
``__call__`` is training step 1.  The optimiser must therefore be fresh (no state yet) and ``capturable``.
"""
from __future__ import annotations

from typing import Callable, Optional

import torch

from . import instrument as _inst
from . import ops
from .models.utils import build_residual_sequence_from_segment
from .parallel import FlatGradBucket

__all__ = ["GraphedStep", "GraphedTrainStep"]


class GraphedStep:
    """Capture machinery: ``forward_backward()`` (any callable that zeroes the bucket, runs forward + ``backward`` on
    static device tensors and returns the loss) and the clip + optimiser update, as graph replays around the bucket's
    all-reduce.  ``replay()`` runs one step and returns the static loss tensor.  Dropout-bearing kernels launched by
    ``forward_backward`` are keyed by ``seed_word``, which the graph bumps first (see the module docstring)."""

    def __init__(self, module: torch.nn.Module, forward_backward: Callable[[], torch.Tensor],
                 optimizer: Optional[torch.optim.Optimizer], bucket: FlatGradBucket, grad_clip: float = 0.0, group=None,
                 warmup: int = 3) -> None:
        import torch.distributed as dist

        dev = next(module.parameters()).device
        if dev.type != "cuda":
            raise ValueError("GraphedStep needs the module on a CUDA device")
        if optimizer is not None:
            if len(optimizer.state):
                raise ValueError("GraphedStep needs a fresh optimizer (its warm-up steps are undone by zeroing the state)")
            for g in optimizer.param_groups:
                if "capturable" not in g:
                    raise ValueError(f"{type(optimizer).__name__} has no capturable mode")
                g["capturable"] = True
        self.optimizer, self.bucket, self.grad_clip, self.group = optimizer, bucket, float(grad_clip), group
        self._fb = forward_backward
        self.loss = torch.zeros((), device=dev)
        self.seed_word = torch.zeros(1, dtype=torch.int64, device=dev)
        self.params = [p for p in module.parameters() if p.requires_grad]
        self.split = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.has_update = self.grad_clip > 0 or optimizer is not None

        timing, _inst._timing = _inst._timing, False               # per-kernel event pairs cannot be captured
        keep = [p.detach().clone() for p in module.parameters()]
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                self._forward_backward()
                bucket.allreduce(group)
                self._update()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph_a = torch.cuda.CUDAGraph()
        self.graph_b = torch.cuda.CUDAGraph() if self.split and self.has_update else None
        counted = _inst.launches
        with ops.capture(self.graph_a):
            self._forward_backward()
            if not self.split:
                self._update()
        if self.graph_b is not None:
            with ops.capture(self.graph_b, pool=self.graph_a.pool()):
                self._update()
        self.kernels_per_replay = _inst.launches - counted       # libltgnn launches recorded into the graph(s)
        ops._release_retired()                                   # graph handles collected during the capture
        # undo the warm-up steps: parameters back, optimiser moments and step counts to zero (addresses unchanged)
        with torch.no_grad():
            for p, k in zip(module.parameters(), keep):
                p.copy_(k)
            if optimizer is not None:
                for st in optimizer.state.values():
                    for v in st.values():
                        if torch.is_tensor(v):
                            v.zero_()
            self.seed_word.zero_()
            bucket.zero()
        _inst._timing = timing

    def _forward_backward(self) -> None:
        self.seed_word.add_(1)
        with ops.device_seed(self.seed_word):
            loss = self._fb()
        self.loss.copy_(loss.detach())

    def _update(self) -> None:
        if self.grad_clip > 0:
            torch.nn.utils.clip_grad_norm_(self.params, self.grad_clip)
        if self.optimizer is not None:
            self.optimizer.step()

    def replay(self) -> torch.Tensor:
        """One step on whatever the static input tensors hold."""
        self.graph_a.replay()
        if self.split:
            self.bucket.allreduce(self.group)
            if self.graph_b is not None:
                self.graph_b.replay()
        _inst.launches += self.kernels_per_replay
        return self.loss


class GraphedTrainStep(GraphedStep):
    """``step = GraphedTrainStep(detector, optimizer, bucket, batch, l_det, ...); loss = step(noisy_seg, time_seg, label)``
    -- the reference's training step (train_detector.py:302-317) for one fixed batch shape.

    ``noisy_seg`` (B, l_pred + l_det, S) and ``time_seg`` (B, l_pred + l_det, F) as ``AbruptLeakDetectorDataset`` yields
    them (with ``predictor=None``: the residual (B, l_det, S) and its time features directly), ``label`` (B,) int64.
    Inputs may live on the host (pinned: the copies are asynchronous) or the device.  Returns the step's loss as a
    0-d device tensor that the next call overwrites."""

    def __init__(self, detector, optimizer: Optional[torch.optim.Optimizer], bucket: FlatGradBucket, batch: int, l_det: int,
                 predictor=None, l_pred: int = 0, grad_clip: float = 0.0, n_time: int = 9,
                 loss_fn: Callable = torch.nn.functional.cross_entropy, group=None, warmup: int = 3) -> None:
        dev = next(detector.parameters()).device
        self.detector, self.predictor, self.loss_fn = detector, predictor, loss_fn
        self.l_pred, self.l_det = int(l_pred), int(l_det)
        seg = self.l_det + (self.l_pred if predictor is not None else 0)
        self.noisy = torch.zeros(batch, seg, len(detector.sensor_node_ids), device=dev)
        self.time = torch.zeros(batch, seg, n_time, device=dev)
        self.label = torch.zeros(batch, dtype=torch.long, device=dev)
        detector.train()
        super().__init__(detector, self._detector_step, optimizer, bucket, grad_clip=grad_clip, group=group, warmup=warmup)

    def _detector_step(self) -> torch.Tensor:
        if self.predictor is not None:
            with torch.no_grad():
                residual = build_residual_sequence_from_segment(self.predictor, self.noisy, self.time, l_pred=self.l_pred,
                                                                l_det=self.l_det)
            tfeat = self.time[:, self.l_pred:, :].contiguous()
        else:
            residual, tfeat = self.noisy, self.time
        self.bucket.zero()
        loss = self.loss_fn(self.detector(residual, tfeat), self.label)
        loss.backward()
        return loss

    def __call__(self, noisy_seg: torch.Tensor, time_seg: torch.Tensor, label: torch.Tensor) -> torch.Tensor:
        self.noisy.copy_(noisy_seg, non_blocking=True)
        self.time.copy_(time_seg, non_blocking=True)
        self.label.copy_(label, non_blocking=True)
        return self.replay()
