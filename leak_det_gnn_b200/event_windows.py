"""Scenario-level ("event") evaluation without one detector call per window (SURVEY.md section 8f rank 3).

The reference slides over every scenario and, for each prediction start ``t0``, builds one (l_pred + l_det)-step segment,
runs the predictor on its l_det windows and calls the detector with B = 1 (eval/event_evaluator.py:478-492): two model
calls, ~60 kernel launches and a device -> host copy per window, thousands of windows per scenario.  Window logits do not
depend on one another (the trigger / aggregation logic that follows only reads them), so here all windows of a scenario
are one strided view of the series and go through the predictor and the detector in large batches:
``scenario_window_logits`` returns exactly the ``records`` the reference accumulates (end index + logits per window).

``GraphedDetector`` covers the case where windows really arrive one at a time (online monitoring): the detector forward
for a fixed batch shape is captured once in a CUDA graph and replayed -- one graph launch instead of ~25 ctypes calls.
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np
import torch

from . import ops
from .models.utils import build_residual_sequence_from_segment, residual_series


@torch.no_grad()
def scenario_window_logits(predictor, detector, pressure_all, tfeat_all, l_pred: int, l_det: int, stride: int, device,
                           batch: int = 1024) -> Tuple[List[int], torch.Tensor]:
    """All windows of one scenario.  pressure_all (T, S), tfeat_all (T, F) -- the standardised series
    event_evaluator.py:455-466 prepares.  Returns (out_end indices, logits (n_windows, C) on the CPU): window i is the
    reference's ``t0 = l_pred + i * stride``, its segment ``[t0 - l_pred, t0 + l_det)`` and its record time
    ``df_sensor.index[out_end - 1]`` (event_evaluator.py:478-492).

    The residual of a step does not depend on the window that reads it, so it is computed once per scenario: at
    stride < l_det the windows read one contiguous range of steps, whose residual series (``residual_series``) every
    window slices; at stride >= l_det no step is read twice and each window's segment goes through the residual builder
    (the steps between windows are never computed).  The detector sees the same batches either way."""
    p = torch.as_tensor(np.asarray(pressure_all), dtype=torch.float32)
    f = torch.as_tensor(np.asarray(tfeat_all), dtype=torch.float32)
    seg_len, n_t = l_pred + l_det, p.shape[0]
    starts = list(range(0, n_t - seg_len + 1, stride))          # in_start = t0 - l_pred
    if not starts:
        return [], torch.empty(0, 0)
    idx = torch.tensor(starts)
    predictor.eval()
    detector.eval()
    out = []
    if stride < l_det:
        end = starts[-1] + seg_len                                # the last step any window reads, + 1
        p_dev, f_dev = p[:end].to(device), f[:end].to(device)
        res = residual_series(predictor, p_dev, f_dev, l_pred)    # row i = step l_pred + i = window start i's first
        res_w = res.unfold(0, l_det, 1)                           # (., S, l_det): window starting at row i
        f_w = f_dev[l_pred:].unfold(0, l_det, 1)
        for lo in range(0, len(starts), batch):
            sel = idx[lo:lo + batch].to(device)
            out.append(detector(res_w[sel].permute(0, 2, 1).contiguous(), f_w[sel].permute(0, 2, 1).contiguous()))
        return [s + seg_len for s in starts], torch.cat(out).cpu()
    seg_p = p.unfold(0, seg_len, 1).permute(0, 2, 1)             # (T - seg_len + 1, seg_len, S) strided view
    seg_f = f.unfold(0, seg_len, 1).permute(0, 2, 1)
    for lo in range(0, len(starts), batch):
        sel = idx[lo:lo + batch]
        noisy = seg_p[sel].contiguous().to(device, non_blocking=True)
        tseg = seg_f[sel].contiguous().to(device, non_blocking=True)
        residual = build_residual_sequence_from_segment(predictor, noisy, tseg, l_pred=l_pred, l_det=l_det, device=device)
        out.append(detector(residual, tseg[:, l_pred:, :].contiguous()))
    return [s + seg_len for s in starts], torch.cat(out).cpu()


class GraphedDetector:
    """``LeakDetector.forward`` (eval mode, no gradients) for ONE fixed input shape as a CUDA graph.

    ``g = GraphedDetector(detector, batch, l_det); logits = g(residual, tfeat)`` copies the inputs into static buffers,
    replays the graph and returns the static output tensor (valid until the next call)."""

    def __init__(self, detector, batch: int, l_det: int, n_time: int = 9) -> None:
        dev = next(detector.parameters()).device
        if dev.type != "cuda":
            raise ValueError("GraphedDetector needs the detector on a CUDA device")
        self.detector = detector.eval()
        self.residual = torch.zeros(batch, l_det, len(detector.sensor_node_ids), device=dev)
        self.tfeat = torch.zeros(batch, l_det, n_time, device=dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side), torch.no_grad():           # warm-up outside the capture: lazy handles, caches
            for _ in range(2):
                self.detector(self.residual, self.tfeat)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), ops.capture(self.graph):
            self.logits = self.detector(self.residual, self.tfeat)

    @torch.no_grad()
    def __call__(self, residual: torch.Tensor, tfeat: torch.Tensor) -> torch.Tensor:
        self.residual.copy_(residual, non_blocking=True)
        self.tfeat.copy_(tfeat, non_blocking=True)
        self.graph.replay()
        return self.logits


__all__ = ["scenario_window_logits", "GraphedDetector"]
