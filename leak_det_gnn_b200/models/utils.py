"""Mirror of reference models/utils.py: the graph builder (lines 18-166) and the residual builder (lines 169-216)."""
from __future__ import annotations

from typing import Any, Optional

import torch

from ..graph import WDNGraph, build_wdn_graph_from_inp, parse_epanet_inp  # noqa: F401

__all__ = ["WDNGraph", "build_wdn_graph_from_inp", "parse_epanet_inp", "build_residual_sequence_from_segment",
           "residual_series"]


def _shares_windows(predictor: Any) -> bool:
    """A frozen predictor (eval mode, no gradients) whose ``forward_windows`` computes overlapping windows' shared rows once."""
    return (getattr(predictor, "forward_windows", None) is not None and getattr(predictor, "share_windows", False)
            and not predictor.training and not torch.is_grad_enabled())


def _differentiates_windows(predictor: Any, noisy_seg: torch.Tensor, time_seg: torch.Tensor) -> bool:
    """A frozen predictor in eval mode whose ``forward_windows`` is differentiable with respect to these inputs."""
    diff = getattr(predictor, "differentiable_windows", None)
    return diff is not None and not predictor.training and diff(noisy_seg, time_seg)


def build_residual_sequence_from_segment(predictor: Any, noisy_seg: torch.Tensor, time_seg: torch.Tensor, l_pred: int,
                                         l_det: int, device: Optional[Any] = None) -> torch.Tensor:
    """Residual sequence for the detector from a (l_pred + l_det)-step segment: same arguments, result and window
    order as reference models/utils.py:169-216 (window kk covers steps [kk, kk + l_pred) and predicts step
    l_pred + kk; the predictor sees the l_det * B windows kk-major; ``residual[b, kk] = noisy[b, l_pred + kk] - y_hat``).

    The reference slices and concatenates l_det copies of every window on the host side of the call; here the windows
    are one strided view of the segment, and a frozen TCN predictor is evaluated only on the dependency cone of its
    last time step (``NormalPredictorTCN.forward_last``: 99 instead of 288 convolution evaluations per window).
    A predictor with ``forward_windows`` and ``share_windows`` on runs the l_det windows of every segment in one call that
    computes what they share once (no window is materialised), with the same result bit for bit.  It does so under
    autograd too when the segment requires grad and the predictor is frozen (``differentiable_windows``): the residual
    is then differentiable with respect to ``noisy_seg`` and ``time_seg`` through the shared windows; with
    ``share_windows`` off the dense ``predictor(x, t)`` on the materialised windows gives the same gradients."""
    squeeze_back = noisy_seg.dim() == 2
    if squeeze_back:
        noisy_seg, time_seg = noisy_seg.unsqueeze(0), time_seg.unsqueeze(0)
    b, seg_len, s = noisy_seg.shape
    assert seg_len == l_pred + l_det, (seg_len, l_pred, l_det)
    if device is not None:
        noisy_seg, time_seg = noisy_seg.to(device), time_seg.to(device)

    if _shares_windows(predictor) or _differentiates_windows(predictor, noisy_seg, time_seg):
        y_hat = predictor.forward_windows(noisy_seg, time_seg, l_pred, count=l_det)              # (B, l_det, S)
        residual = noisy_seg[:, l_pred:, :] - y_hat
        return residual.squeeze(0) if squeeze_back else residual

    def windows(seg: torch.Tensor) -> torch.Tensor:  # (B, l_pred + l_det, C) -> (l_det * B, l_pred, C), kk-major
        w = seg.unfold(1, l_pred, 1)[:, :l_det]      # (B, l_det, C, l_pred) view
        return w.permute(1, 0, 3, 2).reshape(l_det * b, l_pred, seg.shape[-1])

    x, t = windows(noisy_seg), windows(time_seg)
    fast = getattr(predictor, "forward_last", None)
    if fast is not None and not predictor.training and not torch.is_grad_enabled():
        y_hat = fast(x, t)
    else:
        y_hat = predictor(x, t)
    if y_hat.dim() == 3:
        y_hat = y_hat[:, -1, :]
    target = noisy_seg[:, l_pred:, :].transpose(0, 1).reshape(l_det * b, s)
    residual = (target - y_hat).view(l_det, b, s).transpose(0, 1).contiguous()
    return residual.squeeze(0) if squeeze_back else residual


@torch.no_grad()
def residual_series(predictor: Any, x: torch.Tensor, x_time: torch.Tensor, l_pred: int,
                    max_windows: int = 16384) -> torch.Tensor:
    """Residual of every predicted step of whole series: x (T, S) or (B, T, S), x_time (T, F) or (B, T, F) ->
    (T - l_pred, S) or (B, T - l_pred, S), row i = step t = l_pred + i: ``x[t] - y_hat(x[t - l_pred:t])``, the value
    the residual builder gives step t in any segment that holds it.  The windows run ``max_windows`` at a time so that
    long series fit; a predictor with ``forward_windows`` shares the rows of overlapping windows (see
    ``build_residual_sequence_from_segment``), any other runs ``forward_last`` (frozen) or its forward per window."""
    squeeze_back = x.dim() == 2
    if squeeze_back:
        x, x_time = x.unsqueeze(0), x_time.unsqueeze(0)
    b, length, s = x.shape
    n = length - l_pred
    if n <= 0:
        out = x.new_empty(b, 0, s)
        return out.squeeze(0) if squeeze_back else out
    per = max(1, max_windows // b)
    shared = _shares_windows(predictor)
    fast = getattr(predictor, "forward_last", None)
    parts = []
    for j0 in range(0, n, per):
        c = min(per, n - j0)
        xs, ts = x[:, j0:j0 + c + l_pred - 1], x_time[:, j0:j0 + c + l_pred - 1]
        if shared:
            y_hat = predictor.forward_windows(xs, ts, l_pred, count=c)
        else:
            xw, tw = (w.unfold(1, l_pred, 1).permute(0, 1, 3, 2).reshape(b * c, l_pred, w.shape[-1]) for w in (xs, ts))
            frozen = fast is not None and not predictor.training
            y_hat = fast(xw, tw) if frozen else predictor(xw, tw)
            if y_hat.dim() == 3:
                y_hat = y_hat[:, -1, :]
            y_hat = y_hat.view(b, c, s)
        parts.append(x[:, l_pred + j0:l_pred + j0 + c] - y_hat)
    out = torch.cat(parts, dim=1) if len(parts) > 1 else parts[0]
    return out.squeeze(0) if squeeze_back else out
