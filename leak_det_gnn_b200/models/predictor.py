"""Normal-state predictor, API- and checkpoint-compatible with reference models/predictor.py.

The predictor feeds the hot path: detector training runs it frozen on ``l_det`` overlapping windows of every
segment to form the residual sequence (models/utils.py:169-216, train_detector.py:302-307; SURVEY.md section 8f
rank 1).  It contains no graph layers (SURVEY F1).  ``state_dict`` keys equal the reference's
(``input_proj.{weight,bias}``, ``tcn.{i}.conv{1,2}.conv.{weight,bias}``, ``tcn.{i}.norm{1,2}.{weight,bias}``,
``head.{weight,bias}``), so ``predictor_best.ckpt`` files load unchanged.

``forward`` is the reference's dense evaluation (every time step of every layer); ``forward_last`` evaluates only the
dependency cone of the last time step -- the only one the model reads (predictor.py:80): 99 instead of 288
convolution evaluations per window -- and is what the residual builder (models/utils.py) calls.  ``forward_cone`` is
the same cone, differentiable: what ``train_predictor_dp`` trains with.  ``forward_windows`` evaluates every window of a
series from rows computed once; with gradients asked for the inputs of a frozen predictor it is differentiable with
respect to them (``differentiable_windows``), which takes the gradient of the detector's logits back to the raw
sensor series.
"""
from __future__ import annotations

from typing import List, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F


def _differentiable_windows(model: nn.Module, x: torch.Tensor, x_time: torch.Tensor) -> bool:
    """Whether ``forward_windows(x, x_time, ...)`` returns a result differentiable with respect to x and x_time: grad mode
    on, x or x_time requiring grad, the native shared path, and a frozen predictor (no parameter requiring grad: the
    node computes no parameter gradient).  Otherwise ``forward_windows`` runs without gradients."""
    return (torch.is_grad_enabled() and (x.requires_grad or x_time.requires_grad) and model.share_windows
            and model._native_ok(x) and not any(p.requires_grad for p in model.parameters()))


class CausalConv1d(nn.Module):
    """Left-padded dilated convolution: output t sees inputs t, t - d, t - 2 d (predictor.py:17-28)."""

    def __init__(self, in_ch: int, out_ch: int, kernel_size: int, dilation: int = 1) -> None:
        super().__init__()
        self.pad = (kernel_size - 1) * dilation
        self.conv = nn.Conv1d(in_ch, out_ch, kernel_size, dilation=dilation, padding=self.pad)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        y = self.conv(x)
        return y[..., : y.shape[-1] - self.pad] if self.pad > 0 else y


class TCNBlock(nn.Module):
    """x + drop(relu(norm2(conv2(drop(relu(norm1(conv1(x)))))))), LayerNorm over channels (predictor.py:31-52)."""

    def __init__(self, channels: int, kernel_size: int, dilation: int, dropout: float) -> None:
        super().__init__()
        self.conv1 = CausalConv1d(channels, channels, kernel_size, dilation=dilation)
        self.conv2 = CausalConv1d(channels, channels, kernel_size, dilation=dilation)
        self.dropout = nn.Dropout(dropout)
        self.norm1 = nn.LayerNorm(channels)
        self.norm2 = nn.LayerNorm(channels)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        y = x
        for conv, norm in ((self.conv1, self.norm1), (self.conv2, self.norm2)):
            y = self.dropout(F.relu(norm(conv(y).transpose(1, 2)))).transpose(1, 2)
        return x + y


class NormalPredictorTCN(nn.Module):
    """(B, L, S) noisy pressures + (B, L, 9) time features -> (B, S) next-step prediction (predictor.py:55-81)."""

    def __init__(self, num_sensors: int, time_dim: int = 9, hidden_channels: int = 128, kernel_size: int = 3,
                 num_blocks: int = 4, dropout: float = 0.1) -> None:
        super().__init__()
        self.num_sensors = int(num_sensors)
        self.time_dim = int(time_dim)
        self.input_proj = nn.Conv1d(self.num_sensors + self.time_dim, hidden_channels, kernel_size=1)
        self.tcn = nn.Sequential(*[TCNBlock(hidden_channels, kernel_size, 2 ** i, dropout) for i in range(num_blocks)])
        self.head = nn.Linear(hidden_channels, self.num_sensors)

    def forward(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        h = self.input_proj(torch.cat([x, x_time], dim=-1).transpose(1, 2))
        return self.head(self.tcn(h)[:, :, -1])

    # use the hand-written sm_100a kernels for ``forward_last`` on CUDA (csrc/tcn.cu + csrc/linear.cu) where the shapes
    # allow; False = the same cone through torch ops (cuBLAS), kept as the cross-check
    use_native = True
    # ``forward_windows`` computes the rows overlapping windows share once (``shared_cone_plan``); False = ``forward_last``
    # on the materialised windows, kept as the cross-check
    share_windows = True

    def _native_ok(self, x: torch.Tensor) -> bool:
        blk = self.tcn[0]
        return (self.use_native and x.is_cuda and x.dtype == torch.float32 and self.input_proj.out_channels == 128
                and blk.conv1.conv.kernel_size[0] <= 8 and self.num_sensors + self.time_dim <= 64 and self.num_sensors <= 32)

    @torch.no_grad()
    def forward_last(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        """Same result as ``forward`` in eval mode, computing only what the last time step depends on.
        Every convolution becomes one (rows x 3C) @ (3C x C) product over the needed (window, position) rows, with
        zero rows where a tap reaches before the window start (the left padding of CausalConv1d)."""
        if self.training:
            raise RuntimeError("forward_last is the inference path of the frozen predictor (call .eval() first)")
        if self._native_ok(x):
            return self._forward_last_native(x, x_time)
        return self._cone_torch(x, x_time)

    differentiable_windows = _differentiable_windows

    def forward_windows(self, x: torch.Tensor, x_time: torch.Tensor, window: int, count=None) -> torch.Tensor:
        """``forward_last`` of every window of ``window`` steps: x (B, T, S), x_time (B, T, F) -> (B, n, S) with
        ``out[b, j] = forward_last(x[b, j:j + window], x_time[b, j:j + window])``, n = count or T - window + 1.
        On the native path a row of convolution i at window position p >= R_i (the cumulative left reach of convolutions
        0..i) reads no left padding, so it is the same in every window that contains its step: it is computed once per
        (series, step), the input projection once per series row, and only the rows near each window's left edge per
        window (``shared_cone_plan``); the result equals ``forward_last`` on the materialised windows bit for bit.
        When ``differentiable_windows`` holds, the same values come from ONE autograd node (``ops.tcn_windows``) whose
        backward gives d x and d x_time through the shared rows (``_shared_readers``); otherwise no gradient."""
        if self.training:
            raise RuntimeError("forward_windows is the inference path of the frozen predictor (call .eval() first)")
        b, length, _ = x.shape
        n = _window_count(length, window, count)
        if self.differentiable_windows(x, x_time):
            from .. import ops

            dev = x.device
            norms = [(blk.conv1.conv.bias, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps, blk.conv2.conv.bias,
                      blk.norm2.weight, blk.norm2.bias, blk.norm2.eps) for blk in self.tcn]
            return ops.tcn_windows(self._native_input(x, x_time), self._shared_rows(length, window, n, b, dev),
                                   self._shared_readers(length, window, n, b, dev), self._native_weights(dev), norms,
                                   self.num_sensors).view(b, n, -1)
        with torch.no_grad():
            return self._forward_windows(x, x_time, window, n)

    def _forward_windows(self, x: torch.Tensor, x_time: torch.Tensor, window: int, n: int) -> torch.Tensor:
        b, length, _ = x.shape
        if not (self.share_windows and self._native_ok(x)):
            return self.forward_last(windows_of(x, window, n), windows_of(x_time, window, n)).view(b, n, -1)
        from .. import ops

        dev = x.device
        prep = self._native_weights(dev)
        rows = self._shared_rows(length, window, n, b, dev)
        h = ops.linear_tc(self._native_input(x, x_time), prep["w_in"], prep["b_in"])                # (B * T, 128)
        return self._native_stack(h, rows, prep).view(b, n, -1)

    def forward_cone(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        """``forward``'s result, differentiable in train and eval mode, from the dependency cone of the last time step.
        The loss reads only that step, so the parameter gradients are the dense model's (positions outside the cone get
        zero gradient there too), with 34 % of the convolution work at L = 36.  Dropout is the module's (train mode).
        On CUDA at the shapes ``_native_ok`` accepts this is ONE autograd node on the sm_100a kernels
        (``ops.tcn_cone``); otherwise the same cone through torch ops."""
        if not self._native_ok(x):
            return self._cone_torch(x, x_time)
        from .. import ops

        b, length, _ = x.shape
        rows = self._native_rows(length, b, x.device)
        inv = self._native_inverse(length, b, x.device)
        eps = {blk.norm1.eps for blk in self.tcn} | {blk.norm2.eps for blk in self.tcn}
        if len(eps) != 1:
            raise ValueError("forward_cone: the native path takes one LayerNorm eps for all blocks")
        p = self.tcn[0].dropout.p if self.training else 0.0
        params = [self.input_proj.weight, self.input_proj.bias]
        for blk in self.tcn:
            params += [blk.conv1.conv.weight, blk.conv1.conv.bias, blk.norm1.weight, blk.norm1.bias,
                       blk.conv2.conv.weight, blk.conv2.conv.bias, blk.norm2.weight, blk.norm2.bias]
        return ops.tcn_cone(x, x_time, rows, inv, p, eps.pop(), params + [self.head.weight, self.head.bias])

    def _cone_torch(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        """The cone through torch ops: the cross-check of the native kernels and the path of other shapes / devices."""
        b, length, _ = x.shape
        gather = self._cone_plan(length, x.device)
        h = F.linear(torch.cat([x, x_time], dim=-1), self.input_proj.weight[:, :, 0], self.input_proj.bias)  # (B, L, C)
        zero = h.new_zeros(b, 1, h.shape[-1])
        for blk, (taps1, taps2, keep) in zip(self.tcn, gather):
            y = h
            for conv, norm, taps in ((blk.conv1, blk.norm1, taps1), (blk.conv2, blk.norm2, taps2)):
                w = conv.conv.weight.permute(0, 2, 1).reshape(conv.conv.weight.shape[0], -1)   # (C, ks * C), tap-major
                padded = torch.cat([y, zero], dim=1)            # last index = the zero row (left padding)
                rows = padded.index_select(1, taps).view(b, -1, w.shape[1])    # (B, n_out, ks * C)
                y = blk.dropout(F.relu(norm(F.linear(rows, w, conv.conv.bias))))
            h = h.index_select(1, keep) + y
        return self.head(h[:, 0, :])

    def _forward_last_native(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        """The cone on the tensor cores: input projection and output head through ``ops.linear_tc`` (zero-padded to the
        kernel's K / N granularity), every convolution + LayerNorm + ReLU (+ residual) through ``ops.tcn_conv``."""
        from .. import ops

        b, length, _ = x.shape
        dev = x.device
        prep = self._native_weights(dev)
        rows = self._native_rows(length, b, dev)
        h = ops.linear_tc(self._native_input(x, x_time), prep["w_in"], prep["b_in"])                # (B * L, 128)
        return self._native_stack(h, rows, prep)

    def _native_input(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        """cat([x, x_time]) zero-padded to the projection kernel's K = 64: (B * L, 64)."""
        b, length, _ = x.shape
        c_in = self.num_sensors + self.time_dim
        inp = torch.zeros(b, length, 64, device=x.device, dtype=torch.float32)
        inp[:, :, :self.num_sensors] = x
        inp[:, :, self.num_sensors:c_in] = x_time
        return inp.view(b * length, 64)

    def _native_stack(self, h: torch.Tensor, rows, prep) -> torch.Tensor:
        """The blocks and the head on gathered rows: ``rows`` per block (src1, src2, res_row) into the previous row pool
        (``_native_rows`` or ``_shared_rows``), whose last pool holds one row per output, in output order."""
        from .. import ops

        for blk, (w1, w2), (src1, src2, keep_rows) in zip(self.tcn, prep["convs"], rows):
            y = ops.tcn_conv(h, src1, w1, blk.conv1.conv.bias, blk.norm1.weight, blk.norm1.bias, blk.norm1.eps, True)
            h = ops.tcn_conv(y, src2, w2, blk.conv2.conv.bias, blk.norm2.weight, blk.norm2.bias, blk.norm2.eps, True,
                             res=h, res_row=keep_rows)
        return ops.linear_tc(h, prep["w_out"], prep["b_out"])[:, :self.num_sensors]

    def _native_weights(self, device):
        """Weights in the kernels' layouts, rebuilt when a parameter changes (the predictor is frozen in practice)."""
        cache = self.__dict__.setdefault("_native_w", {})
        ver = tuple(p._version for p in self.parameters()) + (str(device),)
        if cache.get("ver") == ver:
            return cache["prep"]
        c_in = self.num_sensors + self.time_dim
        w_in = torch.zeros(128, 64, device=device)
        w_in[:, :c_in] = self.input_proj.weight[:, :, 0]
        w_out = torch.zeros(32, 128, device=device)
        w_out[: self.num_sensors] = self.head.weight
        b_out = torch.zeros(32, device=device)
        b_out[: self.num_sensors] = self.head.bias
        convs = [(blk.conv1.conv.weight.permute(2, 0, 1).contiguous(), blk.conv2.conv.weight.permute(2, 0, 1).contiguous())
                 for blk in self.tcn]                       # (taps, C_out, C_in): tap 0 = the oldest input
        prep = {"w_in": w_in, "b_in": self.input_proj.bias.detach().contiguous(), "w_out": w_out, "b_out": b_out,
                "convs": convs}
        cache.update(ver=ver, prep=prep)
        return prep

    def _native_rows(self, length: int, batch: int, device):
        """Global row indices of the gathered convolutions for ``batch`` windows: per block (src1, src2, keep_rows) with
        src int32 (taps, batch * n_out), -1 = zero padding; activations are laid out (window, position, channel)."""
        cache = self.__dict__.setdefault("_native_r", {})
        key = (length, batch, str(device))
        if key in cache:
            return cache[key]
        ks = self.tcn[0].conv1.conv.kernel_size[0]
        win = torch.arange(batch, device=device, dtype=torch.int64).unsqueeze(1)
        out = []
        n_in = length
        for taps1, taps2, keep in self._cone_plan(length, device):
            rows = []
            n_src = n_in
            for taps in (taps1, taps2):
                rel = taps.view(-1, ks).t()                                   # (ks, n_out), value n_src = the zero row
                n_out = rel.shape[1]
                glob = torch.where(rel.unsqueeze(1) == n_src, torch.full((), -1, device=device, dtype=torch.int64),
                                   win.unsqueeze(0) * n_src + rel.unsqueeze(1))   # (ks, batch, n_out)
                rows.append(glob.reshape(ks, batch * n_out).to(torch.int32).contiguous())
                n_src = n_out
            keep_rows = (win * n_in + keep.unsqueeze(0)).reshape(-1).to(torch.int32).contiguous()
            out.append((rows[0], rows[1], keep_rows))
            n_in = keep.numel()
        if len(cache) > 8:
            cache.clear()
        cache[key] = out
        return out

    def _shared_rows(self, length: int, window: int, count: int, batch: int, device):
        """``shared_cone_plan`` for ``batch`` series in the layout of ``_native_rows`` (int32 on ``device``), built on the
        host once per shape and device: build it outside CUDA-graph capture (a graphed step's warm-up does)."""
        cache = self.__dict__.setdefault("_shared_r", {})
        key = (length, window, count, batch, str(device))
        if key in cache:
            return cache[key]
        plan, _ = shared_cone_plan(length, window, count, batch, self.tcn[0].conv1.conv.kernel_size[0],
                                [blk.conv1.conv.dilation[0] for blk in self.tcn])
        out = [tuple(t.to(device=device, dtype=torch.int32).contiguous() for t in blk) for blk in plan]
        if len(cache) > 8:
            cache.clear()
        cache[key] = out
        return out

    def _shared_readers(self, length: int, window: int, count: int, batch: int, device):
        """The transposes of ``_shared_rows`` for the input gradients (``shared_reader_plan``), int32 on ``device``, per
        block (ptr1, idx1, ptr2, idx2, ptr_res, idx_res, ident1, ident2, ident_res): ident (taps, n) = tap n + r, the
        gather of ``tcn_conv`` over the stacked per-tap sums, and ident_res = arange(n) its residual rows.  Built on the
        host once per shape and device, like ``_shared_rows``: outside CUDA-graph capture."""
        cache = self.__dict__.setdefault("_shared_rd", {})
        key = (length, window, count, batch, str(device))
        if key in cache:
            return cache[key]
        plan, _ = shared_cone_plan(length, window, count, batch, self.tcn[0].conv1.conv.kernel_size[0],
                                   [blk.conv1.conv.dilation[0] for blk in self.tcn])
        out = []
        n_in = batch * length
        for (src1, _, res_row), csr in zip(plan, shared_reader_plan(plan, n_in)):
            ks, n_mid = src1.shape
            ident = [torch.arange(ks * n, dtype=torch.int64).view(ks, n) for n in (n_in, n_mid)]
            out.append(tuple(t.to(device=device, dtype=torch.int32).contiguous()
                             for t in (*csr, *ident, torch.arange(n_in))))
            n_in = res_row.numel()
        if len(cache) > 8:
            cache.clear()
        cache[key] = out
        return out

    def _native_inverse(self, length: int, batch: int, device):
        """Inverses of ``_native_rows`` for the input gradients: per block (inv1, inv2, keep_inv), inv int32 (taps, rows
        of the convolution's input) = the output row that reads input row r through that tap, or -1; keep_inv int32
        (rows of the block input,) = the block output row that keeps input row r as its residual, or -1.  Each map must
        be injective (within a window a fixed tap shifts positions by a constant), which is asserted here."""
        cache = self.__dict__.setdefault("_native_inv", {})
        key = (length, batch, str(device))
        if key in cache:
            return cache[key]

        def invert(idx: torch.Tensor, n_rows: int) -> torch.Tensor:
            idx = idx.view(-1, idx.shape[-1]).long()
            out = torch.full((idx.shape[0], n_rows), -1, device=device, dtype=torch.int64)
            m = torch.arange(idx.shape[1], device=device, dtype=torch.int64)
            for t in range(idx.shape[0]):
                ok = idx[t] >= 0
                hit = idx[t][ok]
                assert hit.unique().numel() == hit.numel(), "gather index is not injective: no gather-form input gradient"
                out[t, hit] = m[ok]
            return out.to(torch.int32).contiguous()

        out = []
        n_in = length
        for (src1, src2, keep_rows), (taps1, _, keep) in zip(self._native_rows(length, batch, device),
                                                              self._cone_plan(length, device)):
            n_mid = taps1.numel() // src1.shape[0]
            out.append((invert(src1, batch * n_in), invert(src2, batch * n_mid), invert(keep_rows, batch * n_in)[0]))
            n_in = keep.numel()
        if len(cache) > 8:
            cache.clear()
        cache[key] = out
        return out

    def _cone_plan(self, length: int, device):
        """Per block: flat tap indices of conv1 / conv2 (oldest tap first, `n_in` = the zero row) and the positions of
        the block input that survive as residual inputs; built once per (length, device)."""
        cache = self.__dict__.setdefault("_cone_cache", {})
        key = (length, str(device))
        if key in cache:
            return cache[key]
        dil = [blk.conv1.conv.dilation[0] for blk in self.tcn]
        ks = self.tcn[0].conv1.conv.kernel_size[0]
        plan = cone_positions(length, ks, dil)
        pos = list(range(length))
        out = []
        for d, (p1, p2) in zip(dil, plan):
            blocks = []
            src = pos
            for out_pos in (p1, p2):
                idx = {t: i for i, t in enumerate(src)}
                sel = [idx.get(t - j * d, len(src)) if t - j * d >= 0 else len(src) for t in out_pos
                       for j in range(ks - 1, -1, -1)]          # weight[:, :, 0] multiplies the OLDEST tap
                blocks.append(torch.tensor(sel, dtype=torch.long, device=device))
                src = out_pos
            idx = {t: i for i, t in enumerate(pos)}
            keep = torch.tensor([idx[t] for t in p2], dtype=torch.long, device=device)
            out.append((blocks[0], blocks[1], keep))
            pos = p2
        assert pos == [length - 1]
        cache[key] = out
        return out


class NormalPredictorGRU(nn.Module):
    """Two-layer GRU baseline (predictor.py:84-111).  ``forward`` is the reference's (cuDNN); ``forward_last`` is the
    frozen predictor's inference path and ``forward_cone`` its differentiable training path, both on the sm_100a kernels
    at hidden 128 (csrc/gru_pred.cu + csrc/linear.cu + csrc/wgrad.cu)."""

    def __init__(self, num_sensors: int, time_dim: int = 9, hidden_size: int = 128, num_layers: int = 2,
                 dropout: float = 0.1) -> None:
        super().__init__()
        self.num_sensors = int(num_sensors)
        self.time_dim = int(time_dim)
        self.gru = nn.GRU(input_size=self.num_sensors + self.time_dim, hidden_size=hidden_size, num_layers=num_layers,
                          batch_first=True, dropout=dropout if num_layers > 1 else 0.0)
        self.head = nn.Linear(hidden_size, self.num_sensors)

    def forward(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        out, _ = self.gru(torch.cat([x, x_time], dim=-1))
        return self.head(out[:, -1, :])

    # use the hand-written sm_100a kernels for ``forward_last`` and ``forward_cone`` on CUDA where the shapes allow;
    # False = the dense cuDNN ``forward``, kept as the cross-check
    use_native = True
    # ``forward_windows`` projects layer 0's input once per series row for all windows; False = ``forward_last`` on the
    # materialised windows, kept as the cross-check
    share_windows = True

    def _native_ok(self, x: torch.Tensor) -> bool:
        g = self.gru
        return (self.use_native and x.is_cuda and x.dtype == torch.float32 and g.hidden_size == 128 and g.bias
                and g.num_layers >= 1 and self.num_sensors + self.time_dim <= 64)

    @torch.no_grad()
    def forward_last(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        """``forward``'s result in eval mode: every layer's recurrence on the tensor cores (``ops.gru_predictor_fwd``),
        the head through ``ops.linear_tc``.  Other shapes and devices run the dense ``forward``."""
        if self.training:
            raise RuntimeError("forward_last is the inference path of the frozen predictor (call .eval() first)")
        if not self._native_ok(x):
            return self.forward(x, x_time)
        from .. import ops

        prep = self._native_weights(x.device)
        h = ops.gru_predictor_fwd(x, x_time, prep["layers"])
        return ops.linear_tc(h, prep["w_out"], prep["b_out"])[:, :self.num_sensors]

    differentiable_windows = _differentiable_windows

    def forward_windows(self, x: torch.Tensor, x_time: torch.Tensor, window: int, count=None) -> torch.Tensor:
        """``forward_last`` of every window of ``window`` steps: x (B, T, S), x_time (B, T, F) -> (B, n, S) with
        ``out[b, j] = forward_last(x[b, j:j + window], x_time[b, j:j + window])``, n = count or T - window + 1.
        Every window restarts the recurrence from a zero state, so only layer 0's input projection is shared: on the
        native path it is computed once per series row and window (b, j) reads rows b T + j .. + window - 1 of it
        (``ops.gru_predictor_windows``), bit for bit the result on the materialised windows.  When
        ``differentiable_windows`` holds, the same values come from ONE autograd node (``ops.gru_windows``) whose
        backward gives d x and d x_time (layer 0's gradient summed over the windows into series rows, ``_window_readers``);
        otherwise no gradient."""
        if self.training:
            raise RuntimeError("forward_windows is the inference path of the frozen predictor (call .eval() first)")
        b, length, _ = x.shape
        n = _window_count(length, window, count)
        if self.differentiable_windows(x, x_time):
            from .. import ops

            prep = self._native_weights(x.device)
            k0 = prep["layers"][0][0].shape[2]
            inp = torch.zeros(b, length, k0, device=x.device, dtype=torch.float32)
            inp[:, :, :self.num_sensors] = x
            inp[:, :, self.num_sensors:self.num_sensors + self.time_dim] = x_time
            return ops.gru_windows(inp.view(b * length, k0), window, self._window_readers(length, window, n, b, x.device),
                                   prep, self.num_sensors).view(b, n, -1)
        with torch.no_grad():
            return self._forward_windows(x, x_time, window, n)

    def _forward_windows(self, x: torch.Tensor, x_time: torch.Tensor, window: int, n: int) -> torch.Tensor:
        b, length, _ = x.shape
        if not (self.share_windows and self._native_ok(x)):
            return self.forward_last(windows_of(x, window, n), windows_of(x_time, window, n)).view(b, n, -1)
        from .. import ops

        prep = self._native_weights(x.device)
        h = ops.gru_predictor_windows(x, x_time, window, n, prep["layers"])
        return ops.linear_tc(h, prep["w_out"], prep["b_out"])[:, :self.num_sensors].view(b, n, -1)

    def forward_cone(self, x: torch.Tensor, x_time: torch.Tensor) -> torch.Tensor:
        """``forward``'s result, differentiable in train and eval mode, with the module's inter-layer dropout in train mode.
        The name is the TCN predictor's: for a GRU the last step's dependency cone is the whole sequence, and
        ``train_predictor_dp`` trains either model through it.  On CUDA at the shapes ``_native_ok`` accepts this is ONE
        autograd node on the sm_100a kernels (``ops.gru_predictor_cone``); otherwise the dense ``forward``."""
        if not self._native_ok(x):
            return self.forward(x, x_time)
        from .. import ops

        g = self.gru
        params = []
        for i in range(g.num_layers):
            params += [getattr(g, f"weight_ih_l{i}"), getattr(g, f"weight_hh_l{i}"), getattr(g, f"bias_ih_l{i}"),
                       getattr(g, f"bias_hh_l{i}")]
        return ops.gru_predictor_cone(x, x_time, g.dropout if self.training else 0.0,
                                      params + [self.head.weight, self.head.bias])

    def _native_weights(self, device):
        """Weights in the kernels' layouts, rebuilt when a parameter changes (the predictor is frozen in practice)."""
        cache = self.__dict__.setdefault("_native_w", {})
        ver = tuple(p._version for p in self.parameters()) + (str(device),)
        if cache.get("ver") == ver:
            return cache["prep"]
        from .. import ops

        g = self.gru
        layers = ops.gru_predictor_weights([(getattr(g, f"weight_ih_l{i}"), getattr(g, f"weight_hh_l{i}"),
                                             getattr(g, f"bias_ih_l{i}"), getattr(g, f"bias_hh_l{i}"))
                                            for i in range(g.num_layers)])
        n_out = (self.num_sensors + 15) // 16 * 16               # the head's N, padded to the kernel's granularity
        w_out = torch.zeros(n_out, g.hidden_size, device=device)
        w_out[: self.num_sensors] = self.head.weight
        b_out = torch.zeros(n_out, device=device)
        b_out[: self.num_sensors] = self.head.bias
        prep = {"layers": layers, "w_out": w_out, "b_out": b_out}
        cache.update(ver=ver, prep=prep)
        return prep

    def _window_readers(self, length: int, window: int, count: int, batch: int, device):
        """(gather, ptr, idx) on ``device``: gather int64 (B * count * window,) = the series row b T + j + p of window row
        (b count + j) window + p, and its transpose ``window_reader_csr`` as int32.  Built on the host once per shape and
        device: outside CUDA-graph capture."""
        cache = self.__dict__.setdefault("_window_rd", {})
        key = (length, window, count, batch, str(device))
        if key in cache:
            return cache[key]
        bs = torch.arange(batch).view(-1, 1, 1)
        gather = (bs * length + torch.arange(count).view(1, -1, 1) + torch.arange(window).view(1, 1, -1)).reshape(-1)
        ptr, idx = window_reader_csr(length, window, count, batch)
        out = (gather.to(device), ptr.to(device=device, dtype=torch.int32), idx.to(device=device, dtype=torch.int32))
        if len(cache) > 8:
            cache.clear()
        cache[key] = out
        return out


def cone_positions(length: int, kernel_size: int, dilations: List[int]) -> List[Tuple[List[int], List[int]]]:
    """Time steps whose values the LAST step depends on, per convolution (two per block), walking backwards:
    element i = (positions needed of conv1's output, positions needed of conv2's output) of block i.
    For L = 36, k = 3, d = 1, 2, 4, 8 that is 36, 18, 18, 9, 9, 5, 3, 1 positions (99) instead of 8 x 36 (288)."""
    need = {length - 1}
    out: List[Tuple[List[int], List[int]]] = []
    for d in reversed(dilations):
        conv2 = sorted(need)                                   # block output positions = conv2 output positions
        conv1 = sorted({t - j * d for t in need for j in range(kernel_size) if t - j * d >= 0})
        need = set(conv1) | need                               # the residual x + y needs x at the block's outputs too
        need = {t - j * d for t in conv1 for j in range(kernel_size) if t - j * d >= 0} | need
        out.append((conv1, conv2))
    return list(reversed(out))


def _window_count(length: int, window: int, count=None) -> int:
    n = length - window + 1 if count is None else int(count)
    if window < 1 or n < 1 or n + window - 1 > length:
        raise ValueError(f"{n} windows of {window} steps do not fit a series of {length} steps")
    return n


def windows_of(x: torch.Tensor, window: int, count: int) -> torch.Tensor:
    """(B, T, C) -> (B * count, window, C): window (b, j) = x[b, j:j + window] at row b * count + j (a copy)."""
    b, _, c = x.shape
    return x.unfold(1, window, 1)[:, :count].permute(0, 1, 3, 2).reshape(b * count, window, c)


def cone_reach(kernel_size: int, dilations: List[int]) -> List[int]:
    """R_i per convolution (two per block): how far left the convolutions 0..i reach together.  A row of convolution i
    at window position p >= R_i reads no left padding, so its value depends on the series alone, not on the window.
    For k = 3 and d = 1, 2, 4, 8: [2, 4, 8, 12, 20, 28, 44, 60]."""
    out, r = [], 0
    for d in dilations:
        for _ in range(2):
            r += (kernel_size - 1) * d
            out.append(r)
    return out


def shared_cone_plan(length: int, window: int, count: int, batch: int, kernel_size: int, dilations: List[int]):
    """Row pools of ``count`` overlapping windows of ``window`` steps per series (window (b, j) = steps j .. j + window - 1
    of series b) that compute every window-independent row once.  The cone of each window is ``cone_positions``; its row
    of convolution i at position p is SHARED, keyed by (series b, step j + p), when p >= R_i (``cone_reach``), and
    WINDOWED, keyed by (window, p), otherwise.  Pool i = [shared rows, series-major then step | windowed rows,
    window-major (b * count + j) then position]; pool -1 = the B * T input-projection rows b * T + t.

    Returns (plan, shared): shared[i] = the shared rows per series of convolution i; plan per block (src1 (k, M1),
    src2 (k, M2), res_row (M2,)) int64 on the CPU, the layout of
    ``NormalPredictorTCN._native_rows``: src1 indexes the block input's pool (oldest tap first, -1 = left padding),
    src2 conv1's pool and res_row the block input's pool.  The last pool holds one row per window in window order:
    windowed when window - 1 < R_last, shared otherwise.  Built with tensor ops over (series, window, position)."""
    if window < 1 or count < 1 or count + window - 1 > length:
        raise ValueError(f"{count} windows of {window} steps do not fit a series of {length} steps")
    cone = [pos for blk in cone_positions(window, kernel_size, dilations) for pos in blk]   # per convolution
    reach = cone_reach(kernel_size, dilations)
    i64 = torch.int64
    bs = torch.arange(batch, dtype=i64).view(-1, 1, 1)        # (B, 1, 1)
    js = torch.arange(count, dtype=i64).view(1, -1, 1)        # (1, n, 1)

    class Pool:
        def __init__(self, shared, windowed, r):
            mask = torch.zeros(length, dtype=torch.bool)
            if shared:
                mask[(torch.tensor(shared, dtype=i64).view(-1, 1) + torch.arange(count, dtype=i64)).view(-1)] = True
            self.steps = mask.nonzero().view(-1)                         # absolute steps of the shared rows
            self.rank_s = torch.cumsum(mask, 0) - 1
            self.rank_s[~mask] = -1
            self.rank_w = torch.full((window,), -1, dtype=i64)
            self.rank_w[torch.tensor(windowed, dtype=i64)] = torch.arange(len(windowed), dtype=i64)
            self.win_pos = torch.tensor(windowed, dtype=i64)
            self.n_s, self.n_w, self.r = self.steps.numel(), len(windowed), r

        def at(self, p):
            """Rows of every window (b, j) at positions p (1-D, may be < 0) -> (B, n, P); -1 for left padding."""
            p = p.view(1, 1, -1)
            pc = p.clamp(min=0)
            rank = torch.where(p >= self.r, self.rank_s[js + pc], self.rank_w[pc])
            assert bool((rank[(p >= 0).expand_as(rank)] >= 0).all()), "a tap reads a row its pool does not hold"
            out = torch.where(p >= self.r, bs * self.n_s + rank, batch * self.n_s + (bs * count + js) * self.n_w + rank)
            return torch.where(p < 0, torch.full_like(out, -1), out)

        def at_steps(self, a):
            """Shared rows of every series at absolute steps a (1-D) -> (B, A)."""
            r = self.rank_s[a]
            assert bool((r >= 0).all()), "a shared row reads a step its pool does not hold"
            return bs.view(-1, 1) * self.n_s + r.view(1, -1)

    def rows(pool_in, pos, r, d):
        """Rows of one convolution: its pool (shared / windowed split of pos at r) and per tap its sources in pool_in."""
        shared = [p for p in pos if p >= r]
        windowed = [p for p in pos if p < r]
        out = Pool(shared, windowed, r)
        taps = []
        for k in range(kernel_size - 1, -1, -1):                # oldest tap first: weight[:, :, 0] multiplies it
            s_rows = pool_in.at_steps(out.steps - k * d).reshape(-1) if out.n_s else torch.empty(0, dtype=i64)
            w_rows = pool_in.at(out.win_pos - k * d).reshape(-1)
            taps.append(torch.cat([s_rows, w_rows]))
        return out, torch.stack(taps)

    def residual(pool_in, out):
        s_rows = pool_in.at_steps(out.steps).reshape(-1) if out.n_s else torch.empty(0, dtype=i64)
        return torch.cat([s_rows, pool_in.at(out.win_pos).reshape(-1)])

    pool = Pool(list(range(window)), [], 0)
    pool.steps, pool.rank_s, pool.n_s = torch.arange(length, dtype=i64), torch.arange(length, dtype=i64), length
    plan, shared = [], []
    for i, d in enumerate(dilations):
        p1, src1 = rows(pool, cone[2 * i], reach[2 * i], d)
        p2, src2 = rows(p1, cone[2 * i + 1], reach[2 * i + 1], d)
        plan.append((src1, src2, residual(pool, p2)))
        shared += [p1.n_s, p2.n_s]
        pool = p2
    # the head reads the last pool as is: one row per window, window-major
    assert (pool.n_w, pool.n_s) == (1, 0) or (pool.n_w == 0 and torch.equal(pool.steps, torch.arange(count) + window - 1))
    return plan, shared


def reader_csr(keys: torch.Tensor, vals: torch.Tensor, n_rows: int):
    """The transpose of a gather as a CSR: row r lists vals[e] for every e with keys[e] == r, in the order of e; keys < 0
    (left padding) are not listed.  keys, vals 1-D int64 -> (ptr (n_rows + 1,), idx) int64 on the CPU."""
    ok = keys >= 0
    keys, vals = keys[ok], vals[ok]
    ptr = torch.zeros(n_rows + 1, dtype=torch.int64)
    ptr[1:] = torch.cumsum(torch.bincount(keys, minlength=n_rows), 0)
    return ptr, vals[torch.sort(keys, stable=True).indices]


def shared_reader_plan(plan, n_input_rows: int):
    """Who reads each row of ``shared_cone_plan``'s pools, for the input gradients: per block (ptr1, idx1, ptr2, idx2,
    ptr_res, idx_res) int64 CSRs.  Convolution c's CSR has one row per (tap, row of its input pool), tap n_src + r, listing
    in ascending order the output rows m with src[tap, m] == r; the residual's has one row per block input row, listing
    the m with res_row[m] == r.  These maps are not injective: a shared row near a window's left edge is read through
    one tap by windowed rows of several neighbouring windows.  ``n_input_rows``: pool -1's rows, B * T."""
    out = []
    n_in = n_input_rows
    for src1, src2, res_row in plan:
        csr = []
        for src, n_src in ((src1, n_in), (src2, src1.shape[1])):
            ks, m = src.shape
            keys = torch.where(src >= 0, src + torch.arange(ks, dtype=torch.int64).view(-1, 1) * n_src, -1)
            csr += reader_csr(keys.reshape(-1), torch.arange(m, dtype=torch.int64).repeat(ks), ks * n_src)
        csr += reader_csr(res_row, torch.arange(res_row.numel(), dtype=torch.int64), n_in)
        out.append(tuple(csr))
        n_in = res_row.numel()
    return out


def window_reader_csr(length: int, window: int, count: int, batch: int):
    """The windows that read each series row: the CSR over series rows b T + t listing the window rows
    (b count + j) window + (t - j), 0 <= t - j < window, in ascending j.  int64 (ptr, idx) on the CPU."""
    bs = torch.arange(batch).view(-1, 1, 1)
    js = torch.arange(count).view(1, -1, 1)
    ps = torch.arange(window).view(1, 1, -1)
    return reader_csr((bs * length + js + ps).reshape(-1), ((bs * count + js) * window + ps).reshape(-1), batch * length)
