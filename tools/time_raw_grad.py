"""Time the gradient of a frozen LeakDetector's target logits with respect to the raw sensor series: noisy segment ->
frozen normal-state predictor (build_residual_sequence_from_segment) -> frozen detector, logits.gather(1, target).sum()
-> torch.autograd.grad(..., (noisy_seg, time_seg)), forward included.

L-TOWN-A (29 sensors, every pipe of the golden graph as a class), sensor and node width 64, eval mode, every parameter
frozen, at (B, l_pred, l_det) = (256, 36, 36) and (1024, 36, 288), TCN and GRU predictor, two arms on the same seeded
weights and inputs:
  native  the predictor's differentiable shared windows (``forward_windows``: one autograd node, ltgnn_row_gather_sum)
  dense   share_windows = False: the dense ``predictor(x, t)`` on the l_det materialised windows, cuDNN with
          torch.backends.cudnn.allow_tf32 = False; cuDNN's RNN backward runs only in training mode, so for the GRU this
          arm puts the predictor in train mode with its dropout set to 0 (the same function)
Device events around back-to-back calls after warm-up calls, and the peak torch.cuda.max_memory_allocated of each arm.
An arm whose peak at the smaller shape, scaled by the number of windows, exceeds 75 % of the card's memory is not run at
the larger one: its line records the estimate instead of a time (an arm that ran out of memory part-way through a call
leaves work in flight on the device).
For the native arm one more instrumented call records the device time of each library kernel of that call, forward
and backward (instrument.summary()),
and the gather-sum's bytes (gathered rows read once per reader, rows written, ptr and idx) over its kernel time.

    python tools/time_raw_grad.py [--out profiles/r10_time_raw_grad.jsonl]

One JSON line per measurement, with the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from leak_det_gnn_b200 import instrument  # noqa: E402
from leak_det_gnn_b200 import ops  # noqa: E402
from leak_det_gnn_b200.models import (LeakDetector, NormalPredictorGRU, NormalPredictorTCN,  # noqa: E402
                                      build_residual_sequence_from_segment)
from tools.time_input_grad import card, timed  # noqa: E402

SHAPES = ((256, 36, 36, 10, 3), (1024, 36, 288, 3, 1))   # B, l_pred, l_det, timed calls, warm-up calls
HBM_BYTES_PER_S = 7.7e12                                 # HGX B200 data sheet, one GPU
FIT = 0.75                                               # share of the card's memory an arm may be estimated to need


def gather_sum_bytes(launches) -> int:
    """Bytes one backward's ltgnn_row_gather_sum launches need: every gathered row read once per reader, every output
    row written once, ptr and idx read once (per plane for the rows)."""
    return sum(p * (nnz + rows) * c * 4 + (rows + 1 + nnz) * 4 for rows, nnz, c, p in launches)


def run(info, dev) -> list:
    z = np.load(REPO / "tests" / "golden" / "graph_LTA.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    s = len(sensors)
    torch.manual_seed(42)
    det = LeakDetector(REPO / "tests" / "golden" / "L-TOWN-A.topo.inp", sensors, pipes, sensor_hidden=64,
                       node_hidden=64).to(dev).eval().requires_grad_(False)
    lines = []
    total = torch.cuda.mem_get_info(dev)[1]
    peaks = {}                                           # (arch, arm) -> (windows, peak bytes) at the smaller shape
    for arch, cls in (("tcn", NormalPredictorTCN), ("gru", NormalPredictorGRU)):
        torch.manual_seed(7)
        pred = cls(s, 9).to(dev).eval().requires_grad_(False)
        for b, l_pred, l_det, steps, warmup in SHAPES:
            g = torch.Generator(device="cpu").manual_seed(b + l_det)
            noisy = torch.randn(b, l_pred + l_det, s, generator=g).to(dev).requires_grad_(True)
            tseg = torch.randn(b, l_pred + l_det, 9, generator=g).to(dev).requires_grad_(True)
            target = torch.randint(0, len(pipes) + 1, (b, 1), generator=g).to(dev)

            def saliency():
                res = build_residual_sequence_from_segment(pred, noisy, tseg, l_pred, l_det)
                logits = det(res, tseg[:, l_pred:])
                return torch.autograd.grad(logits.gather(1, target).sum(), (noisy, tseg))

            for arm in ("native", "dense"):
                pred.share_windows = arm == "native"
                if arch == "gru":
                    pred.gru.dropout = 0.0 if arm == "dense" else 0.1
                    pred.train(arm == "dense")
                torch.backends.cudnn.allow_tf32 = False
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats()
                line = {"workload": "raw_series_grad", "predictor": arch, "arm": arm, "batch": b, "l_pred": l_pred,
                        "l_det": l_det, "sensors": s, "sensor_hidden": 64, "node_hidden": 64}
                prev = peaks.get((arch, arm))
                need = prev[1] * b * l_det / prev[0] if prev else 0.0
                if need > FIT * total:
                    line.update(ms_per_call=None, error=f"does not fit: ~{need / 2**30:.0f} GiB estimated from the peak "
                                f"at {prev[0]} windows, card {total / 2**30:.0f} GiB")
                    line.update(steps=steps, warmup=warmup, **info)
                    print(json.dumps(line), flush=True)
                    lines.append(line)
                    continue
                try:
                    ms = timed(saliency, steps, warmup)
                    peaks[(arch, arm)] = (b * l_det, torch.cuda.max_memory_allocated())
                    line.update(ms_per_call=round(ms, 4),
                                peak_allocated_gib=round(torch.cuda.max_memory_allocated() / 2**30, 2))
                    if arm == "native":
                        launches = []
                        real = ops.row_gather_sum

                        def counted(src, ptr, idx):
                            launches.append((ptr.numel() - 1, idx.numel(), src.shape[-1],
                                             src.shape[0] if src.dim() == 3 else 1))
                            return real(src, ptr, idx)

                        ops.row_gather_sum = counted
                        instrument.reset(timing=True)
                        try:
                            saliency()
                            torch.cuda.synchronize()
                        finally:
                            ops.row_gather_sum = real
                        summ = instrument.summary()
                        instrument.reset()
                        line["kernel_ms"] = {k: round(v["total_ms"], 4) for k, v in sorted(summ.items())}
                        gs_ms = summ.get("row_gather_sum", {}).get("total_ms", 0.0)
                        nbytes = gather_sum_bytes(launches)
                        line["row_gather_sum"] = {"launches": len(launches), "bytes": nbytes, "ms": round(gs_ms, 4),
                                                  "tb_per_s": round(nbytes / (gs_ms * 1e-3) / 1e12, 3) if gs_ms else None,
                                                  "of_7_7_tb_per_s": round(nbytes / (gs_ms * 1e-3) / HBM_BYTES_PER_S, 3)
                                                  if gs_ms else None}
                except torch.cuda.OutOfMemoryError:
                    line.update(ms_per_call=None, error="out of memory")
                    torch.cuda.synchronize()
                line.update(steps=steps, warmup=warmup, **info)
                print(json.dumps(line), flush=True)
                lines.append(line)
            pred.share_windows = True
            pred.eval()
            del noisy, tseg, target
            torch.cuda.empty_cache()
        del pred
    return lines


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_raw_grad: needs a CUDA device")
    info = card()
    lines = run(info, torch.device("cuda"))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
