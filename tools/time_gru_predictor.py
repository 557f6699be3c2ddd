"""Time the residual builder with a frozen GRU normal-state predictor (NormalPredictorGRU(S, 9), hidden 128, two layers)
and one graphed ltown_dp256-shaped detector step with it.

Residual builder (build_residual_sequence_from_segment, l_pred = l_det = 36, S = 29) at B = 128, 256 and 1024 segments
(B x 36 windows), three arms on the same seeded weights and inputs:
  native        forward_last on the sm_100a kernels (csrc/gru_pred.cu + ltgnn_linear)
  cudnn_fp32    the dense cuDNN forward with torch.backends.cudnn.allow_tf32 = False (the fp32 parity setting)
  cudnn_default the dense cuDNN forward with torch's default allow_tf32 = True for cuDNN (TF32 tensor-core math)
and the per-kernel split of the native arm (instrument events, a separate pass).

Detector step: the whole training step of bench.py's ltown_dp256 shape (full L-TOWN, 905 pipes, B = 256, l_det = 36,
hidden 64, clip 1.0, AdamW) as a GraphedTrainStep replay, once with a GRU predictor and once with the TCN predictor.

    python tools/time_gru_predictor.py [--steps 200] [--warmup 20] [--out FILE]

Device events around `steps` back-to-back calls after `warmup` calls; a pool of 4 input batches.  One JSON line per
measurement, with the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from leak_det_gnn_b200 import instrument as inst  # noqa: E402
from leak_det_gnn_b200.models import (LeakDetector, NormalPredictorGRU, NormalPredictorTCN,  # noqa: E402
                                      build_residual_sequence_from_segment)


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = (s.strip() for s in out[0].split(",")) if out else (torch.cuda.get_device_name(), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def timed(fn, pool, steps: int, warmup: int) -> float:
    for i in range(warmup):
        fn(*pool[i % len(pool)])
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        fn(*pool[i % len(pool)])
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def residual_builder(args, info, dev) -> list:
    lines = []
    torch.manual_seed(0)
    pred = NormalPredictorGRU(29, 9).to(dev).eval()
    for b in (128, 256, 1024):
        g = torch.Generator(device="cpu").manual_seed(b)
        pool = [(torch.randn(b, 72, 29, generator=g).to(dev), torch.randn(b, 72, 9, generator=g).to(dev)) for _ in range(4)]

        def build(noisy, tf):
            with torch.no_grad():
                return build_residual_sequence_from_segment(pred, noisy, tf, 36, 36)

        for arm in ("native", "cudnn_fp32", "cudnn_default"):
            pred.use_native = arm == "native"
            torch.backends.cudnn.allow_tf32 = arm == "cudnn_default"
            ms = timed(build, pool, args.steps, args.warmup)
            line = {"workload": "gru_residual_builder", "arm": arm, "segments": b, "windows": b * 36,
                    "ms_per_call": round(ms, 4), "steps": args.steps, "warmup": args.warmup, **info}
            print(json.dumps(line), flush=True)
            lines.append(line)
        pred.use_native = True
        torch.backends.cudnn.allow_tf32 = False
        torch.cuda.synchronize()
        inst.reset(timing=True)
        for i in range(args.steps // 4):
            build(*pool[i % 4])
        torch.cuda.synchronize()
        split = {k: round(v["total_ms"] / (args.steps // 4), 4) for k, v in inst.summary().items()}
        inst.reset()
        line = {"workload": "gru_residual_builder_kernels", "arm": "native", "segments": b, "windows": b * 36,
                "ms_per_call_by_kernel": split, **info}
        print(json.dumps(line), flush=True)
        lines.append(line)
    return lines


def detector_step(args, info, dev) -> list:
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.parallel import FlatGradBucket

    z = np.load(REPO / "tests" / "golden" / "graph_LT.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    b, l_det, l_pred = 256, 36, 36
    g = torch.Generator(device="cpu").manual_seed(198)
    pool = [(torch.randn(b, l_pred + l_det, len(sensors), generator=g).to(dev),
             torch.randn(b, l_pred + l_det, 9, generator=g).to(dev),
             torch.randint(0, len(pipes) + 1, (b,), generator=g).to(dev)) for _ in range(4)]
    lines = []
    for arch in ("tcn", "gru"):
        torch.manual_seed(42)
        model = LeakDetector(REPO / "tests" / "golden" / "L-TOWN.topo.inp", sensors, pipes, sensor_hidden=64, node_hidden=64,
                             gnn_layers=2, dropout=0.1, use_time=True).to(dev).train()
        pred = (NormalPredictorGRU if arch == "gru" else NormalPredictorTCN)(len(sensors), 9).to(dev).eval()
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
        step = GraphedTrainStep(model, opt, FlatGradBucket(model.parameters()), b, l_det, predictor=pred, l_pred=l_pred,
                                grad_clip=1.0)
        ms = timed(step, pool, args.steps, args.warmup)
        line = {"workload": "ltown_dp256_graphed_step", "predictor": arch, "batch": b, "windows": b * l_det,
                "ms_per_step": round(ms, 4), "steps": args.steps, "warmup": args.warmup, **info}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del step, opt, model, pred
    return lines


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_gru_predictor: needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    lines = residual_builder(args, info, dev) + detector_step(args, info, dev)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
