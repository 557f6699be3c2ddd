"""Time one training step of the TCN normal-state predictor (MSE -> backward -> clip 1.0 -> AdamW, train mode, dropout
0.1) in three arms on the same seeded weights and batch:

  dense   the reference's step: NormalPredictorTCN.forward (cuDNN convolutions over all 36 time steps), eager torch
  native  forward_cone on the sm_100a kernels (ops.tcn_cone), eager
  graph   the native step as a CUDA graph replay (graphed.GraphedStep, via train_predictor_dp.PredictorStep)

    python tools/time_predictor_train.py [--batches 256,4096] [--steps 200] [--warmup 20] [--out FILE]

Device events around `steps` back-to-back steps after `warmup` steps; one JSON line per (arm, batch) with the card name and
power limit read in the same run.  The inputs change every step (a pool of 8 batches).
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from leak_det_gnn_b200.models import NormalPredictorTCN  # noqa: E402
from leak_det_gnn_b200.parallel import FlatGradBucket  # noqa: E402
from leak_det_gnn_b200.train_predictor_dp import PredictorStep  # noqa: E402


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = (s.strip() for s in out[0].split(",")) if out else (torch.cuda.get_device_name(), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def make_step(arm: str, batch: int, dev):
    torch.manual_seed(0)
    m = NormalPredictorTCN(29, 9).to(dev).train()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4)   # the reference's; GraphedStep makes it capturable
    if arm == "dense":
        def step(x, xt, y):
            opt.zero_grad(set_to_none=True)
            loss = torch.nn.functional.mse_loss(m(x, xt), y)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            opt.step()
            return loss.detach()
        return step
    return PredictorStep(m, opt, FlatGradBucket(m.parameters()), batch, 1.0, arm == "graph")


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,4096")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_predictor_train: needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    lines = []
    for batch in (int(b) for b in args.batches.split(",")):
        g = torch.Generator(device="cpu").manual_seed(batch)
        pool = [tuple(t.to(dev) for t in (torch.randn(batch, 36, 29, generator=g), torch.randn(batch, 36, 9, generator=g),
                                          torch.randn(batch, 29, generator=g))) for _ in range(8)]
        for arm in ("dense", "native", "graph"):
            step = make_step(arm, batch, dev)
            for i in range(args.warmup):
                step(*pool[i % 8])
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for i in range(args.steps):
                loss = step(*pool[i % 8])
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / args.steps
            line = {"workload": "predictor_train_step", "arm": arm, "batch": batch, "ms_per_step": round(ms, 4),
                    "windows_per_s": round(batch / ms * 1e3, 1), "loss": float(loss), "steps": args.steps,
                    "warmup": args.warmup, **info}
            print(json.dumps(line), flush=True)
            lines.append(line)
            del step
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
