"""Time one training step of a normal-state predictor (MSE -> backward -> clip 1.0 -> AdamW, train mode, dropout 0.1) in
several arms on the same seeded weights and batch.  ``--arch tcn`` (NormalPredictorTCN):

  dense   the reference's step: NormalPredictorTCN.forward (cuDNN convolutions over all 36 time steps), eager torch
  native  forward_cone on the sm_100a kernels (ops.tcn_cone), eager
  graph   the native step as a CUDA graph replay (graphed.GraphedStep, via train_predictor_dp.PredictorStep)

``--arch gru`` (NormalPredictorGRU, 2 layers at hidden 128):

  dense       NormalPredictorGRU.forward (cuDNN GRU) with torch's defaults (cuDNN may use TF32)
  dense_fp32  the same with TF32 off (torch.backends.cudnn.allow_tf32 = False: the fp32 parity setting)
  native      forward_cone on the sm_100a kernels (ops.gru_predictor_cone), eager
  graph       the native step as a CUDA graph replay

    python tools/time_predictor_train.py [--arch tcn|gru] [--batches 256,4096] [--steps 200] [--warmup 20] [--out FILE]

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

from leak_det_gnn_b200.models import NormalPredictorGRU, NormalPredictorTCN  # noqa: E402
from leak_det_gnn_b200.parallel import FlatGradBucket  # noqa: E402
from leak_det_gnn_b200.train_predictor_dp import PredictorStep  # noqa: E402


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = (s.strip() for s in out[0].split(",")) if out else (torch.cuda.get_device_name(), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def make_step(arch: str, arm: str, batch: int, dev):
    torch.manual_seed(0)
    m = (NormalPredictorTCN(29, 9) if arch == "tcn" else NormalPredictorGRU(29, 9)).to(dev).train()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4)   # the reference's; GraphedStep makes it capturable
    torch.backends.cudnn.allow_tf32 = arm != "dense_fp32"                 # torch's default everywhere else
    if arm.startswith("dense"):
        def step(x, xt, y):
            opt.zero_grad(set_to_none=True)
            loss = torch.nn.functional.mse_loss(m(x, xt), y)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            opt.step()
            return loss.detach()
        return step
    return PredictorStep(m, opt, FlatGradBucket(m.parameters()), batch, 1.0, arm == "graph")


def time_recurrence(batch: int, steps: int, warmup: int, dev) -> dict:
    """The GRU's two serial parts alone, one layer at L = 36: the saved-gates forward recurrence and the BPTT."""
    from leak_det_gnn_b200 import ops

    torch.manual_seed(0)
    gru = torch.nn.GRU(128, 128, batch_first=True).to(dev)
    _, _, w_hh, b_hn = ops.gru_predictor_weights([(gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0)],
                                                 k0=128)[0]
    length = 36
    gx = torch.randn(3, batch * length, 128, device=dev)
    dh = torch.randn(batch, 128, device=dev)
    out = {}
    _, hseq, gates = ops.gru_layer_fwd_train(gx, batch, length, w_hh, b_hn)
    for name, fn in (("fwd_train", lambda: ops.gru_layer_fwd_train(gx, batch, length, w_hh, b_hn)),
                     ("bptt", lambda: ops.gru_layer_bwd(batch, length, w_hh, gates, hseq, dh_last=dh))):
        for _ in range(warmup):
            fn()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            fn()
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / steps
        waves = -(-4 * -(-batch // 128) // torch.cuda.get_device_properties(dev).multi_processor_count)
        out[name] = {"ms": round(ms, 4), "us_per_step_and_wave": round(ms * 1e3 / length / waves, 2)}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--arch", default="tcn", choices=["tcn", "gru"])
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
        arms = ("dense", "native", "graph") if args.arch == "tcn" else ("dense", "dense_fp32", "native", "graph")
        for arm in arms:
            step = make_step(args.arch, arm, batch, dev)
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
            line = {"workload": "predictor_train_step" if args.arch == "tcn" else "gru_predictor_train_step", "arm": arm, "batch": batch, "ms_per_step": round(ms, 4),
                    "windows_per_s": round(batch / ms * 1e3, 1), "loss": float(loss), "steps": args.steps,
                    "warmup": args.warmup, **info}
            print(json.dumps(line), flush=True)
            lines.append(line)
            del step
        if args.arch == "gru":
            line = {"workload": "gru_predictor_recurrence", "batch": batch, "L": 36, "hidden": 128,
                    **time_recurrence(batch, args.steps, args.warmup, dev), **info}
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
