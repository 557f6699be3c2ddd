"""Time the gradient of a frozen LeakDetector's target logits with respect to its inputs (residual and time features):
the saliency backward, logits.gather(1, target).sum() -> torch.autograd.grad(..., (residual, tfeat)), forward included.

L-TOWN-A (29 sensors, every pipe of the golden graph as a class), node width 64, eval mode, every parameter frozen, at
(B, L, S) = (256, 36, 29) and (4096, 288, 29), sensor hidden 64 and 128, two arms on the same seeded weights and inputs:
  native      the sensor GRU encoder on the sm_100a kernels (ltgnn_gru_bwd_dx / ltgnn_gru_sensor_bwd_dx after the BPTT)
  cudnn_fp32  the encoder's cuDNN route (use_native = False) with torch.backends.cudnn.allow_tf32 = False; cuDNN's RNN
              backward runs only in training mode, so this arm puts the encoder (one GRU layer, no dropout: the same
              function) in train mode
Device events around back-to-back calls after warm-up calls, and the peak torch.cuda.max_memory_allocated of each arm.
For the native arm one more instrumented call records the device time of each library kernel of the input-gradient
pass (instrument.summary()).

    python tools/time_input_grad.py [--out profiles/r09_time_input_grad.jsonl]

One JSON line per measurement, with the card name and power limit read in the same run.
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

from leak_det_gnn_b200 import instrument  # noqa: E402
from leak_det_gnn_b200.models import LeakDetector  # noqa: E402

SHAPES = ((256, 36, 20, 3), (4096, 288, 3, 1))   # B, L, timed calls, warm-up calls
DX_KERNELS = ("gru_bwd_dg", "gru_bwd_dx", "gru_pred_layer_bwd", "gru_sensor_bwd_dx")


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = (s.strip() for s in out[0].split(",")) if out else (torch.cuda.get_device_name(), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def timed(fn, steps: int, warmup: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def run(info, dev) -> list:
    z = np.load(REPO / "tests" / "golden" / "graph_LTA.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    s = len(sensors)
    lines = []
    for hidden in (64, 128):
        torch.manual_seed(42)
        model = LeakDetector(REPO / "tests" / "golden" / "L-TOWN-A.topo.inp", sensors, pipes, sensor_hidden=hidden,
                             node_hidden=64).to(dev).eval().requires_grad_(False)
        for b, l, steps, warmup in SHAPES:
            g = torch.Generator(device="cpu").manual_seed(b)
            r = torch.randn(b, l, s, generator=g).to(dev).requires_grad_(True)
            tf = torch.randn(b, l, 9, generator=g).to(dev).requires_grad_(True)
            target = torch.randint(0, len(pipes) + 1, (b, 1), generator=g).to(dev)

            def saliency():
                return torch.autograd.grad(model(r, tf).gather(1, target).sum(), (r, tf))

            for arm in ("native", "cudnn_fp32"):
                model.sensor_encoder.use_native = arm == "native"
                model.sensor_encoder.train(arm != "native")
                torch.backends.cudnn.allow_tf32 = False
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats()
                line = {"workload": "detector_input_grad", "arm": arm, "sensor_hidden": hidden, "node_hidden": 64,
                        "batch": b, "l": l, "sensors": s, "sequences": b * s}
                try:
                    ms = timed(saliency, steps, warmup)
                    line.update(ms_per_call=round(ms, 4),
                                peak_allocated_gib=round(torch.cuda.max_memory_allocated() / 2**30, 2))
                    if arm == "native":
                        instrument.reset(timing=True)
                        saliency()
                        torch.cuda.synchronize()
                        summ = instrument.summary()
                        instrument.reset()
                        line["kernel_ms"] = {k: round(v["total_ms"], 4) for k, v in summ.items() if k in DX_KERNELS}
                except torch.cuda.OutOfMemoryError:
                    line.update(ms_per_call=None, error="out of memory")
                line.update(steps=steps, warmup=warmup, **info)
                print(json.dumps(line), flush=True)
                lines.append(line)
            del r, tf, target
        del model
        torch.cuda.empty_cache()
    return lines


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_input_grad: needs a CUDA device")
    info = card()
    lines = run(info, torch.device("cuda"))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
