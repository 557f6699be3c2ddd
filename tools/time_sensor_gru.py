"""Time the shared sensor GRU encoder at hidden 128 (SharedSensorGRUEncoder(hidden_size=128), 9 time features) and one
graphed ltown_dp256-shaped detector step with LeakDetector(sensor_hidden=128).

Encoder, at (B, L, S) = (256, 36, 29) and (4096, 288, 29), with no gradients and forward + backward (a seeded dh), three
arms on the same seeded weights and inputs:
  native        ops.gru_encode on the sm_100a kernels (csrc/gru_pred.cu + ltgnn_linear + ltgnn_wgrad_tc)
  cudnn_fp32    the module's cuDNN route with torch.backends.cudnn.allow_tf32 = False (the fp32 parity setting)
  cudnn_default the cuDNN route with torch's default allow_tf32 = True for cuDNN (TF32 tensor-core math)
The peak torch.cuda.max_memory_allocated of each training arm is recorded; an arm that runs out of memory is recorded
as such.

Detector step: the whole training step of bench.py's ltown_dp256 shape (full L-TOWN, 905 pipes, B = 256, l_det = 36,
node width 64, dropout 0.1, clip 1.0, AdamW, no predictor) as a GraphedTrainStep replay, at sensor_hidden = 128 and, for
comparison, 64.

    python tools/time_sensor_gru.py [--out profiles/r07_time_sensor_gru.jsonl]

Device events around back-to-back calls after warm-up calls.  One JSON line per measurement, with the card name and
power limit read in the same run.
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

from leak_det_gnn_b200.models import LeakDetector  # noqa: E402
from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder  # noqa: E402

SHAPES = ((256, 36, 29, 20, 3), (4096, 288, 29, 3, 1))   # B, L, S, timed calls, warm-up calls


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


def encoder(info, dev) -> list:
    lines = []
    for b, l, s, steps, warmup in SHAPES:
        g = torch.Generator(device="cpu").manual_seed(b)
        r, tf = torch.randn(b, l, s, generator=g).to(dev), torch.randn(b, l, 9, generator=g).to(dev)
        dh = torch.randn(b, s, 128, generator=g).to(dev)
        torch.manual_seed(0)
        enc = SharedSensorGRUEncoder(hidden_size=128).to(dev).train()

        def infer():
            with torch.no_grad():
                enc(r, tf)

        def train():
            (enc(r, tf) * dh).sum().backward()

        for mode, fn in (("no_grad", infer), ("fwd_bwd", train)):
            for arm in ("native", "cudnn_fp32", "cudnn_default"):
                enc.use_native = arm == "native"
                torch.backends.cudnn.allow_tf32 = arm == "cudnn_default"
                enc.zero_grad(set_to_none=True)
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                line = {"workload": "sensor_gru128", "mode": mode, "arm": arm, "batch": b, "l": l, "sensors": s,
                        "sequences": b * s}
                try:
                    ms = timed(fn, steps, warmup)
                    line.update(ms_per_call=round(ms, 4),
                                peak_allocated_gib=round(torch.cuda.max_memory_allocated() / 2**30, 2))
                except torch.cuda.OutOfMemoryError:
                    line.update(ms_per_call=None, error="out of memory")
                line.update(steps=steps, warmup=warmup, **info)
                enc.zero_grad(set_to_none=True)
                torch.cuda.empty_cache()
                print(json.dumps(line), flush=True)
                lines.append(line)
        torch.backends.cudnn.allow_tf32 = False
        del enc, r, tf, dh
        torch.cuda.empty_cache()
    return lines


def detector_step(info, dev, steps: int, warmup: int) -> list:
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.parallel import FlatGradBucket

    z = np.load(REPO / "tests" / "golden" / "graph_LT.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    b, l_det = 256, 36
    g = torch.Generator(device="cpu").manual_seed(198)
    pool = [(torch.randn(b, l_det, len(sensors), generator=g).to(dev), torch.randn(b, l_det, 9, generator=g).to(dev),
             torch.randint(0, len(pipes) + 1, (b,), generator=g).to(dev)) for _ in range(4)]
    lines = []
    for hidden in (128, 64):
        torch.manual_seed(42)
        model = LeakDetector(REPO / "tests" / "golden" / "L-TOWN.topo.inp", sensors, pipes, sensor_hidden=hidden,
                             node_hidden=64, gnn_layers=2, dropout=0.1, use_time=True).to(dev).train()
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
        step = GraphedTrainStep(model, opt, FlatGradBucket(model.parameters()), b, l_det, grad_clip=1.0)
        it = iter(range(10**9))
        ms = timed(lambda: step(*pool[next(it) % 4]), steps, warmup)
        line = {"workload": "ltown_dp256_graphed_step", "sensor_hidden": hidden, "batch": b, "windows": b,
                "ms_per_step": round(ms, 4), "steps": steps, "warmup": warmup, **info}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del step, opt, model
    return lines


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100, help="timed replays of the detector step")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_sensor_gru: needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    lines = encoder(info, dev) + detector_step(info, dev, args.steps, args.warmup)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
