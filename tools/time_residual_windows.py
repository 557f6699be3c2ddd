"""Time ``forward_windows``' sharing of overlapping windows against the per-window path, on both normal-state predictors
(NormalPredictorTCN / NormalPredictorGRU (S = 29, 9 time features), seeded weights), with ``share_windows`` on and off:

  residual builder   build_residual_sequence_from_segment, l_pred = l_det = 36, at B = 128, 256 and 1024 segments
  detector step      bench.py's ltown_dp256 training step (full L-TOWN, B = 256, hidden 64, clip 1.0, AdamW) as a
                     GraphedTrainStep replay
  scenario scoring   scenario_window_logits on one 2 017-step scenario (full L-TOWN-A detector) at strides 1, 3, 12;
                     "off" is the per-segment loop (every window's segment through the residual builder, sharing off)
  plan build         host time of shared_cone_plan (and of the cached device copy) for the shapes above

    python tools/time_residual_windows.py [--steps 200] [--warmup 20] [--out FILE]

Device events around `steps` back-to-back calls after `warmup` calls (scenario scoring: a host clock around calls that
end in a device synchronise); one JSON line per measurement, with the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from leak_det_gnn_b200.event_windows import scenario_window_logits  # noqa: E402
from leak_det_gnn_b200.models import (LeakDetector, NormalPredictorGRU, NormalPredictorTCN,  # noqa: E402
                                      build_residual_sequence_from_segment)
from leak_det_gnn_b200.models.predictor import shared_cone_plan  # noqa: E402
from tools.time_gru_predictor import card, timed  # noqa: E402

ARCH = {"tcn": NormalPredictorTCN, "gru": NormalPredictorGRU}
GOLD = REPO / "tests" / "golden"


def emit(lines, **kw):
    print(json.dumps(kw), flush=True)
    lines.append(kw)


def residual_builder(args, info, dev, lines) -> None:
    for arch in ("tcn", "gru"):
        torch.manual_seed(0)
        pred = ARCH[arch](29, 9).to(dev).eval()
        for b in (128, 256, 1024):
            g = torch.Generator(device="cpu").manual_seed(b)
            pool = [(torch.randn(b, 72, 29, generator=g).to(dev), torch.randn(b, 72, 9, generator=g).to(dev))
                    for _ in range(4)]

            def build(noisy, tf):
                with torch.no_grad():
                    return build_residual_sequence_from_segment(pred, noisy, tf, 36, 36)

            for share in (True, False, True, False):          # alternated: the second pair shows the spread
                pred.share_windows = share
                ms = timed(build, pool, args.steps, args.warmup)
                emit(lines, workload="residual_builder", predictor=arch, share_windows=share, segments=b,
                     windows=b * 36, ms_per_call=round(ms, 4), steps=args.steps, warmup=args.warmup, **info)
            pred.share_windows = True


def detector_step(args, info, dev, lines) -> None:
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.parallel import FlatGradBucket

    z = np.load(GOLD / "graph_LT.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    b, l_det, l_pred = 256, 36, 36
    g = torch.Generator(device="cpu").manual_seed(198)
    pool = [(torch.randn(b, l_pred + l_det, len(sensors), generator=g).to(dev),
             torch.randn(b, l_pred + l_det, 9, generator=g).to(dev),
             torch.randint(0, len(pipes) + 1, (b,), generator=g).to(dev)) for _ in range(4)]
    for arch in ("tcn", "gru"):
        for share in (True, False):
            torch.manual_seed(42)
            model = LeakDetector(GOLD / "L-TOWN.topo.inp", sensors, pipes, sensor_hidden=64, node_hidden=64,
                                 gnn_layers=2, dropout=0.1, use_time=True).to(dev).train()
            pred = ARCH[arch](len(sensors), 9).to(dev).eval()
            pred.share_windows = share
            opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
            step = GraphedTrainStep(model, opt, FlatGradBucket(model.parameters()), b, l_det, predictor=pred,
                                    l_pred=l_pred, grad_clip=1.0)
            ms = timed(step, pool, args.steps, args.warmup)
            emit(lines, workload="ltown_dp256_graphed_step", predictor=arch, share_windows=share, batch=b,
                 ms_per_step=round(ms, 4), steps=args.steps, warmup=args.warmup, **info)
            del step, opt, model, pred


def per_segment(pred, det, pressure, tfeat, stride, dev, batch=1024):
    """Scenario scoring one segment per window (every window's segment through the residual builder)."""
    p, f = torch.as_tensor(pressure), torch.as_tensor(tfeat)
    starts = list(range(0, p.shape[0] - 72 + 1, stride))
    seg_p, seg_f = p.unfold(0, 72, 1).permute(0, 2, 1), f.unfold(0, 72, 1).permute(0, 2, 1)
    out = []
    with torch.no_grad():
        for lo in range(0, len(starts), batch):
            sel = torch.tensor(starts[lo:lo + batch])
            noisy, tseg = seg_p[sel].contiguous().to(dev), seg_f[sel].contiguous().to(dev)
            res = build_residual_sequence_from_segment(pred, noisy, tseg, 36, 36)
            out.append(det(res, tseg[:, 36:].contiguous()))
    return torch.cat(out).cpu()


def scenario(args, info, dev, lines) -> None:
    z = np.load(GOLD / "graph_LTA.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    torch.manual_seed(11)
    det = LeakDetector(GOLD / "L-TOWN-A.topo.inp", sensors, pipes).to(dev).eval()
    rng = np.random.default_rng(2017)
    pressure = rng.standard_normal((2017, len(sensors))).astype(np.float32)
    tfeat = rng.standard_normal((2017, 9)).astype(np.float32)
    reps = max(3, args.steps // 20)
    for arch in ("tcn", "gru"):
        torch.manual_seed(0)
        pred = ARCH[arch](len(sensors), 9).to(dev).eval()
        for stride in (1, 3, 12):
            arms = {"shared": lambda: scenario_window_logits(pred, det, pressure, tfeat, 36, 36, stride, dev)[1],
                    "per_segment": lambda: per_segment(pred, det, pressure, tfeat, stride, dev)}
            res = {}
            for name in ("shared", "per_segment", "shared", "per_segment"):
                pred.share_windows = name == "shared"
                res[name] = arms[name]()                          # warm-up (plans, handles)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(reps):
                    arms[name]()
                torch.cuda.synchronize()
                emit(lines, workload="scenario_scoring", predictor=arch, arm=name, steps_in_scenario=2017,
                     stride=stride, windows=res[name].shape[0], ms_per_call=round((time.perf_counter() - t0) / reps * 1e3, 3),
                     calls=reps, **info)
            emit(lines, workload="scenario_scoring_equal", predictor=arch, stride=stride,
                 bitwise_equal=bool(torch.equal(res["shared"], res["per_segment"])), **info)


def plan_build(info, dev, lines) -> None:
    for length, count, b in ((72, 36, 128), (72, 36, 256), (72, 36, 1024), (2017, 1982, 1)):
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            shared_cone_plan(length, 36, count, b, 3, [1, 2, 4, 8])
            ts.append((time.perf_counter() - t0) * 1e3)
        m = NormalPredictorTCN(29, 9).to(dev).eval()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m._shared_rows(length, 36, count, b, dev)
        torch.cuda.synchronize()
        first = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        m._shared_rows(length, 36, count, b, dev)
        cached = (time.perf_counter() - t0) * 1e3
        emit(lines, workload="tcn_shared_plan_build", series_steps=length, windows_per_series=count, series=b,
             host_ms_median=round(sorted(ts)[2], 3), first_call_with_device_copy_ms=round(first, 3),
             cached_call_ms=round(cached, 4), **info)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_residual_windows: needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    lines: list = []
    plan_build(info, dev, lines)
    residual_builder(args, info, dev, lines)
    detector_step(args, info, dev, lines)
    scenario(args, info, dev, lines)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
