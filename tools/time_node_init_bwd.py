"""Time node init's backward from the first GCN layer's aggregated gradient G1, two ways, on the same seeded operands:
  two_launch  dX0 = G1 W1 stored by ltgnn_linear, then ltgnn_node_init_bwd streams it again (gate, column sums, sensor
              rows) before the two sensor-row GEMMs
  from_layer  ltgnn_node_init_bwd_from_layer: the GEMM gates, sums and extracts in its epilogue, dX0 is never stored
at the lta4096 shape (B = 4096 windows of L-TOWN-A: 661 nodes, 29 sensors, widths 64) and at node width 128.  Device
events around back-to-back calls, the two arms alternated over several rounds (median reported), then one
torch.profiler pass per arm for the device time of each kernel.

    python tools/time_node_init_bwd.py [--out profiles/r14_time_node_init_bwd.jsonl]

One JSON line per measurement, with the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

import bench  # noqa: E402
from leak_det_gnn_b200 import ops  # noqa: E402
from tools.time_input_grad import card, timed  # noqa: E402

SHAPES = ((4096, 64, 64, 64), (2048, 64, 128, 128))   # B, ds, D (node width), K (layer-0 output width)
ROUNDS, STEPS, WARMUP = 5, 20, 3
SCALE = 1.0 / (1.0 - round(0.1 * 65536) / 65536)


def operands(b, ds, d, k, sensor_idx, n):
    gen = torch.Generator(device="cuda").manual_seed(b + d)
    idx = torch.from_numpy(sensor_idx).cuda()
    slot = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    slot[idx] = torch.arange(idx.numel(), dtype=torch.int32, device="cuda")
    h_s = torch.randn(b, idx.numel(), ds, device="cuda", generator=gen)
    w0 = torch.randn(d, ds + 1, device="cuda", generator=gen) * 0.2
    b0 = torch.randn(d, device="cuda", generator=gen) * 0.5
    gz = torch.randn(b, n, k, device="cuda", generator=gen)
    w1 = torch.randn(k, d, device="cuda", generator=gen) * k ** -0.5
    live = ops.new_live_mask(b, n, d, "cuda")
    x0 = ops.node_init_fwd(h_s, slot, n, w0, b0, 0.1, 21, live_out=live)
    return slot, h_s, w0, gz, w1, live, x0


def kernel_times(fn) -> dict:
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count:
            out[e.key[:90]] = round(e.device_time_total / 1e3, 4)   # ms, one call
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r14_time_node_init_bwd.jsonl"))
    args = ap.parse_args()
    info = card()
    net = bench.network("LTA", 764)
    n = net["n_nodes"]
    lines = []
    for b, ds, d, k in SHAPES:
        slot, h_s, w0, gz, w1, live, x0 = operands(b, ds, d, k, net["sensor_idx"], n)

        def two_launch():
            return ops.node_init_bwd(h_s, slot, w0, ops.linear_tc(gz, w1, transposed=True), x0, SCALE, live=live)

        def from_layer():
            return ops.node_init_bwd_from_layer(h_s, slot, w0, gz, w1, live, SCALE)

        arms = {"two_launch": two_launch, "from_layer": from_layer}
        ms = {a: [] for a in arms}
        for _ in range(ROUNDS):
            for a, fn in arms.items():
                ms[a].append(timed(fn, STEPS, WARMUP))
        s = h_s.shape[1]
        g_bytes, live_bytes, dz_bytes = b * n * k * 4, b * n * d // 8, b * s * d * 4
        moved = {"two_launch": g_bytes + 2 * b * n * d * 4 + live_bytes + dz_bytes,
                 "from_layer": g_bytes + live_bytes + dz_bytes}
        for a, fn in arms.items():
            med = statistics.median(ms[a])
            lines.append({**info, "shape": {"B": b, "N": n, "S": s, "ds": ds, "D": d, "K": k}, "arm": a,
                          "ms_median": round(med, 4), "ms_rounds": [round(x, 4) for x in ms[a]],
                          "hbm_bytes": moved[a], "achieved_gbs": round(moved[a] / (med * 1e-3) / 1e9, 1),
                          "kernels_ms": kernel_times(fn)})
        del slot, h_s, w0, gz, w1, live, x0
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    with open(args.out, "w") as f:
        for ln in lines:
            print(json.dumps(ln), flush=True)
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
