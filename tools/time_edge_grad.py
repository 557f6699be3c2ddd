"""Time the per-pipe attribution of a frozen LeakDetector: the gradient of each window's target logit with respect to
that window's edge weights, taken at weight 1 -- ew = ones(B, E) requiring grad, logits.gather(1, target).sum() ->
torch.autograd.grad(..., ew), forward included.

L-TOWN-A (29 sensors, every pipe of the golden graph as a class), sensor and node width 64, eval mode, every parameter
frozen, at (B, L) = (256, 36) and the lta4096 shape (4096, 288), three arms on the same seeded weights and inputs:
  edge_grad       the native path with (B, E) edge weights: device normalisation, weighted aggregation, the
                  adjacency-value gradient (ltgnn_edge_norm_fwd / _bwd, ltgnn_spmm_fused_vals, ltgnn_gcn_adj_grad)
  sensor_saliency the same call without edge weights, differentiated with respect to residual and tfeat instead (the
                  sensor saliency of INTEGRATION section 2: the one-kernel GCN layers)
  oracle_fp32     the fp32 restatement (oracle/pyg_weighted.py over oracle/detector_oracle.py) run on CUDA: gcn_norm
                  of the B-times replicated graph in every conv, torch's index_select / index_add_ message passing,
                  autograd for the edge-weight gradient; its sensor GRU on cuDNN (allow_tf32 = False) in slabs of at most
                  8 192 sequences, as the detector's own cuDNN route runs it (one call over B * S sequences exceeds
                  what cuDNN's RNN takes at the lta4096 shape)
Device events around back-to-back calls after warm-up calls, the peak torch.cuda.max_memory_allocated of each arm, and
for edge_grad one more instrumented call with the device time of each library kernel of the weighted path.

    python tools/time_edge_grad.py [--out profiles/r11_time_edge_grad.jsonl]

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
from leak_det_gnn_b200.models import LeakDetector  # noqa: E402
from oracle.pyg_weighted import WeightedOracleLeakDetector  # noqa: E402
from tools.time_input_grad import card, timed  # noqa: E402

SHAPES = ((256, 36, 20, 3), (4096, 288, 3, 1))   # B, L, timed calls, warm-up calls
EDGE_KERNELS = ("edge_norm_fwd", "edge_norm_bwd", "gcn_adj_grad", "spmm_vals_fwd", "spmm_vals_bwd")


def oracle_on(model: LeakDetector, dev) -> WeightedOracleLeakDetector:
    m = WeightedOracleLeakDetector(len(model.node_names), model.edge_index_single, model.pipe_ends,
                           model.sensor_node_idx.tolist(), 64, 64, 2, 0.1, True)
    m.load_state_dict(model.state_dict(), strict=True)
    m = m.to(dev).eval().requires_grad_(False)
    m.edge_index_single = m.edge_index_single.to(dev)  # plain attributes, not buffers
    m.pipe_ends = m.pipe_ends.to(dev)
    m.sensor_node_idx = m.sensor_node_idx.to(dev)
    return m


def run(info, dev) -> list:
    z = np.load(REPO / "tests" / "golden" / "graph_LTA.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    s = len(sensors)
    torch.manual_seed(42)
    model = LeakDetector(REPO / "tests" / "golden" / "L-TOWN-A.topo.inp", sensors, pipes, sensor_hidden=64,
                         node_hidden=64).to(dev).eval().requires_grad_(False)
    e = model.edge_index_single.shape[1]
    oracle = oracle_on(model, dev)
    torch.backends.cudnn.allow_tf32 = False
    lines = []
    for b, l, steps, warmup in SHAPES:
        g = torch.Generator(device="cpu").manual_seed(b)
        r = torch.randn(b, l, s, generator=g).to(dev)
        tf = torch.randn(b, l, 9, generator=g).to(dev)
        target = torch.randint(0, len(pipes) + 1, (b, 1), generator=g).to(dev)
        ew = torch.ones(b, e, device=dev, requires_grad=True)
        rg, tfg = r.clone().requires_grad_(True), tf.clone().requires_grad_(True)
        slab = max(1, model.sensor_encoder.max_seqs_per_call // s)  # windows per cuDNN call of the oracle's GRU

        def edge_grad():
            return torch.autograd.grad(model(r, tf, edge_weight=ew).gather(1, target).sum(), ew)

        def sensor_saliency():
            return torch.autograd.grad(model(rg, tfg).gather(1, target).sum(), (rg, tfg))

        def oracle_fp32():
            prev = torch.get_default_device()
            torch.set_default_device(dev)  # the restatement allocates its index tensors with the default device
            try:
                h_s = torch.cat([oracle.sensor_encoder(r[w:w + slab], tf[w:w + slab]) for w in range(0, b, slab)])
                return torch.autograd.grad(oracle.gnn_stack(h_s, edge_weight=ew).gather(1, target).sum(), ew)
            finally:
                torch.set_default_device(prev)

        for arm, fn in (("edge_grad", edge_grad), ("sensor_saliency", sensor_saliency), ("oracle_fp32", oracle_fp32)):
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            line = {"workload": "detector_edge_grad", "arm": arm, "sensor_hidden": 64, "node_hidden": 64, "batch": b,
                    "l": l, "sensors": s, "edges": e, "nnz": model.pipe_graph.nnz}
            try:
                ms = timed(fn, steps, warmup)
                line.update(ms_per_call=round(ms, 4), peak_allocated_gib=round(torch.cuda.max_memory_allocated() / 2**30, 2))
                if arm == "edge_grad":
                    instrument.reset(timing=True)
                    fn()
                    torch.cuda.synchronize()
                    summ = instrument.summary()
                    instrument.reset()
                    line["kernel_ms"] = {k: round(v["total_ms"], 4) for k, v in summ.items() if k in EDGE_KERNELS}
            except torch.cuda.OutOfMemoryError:
                line.update(ms_per_call=None, error="out of memory")
            line.update(steps=steps, warmup=warmup, **info)
            print(json.dumps(line), flush=True)
            lines.append(line)
        del r, tf, target, ew, rg, tfg
        torch.cuda.empty_cache()
    return lines


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_edge_grad: needs a CUDA device")
    info = card()
    lines = run(info, torch.device("cuda"))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
