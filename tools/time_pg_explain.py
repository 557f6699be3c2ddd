"""Time PGExplainer on a frozen LeakDetector (leak_det_gnn_b200.explain.PGExplainer) against the batched GNNExplainer.

L-TOWN-A (29 sensors, every pipe of the golden graph as a class), sensor and node width 64, eval mode, at (B, L) =
(256, 36) and the lta4096 shape (4096, 288), on the same seeded inputs and targets:
  train_eager     PGExplainer.train: sensor encoder, embeddings, [P | Q] GEMM, ltgnn_pg_edge_fwd, masked detector,
                  loss, backward (ltgnn_pg_edge_bwd, d W1 on ltgnn_wgrad_tc), Adam -- one step per call
  train_graphed   the same step captured once and replayed (graphed=True)
  explain         PGExplainer.explain end to end (sensor encoder, embeddings, edge network)
  alternated      explain_edges at 100 epochs and the fp32 restatement of PGExplainer's step on CUDA (oracle/
                  pyg_pg_explainer.py: the concatenated MLP input, index_add_ message passing, torch.optim.Adam), in turn
  kernels         device time of ltgnn_pg_edge_fwd (training), ltgnn_pg_edge_bwd and the [P | Q] GEMM over repeated
                  launches, with the bytes each must move (from shapes) over that time, against 7.7 TB/s
Device events around back-to-back calls after warm-up calls.

    python tools/time_pg_explain.py [--out profiles/r13_time_pg_explain.jsonl]

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

from leak_det_gnn_b200 import explain, ops  # noqa: E402
from leak_det_gnn_b200.models import LeakDetector  # noqa: E402
from oracle.pyg_pg_explainer import PGExplainerOracle  # noqa: E402
from tools.time_explain import oracle_on  # noqa: E402
from tools.time_input_grad import card, timed  # noqa: E402

SHAPES = ((256, 36, 20, 3), (4096, 288, 5, 2))   # B, L, timed calls, warm-up calls
HBM = 7.7e12


def kernel_arms(model, ex, h_s, b, n, e) -> list:
    dev = h_s.device
    st = ex._state(dev)
    lin1, lin2 = ex.mlp[0], ex.mlp[2]
    with torch.no_grad():
        z = model.embeddings(h_s)
        w_stack = torch.cat([lin1.weight[:, :64], lin1.weight[:, 64:]], 0).contiguous()
        pq = ops.linear_tc(z, w_stack)
        mask, s, gate = ops.pg_edge_fwd(pq, st["idx"], lin1.bias, lin2.weight, lin2.bias, st["inv_t"], 0.01, 1)
        dmask = torch.randn_like(mask)
        reps = 50 if b == 256 else 10
        arms = {
            "pq_gemm": (lambda: ops.linear_tc(z, w_stack, out=pq), 4 * b * n * (64 + 128)),
            "pg_edge_fwd": (lambda: ops.pg_edge_fwd(pq, st["idx"], lin1.bias, lin2.weight, lin2.bias, st["inv_t"], 0.01, 1),
                            4 * b * n * 128 + 16 * b * e),
            "pg_edge_bwd": (lambda: ops.pg_edge_bwd(pq, st["idx"], lin1.bias, lin2.weight, st["inv_t"], mask, dmask, gate),
                            4 * b * n * 128 * 2 + 16 * b * e),
        }
        out = []
        for name, (fn, nbytes) in arms.items():
            ms = timed(fn, reps, 2)
            out.append({"arm": f"kernel_{name}", "ms_per_call": round(ms, 4), "bytes": nbytes,
                        "achieved_tb_s": round(nbytes / (ms * 1e-3) / 1e12, 3),
                        "share_of_hbm_peak": round(nbytes / (ms * 1e-3) / HBM, 3), "calls": reps})
    return out


def oracle_step(oracle_model, ox, h_s, target, u):
    prev = torch.get_default_device()
    torch.set_default_device(h_s.device)  # the restatement allocates its index tensors with the default device
    try:
        return ox.train(3, oracle_model, h_s, target, u)
    finally:
        torch.set_default_device(prev)


def run(info, dev) -> list:
    z = np.load(REPO / "tests" / "golden" / "graph_LTA.npz")
    sensors, pipes = [str(s) for s in z["sensor_node_ids"]], [str(p) for p in z["pipe_ids"]]
    s = len(sensors)
    torch.manual_seed(42)
    model = LeakDetector(REPO / "tests" / "golden" / "L-TOWN-A.topo.inp", sensors, pipes, sensor_hidden=64,
                         node_hidden=64).to(dev).eval().requires_grad_(False)
    e, n = model.edge_index_single.shape[1], len(model.node_names)
    oracle = oracle_on(model, dev)
    torch.backends.cudnn.allow_tf32 = False
    lines = []

    def emit(line):
        line.update(info)
        print(json.dumps(line), flush=True)
        lines.append(line)

    for b, l, steps, warmup in SHAPES:
        g = torch.Generator(device="cpu").manual_seed(b)
        r = torch.randn(b, l, s, generator=g).to(dev)
        tf = torch.randn(b, l, 9, generator=g).to(dev)
        target = torch.randint(0, len(pipes) + 1, (b,), generator=g).to(dev)
        base = {"workload": "detector_pg_explain", "sensor_hidden": 64, "node_hidden": 64, "batch": b, "l": l,
                "sensors": s, "nodes": n, "edges": e}
        for graphed in (False, True):
            torch.manual_seed(1)
            ex = explain.PGExplainer(model, epochs=1000, graphed=graphed)
            ex.train(0, r, tf, target)  # the capture (graphed) or the first eager step
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            ms = timed(lambda: ex.train(500, r, tf, target), steps, warmup)
            emit(dict(base, arm="train_graphed" if graphed else "train_eager", ms_per_step=round(ms, 4),
                      peak_allocated_gib=round(torch.cuda.max_memory_allocated() / 2**30, 2), steps=steps, warmup=warmup))
        ex._curr_epoch = ex.epochs - 1
        ms = timed(lambda: ex.explain(r, tf), steps, warmup)
        emit(dict(base, arm="explain", ms_per_call=round(ms, 4), steps=steps, warmup=warmup))
        with torch.no_grad():
            h_s = model.sensor_encoder(r, tf)
        for k in kernel_arms(model, ex, h_s, b, n, e):
            emit(dict(base, **k))

        # explain_edges at 100 epochs and the fp32 restatement's step on CUDA, alternated
        ox = PGExplainerOracle(64, 1000).to(dev)
        ox.mlp.load_state_dict(ex.mlp.state_dict())
        u = torch.rand(b, e, device=dev)
        reps = {"explain_edges_100": [], "oracle_fp32_step": []}
        for _ in range(2):
            reps["explain_edges_100"].append(timed(
                lambda: explain.explain_edges(model, r, tf, target, epochs=100, generator=torch.Generator().manual_seed(1)),
                1, 1))
            try:
                reps["oracle_fp32_step"].append(timed(lambda: oracle_step(oracle, ox, h_s, target, u), 1, 1))
            except torch.cuda.OutOfMemoryError:
                reps["oracle_fp32_step"].append(None)
            torch.cuda.empty_cache()
        for arm, ms_list in reps.items():
            emit(dict(base, arm=arm, ms_per_call=[None if x is None else round(x, 3) for x in ms_list]))
        del r, tf, target, h_s, ex, ox, u
        torch.cuda.empty_cache()
    return lines


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_pg_explain: needs a CUDA device")
    info = card()
    lines = run(info, torch.device("cuda"))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
