"""Time the batched GNNExplainer of a frozen LeakDetector (leak_det_gnn_b200.explain.explain_edges) and what pruning
the frozen backward saves on the existing per-pipe attribution call.

L-TOWN-A (29 sensors, every pipe of the golden graph as a class), sensor and node width 64, eval mode, at (B, L) =
(256, 36) and the lta4096 shape (4096, 288), 100 epochs, on the same seeded inputs and targets:
  explain_native  explain_edges: sensor encoder once, eager epoch 0, epoch 1 captured as a CUDA graph and replayed 99
                  times (ltgnn_edge_mask_fwd / _bwd, the weighted layers, ltgnn_gcn_adj_grad, ltgnn_explain_step); the
                  device time of each library kernel from one more instrumented eager epoch
  explain_oracle  the fp32 restatement on CUDA: oracle/pyg_explain.py's masked detector (gcn_norm of the replicated graph
                  in every conv, index_select / index_add_ message passing), autograd, torch.optim.Adam, the regularisers
                  vectorised over windows; fewer epochs, reported per epoch
  edge_grad       the d edge_weight recipe of tools/time_edge_grad.py, frozen (no parameter requires grad) and with
                  trainable parameters, alternated in the same run: what the pruned backward saves
Device events around back-to-back calls after warm-up calls, and the peak torch.cuda.max_memory_allocated of each arm.

    python tools/time_explain.py [--out profiles/r12_time_explain.jsonl]

One JSON line per measurement, with the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch
import torch.nn.functional as F

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))

from leak_det_gnn_b200 import explain, instrument  # noqa: E402
from leak_det_gnn_b200.models import LeakDetector  # noqa: E402
from oracle.pyg_explain import MaskedOracleLeakDetector  # noqa: E402
from tools.time_input_grad import card, timed  # noqa: E402

EPOCHS = 100
SHAPES = ((256, 36, 3, 1, 10), (4096, 288, 2, 1, 3))   # B, L, timed calls, warm-up calls, oracle epochs


def oracle_on(model: LeakDetector, dev) -> MaskedOracleLeakDetector:
    m = MaskedOracleLeakDetector(len(model.node_names), model.edge_index_single, model.pipe_ends,
                                 model.sensor_node_idx.tolist(), 64, 64, 2, 0.1, True)
    m.load_state_dict(model.state_dict(), strict=True)
    m = m.to(dev).eval().requires_grad_(False)
    m.edge_index_single = m.edge_index_single.to(dev)  # plain attributes, not buffers
    m.pipe_ends = m.pipe_ends.to(dev)
    m.sensor_node_idx = m.sensor_node_idx.to(dev)
    return m


def oracle_explain(oracle, h_s, target, m0, epochs, lr=0.01, edge_size=0.005, edge_ent=1.0):
    """The batched restatement in fp32 on the device, regularisers as masked sums over windows."""
    p = torch.nn.Parameter(m0.clone())
    opt = torch.optim.Adam([p], lr=lr)
    hard = n_hard = None
    for i in range(epochs):
        opt.zero_grad()
        s = p.sigmoid()
        loss = F.cross_entropy(oracle.gnn_stack(h_s, edge_mask=s), target, reduction="sum")
        if hard is not None:
            ent = -s * torch.log(s + 1e-15) - (1 - s) * torch.log(1 - s + 1e-15)
            loss = loss + edge_size * (s * hard).sum() + edge_ent * ((ent * hard).sum(1) / n_hard.clamp(min=1)).sum()
        loss.backward()
        opt.step()
        if i == 0:
            hard = p.grad != 0
            n_hard = hard.sum(1)
    return torch.where(hard, p.detach().sigmoid(), 0.0)


def kernel_times(model, h_s, target, b, e, n) -> dict:
    """One instrumented eager epoch (after the recording epoch 0) of explain_edges' loop."""
    st = explain._MaskState(explain.initial_mask_logits(b, e, n, torch.Generator().manual_seed(1)).to(h_s.device))
    st.epoch(model, h_s, target, True, 0.01, 0.005, 1.0)
    torch.cuda.synchronize()
    instrument.reset(timing=True)
    st.epoch(model, h_s, target, False, 0.01, 0.005, 1.0)
    torch.cuda.synchronize()
    summ = instrument.summary()
    instrument.reset()
    return {k: round(v["total_ms"], 4) for k, v in summ.items()}


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

    for b, l, steps, warmup, oracle_epochs in SHAPES:
        g = torch.Generator(device="cpu").manual_seed(b)
        r = torch.randn(b, l, s, generator=g).to(dev)
        tf = torch.randn(b, l, 9, generator=g).to(dev)
        target = torch.randint(0, len(pipes) + 1, (b,), generator=g).to(dev)
        base = {"workload": "detector_explain", "sensor_hidden": 64, "node_hidden": 64, "batch": b, "l": l,
                "sensors": s, "edges": e, "nnz": model.pipe_graph.nnz}

        def native():
            return explain.explain_edges(model, r, tf, target, epochs=EPOCHS, generator=torch.Generator().manual_seed(1))

        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        ms = timed(native, steps, warmup)
        line = dict(base, arm="explain_native", epochs=EPOCHS, ms_per_call=round(ms, 3), ms_per_epoch=round(ms / EPOCHS, 4),
                    peak_allocated_gib=round(torch.cuda.max_memory_allocated() / 2**30, 2), steps=steps, warmup=warmup)
        with torch.no_grad():
            h_s = model.sensor_encoder(r, tf)
        line["eager_epoch_kernel_ms"] = kernel_times(model, h_s, target, b, e, n)
        emit(line)

        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        line = dict(base, arm="explain_oracle", epochs=oracle_epochs)
        try:
            m0 = explain.initial_mask_logits(b, e, n, torch.Generator().manual_seed(1)).to(dev)
            prev = torch.get_default_device()
            torch.set_default_device(dev)  # the restatement allocates its index tensors with the default device
            try:
                ms = timed(lambda: oracle_explain(oracle, h_s, target, m0, oracle_epochs), 1, 1)
            finally:
                torch.set_default_device(prev)
            line.update(ms_per_call=round(ms, 3), ms_per_epoch=round(ms / oracle_epochs, 4),
                        peak_allocated_gib=round(torch.cuda.max_memory_allocated() / 2**30, 2))
        except torch.cuda.OutOfMemoryError:
            line.update(ms_per_call=None, error="out of memory")
        emit(line)

        # the existing d edge_weight recipe, frozen against trainable parameters, alternated
        ew = torch.ones(b, e, device=dev, requires_grad=True)
        tcol = target[:, None]

        def edge_grad():
            return torch.autograd.grad(model(r, tf, edge_weight=ew).gather(1, tcol).sum(), ew)

        reps = {"frozen": [], "trainable": []}
        for _ in range(3):
            for arm in ("frozen", "trainable"):
                model.requires_grad_(arm == "trainable")
                reps[arm].append(timed(edge_grad, steps * 5 if b == 256 else steps, 1))
        model.requires_grad_(False)
        for arm, ms_list in reps.items():
            emit(dict(base, workload="detector_edge_grad", arm=f"edge_grad_{arm}", ms_per_call=[round(x, 4) for x in ms_list],
                      steps=steps * 5 if b == 256 else steps, warmup=1))
        del r, tf, target, ew, h_s
        torch.cuda.empty_cache()
    return lines


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_explain: needs a CUDA device")
    info = card()
    lines = run(info, torch.device("cuda"))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
