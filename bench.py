#!/usr/bin/env python
"""bench.py -- window-graphs/s, forward+backward, of the detector's message-passing path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json configs as restated by SURVEY.md 8d); synthetic inputs (residual ~ N(0,1), seed 198 + rank;
time features on a 5-minute grid from 2018-01-02), random-init weights (seed 42), train mode (dropout on), fp32:

  lta4096      (default; configs[2]) real L-TOWN-A topology (N=661, E=1532, nnz=2193), B = 4096 windows x 288 steps per
               GPU, hidden 64, all P = 764 pipes as classes.
  lta128       (configs[1] shape) same network at the reference's training batch B = 128, l_det = 36
               (train_detector.py:142,147-148); also reports the B = 1 forward latency of event_evaluator.py:486.
  ltown_dp256  (configs[3]) full L-TOWN (N=785, nnz=2603, P=905), B = 256 per GPU: the reference's whole training step
               (train_detector.py:296-317) -- frozen TCN predictor forward on B * l_det windows under no_grad (residual
               builder), detector forward/backward, gradient all-reduce, clip_grad_norm_, AdamW.
  scaled100k   (configs[4]) synthetic pipe network, N = 100 000, 115 000 links (mean degree 2.3), hidden 128, B = 16.

One STEP = one pass of the hot path over one batch of B windows:
  * `value`  : lta4096 / lta128 / scaled100k: the GNN stack -- node init -> 2 x (GCN conv, ReLU, dropout) -> pipe head +
               mean-pool no-leak head -> cross-entropy -> backward to every non-GRU parameter and to the sensor embeddings
               (reference detector.py:178-218 + autograd; SURVEY 8a rows a4-a13), sensor embeddings h_s resident in HBM.
               ltown_dp256: the whole training step with the segment batch resident in HBM.
               At N > 1 the step also averages the gradients with one flat-bucket NCCL all-reduce.
  * `e2e`    : the call a user makes -- LeakDetector.forward(residual, tfeat) (sensor GRU encoder included), cross-entropy,
               backward (ltown_dp256: + residual builder, clip, AdamW) -- with the inputs copied from pinned host memory
               and the loss read back to the host inside the timed region.
The reference arm (--impl reference) reports the SAME scopes on the host cores (oracle port; bounded sample).
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))
GOLDEN = REPO / "tests" / "golden"

METRIC = "window_graphs_per_sec_fwd_bwd"
UNIT = "window-graphs/s"
SENSORS = 29
DUMP_LIMIT = 64_000_000   # bytes that --dump-outputs writes at most

WORKLOADS = {
    "lta4096": dict(net="LTA", batch=4096, l_det=288, pipes=764, hidden=64, full_step=False, cpu_sample=32,
                    cfg="BASELINE configs[2] per SURVEY 8d"),
    "lta128": dict(net="LTA", batch=128, l_det=36, pipes=764, hidden=64, full_step=False, cpu_sample=32, graphed=True,
                   cfg="BASELINE configs[1] shape: the reference's training batch"),
    "ltown_dp256": dict(net="LT", batch=256, l_det=36, pipes=905, hidden=64, full_step=True, cpu_sample=16, graphed=True,
                        cfg="BASELINE configs[3]: whole training step incl. frozen predictor, clip, AdamW"),
    "predictor_train": dict(net="LTA", batch=256, l_det=36, pipes=2, hidden=64, full_step=False, cpu_sample=256,
                            cfg="BASELINE configs[0]: train_predictor (TCN, batch 256) -- the reference's CPU-runnable case; "
                                "no graph work, baseline only: --impl reference"),
    "scaled100k": dict(net="SYN100K", batch=16, l_det=36, pipes=2000, hidden=128, full_step=False, cpu_sample=1,
                       cfg="BASELINE configs[4]: N=100k, mean degree 2.3, hidden 128"),
}


def time_features(n_steps: int, start_step: int = 0) -> np.ndarray:
    """(n_steps, 9): hour sin/cos + day-of-week one-hot on a 5-minute grid from 2018-01-02 00:00
    (Tuesday) -- the arithmetic of reference models/datasets.py:49-59."""
    minutes = 5 * (start_step + np.arange(n_steps))
    hour = ((minutes // 60) % 24).astype(np.float32) + ((minutes % 60).astype(np.float32) / 60.0)
    angle = (2.0 * np.pi) * (hour / 24.0)
    dow = (1 + minutes // 1440) % 7
    return np.concatenate([np.sin(angle).astype(np.float32)[:, None], np.cos(angle).astype(np.float32)[:, None],
                           np.eye(7, dtype=np.float32)[dow]], axis=1).astype(np.float32)


def synthetic_batch(batch: int, n_steps: int, n_sensors: int, n_classes: int, seed: int):
    """(signal (B, n_steps, S), time features (B, n_steps, 9), labels (B,)); window b starts at grid step b."""
    gen = torch.Generator().manual_seed(seed)
    signal = torch.randn(batch, n_steps, n_sensors, generator=gen)
    tf = torch.from_numpy(time_features(n_steps + batch))
    idx = torch.arange(n_steps).unsqueeze(0) + torch.arange(batch).unsqueeze(1)
    label = torch.randint(0, n_classes, (batch,), generator=gen)
    return signal, tf[idx], label


def scaled_network(n_nodes: int = 100_000, n_links: int = 115_000, n_sensors: int = 1000, n_pipes: int = 2000):
    """SURVEY 8d config 5 generator (numpy default_rng(198)): a random tree (node i > 0 hangs off one of its 64
    predecessors) plus chords (i, i +- [2, 64)) without duplicates or self loops, up to n_links links."""
    rng = np.random.default_rng(198)
    i = np.arange(1, n_nodes)
    parent = i - 1 - rng.integers(0, np.minimum(i, 64))
    links = {(int(min(a, b)), int(max(a, b))) for a, b in zip(i, parent)}
    while len(links) < n_links:
        a = rng.integers(0, n_nodes, 4096)
        b = a + rng.integers(2, 64, 4096) * rng.choice([-1, 1], 4096)
        for u, v in zip(a, b):
            if 0 <= v < n_nodes and u != v and len(links) < n_links:
                links.add((int(min(u, v)), int(max(u, v))))
    links = sorted(links)
    names = [f"n{k:06d}" for k in range(n_nodes)]                # lexicographic == numeric order
    sensors = [names[k] for k in np.sort(rng.choice(n_nodes, n_sensors, replace=False))]
    pipe_ids = [f"p{k:06d}" for k in range(len(links))]
    classes = [pipe_ids[k] for k in np.sort(rng.choice(len(links), n_pipes, replace=False))]
    return names, links, pipe_ids, sensors, classes


def write_inp(path: Path, names, links, pipe_ids) -> None:
    with open(path, "w") as f:
        f.write("[JUNCTIONS]\n" + "".join(f" {n}\n" for n in names))
        f.write("[PIPES]\n" + "".join(f" {p} {names[u]} {names[v]}\n" for p, (u, v) in zip(pipe_ids, links)))
        f.write("[END]\n")


def network(net: str, n_pipes: int):
    """-> dict(inp, sensors, pipe_ids, n_nodes, n_edges, nnz, edge_index, pipe_ends, sensor_idx)."""
    if net in ("LTA", "LT"):
        z = np.load(GOLDEN / f"graph_{net}.npz")
        g = {k: z[k] for k in z.files}
        n = len(g["node_names"])
        e = int(g["edge_index"].shape[1])
        return dict(inp=GOLDEN / ("L-TOWN-A.topo.inp" if net == "LTA" else "L-TOWN.topo.inp"),
                    sensors=[str(s) for s in g["sensor_node_ids"]], pipe_ids=[str(p) for p in g["pipe_ids"]][:n_pipes],
                    n_nodes=n, n_edges=e, nnz=e + n, edge_index=g["edge_index"], pipe_ends=g["pipe_ends"][:n_pipes],
                    sensor_idx=g["sensor_node_idx"])
    names, links, pipe_ids, sensors, classes = scaled_network(n_pipes=n_pipes)
    inp = Path(tempfile.gettempdir()) / f"ltgnn_syn100k_{os.getpid()}.inp"
    write_inp(inp, names, links, pipe_ids)
    ei = np.empty((2, 2 * len(links)), dtype=np.int64)
    lk = np.asarray(links, dtype=np.int64)
    ei[0, 0::2], ei[1, 0::2], ei[0, 1::2], ei[1, 1::2] = lk[:, 0], lk[:, 1], lk[:, 1], lk[:, 0]
    pidx = {p: k for k, p in enumerate(pipe_ids)}
    return dict(inp=inp, sensors=sensors, pipe_ids=classes, n_nodes=len(names), n_edges=2 * len(links),
                nnz=2 * len(links) + len(names), edge_index=ei, pipe_ends=lk[[pidx[p] for p in classes]],
                sensor_idx=np.asarray([int(s[1:]) for s in sensors], dtype=np.int64))


def dump_outputs(out_dir, arrays: dict, limit: int = DUMP_LIMIT) -> None:
    """Write every array as out_dir/<name>.npy in float32.  If they add up to more than `limit` bytes, each array above
    1/64 of the limit keeps the same share of its first-axis rows, drawn by a fixed seed and kept in order.  The sample
    depends on the shapes alone: arrays with as many rows keep the same rows, and two builds keep the same sample."""
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > limit:
        big = [k for k, a in arrays.items() if a.ndim > 0 and a.shape[0] > 1 and a.nbytes > limit // 64]
        rest = total - sum(arrays[k].nbytes for k in big)
        share = (limit - rest) / (total - rest)
        for k in big:
            n = arrays[k].shape[0]
            rows = np.sort(np.random.default_rng(0).choice(n, int(n * share), replace=False))
            arrays[k] = arrays[k][rows]
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out / f"{k}.npy", a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int) -> None:
        self.index, self.proc, self.path = index, None, None

    def __enter__(self):
        if os.environ.get("BENCH_NO_CLOCKS"):
            return self
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=f, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def result(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.path:
            return out
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in Path(self.path).read_text().splitlines():
                c = [t.strip() for t in line.split(",")]
                if len(c) < 7:
                    continue
                try:
                    sm.append(float(c[0]))
                    mx.append(float(c[1]))
                except ValueError:
                    continue
                for nm, v in zip(names, c[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def peaks() -> dict:
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json; HBM copy, sustained bf16 GEMM)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def workload_config(args, wl: dict, net: dict, world: int) -> dict:
    unit_mb = net["n_nodes"] * wl["hidden"] * 4 * args.batch / 1e6
    scope = ("whole training step: frozen TCN predictor forward on B x l_det windows + detector fwd/bwd + clip + AdamW"
             if wl["full_step"] else "detector GNN stack fwd+bwd")
    return {
        "workload": f"{args.workload}: {wl['net']} graph (N={net['n_nodes']}, E={net['n_edges']}, nnz={net['nnz']}), "
                    f"{args.batch} windows x {args.l_det} timesteps per GPU, hidden {wl['hidden']}, P={args.pipes} pipe "
                    f"classes, {scope} ({wl['cfg']})",
        "windows_per_gpu": args.batch, "global_windows": args.batch * world, "l_det": args.l_det,
        "nodes": net["n_nodes"], "nnz": net["nnz"], "hidden": wl["hidden"], "pipes": args.pipes,
        "mode": "train (dropout 0.1)",
        "launch": ("CUDA-graph replay of the step (leak_det_gnn_b200.graphed; fresh dropout masks per replay through the "
                   "device-resident seed word)" if wl.get("graphed") and not args.eager else "eager: one ctypes call per kernel"),
        "parallelism": f"dp{world}" if world > 1 else "single",
        "l2": (f"one activation tensor is {unit_mb:.0f} MB and a step touches ~8 of them: "
               + ("far above the 126 MB L2, nothing survives between steps"
                  if unit_mb * 8 > 400 else "comparable to the 126 MB L2, so 256 MB are written between timed steps to flush it")),
    }


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle (a port of the reference path; PyG is not installable here) on host cores
# ----------------------------------------------------------------------------------------------
def build_oracle(net: dict, hidden: int):
    from oracle.detector_oracle import OracleLeakDetector

    torch.manual_seed(42)
    m = OracleLeakDetector(net["n_nodes"], torch.from_numpy(net["edge_index"]), torch.from_numpy(net["pipe_ends"]),
                           net["sensor_idx"].tolist(), 64, hidden, 2, 0.1, True)
    return m.train()


def cpu_stack_time(net: dict, wl: dict, sample_b: int, iters: int):
    """Oracle GNN stack fwd+bwd from resident h_s -- the scope of the product arm's `value`."""
    m = build_oracle(net, wl["hidden"])
    gen = torch.Generator().manual_seed(198)
    h_s = torch.randn(sample_b, len(net["sensors"]), 64, generator=gen).requires_grad_(True)
    label = torch.randint(0, len(net["pipe_ids"]) + 1, (sample_b,), generator=gen)

    def step():
        m.zero_grad(set_to_none=True)
        h_s.grad = None
        torch.nn.functional.cross_entropy(m.gnn_stack(h_s), label).backward()

    step()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def cpu_full_step_fn(net: dict, wl: dict, sample_b: int, l_det: int, with_predictor: bool):
    """Oracle full call: (residual builder with the reference-equivalent torch TCN,) detector forward, CE, backward
    (, clip, AdamW) -- the scope of the product arm's `e2e` (and of `value` for ltown_dp256)."""
    from leak_det_gnn_b200.models.predictor import NormalPredictorTCN

    m = build_oracle(net, wl["hidden"])
    n_s = len(net["sensors"])
    if with_predictor:
        pred = NormalPredictorTCN(n_s, 9).eval()
        seg, tseg, label = synthetic_batch(sample_b, 36 + l_det, n_s, len(net["pipe_ids"]) + 1, 198)
        opt = torch.optim.AdamW(m.parameters(), lr=1e-3)

        def step():
            with torch.no_grad():  # the reference's dense evaluation (models/utils.py:197-207)
                x = torch.cat([seg[:, k:k + 36] for k in range(l_det)], dim=0)
                t = torch.cat([tseg[:, k:k + 36] for k in range(l_det)], dim=0)
                y = pred(x, t)
                residual = (torch.cat([seg[:, 36 + k] for k in range(l_det)], dim=0) - y).view(l_det, sample_b, n_s)
                residual = residual.transpose(0, 1).contiguous()
            loss = torch.nn.functional.cross_entropy(m(residual, tseg[:, 36:]), label)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            opt.step()
            return loss.item()
    else:
        residual, tfeat, label = synthetic_batch(sample_b, l_det, n_s, len(net["pipe_ids"]) + 1, 198)

        def step():
            m.zero_grad(set_to_none=True)
            loss = torch.nn.functional.cross_entropy(m(residual, tfeat), label)
            loss.backward()
            return loss.item()
    return step


def run_predictor_train(args, wl: dict) -> None:
    """BASELINE configs[0]: one optimisation step of reference models/train_predictor.py:203-228 (TCN, MSE, AdamW lr 1e-3,
    weight decay 1e-4, clip 1.0, batch 256) on synthetic normal windows in the dataset's batch layout (x (B, 36, S),
    x_time (B, 36, 9), y (B, S)), on the host cores.  The predictor has no graph layers (SURVEY F1): nothing of this step
    is on the sm_100a path; the line exists so that every BASELINE config has a number on this box."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from leak_det_gnn_b200.models import NormalPredictorTCN   # state_dict-compatible mirror of models/predictor.py:55-81

    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(198)
    b, l, n_s = args.batch, 36, SENSORS
    model = NormalPredictorTCN(n_s, 9).train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=1e-4)
    rng = np.random.default_rng(198)
    hour = (np.arange(l)[None, :] * 5 / 60.0 + rng.uniform(0, 24, (b, 1))) % 24
    x = torch.from_numpy((8 * np.sin(2 * np.pi * hour / 24)[:, :, None] / 8 + 0.05 * rng.standard_normal((b, l, n_s))).astype(np.float32))
    xt = torch.from_numpy(np.stack([time_features(l, int(i)) for i in rng.integers(0, 2016, b)]))
    y = x[:, -1, :] + 0.01

    def step():
        opt.zero_grad(set_to_none=True)
        loss = torch.nn.functional.mse_loss(model(x, xt), y)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()

    for _ in range(max(1, args.warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    t = (time.perf_counter() - t0) / args.steps
    line = {"impl": "reference", "metric": "predictor_windows_per_sec_train_step", "value": b / t, "unit": "windows/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"predictor_train: NormalPredictorTCN (405 021 parameters), batch {b} x 36 steps x {n_s} sensors, "
                                   f"one AdamW step ({wl['cfg']})"},
            "cpu_baseline": {"value": b / t, "unit": "windows/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"{args.steps} steps of batch {b}, {t * 1e3:.0f} ms/step"},
            "e2e": {"value": b / t, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_reference(args, wl: dict) -> None:
    """--impl reference: the reference path on the host cores (oracle port) at the product arm's scopes: `value` = GNN
    stack from resident sensor embeddings (whole training step for ltown_dp256), `e2e` = the full detector call, each on a
    bounded sample of the workload per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    net = network(wl["net"], args.pipes)
    sample_b = args.cpu_sample
    full = cpu_full_step_fn(net, wl, sample_b, args.l_det, with_predictor=wl["full_step"])
    if wl["full_step"]:
        for _ in range(max(1, min(args.warmup, 2))):
            full()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            full()
        t_value = t_e2e = (time.perf_counter() - t0) / args.steps
    else:
        t_value = cpu_stack_time(net, wl, sample_b, max(3, min(args.steps, 10)))
        full()
        k = max(1, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(k):
            full()
        t_e2e = (time.perf_counter() - t0) / k
    value, e2e = sample_b / t_value, sample_b / t_e2e
    sample = (f"B={sample_b} windows x L={args.l_det} per step (bounded sample of the B={args.batch} workload); value: oracle "
              + ("whole training step" if wl["full_step"] else "GNN stack fwd+bwd from resident sensor embeddings")
              + f" ({t_value * 1e3:.0f} ms/step); e2e: full detector call incl. the sensor GRU ({t_e2e * 1e3:.0f} ms/step)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_value * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, wl, net, 1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "torch_geometric is not installable offline; this arm runs oracle/ (CPU restatement of the reference "
                "LeakDetector + PyG GCNConv/global_mean_pool) on all host threads; rank 0 only",
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_ours(args, wl: dict) -> None:
    import torch.distributed as dist

    from leak_det_gnn_b200 import instrument as inst
    from leak_det_gnn_b200.models import LeakDetector, NormalPredictorTCN, build_residual_sequence_from_segment
    from leak_det_gnn_b200.parallel import FlatGradBucket

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    net = network(wl["net"], args.pipes)
    n_s, hidden, l_pred = len(net["sensors"]), wl["hidden"], 36
    torch.manual_seed(42)
    model = LeakDetector(net["inp"], net["sensors"], net["pipe_ids"], sensor_hidden=64, node_hidden=hidden, gnn_layers=2,
                         dropout=0.1, use_time=True).to(dev).train()
    params = [p for p in model.parameters()]
    n_classes = len(net["pipe_ids"]) + 1

    full_step = wl["full_step"]
    seg_len = args.l_det + (l_pred if full_step else 0)
    signal_h, tfeat_h, label_h = synthetic_batch(args.batch, seg_len, n_s, n_classes, 198 + rank)
    signal_h, tfeat_h = signal_h.pin_memory(), tfeat_h.pin_memory()
    label = label_h.to(dev)
    loss_h = torch.empty((), dtype=torch.float32).pin_memory()
    predictor = NormalPredictorTCN(n_s, 9).to(dev).eval() if full_step else None
    opt = torch.optim.AdamW(params, lr=1e-3) if full_step else None

    # data parallel over windows: every p.grad is a view into ONE flat bucket (242 KB); backward accumulates
    # straight into it and a single NCCL all-reduce averages it (leak_det_gnn_b200/parallel.py)
    bucket = FlatGradBucket(params)
    unit_bytes = net["n_nodes"] * hidden * 4 * args.batch
    flush = torch.empty(64 * 1024 * 1024, device=dev) if unit_bytes * 8 < 400e6 else None  # 256 MB > L2
    last = {}   # the logits and loss of the latest step (graph replays: their static tensors), for --dump-outputs

    def detector_step(residual, tfeat):
        """reference train_detector.py:310-317 from the detector call on"""
        bucket.zero()
        logits = model(residual, tfeat)
        loss = torch.nn.functional.cross_entropy(logits, label)
        last.update(logits=logits.detach(), loss=loss.detach())
        loss.backward()
        bucket.allreduce()
        if full_step:
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
        return loss

    def call_from_device_inputs(sig, tf):
        if full_step:
            with torch.no_grad():
                residual = build_residual_sequence_from_segment(predictor, sig, tf, l_pred, args.l_det)
            return detector_step(residual, tf[:, l_pred:, :].contiguous())
        return detector_step(sig, tf)

    # ---- scope `value` ----
    sig_d, tf_d = signal_h.to(dev), tfeat_h.to(dev)
    graphed = bool(wl.get("graphed")) and not args.eager
    g_value = g_e2e = None
    if graphed:
        # small-batch workloads: the step is launch-bound when issued kernel by kernel, so the product path is a
        # CUDA-graph replay of the whole step (leak_det_gnn_b200/graphed.py); --eager times the call-by-call form
        from leak_det_gnn_b200.graphed import GraphedStep, GraphedTrainStep

        def recorded_ce(logits, target):
            last["logits"] = logits.detach()
            return torch.nn.functional.cross_entropy(logits, target)

        g_e2e = GraphedTrainStep(model, opt, bucket, args.batch, args.l_det, predictor=predictor,
                                 l_pred=l_pred if full_step else 0, grad_clip=1.0 if full_step else 0.0,
                                 loss_fn=recorded_ce)
        g_e2e.label.copy_(label)
    if full_step:
        def eager_value_step():
            if flush is not None:
                flush.fill_(0.0)
            call_from_device_inputs(sig_d, tf_d)
    else:
        with torch.no_grad():
            h_s = model.sensor_encoder(sig_d, tf_d)
        h_s = h_s.detach().clone().requires_grad_(True)

        def eager_value_step():
            if flush is not None:
                flush.fill_(0.0)
            bucket.zero()
            h_s.grad = None
            logits = model.gnn_stack(h_s)
            loss = torch.nn.functional.cross_entropy(logits, label)
            last.update(logits=logits.detach(), loss=loss.detach(), h_s=h_s)
            loss.backward()
            bucket.allreduce()

    if graphed:
        if full_step:
            g_value = g_e2e
            g_value.noisy.copy_(sig_d)
            g_value.time.copy_(tf_d)
        else:
            def stack_fwd_bwd():
                bucket.zero()
                leaf = h_s.detach().requires_grad_(True)
                logits = model.gnn_stack(leaf)
                loss = torch.nn.functional.cross_entropy(logits, label)
                last.update(logits=logits.detach(), h_s=leaf)   # captured: every replay rewrites them and leaf.grad
                loss.backward()
                return loss
            g_value = GraphedStep(model, stack_fwd_bwd, None, bucket)

        def value_step():
            if flush is not None:
                flush.fill_(0.0)
            g_value.replay()
    else:
        value_step = eager_value_step

    # e2e input pipeline: like a DataLoader with pinned memory and a prefetch depth of one, the H2D copy of the NEXT
    # step's batch runs on a copy stream while the current step computes.  Every step still copies its own
    # inputs from pinned host memory inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    dev_bufs = [(torch.empty(signal_h.shape, device=dev), torch.empty(tfeat_h.shape, device=dev)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"step": 0, "prefetched": -1}

    def prefetch(i):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])      # the step that last read this buffer has finished with it
            dev_bufs[slot][0].copy_(signal_h, non_blocking=True)
            dev_bufs[slot][1].copy_(tfeat_h, non_blocking=True)
            ready[slot].record(copy_stream)
        state["prefetched"] = i

    def e2e_step():
        i = state["step"]
        if state["prefetched"] < i:
            prefetch(i)
        prefetch(i + 1)
        slot = i % 2
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(ready[slot])
        if flush is not None:
            flush.fill_(0.0)
        if g_e2e is not None:
            loss = g_e2e(dev_bufs[slot][0], dev_bufs[slot][1], label)   # device-to-device into the graph's static inputs
        else:
            loss = call_from_device_inputs(*dev_bufs[slot])
        consumed[slot].record(cur)
        loss_h.copy_(loss.detach(), non_blocking=True)
        state["step"] = i + 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, timing_kernels=False, finish=None):
        for _ in range(warmup):
            fn()
        barrier()
        inst.reset(timing=timing_kernels)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, inst.launches, inst.summary()

    # rank 0 alone samples clocks and brackets kernels with events: 8 nvidia-smi pollers + per-kernel events on
    # every rank measurably slow the host side of an 8-process run
    if rank == 0:
        with ClockSampler(local) as clk:
            ms_stack, launches, ksum = timed(value_step, args.steps, args.warmup, timing_kernels=not graphed)
        clocks = clk.result()
    else:
        ms_stack, launches, ksum = timed(value_step, args.steps, args.warmup)
        clocks = None
    if rank == 0 and args.dump_outputs:
        # what the last timed step of `value` handed its caller, before the passes below overwrite it: the logits and
        # loss, the gradient of every parameter and (GNN stack) of the sensor embeddings, the parameters after the update
        if graphed:
            last["loss"] = g_value.loss
        outs = {"logits": last["logits"], "loss": last["loss"]}
        if not full_step:
            outs["grad_h_s"] = last["h_s"].grad
        for name, p in model.named_parameters():
            outs[f"grad.{name}"] = p.grad
            if full_step:
                outs[f"param.{name}"] = p
        dump_outputs(args.dump_outputs, {k: v.detach().cpu().numpy() for k, v in outs.items()})
    ms_kernel_pass = ms_stack
    if graphed:   # kernels inside a graph replay cannot be bracketed by events: per-kernel durations from an eager pass
        ms_kernel_pass, _, ksum = timed(eager_value_step, args.steps, args.warmup, timing_kernels=(rank == 0))
    if flush is not None:  # the flush fill is not part of the step: time it alone and take it out
        fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fe0.record()
        for _ in range(args.steps):
            flush.fill_(0.0)
        fe1.record()
        torch.cuda.synchronize()
        flush_ms = fe0.elapsed_time(fe1)
    else:
        flush_ms = 0.0
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    # the end event also waits for the copy stream: all K copies issued inside the region are inside the time
    ms_e2e, launches_e2e, ksum_e2e = timed(e2e_step, e2e_steps, max(3, min(args.warmup, 3)), timing_kernels=(rank == 0),
                                            finish=lambda: torch.cuda.current_stream(dev).wait_stream(copy_stream))

    ms_stack_net = max(ms_stack - flush_ms, 1e-6)
    ms_e2e_net = max(ms_e2e - flush_ms * e2e_steps / args.steps, 1e-6)
    value = args.batch * world * args.steps / (ms_stack_net * 1e-3)
    e2e_value = args.batch * world * e2e_steps / (ms_e2e_net * 1e-3)

    # B = 1 forward latency (event_evaluator.py:486 calls the detector one window at a time)
    latency = None
    if rank == 0 and args.workload == "lta128":
        model.eval()
        r1, t1 = sig_d[:1].contiguous(), tf_d[:1].contiguous()
        with torch.no_grad():
            for _ in range(5):
                model(r1, t1)
            torch.cuda.synchronize()
            le0, le1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            le0.record()
            for _ in range(50):
                model(r1, t1)
            le1.record()
            torch.cuda.synchronize()
        from leak_det_gnn_b200.event_windows import GraphedDetector

        graphed = GraphedDetector(model, 1, args.l_det)
        for _ in range(5):
            graphed(r1, t1)
        torch.cuda.synchronize()
        ge0, ge1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ge0.record()
        for _ in range(200):
            graphed(r1, t1)
        ge1.record()
        torch.cuda.synchronize()
        latency = {"b1_forward_ms": le0.elapsed_time(le1) / 50, "b1_forward_cuda_graph_ms": ge0.elapsed_time(ge1) / 200,
                   "calls": 50,
                   "scope": "LeakDetector.forward at B = 1, eval mode, device inputs (event_evaluator.py:486): eager "
                            "(one ctypes call per kernel) and replayed as a CUDA graph (event_windows.GraphedDetector)"}
        model.train()

    # ---- scope (i): the aggregation kernels alone (BASELINE metric "SpMM HBM GB/s vs peak"), outside the step ----
    agg_alone = None
    if rank == 0 and hidden % 32 == 0:
        from leak_det_gnn_b200 import ops

        xa = torch.randn(args.batch, net["n_nodes"], hidden, device=dev)
        staged = ops._staged_ok(model.pipe_graph, hidden)
        live = ops.new_live_mask(args.batch, net["n_nodes"], hidden, dev) if staged and net["n_nodes"] <= 1024 else None
        bias = torch.zeros(hidden, device=dev)
        forms = {
            "aggregate": lambda: ops.spmm(model.pipe_graph, xa),
            "aggregate_transpose": lambda: ops.spmm(model.pipe_graph, xa, transpose=True),
            "aggregate+bias+relu+dropout+mask": lambda: ops.spmm_fused(model.pipe_graph, xa, bias=bias, relu=True, drop_p=0.1,
                                                                       drop_seed=7, live_out=live),
        }
        if live is not None:
            forms["gate+aggregate_transpose+colsum"] = lambda: ops.spmm_fused(model.pipe_graph, xa, transpose=True,
                                                                              live_in=live, gate_scale=1.1, want_colsum=True)
        agg_alone = []
        for name, fn in forms.items():
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(10):
                fn()
            a1.record()
            torch.cuda.synchronize()
            ms = a0.elapsed_time(a1) / 10
            gbs = 2 * unit_bytes / (ms * 1e-3) / 1e9
            agg_alone.append({"kernel": name, "ms": ms, "achieved": gbs, "unit": "GB/s", "peak": peaks()["hbm_gbs"],
                              "frac": gbs / peaks()["hbm_gbs"], "algorithmic_bytes": 2 * unit_bytes,
                              "path": "STAGED (TMA + shared-memory topology)" if staged else "GATHER (L2)"})
        del xa, live

    # ---- rooflines, from the CUDA-event durations recorded live inside the timed region ----
    pk = peaks()
    unit_b = unit_bytes                                      # one (B, N, D) fp32 tensor
    rows_p = args.batch * args.pipes
    head_flops = 2.0 * rows_p * (3 * hidden) * 128           # EdgeHead first layer, fp32-equivalent flops
    # algorithmic bytes / flops per launch (SURVEY.md 8d; DESIGN.md "Kernels")
    model_of = {
        "spmm_fwd": ("hbm", 2 * unit_b), "spmm_bwd": ("hbm", 2 * unit_b),
        "spmm_fused_fwd": ("hbm", 2 * unit_b + unit_b // 32),   # read XW, write X_l and its 1-bit live mask
        "spmm_fused_bwd": ("hbm", 2 * unit_b + unit_b // 32),   # read dX_l and the live mask of X_l (gate), write G
        "gcn_layer_fwd": ("hbm", 2 * unit_b + unit_b // 32),     # fused layer: read X_{l-1}, write X_l and its live mask
        "linear_tc": ("hbm", 2 * unit_b), "wgrad_tc": ("hbm", 2 * unit_b), "wgrad": ("hbm", 2 * unit_b),
        "node_init_fwd": ("hbm", unit_b + unit_b // 32),          # write X_0 and its live mask
        "node_init_bwd": ("hbm", unit_b + unit_b // 32),          # read dX_0 and the live mask (sensor rows: 4 %)
        "mean_pool_fwd": ("hbm", unit_b), "mean_pool_bwd": ("hbm", unit_b),
        "pipe_head_fwd": ("tensor", head_flops), "pipe_head_bwd_dx": ("tensor", head_flops),
        "pipe_head_bwd_w": ("tensor", head_flops),
    }
    # e2e-only kernels (sensor GRU encoder): fp32-equivalent flops of the fused [h|x|tf|1] x [4H, 96] step GEMM
    q_seq = args.batch * n_s
    model_of["gru_fwd"] = ("tensor", 2.0 * q_seq * args.l_det * 256 * 75)
    model_of["gru_bwd_dg"] = ("tensor", 2.0 * q_seq * args.l_det * (192 * 64 + 64 * 64))  # dh GEMM + rebuilt hn
    model_of["gru_bwd_w"] = ("tensor", 2.0 * q_seq * args.l_det * 256 * 75)
    traffic = {}
    tpath = REPO / "profiles" / "ncu_traffic.json"
    if tpath.exists():
        traffic = json.loads(tpath.read_text()).get(f"B{args.batch}_P{args.pipes}", {})
    roofs = []
    for name, v in ksum.items():
        if name not in model_of or v["count"] == 0:
            continue
        bound, work = model_of[name]
        sec = v["mean_ms"] * 1e-3
        if bound == "hbm":
            ach, peak, unit = work / sec / 1e9, pk["hbm_gbs"], "GB/s"
        else:
            ach, peak, unit = work / sec / 1e12, pk["bf16_tflops"], "TFLOP/s"
        roofs.append({"kernel": name, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                      "traffic": traffic.get(name), "algorithmic_per_launch": work, "mean_launch_ms": v["mean_ms"],
                      "launches_timed": v["count"],
                      "share_of_step": v["total_ms"] / max(ms_kernel_pass - flush_ms, 1e-6)})
    roofs.sort(key=lambda r: -r["share_of_step"])
    roof = dict(roofs[0]) if roofs else None
    if roof:
        roof["peak_source"] = pk["source"]
        if graphed:
            roof["timed_in"] = ("an eager pass of the same step after the graph-replay timing (events cannot bracket kernels "
                                "inside a replay); share_of_step is relative to that pass")
        if roof["bound"] == "tensor":
            roof["note"] = ("achieved counts fp32-equivalent flops (2*M*K*N); the fp32-faithful 3xTF32 scheme issues 3 "
                            "TF32 MMAs per product and TF32 runs at half the bf16 rate, so the attainable ceiling is "
                            "peak/6; peak is the measured sustained bf16 GEMM rate")
    agg = [r for r in roofs if r["kernel"].startswith("spmm")]

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            torch.set_num_threads(os.cpu_count() or 1)
            if full_step:
                fn = cpu_full_step_fn(net, wl, args.cpu_sample, args.l_det, with_predictor=True)
                fn()
                t0 = time.perf_counter()
                for _ in range(2):
                    fn()
                t_cpu = (time.perf_counter() - t0) / 2
                what = "oracle whole training step (reference-equivalent torch TCN predictor + detector + clip + AdamW)"
            else:
                t_cpu = cpu_stack_time(net, wl, args.cpu_sample, 3)
                what = "oracle (torch CPU restatement of reference detector.py:178-218 + PyG GCNConv) GNN stack fwd+bwd"
            cpu = {"value": args.cpu_sample / t_cpu, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                   "sample": f"{what}, B={args.cpu_sample} windows of the same workload, {t_cpu * 1e3:.1f} ms/iter"}
        h2d = signal_h.numel() * 4 + tfeat_h.numel() * 4
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_stack_net / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, wl, net, world),
            "roofline": roof, "roofline_aggregation": agg, "aggregation_alone": agg_alone, "roofline_all": roofs,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e_net / e2e_steps, "steps": e2e_steps,
                    "scope": ("build_residual_sequence_from_segment (frozen TCN) + " if full_step else "")
                             + "LeakDetector.forward(residual, tfeat) incl. the sensor GRU encoder over L + CE + backward"
                             + (" + all-reduce + clip_grad_norm_ + AdamW" if full_step else "")
                             + ", pinned-host inputs copied H2D every step (on a copy stream, one step ahead of the "
                               "compute, like a prefetching data loader) and loss copied D2H every step"},
            "gpu_launches": launches, "clocks": clocks, "latency": latency,
            "kernels": {k: {"count": v["count"], "mean_ms": round(v["mean_ms"], 4)} for k, v in ksum.items()},
            "kernels_e2e": {k: {"count": v["count"], "mean_ms": round(v["mean_ms"], 4)} for k, v in ksum_e2e.items()},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="lta4096")
    ap.add_argument("--batch", type=int, default=None, help="windows per GPU (default: the workload's)")
    ap.add_argument("--l-det", type=int, default=None)
    ap.add_argument("--pipes", type=int, default=None)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-sample", type=int, default=None, help="windows per CPU-arm step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true", help="time the call-by-call step where the workload defaults to graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step of `value` computed as DIR/<name>.npy (float32, "
                         "at most 64 MB: larger outputs as a fixed sample of their rows); the inputs depend on the "
                         "arguments alone, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        raise SystemExit("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    wl = WORKLOADS[args.workload]
    args.batch = wl["batch"] if args.batch is None else args.batch
    args.l_det = wl["l_det"] if args.l_det is None else args.l_det
    args.pipes = wl["pipes"] if args.pipes is None else args.pipes
    args.cpu_sample = wl["cpu_sample"] if args.cpu_sample is None else args.cpu_sample
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload == "predictor_train":
        if args.impl != "reference":
            raise SystemExit("predictor_train is BASELINE configs[0], the reference's CPU baseline: run it with --impl reference "
                             "(the predictor has no graph layers; its training step is not on the sm_100a path)")
        run_predictor_train(args, wl)
        return
    if args.impl == "reference":
        run_reference(args, wl)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29541", __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_ours(args, wl)


if __name__ == "__main__":
    main()
