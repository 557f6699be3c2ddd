"""bench.py contract: the reference arm (the oracle port on the host cores) prints ONE JSON line with the keys a caller
reads, and --dump-outputs writes what the GPU arm's last timed step computed, the same for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import REPO


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, str(REPO / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-sample", "2", "--l-det", "36"], capture_output=True, text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "window_graphs_per_sec_fwd_bwd" and d["unit"] == "window-graphs/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    # same scopes as the product arm: value = GNN stack from resident sensor embeddings, e2e = the full detector call
    # (sensor GRU included), so value / value and e2e / e2e ratios are like for like
    assert 0 < d["e2e"]["value"] <= d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]


def test_dump_outputs_keeps_the_total_under_the_limit_with_a_fixed_row_sample(tmp_path):
    big = np.arange(4000 * 300, dtype=np.float64).reshape(4000, 300)     # row r holds 300 r .. 300 r + 299
    other = 2.0 * big[:, :100]
    small = np.ones((3, 5))
    arrays = {"big": big, "other": other, "small": small, "loss": np.float64(2.5)}
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, arrays, limit=2_000_000)
    a = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    b = {p.stem: np.load(p) for p in (tmp_path / "b").glob("*.npy")}
    assert set(a) == set(arrays) and all(v.dtype == np.float32 for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 2_000_000
    assert all(np.array_equal(a[k], b[k]) for k in a)                    # the sample is fixed
    assert np.array_equal(a["small"], small) and a["loss"] == 2.5         # small arrays whole
    rows = (a["big"][:, 0] / 300).astype(np.int64)
    assert 1000 < len(rows) < 4000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["big"], big[rows]) and np.array_equal(a["other"], other[rows])   # same rows, in order
    bench.dump_outputs(tmp_path / "c", arrays)
    assert np.array_equal(np.load(tmp_path / "c" / "big.npy"), big)       # under the limit: everything


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """Two runs with the same arguments dump the same arrays (seeded inputs, deterministic kernels), and they belong to
    one step: the loss and the gradients of the two output biases follow from the dumped logits and the seeded labels."""
    args = [sys.executable, str(REPO / "bench.py"), "--workload", "lta128", "--batch", "8", "--steps", "2", "--warmup", "3",
            "--no-cpu-baseline"]
    runs = []
    for k in range(2):
        r = subprocess.run(args + ["--dump-outputs", str(tmp_path / str(k))], capture_output=True, text=True, timeout=600,
                           cwd=REPO, env={**os.environ, "BENCH_NO_CLOCKS": "1"})
        assert r.returncode == 0, r.stderr[-2000:]
        runs.append({p.stem: np.load(p) for p in (tmp_path / str(k)).glob("*.npy")})
    a, b = runs
    assert set(a) == set(b) and {"logits", "loss", "grad_h_s", "grad.convs.0.lin.weight"} <= set(a)
    for k in a:
        assert a[k].dtype == np.float32 and np.array_equal(a[k], b[k]), k
    assert a["logits"].shape == (8, 765) and a["grad_h_s"].shape == (8, 29, 64) and np.abs(a["grad_h_s"]).max() > 0
    _, _, label = bench.synthetic_batch(8, 36, 29, 765, 198)
    logits = torch.from_numpy(a["logits"]).double().requires_grad_(True)
    loss = torch.nn.functional.cross_entropy(logits, label)
    loss.backward()
    assert abs(loss.item() - float(a["loss"])) <= 1e-6 * loss.item()
    d = logits.grad
    assert abs(d[:, :764].sum().item() - float(a["grad.edge_head.mlp.3.bias"][0])) <= 1e-6
    assert abs(d[:, 764].sum().item() - float(a["grad.noleak_head.mlp.3.bias"][0])) <= 1e-6
