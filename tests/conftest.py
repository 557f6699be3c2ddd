import sys
from pathlib import Path

import numpy as np
import pytest
import torch

REPO = Path(__file__).resolve().parents[1]
GOLDEN = REPO / "tests" / "golden"
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))

TOPO = {"LTA": GOLDEN / "L-TOWN-A.topo.inp", "LT": GOLDEN / "L-TOWN.topo.inp"}


# fp32 parity: cuDNN's RNN may otherwise run TF32 tensor-core math (torch default allow_tf32=True for
# cuDNN), which alone costs ~1e-3 on the GRU gradients; torch.matmul already defaults to full fp32.
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    # a gpu-marked test on a machine without CUDA is a skip, not a failure
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def graph_golden():
    def load(net: str):
        z = np.load(GOLDEN / f"graph_{net}.npz")
        return {k: z[k] for k in z.files}
    return load


@pytest.fixture(scope="session")
def detector_golden():
    def load(case: str):
        return torch.load(GOLDEN / f"detector_{case}.pt", map_location="cpu")
    return load


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    """max|a-b| / max|b| -- the norm-relative measure the fp32 tolerance is stated in (SURVEY 8c)."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    denom = b.abs().max().item()
    return (a - b).abs().max().item() / (denom if denom > 0 else 1.0)


def parity_log(tag: str, report: dict) -> None:
    """Per-tensor error report of a parity comparison: printed (pytest -s / -rP) and appended to
    gpurun_out/parity_report.jsonl so that the margins against the stated tolerances are on record."""
    import json
    line = json.dumps({"case": tag, "errors": report})
    print(line)
    out = REPO / "gpurun_out"
    try:
        out.mkdir(exist_ok=True)
        with open(out / "parity_report.jsonl", "a") as f:
            f.write(line + "\n")
    except OSError:
        pass
