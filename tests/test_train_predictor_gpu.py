"""The predictor training launcher (leak_det_gnn_b200/train_predictor_dp.py): checkpoint layout of the reference's
train_predictor.py (SURVEY section 5), loadable by the detector launcher, and two NCCL ranks computing the gradients of one
process on the concatenated batch."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

from conftest import REPO, TOPO, rel_err

pytestmark = pytest.mark.gpu


def test_synthetic_run_writes_checkpoints_the_detector_launcher_loads(tmp_path, graph_golden):
    from leak_det_gnn_b200 import train_detector_dp
    from leak_det_gnn_b200.train_predictor_dp import main

    sensors = ",".join(str(s) for s in graph_golden("LTA")["sensor_node_ids"])
    pdir = tmp_path / "pred"
    metrics = main(["--out_dir", str(pdir), "--synthetic", "256", "--synthetic_sensors", sensors, "--batch_size", "64",
                    "--epochs", "2", "--val_steps", "128", "--log_every", "2"])
    assert set(metrics) == {"val_mae", "val_rmse"} and metrics["val_rmse"] > 0
    for name in ("predictor_best.ckpt", "predictor_last.ckpt", "predictor_meta.json"):
        assert (pdir / name).exists(), name
    ckpt = torch.load(pdir / "predictor_last.ckpt", map_location="cpu", weights_only=False)
    assert set(ckpt) == {"epoch", "arch", "model_state", "standardizer_mean", "standardizer_std", "sensor_ids", "args"}
    assert ckpt["epoch"] == 2 and ckpt["arch"] == "tcn" and len(ckpt["model_state"]) == 36
    assert json.loads((pdir / "predictor_meta.json").read_text())["sensor_ids"] == sensors.split(",")
    model, _ = train_detector_dp.load_predictor(pdir / "predictor_best.ckpt", torch.device("cuda"))
    assert model.num_sensors == len(sensors.split(","))
    train_detector_dp.main(["--inp_path", str(TOPO["LTA"]), "--out_dir", str(tmp_path / "det"), "--synthetic", "32",
                            "--predictor_ckpt", str(pdir / "predictor_best.ckpt"), "--synthetic_pipes", "40",
                            "--batch_size", "32", "--epochs", "1", "--val_steps", "32"])
    assert (tmp_path / "det" / "detector_last.ckpt").exists()


def test_gru_arch_points_to_the_reference(tmp_path):
    from leak_det_gnn_b200.train_predictor_dp import main

    with pytest.raises(SystemExit, match="models/train_predictor.py"):
        main(["--out_dir", str(tmp_path), "--arch", "gru", "--synthetic", "8"])


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {repo!r})
from leak_det_gnn_b200.models import NormalPredictorTCN
from leak_det_gnn_b200.parallel import FlatGradBucket
rank = int(os.environ["RANK"]); torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
blob = torch.load({blob!r})
m = NormalPredictorTCN(29, 9).cuda().eval()        # eval: no dropout, so the split is exact
m.load_state_dict(blob["state"])
bucket = FlatGradBucket(m.parameters())
lo, hi = (0, 128) if rank == 0 else (128, 256)
pred = m.forward_cone(blob["x"][lo:hi].cuda(), blob["xt"][lo:hi].cuda())
torch.nn.functional.mse_loss(pred, blob["y"][lo:hi].cuda()).backward()
bucket.allreduce()
if rank == 0:
    torch.save({{n: p.grad.cpu() for n, p in m.named_parameters()}}, {out!r})
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_gradients_equal_single_gpu_on_concatenated_batch(tmp_path):
    from leak_det_gnn_b200.models import NormalPredictorTCN

    torch.manual_seed(7)
    m = NormalPredictorTCN(29, 9).cuda().eval()
    gen = torch.Generator().manual_seed(8)
    blob = {"state": {k: v.cpu() for k, v in m.state_dict().items()}, "x": torch.randn(256, 36, 29, generator=gen),
            "xt": torch.randn(256, 36, 9, generator=gen), "y": torch.randn(256, 29, generator=gen)}
    torch.save(blob, tmp_path / "blob.pt")
    torch.nn.functional.mse_loss(m.forward_cone(blob["x"].cuda(), blob["xt"].cuda()), blob["y"].cuda()).backward()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(repo=str(REPO), blob=str(tmp_path / "blob.pt"), out=str(tmp_path / "g.pt")))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=600,
                       env={**os.environ, "PYTHONPATH": str(REPO)})
    assert r.returncode == 0, r.stderr[-3000:]
    got = torch.load(tmp_path / "g.pt")
    errs = {n: rel_err(got[n], p.grad) for n, p in m.named_parameters()}
    assert all(e <= 3e-6 for e in errs.values()), {n: e for n, e in errs.items() if e > 3e-6}
