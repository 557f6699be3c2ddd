"""SURVEY 8f rank 3: the data-parallel training entry point (leak_det_gnn_b200/train_detector_dp.py) keeps the
reference's flags and checkpoint layout (models/train_detector.py:131-155, 346-361), and with the REAL kernels two ranks
produce the gradients of one process on the concatenated batch (SURVEY 8d config 4)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

from conftest import REPO, TOPO, rel_err

pytestmark = pytest.mark.gpu


def test_launcher_trains_and_writes_reference_checkpoints(tmp_path, graph_golden):
    from leak_det_gnn_b200.models import LeakDetector
    from leak_det_gnn_b200.train_detector_dp import build_argparser, main

    ref_flags = {"leak_root", "inp_path", "predictor_ckpt", "out_dir", "epochs", "steps_per_epoch", "val_steps", "test_steps",
                 "batch_size", "lr", "weight_decay", "grad_clip", "l_pred", "l_det", "topk", "seed", "device", "num_workers",
                 "log_every"}                                               # models/train_detector.py:131-155
    assert ref_flags <= {a.dest for a in build_argparser()._actions}
    g = graph_golden("LTA")
    sensors = ",".join(str(s) for s in g["sensor_node_ids"])
    metrics = main(["--inp_path", str(TOPO["LTA"]), "--out_dir", str(tmp_path), "--synthetic", "192", "--synthetic_sensors",
                    sensors, "--synthetic_pipes", "40", "--batch_size", "32", "--epochs", "2", "--log_every", "3", "--val_steps",
                    "64"])
    assert {"acc_top1", "acc_top5", "det_f1", "early_n", "noleak_acc"} <= set(metrics) and metrics["n_total"] == 64
    for name in ("detector_best.ckpt", "detector_last.ckpt", "detector_meta.json"):
        assert (tmp_path / name).exists(), name
    ckpt = torch.load(tmp_path / "detector_last.ckpt", map_location="cpu", weights_only=False)
    assert set(ckpt) == {"epoch", "detector_state", "sensor_ids", "pipe_ids_in_order", "num_classes", "predictor_ckpt", "args"}
    assert ckpt["epoch"] == 2 and ckpt["num_classes"] == 41 and len(ckpt["detector_state"]) == 18
    # what eval/event_evaluator.py:249-259 does with such a file
    m = LeakDetector(TOPO["LTA"], ckpt["sensor_ids"], ckpt["pipe_ids_in_order"], sensor_hidden=64, node_hidden=64, gnn_layers=2,
                     dropout=0.1, use_time=True)
    m.load_state_dict(ckpt["detector_state"])


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {repo!r})
from leak_det_gnn_b200.models import LeakDetector
from leak_det_gnn_b200.parallel import FlatGradBucket
rank = int(os.environ["RANK"]); torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
blob = torch.load({blob!r})
m = LeakDetector({inp!r}, blob["sensors"], blob["pipes"]).cuda().eval()   # eval: no dropout, so the split is exact
m.load_state_dict(blob["state"])
bucket = FlatGradBucket(m.parameters())
lo, hi = (0, 24) if rank == 0 else (24, 48)
logits = m(blob["residual"][lo:hi].cuda(), blob["tfeat"][lo:hi].cuda())
torch.nn.functional.cross_entropy(logits, blob["label"][lo:hi].cuda()).backward()
bucket.allreduce()
if rank == 0:
    torch.save({{n: p.grad.cpu() for n, p in m.named_parameters()}}, {out!r})
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_gradients_equal_single_gpu_on_concatenated_batch(tmp_path, graph_golden):
    from leak_det_gnn_b200.models import LeakDetector

    g = graph_golden("LT")
    sensors, pipes = [str(s) for s in g["sensor_node_ids"]], [str(p) for p in g["pipe_ids"]]
    torch.manual_seed(7)
    m = LeakDetector(TOPO["LT"], sensors, pipes).cuda().eval()
    gen = torch.Generator().manual_seed(8)
    blob = {"sensors": sensors, "pipes": pipes, "state": {k: v.cpu() for k, v in m.state_dict().items()},
            "residual": torch.randn(48, 36, 29, generator=gen), "tfeat": torch.randn(48, 36, 9, generator=gen),
            "label": torch.randint(0, len(pipes) + 1, (48,), generator=gen)}
    torch.save(blob, tmp_path / "blob.pt")
    logits = m(blob["residual"].cuda(), blob["tfeat"].cuda())
    torch.nn.functional.cross_entropy(logits, blob["label"].cuda()).backward()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(repo=str(REPO), blob=str(tmp_path / "blob.pt"), inp=str(TOPO["LT"]), out=str(tmp_path / "g.pt")))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=600,
                       env={**os.environ, "PYTHONPATH": str(REPO)})
    assert r.returncode == 0, r.stderr[-3000:]
    got = torch.load(tmp_path / "g.pt")
    # equal halves: mean over 48 = average of the two means over 24.  Only the summation order differs (the row ranges of
    # the weight-gradient CTAs, torch's reduction trees, the NCCL average); measured 3e-7 .. 3e-6.  The scalar bias of the
    # last head layer is the exception: its gradient is the sum of all 48 x 905 pipe-logit gradients, which cancel to
    # 5e-4 of their absolute sum, so a reordering of torch's own fp32 sum moves it by 1e-5 (absolute: 2e-8).  As in
    # test_benchscale_gpu.py such ill-conditioned sums get 3e-5, and there may be at most two of them.
    errs = {n: rel_err(got[n], p.grad) for n, p in m.named_parameters()}
    loose = [n for n, e in errs.items() if e > 5e-6]
    assert len(loose) <= 2 and all(errs[n] <= 3e-5 for n in loose), {n: errs[n] for n in loose}
