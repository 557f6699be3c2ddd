"""Data-parallel training of the TCN normal-state predictor: the reference's ``python models/train_predictor.py`` with one
process per GPU.

    torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 -m leak_det_gnn_b200.train_predictor_dp \
        --normal_root DATA --out_dir OUT --reference_root /path/to/Leak-det-gnn [flags ...]

The step is the reference's loop (train_predictor.py:203-228): prediction of the next step -> MSE -> backward -> clip_grad_norm_
-> AdamW (lr 1e-3, weight decay 1e-4, clip 1.0, batch 256, 15 epochs x 100 000 steps by default).  What changes:

* the prediction is ``NormalPredictorTCN.forward_cone``: only the dependency cone of the last time step (the only one the
  loss reads) on the sm_100a kernels, the same gradients as the dense model (up to the random dropout masks);
* gradients live in one flat 1.62 MB bucket (405 021 parameters) averaged by ONE NCCL all-reduce per step, before the clip;
  rank r takes samples r, r + W, ... so W ranks with ``--batch_size B`` reproduce one process with batch W * B;
* the step is one fixed launch sequence, captured once and replayed as a CUDA graph (graphed.GraphedStep;
  ``--cuda_graph 0`` issues it call by call);
* validation MAE / RMSE in original units are accumulated on the device through ``forward_last``.

Checkpoints (rank 0): ``predictor_best.ckpt``, ``predictor_last.ckpt`` with the keys ``epoch, arch, model_state,
standardizer_mean, standardizer_std, sensor_ids, args`` and ``predictor_meta.json`` -- what ``train_detector_dp
--predictor_ckpt`` loads.  ``predictor_best.ckpt`` is selected on validation RMSE (original units).  This selection
metric is this launcher's choice: the reference's could not be confirmed from the sources available here.

Data: ``--reference_root`` puts the reference checkout on ``sys.path``; its ``models.datasets.NormalPredictorDataset`` and
``compute_sensor_stats_from_normal`` are used unchanged (the keyword arguments passed to them are not confirmed against
the reference source either).  **Validation is NOT on held-out scenes here.**  The reference splits the normal scenes
80/10/10 into train / validation / test (``split_ids``, train_predictor.py:44-55) and builds a dataset per split; how
those scene lists are handed to ``NormalPredictorDataset`` cannot be confirmed, so this launcher builds the training and
validation datasets over ALL scenes of ``--normal_root`` (different seeds, i.e. different windows of the same scenes) and
computes the standardiser over all of them.  Validation MAE / RMSE -- and with them the choice of
``predictor_best.ckpt`` -- therefore measure in-distribution error; the launcher says so when it starts.  To select on
held-out scenes, give the validation dataset a separate normal root (``--val_normal_root``).  ``--synthetic N`` instead generates N seeded normal windows per epoch in the dataset's
batch layout (``x (36, S)``, ``x_time (36, 9)``, ``y (S,)``), which is what the tests and smoke runs use.  Only the TCN is
built here: ``--arch gru`` exits with a pointer to the reference script.
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch.utils.data import DataLoader, Dataset, Subset

from .graphed import GraphedStep
from .models import NormalPredictorTCN
from .parallel import FlatGradBucket, broadcast_parameters, shard_indices
from .train_detector_dp import _dist_env, now

L_IN = 36   # the reference's hard-coded window length (train_predictor.py:135)


def build_argparser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--normal_root", type=str, default=None, help="Path to the normal-operation dataset root")
    ap.add_argument("--out_dir", type=str, required=True, help="Output directory for predictor checkpoints")
    ap.add_argument("--arch", type=str, default="tcn", choices=["tcn", "gru"])
    ap.add_argument("--epochs", type=int, default=15)
    ap.add_argument("--steps_per_epoch", type=int, default=100000)
    ap.add_argument("--val_steps", type=int, default=10000)
    ap.add_argument("--batch_size", type=int, default=256, help="per process (global batch = world size x this)")
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--weight_decay", type=float, default=1e-4)
    ap.add_argument("--grad_clip", type=float, default=1.0)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--num_workers", type=int, default=0)
    ap.add_argument("--log_every", type=int, default=200)
    # ---- additions
    ap.add_argument("--reference_root", type=str, default=None, help="checkout of the reference (for models.datasets)")
    ap.add_argument("--val_normal_root", type=str, default=None,
                    help="normal-operation root of held-out validation scenes (default: --normal_root, NOT held out)")
    ap.add_argument("--synthetic", type=int, default=0, help="use N synthetic windows per epoch instead of --normal_root")
    ap.add_argument("--synthetic_sensors", type=str, default=None,
                    help="comma-separated sensor node ids (synthetic mode; default 29 placeholder ids)")
    ap.add_argument("--cuda_graph", type=int, default=1, help="1: replay the training step as a CUDA graph; 0: eager")
    return ap


class SyntheticNormalWindows(Dataset):
    """Seeded normal windows in ``NormalPredictorDataset``'s item layout: ``x (36, S)`` standardised pressures with a daily
    cycle, ``x_time (36, 9)`` (hour sin / cos + day-of-week one-hot), ``y (S,)`` the next step; item ``idx`` depends only
    on ``seed + idx``."""

    def __init__(self, n: int, n_sensors: int, seed: int) -> None:
        self.n, self.s, self.seed = n, n_sensors, seed

    def __len__(self) -> int:
        return self.n

    def __getitem__(self, idx: int) -> Dict:
        rng = np.random.default_rng(self.seed + idx)
        minutes = 5 * (int(rng.integers(0, 288 * 7)) + np.arange(L_IN + 1))
        hour = ((minutes // 60) % 24 + (minutes % 60) / 60.0).astype(np.float32)
        ang = 2.0 * np.pi * hour / 24.0
        phase = rng.uniform(0, 2 * np.pi, self.s).astype(np.float32)
        seq = (np.sin(ang[:, None] + phase[None, :]) + 0.1 * rng.standard_normal((L_IN + 1, self.s))).astype(np.float32)
        tfeat = np.concatenate([np.sin(ang)[:, None], np.cos(ang)[:, None], np.eye(7, dtype=np.float32)[(minutes // 1440) % 7]],
                               axis=1).astype(np.float32)
        return {"x": torch.from_numpy(seq[:L_IN]), "x_time": torch.from_numpy(tfeat[:L_IN]), "y": torch.from_numpy(seq[L_IN])}


def predictor_loss(model: NormalPredictorTCN, x: torch.Tensor, x_time: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    return F.mse_loss(model.forward_cone(x, x_time), y)


class PredictorStep:
    """One training step (forward_cone -> MSE -> backward into the bucket -> all-reduce -> clip -> AdamW) for a fixed
    batch shape, eager or as graph replays (``cuda_graph``).  ``step(x, x_time, y)`` returns the device loss.
    ``opt = None`` (with ``grad_clip = 0``) leaves the weights alone: forward and backward only."""

    def __init__(self, model: NormalPredictorTCN, opt, bucket: FlatGradBucket, batch: int, grad_clip: float,
                 cuda_graph: bool, warmup: int = 3) -> None:
        dev = next(model.parameters()).device
        self.model, self.opt, self.bucket, self.grad_clip = model, opt, bucket, float(grad_clip)
        s = model.num_sensors
        self.x = torch.zeros(batch, L_IN, s, device=dev)
        self.x_time = torch.zeros(batch, L_IN, model.time_dim, device=dev)
        self.y = torch.zeros(batch, s, device=dev)
        model.train()
        self.graphed = (GraphedStep(model, self._fb, opt, bucket, grad_clip=grad_clip, warmup=warmup) if cuda_graph
                        else None)

    def _fb(self) -> torch.Tensor:
        self.bucket.zero()
        loss = predictor_loss(self.model, self.x, self.x_time, self.y)
        loss.backward()
        return loss

    def __call__(self, x: torch.Tensor, x_time: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
        self.x.copy_(x, non_blocking=True)
        self.x_time.copy_(x_time, non_blocking=True)
        self.y.copy_(y, non_blocking=True)
        if self.graphed is not None:
            return self.graphed.replay()
        loss = self._fb()
        self.bucket.allreduce()
        if self.grad_clip > 0:
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.grad_clip)
        if self.opt is not None:
            self.opt.step()
        return loss.detach()


@torch.no_grad()
def evaluate(model: NormalPredictorTCN, loader: DataLoader, std: torch.Tensor, device) -> Dict[str, float]:
    """Validation MAE / RMSE in original units (errors times the per-sensor standard deviation), summed on the device."""
    model.eval()
    abs_sum = torch.zeros((), device=device, dtype=torch.float64)
    sq_sum = torch.zeros((), device=device, dtype=torch.float64)
    n = 0
    for batch in loader:
        x, xt, y = (batch[k].to(device, non_blocking=True) for k in ("x", "x_time", "y"))
        err = (model.forward_last(x, xt) - y) * std
        abs_sum += err.abs().double().sum()
        sq_sum += err.double().square().sum()
        n += err.numel()
    model.train()
    n = max(n, 1)
    return {"val_mae": float(abs_sum) / n, "val_rmse": (float(sq_sum) / n) ** 0.5}


def main(argv: Optional[List[str]] = None) -> Dict[str, float]:
    args = build_argparser().parse_args(argv)
    if args.arch != "tcn":
        raise SystemExit("train_predictor_dp trains the TCN predictor only; train the GRU baseline with the reference's "
                         "`python models/train_predictor.py --arch gru`")
    rank, world, local = _dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("train_predictor_dp: needs a CUDA device (the native predictor training has no CPU path)")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    torch.manual_seed(args.seed)
    np.random.seed(args.seed)
    out_dir = Path(args.out_dir)
    if rank == 0:
        out_dir.mkdir(parents=True, exist_ok=True)
        print(f"{now()} [predictor] device={device} seed={args.seed} world={world}")

    if args.synthetic:
        sensor_ids = args.synthetic_sensors.split(",") if args.synthetic_sensors else [f"S{i}" for i in range(29)]
        mean = np.zeros(len(sensor_ids), dtype=np.float32)
        std = np.ones(len(sensor_ids), dtype=np.float32)
        train_ds = SyntheticNormalWindows(args.synthetic, len(sensor_ids), args.seed)
        val_ds = SyntheticNormalWindows(max(args.batch_size, min(args.val_steps, args.synthetic)), len(sensor_ids),
                                        args.seed + 1)
    else:
        if not (args.normal_root and args.reference_root):
            raise SystemExit("need --normal_root and --reference_root (or --synthetic N)")
        sys.path.insert(0, str(Path(args.reference_root)))
        from models.datasets import NormalPredictorDataset, compute_sensor_stats_from_normal  # the reference's loaders

        stdzr, sensor_ids = compute_sensor_stats_from_normal(args.normal_root)
        mean, std = np.asarray(stdzr.mean, dtype=np.float32), np.asarray(stdzr.std, dtype=np.float32)
        mk = lambda root, steps, seed: NormalPredictorDataset(normal_root=root, l_in_steps=L_IN, horizon_steps=1,
                                                              steps_per_epoch=steps, seed=seed, sensor_ids=sensor_ids,
                                                              standardizer=stdzr)
        train_ds = mk(args.normal_root, args.steps_per_epoch, args.seed)
        val_ds = mk(args.val_normal_root or args.normal_root, args.val_steps, args.seed + 1)
        if rank == 0 and not args.val_normal_root:
            print(f"{now()} [predictor] NOTE: validation windows come from the training scenes (no held-out scene split; "
                  "pass --val_normal_root for held-out validation): predictor_best.ckpt is chosen on in-distribution error")

    shard = Subset(train_ds, list(shard_indices(len(train_ds), rank, world)))
    train_loader = DataLoader(shard, batch_size=args.batch_size, num_workers=args.num_workers, pin_memory=True, drop_last=True)
    val_loader = DataLoader(val_ds, batch_size=args.batch_size, num_workers=args.num_workers, pin_memory=True)

    model = NormalPredictorTCN(num_sensors=len(sensor_ids), time_dim=9).to(device)
    broadcast_parameters(list(model.parameters()))
    bucket = FlatGradBucket(model.parameters())
    opt = torch.optim.AdamW(model.parameters(), lr=args.lr, weight_decay=args.weight_decay)
    step = PredictorStep(model, opt, bucket, args.batch_size, args.grad_clip, bool(args.cuda_graph))
    std_dev = torch.as_tensor(std, device=device)
    if rank == 0:
        meta = {"arch": "tcn", "sensor_ids": sensor_ids, "standardizer_mean": mean.tolist(),
                "standardizer_std": std.tolist(), "world_size": world, "args": vars(args)}
        (out_dir / "predictor_meta.json").write_text(json.dumps(meta, indent=2, ensure_ascii=False), encoding="utf-8")
    best, metrics = float("inf"), {}
    for epoch in range(1, args.epochs + 1):
        model.train()
        running = torch.zeros((), device=device)
        seen = 0
        for it, batch in enumerate(train_loader, start=1):
            loss = step(batch["x"], batch["x_time"], batch["y"])
            running += loss * batch["x"].size(0)
            seen += batch["x"].size(0)
            if rank == 0 and it % args.log_every == 0:
                print(f"{now()} [predictor][epoch {epoch:02d}] step {it:05d}/{len(train_loader):05d} "
                      f"loss={running.item() / max(seen, 1):.6f}")
        if rank == 0:
            metrics = evaluate(model, val_loader, std_dev, device)
            print(f"{now()} [predictor][epoch {epoch:02d}] train_loss={running.item() / max(seen, 1):.6f} "
                  f"val_mae={metrics['val_mae']:.6f} val_rmse={metrics['val_rmse']:.6f}")
            ckpt = {"epoch": epoch, "arch": "tcn", "model_state": model.state_dict(), "standardizer_mean": mean,
                    "standardizer_std": std, "sensor_ids": sensor_ids, "args": vars(args)}
            torch.save(ckpt, out_dir / "predictor_last.ckpt")
            if metrics["val_rmse"] < best:
                best = metrics["val_rmse"]
                torch.save(ckpt, out_dir / "predictor_best.ckpt")
        if world > 1:
            dist.barrier()
    if world > 1 and argv is None:
        dist.destroy_process_group()
    return metrics


if __name__ == "__main__":
    main()
