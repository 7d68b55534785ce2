#!/usr/bin/env python
"""BASELINE.json configs[2]: ScanNet-shaped training step (21 classes, 180 GWs, base_num 15, batch 32 blocks / GPU),
forward + backward + Adam, data-parallel with one flat-bucket NCCL gradient all-reduce per step.

    python scripts/bench_train.py [--batch 32] [--steps 10]
    torchrun --nproc-per-node N scripts/bench_train.py
    python scripts/bench_train.py --deterministic

Prints one JSON line (ms/step max over ranks, blocks/s whole job).  Attention dropout stays ON (p = 0.1) as in training.
--deterministic (one GPU): times the default step and the step under torch.use_deterministic_algorithms(True, warn_only=True),
with torch's NaN fill of uninitialised memory on and off, alternately for three rounds, and reports the ordered-scatter
entry points' times next to the atomic scatter's."""
import argparse
import json
import os
import random
import sys
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gfs-3dseg_gws_b200"))
from gfs3d import ops  # noqa: E402
from gfs3d.dist import allreduce_gradients  # noqa: E402
from gfs3d.synthetic import randomize_bn_, synthetic_blocks  # noqa: E402
from model.capl import mpti_net_Point_GeoAsWeight_v2  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=32)
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--npts", type=int, default=2048)
ap.add_argument("--deterministic", action="store_true", help="compare the default and the deterministic step (one GPU)")
a = ap.parse_args()
world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist = None
if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
CLASSES, BASE, G = 21, 15, 180
args = SimpleNamespace(edgeconv_widths=[[64, 64]] * 3, dgcnn_mlp_widths=[512, 256], pc_in_dim=9, dgcnn_k=20, base_widths=[128, 64],
                       output_dim=64, eval_weight=1.2)
torch.manual_seed(321)
import contextlib
with contextlib.redirect_stdout(sys.stderr):
    m = mpti_net_Point_GeoAsWeight_v2(classes=CLASSES, criterion=torch.nn.CrossEntropyLoss(ignore_index=255), args=args, base_num=BASE,
                                      gp=torch.randn(G, 192, generator=torch.Generator().manual_seed(7)).to(dev), energy=0.9)
randomize_bn_(m, seed=6)
m = m.to(dev).train()
opt = torch.optim.Adam(m.parameters(), lr=1e-3)
xs = [synthetic_blocks(a.batch, a.npts, seed=1000 * rank + 7 * i).to(dev) for i in range(2)]
ys = [torch.randint(0, BASE + 1, (a.batch, a.npts), generator=torch.Generator().manual_seed(i + rank)).to(dev) for i in range(2)]
random.seed(1 + rank)


def step(i):
    opt.zero_grad(set_to_none=True)
    pred, loss = m(x=xs[i % 2], y=ys[i % 2])
    loss.backward()
    n = allreduce_gradients(m.parameters()) if world > 1 else 0
    opt.step()
    return loss, n


def bench_deterministic():
    import subprocess
    import warnings
    warnings.filterwarnings("ignore", message=".*deterministic.*")        # torch's alerts for its own ops (warn_only)
    modes = {"default": (False, True), "deterministic": (True, True), "deterministic_no_fill": (True, False)}

    def set_mode(name):
        on, fill = modes[name]
        torch.use_deterministic_algorithms(on, warn_only=True)
        torch.utils.deterministic.fill_uninitialized_memory = fill

    for name in modes:
        set_mode(name)
        for i in range(a.warmup):
            step(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rounds = {name: [] for name in modes}
    for _ in range(3):
        for name in modes:
            set_mode(name)
            torch.cuda.synchronize()
            e0.record()
            for i in range(a.steps):
                step(i)
            e1.record()
            torch.cuda.synchronize()
            rounds[name].append(round(e0.elapsed_time(e1) / a.steps, 3))
    scatter = {}
    for name in ("default", "deterministic"):
        set_mode(name)
        ops.PROFILE = {}
        step(0)
        torch.cuda.synchronize()
        scatter[name] = {k: round(sum(s_.elapsed_time(e_) for s_, e_ in v), 3) for k, v in ops.PROFILE.items()
                         if k.startswith(("gfs_edge_scatter", "gfs_edge_reverse"))}
        ops.PROFILE = None
    set_mode("default")
    smi = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    print(json.dumps({"metric": "gfs_train_step_ms_deterministic", "ms_per_step_rounds": rounds,
                      "ms_per_step_median": {k: sorted(v)[1] for k, v in rounds.items()},
                      "scatter_entry_ms_per_step": scatter, "steps_per_round": a.steps, "batch": a.batch, "npts": a.npts,
                      "gpu": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": smi,
                      "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9,
                      "config": "ScanNet-shaped: 21 classes, 180 GWs, base_num 15, fwd+bwd+Adam, attention dropout 0.1"}))


if a.deterministic:
    if world > 1:
        sys.exit("--deterministic runs on one GPU")
    bench_deterministic()
    sys.exit(0)

for i in range(a.warmup):
    step(i)
if dist:
    dist.barrier()
torch.cuda.synchronize()
l0 = ops.LAUNCHES
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(a.steps):
    loss, nred = step(i)
e1.record()
if dist:
    dist.barrier()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / a.steps
ops.PROFILE = {}
ops.PROFILE_SHAPES = True
step(0)
torch.cuda.synchronize()
prof = {k: round(sum(s_.elapsed_time(e_) for s_, e_ in v), 3) for k, v in ops.PROFILE.items()}
calls = {k: len(v) for k, v in ops.PROFILE.items()}
ops.PROFILE = None
t = torch.tensor([ms], dtype=torch.float64, device=dev)
if dist:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
if rank == 0:
    print(json.dumps({"metric": "gfs_train_step_blocks_per_sec", "value": a.batch * world / (float(t[0]) / 1e3), "unit": "blocks/s",
                      "ms_per_step": float(t[0]), "n_gpus": world, "batch_per_gpu": a.batch, "npts": a.npts, "classes": CLASSES, "gws": G,
                      "loss_last": float(loss.detach()), "gpu_launches_per_step": (ops.LAUNCHES - l0) / a.steps,
                      "allreduce_floats_per_step": nred, "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9,
                      "entry_point_ms": prof, "entry_point_calls": calls, "dtype": "f32", "config": "ScanNet-shaped: 21 classes, 180 GWs, base_num 15, fwd+bwd+Adam, attention dropout 0.1"}))
if dist:
    dist.destroy_process_group()
