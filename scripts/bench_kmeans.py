#!/usr/bin/env python
"""BASELINE.json configs[3]: global k-means (150 centroids, 192-d) over EdgeConv123-shaped features, per-GPU shard timing.

    python scripts/bench_kmeans.py [--n 500000] [--iters 10]          (one GPU: one shard of the 4 M / 8 split)
    torchrun --nproc-per-node N scripts/bench_kmeans.py --n 4000000   (points sharded over N GPUs, NCCL all-reduce)
    python scripts/bench_kmeans.py --weighted [--n 4194304]          (one GPU: weighted vs unweighted Lloyd iteration,
                                                                      the inertia pass, weighted k-means++ seeding)
    python scripts/bench_kmeans.py --clusters 150,256,512 --n 4000000  (one GPU: Lloyd iteration and E-step alone per K, the
                                                                      GW projection at G = 150 / 256 / 512 over 32 x 2048 rows)

Prints one JSON line: ms per Lloyd iteration (E-step + M-step + all-reduce), kernel times, achieved GB/s / TFLOP/s,
and sklearn's Lloyd iteration on a bounded sample of the host cores for comparison."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gfs-3dseg_gws_b200"))
from gfs3d import ops  # noqa: E402
from gfs3d.dist import allreduce_centroid_stats, shard_range  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=500000)
ap.add_argument("--iters", type=int, default=10)
ap.add_argument("--cpu-sample", type=int, default=200000)
ap.add_argument("--weighted", action="store_true", help="time the sample_weight path against the unweighted one (one GPU)")
ap.add_argument("--clusters", default=None, help="comma-separated K: time one Lloyd iteration (E + M) and the E-step alone per K, "
                "and the GW projection at the same widths (one GPU)")
a = ap.parse_args()
world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
D, K = 192, 150
lo, hi = shard_range(a.n, rank, world)
n = (hi - lo + 3) // 4 * 4
g = torch.Generator(device=dev).manual_seed(99 + rank)
cent = torch.randn(K, D, device=dev, generator=g)
X = cent[torch.randint(0, K, (n,), device=dev, generator=g)] + 0.35 * torch.randn(n, D, device=dev, generator=g)
xt = X.t().contiguous()
centers = X[torch.randperm(n, device=dev, generator=g)[:K]].clone()
Kp = (K + 3) // 4 * 4


def lloyd(centers):
    ct = torch.zeros(D, Kp, device=dev)
    ct[:, :K] = centers.t()
    labels = ops.kmeans_assign(xt, ct, K)
    sums, counts = ops.kmeans_accumulate(X, labels, K)
    if world > 1:
        sums, counts = allreduce_centroid_stats(sums, counts)
    return (sums / counts.clamp_min(1)[:, None]).float(), labels


def bench_weighted():
    """KMeans' Lloyd iteration as the fit issues it (E-step, M-step sums, pack, centre update, one 24-byte read), weighted and
    unweighted alternately in rounds; the inertia pass; weighted k-means++ seeding.  Prints the card and its power limit."""
    import subprocess
    from gfs3d.kmeans import KMeans as GKMeans
    w = torch.rand(n, device=dev, generator=g) * 2
    npad = xt.shape[1]
    ct = torch.zeros(D, Kp, device=dev)
    ct[:, :K] = centers.t()
    cnew, cold = torch.empty(K, D, device=dev), centers.clone()
    packed = torch.empty(K * D + K + 1, dtype=torch.float64, device=dev)
    counts = torch.empty(K, dtype=torch.int64, device=dev)
    ws_u, ws_w = ops.kmeans_accumulate_workspace(K, D, dev), ops.kmeans_accumulate_weighted_workspace(K, D, dev)
    scratch = torch.zeros(2, dtype=torch.int64, device=dev)
    result = torch.empty(3, dtype=torch.float64, device=dev)
    labels_old = torch.full((npad,), -1, dtype=torch.int32, device=dev)
    sums = packed[:K * D].view(K, D)

    def iteration(weighted):
        labels = ops.kmeans_assign(xt, ct, K)
        if weighted:
            ops.kmeans_accumulate_weighted(X, labels, w, K, sums=sums, wsums=packed[K * D:K * D + K], ws=ws_w)
        else:
            ops.kmeans_accumulate(X, labels, K, sums=sums, counts=counts, ws=ws_u)
        ops.kmeans_pack(labels, labels_old, n, K, D, packed, scratch, counts=None if weighted else counts)
        ops.kmeans_update(packed, cold, K, D, Kp, cnew, ct, result)
        result.tolist()
        return labels

    def timed(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, out

    for flag in (False, True, False, True):
        iteration(flag)                                    # warm-up
    rounds = {"unweighted": [], "weighted": []}
    for _ in range(5):
        rounds["unweighted"].append(timed(lambda: iteration(False), a.iters)[0])
        rounds["weighted"].append(timed(lambda: iteration(True), a.iters)[0])
    ops.PROFILE = {}
    iteration(False)
    labels = iteration(True)
    torch.cuda.synchronize()
    entries = {k: round(sum(s_.elapsed_time(e_) for s_, e_ in v), 4) for k, v in ops.PROFILE.items()}
    ops.PROFILE = None
    ops.kmeans_inertia(X, labels, cnew, w)
    inert = {"weighted_ms": timed(lambda: ops.kmeans_inertia(X, labels, cnew, w), 20)[0],
             "unweighted_ms": timed(lambda: ops.kmeans_inertia(X, labels, cnew), 20)[0]}
    inert["algorithmic_gbs"] = (n * D * 4 + n * 8) / inert["weighted_ms"] / 1e6
    seeder = GKMeans(n_clusters=K, init="k-means++", random_state=0)
    seeder._seed_plusplus(X[:40000], xt[:, :40000].contiguous(), np.random.RandomState(0), w=w[:40000].contiguous())   # warm-up
    seed_s = {}
    for name, ww in (("unweighted", None), ("weighted", w), ("unweighted_again", None), ("weighted_again", w)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        seeder._seed_plusplus(X, xt, np.random.RandomState(0), w=ww)
        torch.cuda.synchronize()
        seed_s[name] = time.perf_counter() - t0
    smi = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    med = {k: sorted(v)[len(v) // 2] for k, v in rounds.items()}
    print(json.dumps({"metric": "kmeans_weighted_lloyd_iteration_ms", "ms_per_iteration_median": med,
                      "ms_per_iteration_rounds": rounds, "weighted_over_unweighted": med["weighted"] / med["unweighted"],
                      "entry_ms_one_iteration_each": entries, "inertia": inert, "seeding_seconds": seed_s,
                      "points": n, "centroids": K, "dim": D, "gpu": torch.cuda.get_device_name(dev),
                      "nvidia_smi_name_power_limit": smi}))


def bench_clusters(ks):
    """K beyond 192 runs the panelled E-step (ceil(K / 192) passes over X) and, past the shared-memory table, the centre-split
    M-step.  Per K: KMeans' E-step (gfs_kmeans_assign_tc) alone and a whole Lloyd iteration as the fit issues it (E-step,
    M-step sums, pack, centre update, one read); then gfs_gw_project_tc with act tiles at B x N = 32 x 2048 and G = K.
    X (n x 192 fp32, 3 GB at 4 M points) is far larger than L2.  Prints the card and its power limit."""
    import subprocess
    import torch.nn.functional as F
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    out = {"metric": "kmeans_wide_dictionary_ms", "points": n, "dim": D, "gpu": torch.cuda.get_device_name(dev),
           "nvidia_smi_name_power_limit_max_sm_clock": smi, "kmeans": {}, "gw_project": {}}
    for k in ks:
        kp = (k + 3) // 4 * 4
        c = X[torch.randperm(n, device=dev, generator=g)[:k]].clone()
        ct = torch.zeros(D, kp, device=dev)
        ct[:, :k] = c.t()
        packed = torch.empty(k * D + k + 1, dtype=torch.float64, device=dev)
        sums = packed[:k * D].view(k, D)
        counts = torch.empty(k, dtype=torch.int64, device=dev)
        ws = ops.kmeans_accumulate_workspace(k, D, dev)
        scratch = torch.zeros(2, dtype=torch.int64, device=dev)
        result = torch.empty(3, dtype=torch.float64, device=dev)
        cnew, lold = torch.empty_like(c), torch.full((n,), -1, dtype=torch.int32, device=dev)

        def iteration():
            labels = ops.kmeans_assign(xt, ct, k)
            ops.kmeans_accumulate(X, labels, k, sums=sums, counts=counts, ws=ws)
            ops.kmeans_pack(labels, lold, n, k, D, packed, scratch, counts=counts)
            ops.kmeans_update(packed, c, k, D, kp, cnew, ct.clone(), result)
            result.tolist()
        labels = ops.kmeans_assign(xt, ct, k)
        e_ms = timed(lambda: ops.kmeans_assign(xt, ct, k), a.iters)
        m_ms = timed(lambda: ops.kmeans_accumulate(X, labels, k, sums=sums, counts=counts, ws=ws), a.iters)
        out["kmeans"][k] = {"lloyd_iteration_ms": timed(iteration, a.iters), "estep_ms": e_ms, "mstep_ms": m_ms,
                            "estep_passes_over_x": (kp + 191) // 192 if kp > 192 else 1}
    B, N = 32, 2048
    ec = torch.randn(B, D, N, device=dev, generator=g)
    for G in ks:
        Gp = (G + 63) // 64 * 64
        gp_l2t = torch.zeros(D, Gp, device=dev)
        gp_l2t[:, :G] = F.normalize(torch.randn(G, D, device=dev, generator=g), dim=1).t()
        act = ops.new_act(B * N, 3 + Gp // 64, dev)
        out["gw_project"][G] = {"ms": timed(lambda: ops.gw_project(ec, gp_l2t, G, cosine_act=act, kb0=3), 20), "rows": B * N}
    print(json.dumps(out))


if a.clusters:
    assert world == 1, "--clusters runs on one GPU"
    bench_clusters([int(v) for v in a.clusters.split(",")])
    sys.exit(0)

if a.weighted:
    assert world == 1, "--weighted runs on one GPU"
    bench_weighted()
    sys.exit(0)

for _ in range(3):
    centers, _ = lloyd(centers)
torch.cuda.synchronize()
ops.PROFILE = {}
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(a.iters):
    centers, labels = lloyd(centers)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / a.iters
prof = {k: sum(s.elapsed_time(e) for s, e in v) / a.iters for k, v in ops.PROFILE.items()}
t = torch.tensor([ms], dtype=torch.float64, device=dev)
if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
if rank == 0:
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    am = prof.get("gfs_kmeans_assign_tc", prof.get("gfs_kmeans_assign"))      # tensor-core E-step when the shape is eligible
    cm = prof["gfs_kmeans_accumulate"]
    line = {"metric": "kmeans_lloyd_iteration_ms", "value": float(t[0]), "unit": "ms", "n_gpus": world, "points_total": a.n,
            "points_per_gpu": n, "centroids": K, "dim": D, "higher_is_better": False,
            "assign": {"ms": am, "fp32_tflops": 2.0 * n * D * 192 / am / 1e9, "algorithmic_gbs": (n * D * 4 + n * 4) / am / 1e6},
            "accumulate": {"ms": cm, "algorithmic_gbs": (n * D * 4 + n * 4) / cm / 1e6, "hbm_peak_gbs": peaks.get("hbm_gbs")},
            "allreduce_bytes": (K * D + K) * 8 if world > 1 else 0}
    # k-means++ seeding (SURVEY 8f N3): one pass over the resident channel-major copy per centre (gfs_kmeans_pp_trial)
    from gfs3d.kmeans import KMeans as GKMeans
    seeder = GKMeans(n_clusters=K, init="k-means++", random_state=0)
    seeder._seed_plusplus(X[:40000], xt[:, :40000].contiguous(), np.random.RandomState(0))      # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    seeder._seed_plusplus(X, xt, np.random.RandomState(0))
    torch.cuda.synchronize()
    seed_s = time.perf_counter() - t0
    line["seeding"] = {"seconds": seed_s, "ms_per_centre": 1e3 * seed_s / K, "trials_per_centre": 2 + int(np.log(K)),
                       "algorithmic_gbs": K * n * D * 4 / 1e9 / seed_s, "hbm_peak_gbs": peaks.get("hbm_gbs")}
    if a.cpu_sample:
        from sklearn.cluster import KMeans
        rs = np.random.RandomState(0)
        c = rs.randn(K, D).astype(np.float32)
        Xc = (c[rs.randint(0, K, a.cpu_sample)] + 0.35 * rs.randn(a.cpu_sample, D)).astype(np.float32)
        init = Xc[rs.choice(a.cpu_sample, K, replace=False)]
        t0 = time.perf_counter()
        km = KMeans(n_clusters=K, init=init, n_init=1, max_iter=5, tol=0).fit(Xc)
        dt = time.perf_counter() - t0
        from sklearn.cluster import kmeans_plusplus
        t0 = time.perf_counter()
        kmeans_plusplus(Xc, K, random_state=np.random.RandomState(0))
        line["seeding"]["cpu_sklearn_seconds_scaled_to_points_per_gpu"] = (time.perf_counter() - t0) * n / a.cpu_sample
        line["cpu_sklearn"] = {"ms_per_iter": 1e3 * dt / max(1, km.n_iter_), "points": a.cpu_sample, "cores": os.cpu_count(),
                               "ms_per_iter_scaled_to_points_per_gpu": 1e3 * dt / max(1, km.n_iter_) * n / a.cpu_sample}
    print(json.dumps(line))
if world > 1:
    dist.destroy_process_group()
