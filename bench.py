#!/usr/bin/env python
"""bench.py -- DGCNN+GW inference throughput (blocks/s) on synthetic S3DIS-shaped blocks, BASELINE.json configs[1]:
full GFS model eval forward (DGCNN + attention + GW head, 13 classes, 150 geometric words), batch = 32 blocks of
2048 points x 9 channels per GPU, k = 20, random-init weights.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl gfs3d|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one eval forward of the model over one batch of 32 blocks.  Blocks are independent (SURVEY.md section 8e): every
rank processes its own 32 blocks, no data-path collective (weak scaling).  Prints ONE JSON line on rank 0.

--dump-outputs DIR writes the logits of the last timed step as DIR/logits.npy (float32, (blocks, classes, points);
DIR/logits_rank<r>.npy per rank when N > 1).  Inputs and weights come from fixed seeds, so two builds run with the same
arguments can be compared output for output.  Above 64 MB in all, a fixed seeded sample of whole blocks is written.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "gfs-3dseg_gws_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "dgcnn_gw_inference_blocks_per_sec"
UNIT = "blocks/s"
CLASSES, BASE_NUM, G, NPTS, KNN = 13, 7, 150, 2048, 20


def workload_name(batch):
    """config.workload of both arms (the reference arm runs the same workload on the host cores)"""
    return (f"BASELINE.json configs[1]: full GFS eval forward, batch={batch} S3DIS-shaped blocks/GPU, N={NPTS}, C=9, k={KNN}, "
            f"{CLASSES} classes, {G} GWs, random-init weights")


def model_args():
    return SimpleNamespace(edgeconv_widths=[[64, 64]] * 3, dgcnn_mlp_widths=[512, 256], pc_in_dim=9, dgcnn_k=KNN,
                           base_widths=[128, 64], output_dim=64, eval_weight=1.2)


def head_inputs(device):
    g = torch.Generator().manual_seed(11)
    gened = torch.nn.functional.normalize(torch.randn(CLASSES, 128, generator=g), dim=1)
    coding = (torch.rand(CLASSES, G, generator=g) < 0.3).float()
    return gened.to(device), coding[:BASE_NUM].to(device), coding[BASE_NUM:].to(device)


def build_model(device):
    from gfs3d.synthetic import randomize_bn_
    from model.capl import mpti_net_Point_GeoAsWeight_v2
    import contextlib
    torch.manual_seed(321)
    gp = torch.randn(G, 192, generator=torch.Generator().manual_seed(7))
    with contextlib.redirect_stdout(sys.stderr):      # the constructor prints (as the reference's does); stdout carries ONE JSON line
        m = mpti_net_Point_GeoAsWeight_v2(classes=CLASSES, criterion=torch.nn.CrossEntropyLoss(ignore_index=255), args=model_args(),
                                          base_num=BASE_NUM, gp=gp.to(device), energy=0.9)
    randomize_bn_(m, seed=6)
    return m.to(device).eval(), gp


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def reference_forward(device, state_dict, gp):
    """(kind, fn): fn(x) -> logits through the reference's OWN model classes (model/capl.py:144-192, unmodified byte copies
    staged by oracle/make_ref.py under oracle/_ref/reference; kind "reference") or, when they have not been staged, through the
    oracle port (oracle/gfs_oracle.py:forward_eval, the same ATen ops in the same order; kind "port")."""
    import contextlib
    import importlib
    from oracle import make_ref
    gened, bc, nc = head_inputs(device)
    ref = make_ref.ref_dir()
    if ref is None:
        from oracle import gfs_oracle as O
        sd = {k: v.detach().float().to(device) for k, v in state_dict.items()}
        gpd = gp.to(device)
        return "port", lambda x: O.forward_eval(sd, gpd, x, gened, bc, nc, BASE_NUM, 1.2, k=KNN)[0]
    ours = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "model" or k.startswith("model.")}
    import types
    pkg = types.ModuleType("model")                                  # the reference's model/ has no __init__.py (namespace package):
    pkg.__path__ = [os.path.join(ref, "model")]                      # a regular package of the same name would shadow it
    sys.modules["model"] = pkg
    try:
        capl = importlib.import_module("model.capl")                 # the reference's model package, not this repo's
    finally:
        for k in [k for k in sys.modules if k == "model" or k.startswith("model.")]:
            del sys.modules[k]
        sys.modules.update(ours)
    assert os.path.abspath(capl.__file__).startswith(os.path.abspath(ref))
    with contextlib.redirect_stdout(sys.stderr):
        m = capl.mpti_net_Point_GeoAsWeight_v2(classes=CLASSES, criterion=torch.nn.CrossEntropyLoss(ignore_index=255), args=model_args(),
                                               base_num=BASE_NUM, gp=gp.to(device), energy=0.9)
    m.load_state_dict({k: v.detach().float().cpu() for k, v in state_dict.items()})
    m = m.to(device).eval()
    return "reference", lambda x: m(x=x, y=None, eval_model=True, gen_proto=False, gened_proto=gened, base_class_coding=bc,
                                    novel_class_coding=nc)[0]


def cpu_port_blocks_per_sec(state_dict, gp, sample_blocks, iters, threads):
    """the reference's CPU path on the host cores: (blocks/s, kind) -- see reference_forward"""
    from gfs3d.synthetic import synthetic_blocks
    torch.set_num_threads(threads)
    kind, fwd = reference_forward("cpu", state_dict, gp)
    x = synthetic_blocks(sample_blocks, NPTS, seed=999)
    with torch.no_grad():
        fwd(x[:1])     # warm-up
        t0 = time.perf_counter()
        for _ in range(iters):
            fwd(x)
        dt = time.perf_counter() - t0
    return sample_blocks * iters / dt, kind


def run_reference(a):
    """--impl reference: the reference's own CPU implementation of the path -- its unmodified model classes when
    oracle/make_ref.py staged them (oracle/_ref, git-ignored, travels with the snapshot), else the oracle port --
    all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    m, gp = build_model("cpu")
    # each step is the workload's own batch (32 blocks, ~1.6 s on 16 cores) unless that would take more than a few minutes
    sample = a.batch if (a.steps + a.warmup) * a.batch <= 2400 else 4
    t0 = time.perf_counter()
    v, kind = cpu_port_blocks_per_sec(m.state_dict(), gp, sample, max(1, a.steps), threads)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * sample / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(a.batch),
                       "blocks_per_step": sample, "blocks_per_gpu_per_step": sample,
                       "note": "the reference's CPU path on the host cores" + ("" if sample == a.batch else ", bounded sample of the batch=32 workload")},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": f"{sample} blocks x {max(1, a.steps)} steps"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t0}
    emit(line)


SCANNET = dict(classes=21, base_num=15, G=180)


def build_train_model(device):
    """BASELINE.json configs[2]: ScanNet-shaped model (21 classes, 180 GWs, base_num 15), random init, train mode"""
    from gfs3d.synthetic import randomize_bn_
    from model.capl import mpti_net_Point_GeoAsWeight_v2
    import contextlib
    torch.manual_seed(321)
    gp = torch.randn(SCANNET["G"], 192, generator=torch.Generator().manual_seed(7))
    with contextlib.redirect_stdout(sys.stderr):
        m = mpti_net_Point_GeoAsWeight_v2(classes=SCANNET["classes"], criterion=torch.nn.CrossEntropyLoss(ignore_index=255),
                                          args=model_args(), base_num=SCANNET["base_num"], gp=gp.to(device), energy=0.9)
    randomize_bn_(m, seed=6)
    return m.to(device).train()


def train_leg(dev, rank, world, dist, batch, steps, warmup):
    """configs[2]: data-parallel training step, forward + backward + ONE flat-bucket NCCL all-reduce + Adam (train.py:616-631)"""
    import random
    from gfs3d import ops
    from gfs3d.dist import GradBucket
    from gfs3d.synthetic import synthetic_blocks
    m = build_train_model(dev)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    bucket = GradBucket(m.parameters())
    xs = [synthetic_blocks(batch, NPTS, seed=5000 + 1000 * rank + 7 * i).to(dev) for i in range(2)]
    ys = [torch.randint(0, SCANNET["base_num"] + 1, (batch, NPTS), generator=torch.Generator().manual_seed(i + 10 * rank)).to(dev) for i in range(2)]
    random.seed(1 + rank)
    ar_ev = []

    def step(i, timed=False):
        bucket.zero()
        _, loss = m(x=xs[i % 2], y=ys[i % 2])
        loss.backward()
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        nfl = bucket.allreduce() if world > 1 else 0
        if timed:
            e1.record()
            ar_ev.append((e0, e1))
        opt.step()
        return loss, nfl

    for i in range(warmup):
        step(i)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    l0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        loss, nfl = step(i, timed=True)
    e1.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps, sum(a.elapsed_time(b) for a, b in ar_ev) / steps], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ok = bucket.views_intact() and bool(torch.isfinite(loss.detach()))
    del opt, bucket, m
    torch.cuda.empty_cache()
    return {"config": f"BASELINE.json configs[2]: ScanNet-shaped ({SCANNET['classes']} classes, {SCANNET['G']} GWs, base_num {SCANNET['base_num']}), "
                      f"batch {batch} blocks/GPU x {NPTS} points, fwd + bwd + flat-bucket all-reduce + Adam, attention dropout 0.1",
            "blocks_per_s": batch * world / (float(t[0]) / 1e3), "ms_per_step": float(t[0]), "allreduce_ms": float(t[1]),
            "allreduce_floats": nfl, "steps": steps, "gpu_launches_per_step": (ops.LAUNCHES - l0) / steps,
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9, "loss_last": float(loss.detach()), "dtype": "f32", "finite": ok}


def kmeans_leg(dev, rank, world, dist, n_total, iters):
    """configs[3]: get_basis global k-means (150 centroids, 192-d) over n_total synthetic points sharded over the ranks; Lloyd
    iterations through the product's KMeans.fit (E-step, M-step, one packed all-reduce, centre update, one host read each)"""
    from gfs3d.dist import shard_range
    from gfs3d.kmeans import KMeans
    D, K = 192, 150
    lo, hi = shard_range(n_total, rank, world)
    n = hi - lo
    g = torch.Generator(device=dev).manual_seed(99)
    cent = torch.randn(K, D, device=dev, generator=g)                     # the same mixture on every rank
    g2 = torch.Generator(device=dev).manual_seed(1000 + rank)
    X = cent[torch.randint(0, K, (n,), device=dev, generator=g2)] + 0.35 * torch.randn(n, D, device=dev, generator=g2)
    init = (cent + 0.2 * torch.randn(K, D, device=dev, generator=g)).cpu().numpy()
    km = KMeans(n_clusters=K, init=init, max_iter=2, tol=0.0, shard=world > 1)
    km.fit(X)                                                             # warm-up (allocator, lazy module loading)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    km = KMeans(n_clusters=K, init=init, max_iter=iters, tol=0.0, shard=world > 1).fit(X)
    # the collective alone: the packed fp64 [sums | counts | changed] vector of one iteration
    ar_ms = 0.0
    if dist is not None:
        buf = torch.zeros(K * D + K + 1, dtype=torch.float64, device=dev)
        for _ in range(3):
            dist.all_reduce(buf)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            dist.all_reduce(buf)
        e1.record()
        torch.cuda.synchronize()
        ar_ms = e0.elapsed_time(e1) / 20
    t = torch.tensor([km.lloyd_ms_ / max(1, km.n_iter_), ar_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    del X, km
    torch.cuda.empty_cache()
    return {"config": f"BASELINE.json configs[3]: Lloyd iterations of the global k-means, {n_total} points x {D}, {K} centroids, "
                      f"points sharded over {world} GPU(s)", "ms_per_iter": float(t[0]), "allreduce_ms": float(t[1]),
            "allreduce_bytes": (K * D + K + 1) * 8 if world > 1 else 0, "points_per_gpu": n, "points_total": n_total, "iters": iters,
            "points_per_s": n_total / (float(t[0]) / 1e3)}


def multi_gpu_check(dev, rank, world, dist):
    """N ranks against one: (a) sharded k-means (k-means++ seeding included) labels == single-GPU labels on a small problem,
    (b) the all-reduced flat gradient bucket == the average of the N per-rank gradients recomputed on rank 0"""
    if world == 1:
        return {"kmeans_sharded_equals_single": "n/a (1 rank)", "grad_allreduce_equals_replica_average": "n/a (1 rank)"}
    import random
    import numpy as np
    from gfs3d.dist import GradBucket, shard_range
    from gfs3d.kmeans import KMeans
    from gfs3d.synthetic import synthetic_blocks
    out = {}
    rs = np.random.RandomState(5)
    n, D, K = 24000, 192, 24
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    lo, hi = shard_range(n, rank, world)
    sh = KMeans(n_clusters=K, init="k-means++", random_state=11, shard=True).fit(X[lo:hi])
    one = KMeans(n_clusters=K, init="k-means++", random_state=11).fit(X)
    bad = torch.tensor([float((sh.labels_ != one.labels_[lo:hi]).sum()), float(abs(sh.n_iter_ - one.n_iter_))], dtype=torch.float64, device=dev)
    dist.all_reduce(bad)
    out["kmeans_sharded_equals_single"] = "ok" if float(bad.sum()) == 0 else f"MISMATCH: {int(bad[0])} labels, iteration count differs by {int(bad[1])}"
    # gradients
    m = build_train_model(dev)
    m.att_learner.dropout.p = 0.0
    bucket = GradBucket(m.parameters())
    B, N = 2, 256

    def batch_of(r):
        return (synthetic_blocks(B, N, seed=77 + 13 * r).to(dev),
                torch.randint(0, SCANNET["base_num"] + 1, (B, N), generator=torch.Generator().manual_seed(5 + r)).to(dev))

    def grad_of(r):
        bucket.zero()
        random.seed(1000 + r)
        x, y = batch_of(r)
        _, loss = m(x=x, y=y)
        loss.backward()
        return bucket.flat.clone()

    grad_of(rank)
    bucket.allreduce()
    got = bucket.flat.clone()
    err = torch.zeros(1, dtype=torch.float64, device=dev)
    if rank == 0:
        ref = torch.stack([grad_of(r) for r in range(world)]).double().mean(0)
        err[0] = float((got.double() - ref).norm() / ref.norm())
    dist.all_reduce(err)
    out["grad_allreduce_equals_replica_average"] = "ok" if float(err[0]) <= 1e-4 else f"MISMATCH: relative L2 {float(err[0]):.3e}"
    out["grad_rel_l2"] = float(err[0])
    del bucket, m
    torch.cuda.empty_cache()
    return out


def reference_on_b200(dev, state_dict, gp, B, iters=3):
    """context number (SURVEY.md section 2b): the reference's stock-PyTorch path (the oracle port executes the same ATen ops in
    the same order as model/capl.py:144-192) eager on the SAME B200, fp32 with TF32 off"""
    from gfs3d.synthetic import synthetic_blocks
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        kind, fwd = reference_forward(dev, state_dict, gp)
        x = synthetic_blocks(B, NPTS, seed=999).to(dev)
        with torch.no_grad():
            fwd(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fwd(x)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        return {"value": B / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "batch": B, "kind": kind,
                "what": "stock PyTorch eager (ATen / cuBLAS / cuDNN ops of the reference, fp32, TF32 off) on this B200, inputs resident"}
    except Exception as e:                                            # noqa: BLE001  (a context number must not kill the bench line)
        return {"error": f"{type(e).__name__}: {e}"[:200]}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
        torch.cuda.empty_cache()


_JSON_OUT = None


def claim_stdout():
    """stdout carries ONE JSON line: keep a private handle on it and send everything else that writes to file descriptor 1 --
    NCCL's version / debug lines, the reference constructors' prints -- to stderr"""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


DUMP_BYTES = 63_000_000                  # under 64 MB (either unit) with the .npy headers


def dump_logits(out_dir, logits, name, budget):
    """logits (B, classes, N) -> out_dir/<name>.npy as float32; whole blocks, a fixed seeded sample of them when the batch is
    larger than `budget` bytes (the kept block indices go to out_dir/<name>_blocks.npy as float64)"""
    import numpy as np
    a = logits.detach().float().cpu().numpy()
    keep = max(1, budget // (a[0].nbytes + 8))
    if a.shape[0] > keep:
        blocks = np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))
        a = a[blocks]
        np.save(os.path.join(out_dir, name + "_blocks.npy"), blocks.astype(np.float64))
    np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="gfs3d", choices=["gfs3d", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="blocks per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--skip-train", action="store_true", help="skip the configs[2] data-parallel training leg")
    ap.add_argument("--skip-kmeans", action="store_true", help="skip the configs[3] sharded k-means leg")
    ap.add_argument("--kmeans-points", type=int, default=4_000_000, help="total points of the k-means leg (sharded over the ranks)")
    ap.add_argument("--e2e-serial", action="store_true",
                    help="end-to-end leg without prefetch: H2D, forward and D2H of a step strictly one after the other")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the logits of the last timed step to DIR as .npy (float32), for comparing two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference" and a.dump_outputs:
        ap.error("--dump-outputs writes what the gfs3d path computed; --impl reference does not support it")
    if a.impl == "reference":
        return run_reference(a)
    a.warmup = max(a.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from gfs3d import ops
    from gfs3d.synthetic import synthetic_blocks
    m, gp = build_model(dev)
    gened, bc, nc = head_inputs(dev)
    B = a.batch
    NROT = 4     # distinct input batches, rotated
    host = [synthetic_blocks(B, NPTS, seed=1234 + 1000 * rank + 100 * i).pin_memory() for i in range(NROT)]
    xs = [h.to(dev) for h in host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    labels_host = torch.empty(B, NPTS, dtype=torch.int32).pin_memory()

    def step(x):
        with torch.no_grad():
            logits, _, _ = m(x=x, y=None, eval_model=True, gened_proto=gened, base_class_coding=bc, novel_class_coding=nc)
        return logits

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(a.warmup):
        step(xs[i % NROT])
    barrier()
    graphed = None
    if not a.no_graph:
        from gfs3d.graph import GraphedEval
        graphed = GraphedEval(step, xs[0])
        for i in range(a.warmup):
            graphed(xs[i % NROT])
        barrier()
    run = graphed if graphed is not None else step

    # ---- timed region 1: inputs resident in HBM; per-step CUDA events, L2 flushed between steps ----
    clocks = ClockSampler(local) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    l0 = ops.LAUNCHES
    barrier()
    w0 = time.perf_counter()
    for i in range(a.steps):
        flush.zero_()
        ev[i][0].record()
        last = run(xs[i % NROT])
        ev[i][1].record()
    barrier()
    wall = time.perf_counter() - w0
    if a.dump_outputs:                          # before the next replay overwrites the graph's static output
        os.makedirs(a.dump_outputs, exist_ok=True)
        dump_logits(a.dump_outputs, last, "logits" if world == 1 else f"logits_rank{rank}", DUMP_BYTES // world)
    last = None
    launches = (ops.LAUNCHES - l0) if graphed is None else graphed.kernels_per_replay * a.steps
    dev_ms = sum(s.elapsed_time(e) for s, e in ev)

    # ---- timed region 2: end to end through the public module API with HOST buffers (H2D + forward + D2H labels) ----
    # Default: the next batch's pinned host -> device copy is issued (on a copy stream, into a second device buffer) at the
    # START of a step's timed interval, so it runs under that step's kernels; every interval contains exactly one H2D, one
    # forward and one D2H of the labels.  --e2e-serial keeps the three strictly one after the other.
    xdev = [torch.empty(B, 9, NPTS, device=dev) for _ in range(2)]
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]     # H2D into xdev[j] finished
    freed = [torch.cuda.Event(), torch.cuda.Event()]     # the forward that read xdev[j] finished
    # warm-up of THIS leg's own operations (arg-max / int32 conversion / pinned device->host copy are first used here: their
    # one-time module loading must not land in the timed region)
    for i in range(a.warmup):
        lg = graphed(host[i % NROT]) if graphed is not None else step(host[i % NROT].to(dev, non_blocking=True))
        labels_host.copy_(lg.argmax(1).to(torch.int32), non_blocking=True)
    barrier()
    if not a.e2e_serial:
        with torch.cuda.stream(copy_stream):             # prologue: the first batch (its copy is the one step K-1 would prefetch)
            xdev[0].copy_(host[0], non_blocking=True)
            ready[0].record(copy_stream)
        freed[1].record(main_stream)
    for i in range(a.steps):
        flush.zero_()
        ev2[i][0].record()
        if a.e2e_serial:
            if graphed is not None:
                lg = graphed(host[i % NROT])                 # pinned host -> static device input, then one graph launch
            else:
                xdev[0].copy_(host[i % NROT], non_blocking=True)
                lg = step(xdev[0])
        else:
            cur, nxt = i & 1, (i + 1) & 1
            copy_stream.wait_event(ev2[i][0])                # the prefetch belongs to this interval
            copy_stream.wait_event(freed[nxt])
            with torch.cuda.stream(copy_stream):
                xdev[nxt].copy_(host[(i + 1) % NROT], non_blocking=True)
                ready[nxt].record(copy_stream)
            main_stream.wait_event(ready[cur])
            lg = graphed(xdev[cur]) if graphed is not None else step(xdev[cur])
            freed[cur].record(main_stream)
        labels_host.copy_(lg.argmax(1).to(torch.int32), non_blocking=True)
        if not a.e2e_serial:
            main_stream.wait_event(ready[(i + 1) & 1])       # the interval ends after ITS host -> device copy as well
        ev2[i][1].record()
    barrier()
    e2e_ms = sum(s.elapsed_time(e) for s, e in ev2)
    clk = clocks.stop() if clocks else None

    # ---- instrumented replay of the same steps: per-entry-point CUDA events for the roofline ----
    ops.PROFILE = {}
    for i in range(a.steps):
        flush.zero_()
        step(xs[i % NROT])
    torch.cuda.synchronize()
    prof = {k: sum(s.elapsed_time(e) for s, e in v) / a.steps for k, v in ops.PROFILE.items()}   # ms per step per entry point
    calls = {k: len(v) // a.steps for k, v in ops.PROFILE.items()}
    ops.PROFILE = None

    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])

    # ---- BASELINE.json configs[2] / configs[3] at the same N (the only places the path has a collective), and the N-rank checks
    used_graph = graphed is not None
    graphed = run = None                        # drop the captured graph's memory pool before the training leg
    torch.cuda.empty_cache()
    train = None if a.skip_train else train_leg(dev, rank, world, dist, B, steps=5, warmup=3)
    kmeans = None if a.skip_kmeans else kmeans_leg(dev, rank, world, dist, a.kmeans_points, iters=8)
    checks = multi_gpu_check(dev, rank, world, dist) if not (a.skip_train and a.skip_kmeans) else None
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"

    # dominant kernel: the fused kNN (3 launches per step; the two C=64 layers dominate)
    knn_ms = prof.get("gfs_knn_tc_set_f32", 0.0) + prof.get("gfs_knn_tc_f32", 0.0) + prof.get("gfs_knn_f32", 0.0)
    knn_bytes = sum(B * NPTS * (c * 4 + KNN * 4) for c in (9, 64, 64))                  # read x once + write idx, per step
    knn_flops = sum(2.0 * c * NPTS * NPTS * B for c in (9, 64, 64))
    ec_ms = prof.get("gfs_edgeconv_fwd", 0.0)
    ec_bytes = 3 * B * NPTS * (128 * 4 + KNN * 4 + 64 * 4)                              # read P',Q',idx + write y (SURVEY 8d)
    ec123_ms = knn_ms + ec_ms + prof.get("gfs_pointwise_f32", 0.0)
    ec123_bytes = 1316 * NPTS * B                                                        # compulsory bytes (SURVEY 8d)
    gbs = lambda byt, ms: (byt / 1e9) / (ms / 1e3) if ms > 0 else None
    traffic = None          # dram__bytes_read+write of the kNN kernels of a step (3 x prep, filter, finish), from the committed ncu captures
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["knn_bytes_per_step_b32"] * B / 32.0
    except Exception:
        pass
    roof = {"kernel": "kNN graph: knn_prep + knn_tc (two-pass tcgen05 filter) + knn_finish (gfs_knn_tc_set_f32, 3 calls/step)", "bound": "hbm", "achieved": gbs(knn_bytes, knn_ms), "peak": hbm_peak,
            "unit": "GB/s", "frac": (gbs(knn_bytes, knn_ms) or 0) / hbm_peak, "traffic": traffic, "peak_source": peak_src,
            "ms_per_step": knn_ms, "share_of_step": knn_ms / (sum(prof.values()) or 1),
            "binding_roof": "per-row top-k selection out of TMEM (dependent-issue latency), not HBM or the tensor pipe",
            "distance_tflops_algorithmic": knn_flops / 1e12 / (knn_ms / 1e3) if knn_ms else None,
            "timing": "CUDA events around every C-ABI call on the launch stream, instrumented replay of the same K steps"}
    # the same entry point against the tensor roof: algorithmic flops = 2 C N^2 per block and layer (the distance matrix); the
    # filter EXECUTES 12 C' N^2 (three bf16 products of the hi/lo split, candidates streamed twice, C' = C padded to 16)
    bf16_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1405.0)))
    knn_exec_flops = 12.0 * (16 + 64 + 64) * NPTS * NPTS * B
    knn_tensor = {"bound": "tensor", "achieved": knn_flops / 1e12 / (knn_ms / 1e3) if knn_ms else None, "peak": bf16_peak, "unit": "TFLOP/s",
                  "frac": (knn_flops / 1e12 / (knn_ms / 1e3) / bf16_peak) if knn_ms else None,
                  "executed_tflops": knn_exec_flops / 1e12 / (knn_ms / 1e3) if knn_ms else None,
                  "executed_frac": (knn_exec_flops / 1e12 / (knn_ms / 1e3) / bf16_peak) if knn_ms else None,
                  "note": "over the whole kNN entry point (preparation + filter + exact finish); the filter kernel alone runs the "
                          "tensor pipe at 43-46 % (ncu, profiles/r2_summary.md)"}
    extra = {
        "knn_graph_tensor": knn_tensor,
        "edgeconv_given_graph": {"bound": "hbm", "achieved": gbs(ec_bytes, ec_ms), "peak": hbm_peak, "unit": "GB/s",
                                 "frac": (gbs(ec_bytes, ec_ms) or 0) / hbm_peak, "ms_per_step": ec_ms},
        "edgeconv123_fused_knn": {"bound": "hbm", "achieved": gbs(ec123_bytes, ec123_ms), "peak": hbm_peak, "unit": "GB/s",
                                  "frac": (gbs(ec123_bytes, ec123_ms) or 0) / hbm_peak, "ms_per_step": ec123_ms,
                                  "note": "compulsory bytes 1316*N per block; ceiling with brute-force fp32 kNN is ~2.5 % (SURVEY 8d)"},
        "entry_point_ms_per_step": prof, "entry_point_calls_per_step": calls,
    }

    cpu = None
    if not a.no_cpu_baseline:
        threads = os.cpu_count() or 1
        sample, iters = B, 8                                  # ~13 s of CPU work on 16 cores
        v, kind = cpu_port_blocks_per_sec(m.state_dict(), gp, sample, iters, threads)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": f"{sample} blocks x {iters} iterations of the same workload"}

    ref_gpu = None if a.no_cpu_baseline else reference_on_b200(dev, m.state_dict(), gp, B)
    total_blocks = B * a.steps * world
    h2d = B * 9 * NPTS * 4
    d2h = B * NPTS * 4
    line = {"metric": METRIC, "value": total_blocks / (dev_ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+bf16",
            "data": "synthetic",
            "config": {"workload": workload_name(B), "blocks_per_gpu_per_step": B,
                       "l2": "flushed between steps (256 MiB write outside the per-step event pair); 4 rotating input batches",
                       "parallelism": f"block-sharded x{world}, no data-path collective",
                       "launch": "CUDA graph replay of the eager step (gfs3d/graph.py)" if used_graph else "eager",
                       "attention": "hand-written tcgen05 flash kernel (gfs_attention_fwd)"},
            "clocks": clk, "e2e": {"value": total_blocks / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                   "ms_per_step": e2e_ms / a.steps,
                                   "mode": "serial: H2D, forward, D2H one after the other" if a.e2e_serial else
                                           "prefetch: each step's timed interval holds one pinned H2D (the next batch, on a copy "
                                           "stream, into a second device buffer), one forward and one D2H of the labels"},
            "gpu_launches": launches, "roofline": roof, "roofline_detail": extra, "cpu_baseline": cpu, "reference_pytorch_on_this_gpu": ref_gpu,
            "train": train, "kmeans": kmeans, "multi_gpu_check": checks, "wall_s_timed_region": wall}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
