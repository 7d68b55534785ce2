"""CPU suite: the C-ABI library loads and exports every symbol include/gfs3d.h declares, its argument validation
follows the documented error convention (these calls return before touching CUDA), and the host-side sharding /
collective helpers work at world_size 2 over gloo."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "gfs3d.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gfs_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from gfs3d._lib import LIB_PATH, SIGNATURES, UTILITIES
    assert os.path.exists(LIB_PATH), "build the library first: python gfs-3dseg_gws_b200/build.py"
    l = ctypes.CDLL(LIB_PATH)
    names = _declared()
    assert len(names) >= 14
    for n in names:
        assert hasattr(l, n), f"{n} is declared in include/gfs3d.h but not exported"
    bound = set(SIGNATURES) | set(UTILITIES)
    assert set(names) == bound, f"ctypes table and header disagree: {set(names) ^ bound}"


def test_error_convention_without_gpu():
    from gfs3d._lib import lib
    l = lib()
    assert l.gfs_version() >= 100
    rc = l.gfs_knn_f32(None, 0, 1, 9, 128, 20, None, None, None, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    rc = l.gfs_knn_f32(p, 0, 1, 9, 128, 65, p, p, None, None)
    assert rc == 2 and b"k=65" in l.gfs_last_error_string()
    rc = l.gfs_knn_f32(p, 0, 1, 9, 16, 20, p, p, None, None)
    assert rc == 1 and b"exceeds N" in l.gfs_last_error_string()
    rc = l.gfs_linear_bf16(p, 3, 0, 3, p, None, 100, 1, 1, 128, p, 2, 0, None, 0, None)
    assert rc == 2 and b"multiple of 32" in l.gfs_last_error_string()
    # launch-policy switches are host state only: callable without a device
    assert l.gfs_set_pdl(0) == 0 and l.gfs_set_pdl(3) == 0
    assert l.gfs_knn_tc_set_split(-1) == 0


def test_product_path_has_no_cpu_fallback():
    from gfs3d import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.knn(torch.randn(1, 9, 128), 20)
    from model.dgcnn import DGCNN
    m = DGCNN([[64, 64]] * 3, [512, 256], 9).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 9, 128))
    with pytest.raises(NotImplementedError):
        DGCNN([[64, 128]], [256], 9).eval()._check_supported()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gfs-3dseg_gws_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                txt = open(os.path.join(d, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "oracle/" not in txt.replace("oracle/gfs_oracle.c", ""), f


def test_state_dict_contract_matches_reference_keys(golden_sd):
    from types import SimpleNamespace
    from model.capl import mpti_net_Point_GeoAsWeight_v2
    args = SimpleNamespace(edgeconv_widths=[[64, 64]] * 3, dgcnn_mlp_widths=[512, 256], pc_in_dim=9, dgcnn_k=20,
                           base_widths=[128, 64], output_dim=64, eval_weight=1.0)
    m = mpti_net_Point_GeoAsWeight_v2(classes=13, args=args, base_num=7, gp=torch.randn(150, 192), energy=0.9)
    ref = golden_sd("gfs_s3dis_weights")          # keys and shapes of the real reference model's state_dict
    mine = m.state_dict()
    assert list(mine.keys()) == list(ref.keys())
    for k in ref:
        assert tuple(mine[k].shape) == tuple(ref[k].shape), k
    assert "gp" not in mine                        # the GW basis is a plain attribute (model/capl.py:49-50)
    assert sum(p.numel() for p in m.parameters()) == 398144


def test_invalidate_folded_drops_every_weight_cache():
    """ADVICE r1: the folded-weight caches are keyed on tensor._version, which `.data` edits do not bump -> explicit hook"""
    from types import SimpleNamespace
    from model.capl import mpti_net_Point_GeoAsWeight_v2
    args = SimpleNamespace(edgeconv_widths=[[64, 64]] * 3, dgcnn_mlp_widths=[512, 256], pc_in_dim=9, dgcnn_k=20,
                           base_widths=[128, 64], output_dim=64, eval_weight=1.0)
    m = mpti_net_Point_GeoAsWeight_v2(classes=13, args=args, base_num=7, gp=torch.randn(150, 192), energy=0.9)
    caches = [mod._folded for mod in m.modules() if hasattr(mod, "_folded")]
    assert len(caches) >= 3                        # head, encoder, base learner
    for c in caches:
        c.key, c.data = ("stale",), object()
    m.att_learner._key, m.att_learner._wp = ("stale",), object()
    m.invalidate_folded()
    assert all(c.key is None and c.data is None for c in caches)
    assert m.att_learner._key is None and m.att_learner._wp is None


def test_act_layout_roundtrip_on_cpu():
    """the documented tile formula byte(r,c) = r*128 + (((c/8) ^ (r&7)) << 4) + (c%8)*2 vs ops.act_to_dense"""
    from gfs3d import ops
    M, kb = 256, 2
    dense = torch.arange(M * kb * 64, dtype=torch.float32).reshape(M, kb * 64) % 251
    act = torch.zeros(M // 128, kb, 128 * 64, dtype=torch.bfloat16)
    for mt in range(M // 128):
        for b in range(kb):
            tile = act[mt, b]
            for r in range(128):
                for q in range(8):
                    off = (r * 128 + ((q ^ (r & 7)) << 4)) // 2
                    tile[off:off + 8] = dense[mt * 128 + r, b * 64 + q * 8: b * 64 + q * 8 + 8].bfloat16()
    assert torch.equal(ops.act_to_dense(act, M).float(), dense)


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from gfs3d.dist import all_same, allreduce_centroid_stats, max_over_ranks, shard_range
    n, D, K = 1001, 8, 5
    rs = np.random.RandomState(0)
    X = rs.randn(n, D)
    labels = rs.randint(0, K, n)
    lo, hi = shard_range(n, rank, world)
    sums = torch.zeros(K, D, dtype=torch.float64)
    counts = torch.zeros(K, dtype=torch.int64)
    for i in range(lo, hi):
        sums[labels[i]] += torch.from_numpy(X[i])
        counts[labels[i]] += 1
    gs, gc = allreduce_centroid_stats(sums, counts)
    ref = np.zeros((K, D))
    for i in range(n):
        ref[labels[i]] += X[i]
    ok = np.allclose(gs.numpy(), ref) and gc.tolist() == np.bincount(labels, minlength=K).tolist()
    ok = ok and max_over_ranks(float(rank + 1), "cpu") == float(world)
    ok = ok and all_same(True, "cpu") and not all_same(rank == 0, "cpu")
    # flat-bucket gradient all-reduce (data-parallel training): average over ranks, written back in place
    from gfs3d.dist import allreduce_gradients
    ps = [torch.nn.Parameter(torch.zeros(3, 4)), torch.nn.Parameter(torch.zeros(5)), torch.nn.Parameter(torch.zeros(2))]
    ps[0].grad = torch.full((3, 4), float(rank + 1))
    ps[1].grad = torch.arange(5.0) * (rank + 1)
    n = allreduce_gradients(ps)
    ok = ok and n == 17 and torch.allclose(ps[0].grad, torch.full((3, 4), 1.5)) and torch.allclose(ps[1].grad, torch.arange(5.0) * 1.5)
    ok = ok and ps[2].grad is None
    # GradBucket: the gradients LIVE in one flat buffer, autograd accumulates into the views, one in-place all-reduce
    from gfs3d.dist import GradBucket
    lin = torch.nn.Linear(4, 3)
    with torch.no_grad():
        lin.weight.fill_(0.5)
        lin.bias.zero_()
    bucket = GradBucket(lin.parameters())
    bucket.zero()
    xin = torch.full((2, 4), float(rank + 1))
    lin(xin).sum().backward()
    ok = ok and bucket.views_intact() and torch.allclose(lin.weight.grad, torch.full((3, 4), 2.0 * (rank + 1)))
    nfl = bucket.allreduce()
    ok = ok and nfl == 15 and torch.allclose(lin.weight.grad, torch.full((3, 4), 3.0)) and torch.allclose(lin.bias.grad, torch.full((3,), 2.0))
    bucket.zero()
    lin(xin).sum().backward()                      # second step: still accumulating into the same storage
    ok = ok and bucket.views_intact() and torch.allclose(bucket.flat[:12], torch.full((12,), 2.0 * (rank + 1)))
    # sharded k-means++ seeding, unweighted and weighted (host logic of gfs3d.kmeans.KMeans._seed_plusplus; the scoring kernel
    # is replaced by a torch stand-in with the same contract): the picks of the 2-rank run must equal the single-process picks
    from gfs3d import kmeans as km_mod
    from gfs3d.kmeans import KMeans

    def trial_stub(xt, n_, xsq, cand, closest, m_out, pots, weights=None):
        X_ = xt[:, :n_].t().double()
        d = (xsq[:n_][None, :] - 2.0 * (cand.double() @ X_.t()) + (cand.double() ** 2).sum(1)[:, None]).float().clamp_min(0)
        if closest is not None:
            d = torch.minimum(d, closest[:n_][None, :])
        T = cand.shape[0]
        m_out[:T, :n_] = d
        pots[:T] += (d.double() * (1.0 if weights is None else weights[:n_].double())).sum(1)

    real = km_mod.ops.kmeans_pp_trial
    km_mod.ops.kmeans_pp_trial = trial_stub
    try:
        rs2 = np.random.RandomState(3)
        Xs = torch.from_numpy(rs2.randn(403, 6).astype(np.float32))
        lo2, hi2 = shard_range(403, rank, world)

        def seed(Xpart, shard, w=None):
            k = KMeans(n_clusters=9, init="k-means++", shard=shard)
            npad = (Xpart.shape[0] + 3) // 4 * 4
            xt = torch.zeros(6, npad)
            xt[:, :Xpart.shape[0]] = Xpart.t()
            return k._seed_plusplus(Xpart, xt, np.random.RandomState(17), w=w)
        c_sharded = seed(Xs[lo2:hi2].contiguous(), True)
        c_single = seed(Xs, False)
        ok = ok and torch.equal(c_sharded, c_single)
        # weighted: an even split (gloo's all-gather of the weights takes equal sizes only; NCCL takes uneven ones)
        ws = torch.from_numpy(rs2.lognormal(0.0, 0.75, 402).astype(np.float32))
        ws[::7] = 0.0
        lo3, hi3 = shard_range(402, rank, world)
        c_sharded = seed(Xs[lo3:hi3].contiguous(), True, ws[lo3:hi3].contiguous())
        c_single = seed(Xs[:402], False, ws)
        ok = ok and torch.equal(c_sharded, c_single) and not torch.equal(c_single, seed(Xs[:402], False))
    finally:
        km_mod.ops.kmeans_pp_trial = real
    out[rank] = bool(ok)
    dist.destroy_process_group()


def test_sharded_centroid_allreduce_and_seeding_gloo_world2():
    from gfs3d.dist import shard_range
    assert [shard_range(10, r, 4) for r in range(4)] == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert shard_range(3, 3, 4) == (3, 3)
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Manager().dict()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert all(out.get(r) for r in range(world))
