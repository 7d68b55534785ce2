"""GPU suite: weighted k-means and the rest of sklearn's KMeans interface (sample_weight, inertia_, predict, transform, score,
n_init, init='random') against committed sklearn 1.9.0 runs (tests/golden/make_kmeans_weighted.py), against fp64,
and against exact invariants of the kernels."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import gfs_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24


def _problem(g):
    """kmeans_weighted_problem of make_kmeans_weighted.py, regenerated from the fixture's seed"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    rs = np.random.RandomState(int(g["seed"]))
    n, D, K = int(g["n"]), int(g["D"]), int(g["K"])
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    w = rs.lognormal(0.0, 0.75, n).astype(np.float32)
    ints = rs.rand(n) < 0.2
    w[ints] = rs.randint(1, 5, int(ints.sum())).astype(np.float32)
    w[rs.rand(n) < 0.05] = 0.0
    assert abs(float(X.astype(np.float64).sum()) - float(g["x_checksum"])) < 1e-9
    return X, w, cent, rs


def _mixture(n, D, K, seed):
    rs = np.random.RandomState(seed)
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    return X, rs


def _xt(Xd):
    n, D = Xd.shape
    xt = torch.zeros(D, (n + 3) // 4 * 4, device=Xd.device)
    xt[:, :n] = Xd.t()
    return xt


def _fit_checks(km, X, labels, centers, n_iter, inertia):
    assert km.labels_.shape == (X.shape[0],) and km.labels_.dtype == np.int32
    assert (km.labels_ == labels).mean() >= 0.999
    assert np.abs(km.cluster_centers_ - centers).max() <= 1e-4
    assert km.n_iter_ == int(n_iter)
    assert abs(km.inertia_ / float(inertia) - 1.0) <= 1e-5


def test_weighted_lloyd_predict_transform_score_vs_sklearn_fixture(golden):
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_weighted_n6000_k150")
    X, w, cent, rs = _problem(g)
    K, D = int(g["K"]), int(g["D"])
    rs.choice(X.shape[0], K, replace=False)
    Xh = (cent[rs.randint(0, K, 2000)] + 0.35 * rs.randn(2000, D)).astype(np.float32)
    wh = rs.lognormal(0.0, 0.75, 2000).astype(np.float32)
    assert abs(float(Xh.astype(np.float64).sum()) - float(g["xh_checksum"])) < 1e-9
    km = KMeans(n_clusters=K, init=g["init"], n_init=1).fit(X, sample_weight=w)
    _fit_checks(km, X, g["labels"], g["centers"], g["n_iter"], g["inertia"])
    # predict: sklearn labels uncentred data, so agreement is statistical; every mismatch must be a near-tie in fp64
    p = km.predict(Xh)
    assert isinstance(p, np.ndarray) and p.shape == (2000,)
    miss = np.nonzero(p != g["predict"])[0]
    assert len(miss) <= 0.001 * len(p)
    C64 = km.cluster_centers_.astype(np.float64)
    for i in miss:
        d = ((Xh[i].astype(np.float64) - C64) ** 2).sum(1)
        assert abs(d[p[i]] - d[g["predict"][i]]) <= 1e-5 * d.min()
    t = km.transform(Xh[:500])
    assert t.shape == (500, K) and t.dtype == np.float32
    assert np.all(np.abs(t - g["transform"]) <= 1e-5 * np.abs(g["transform"]) + 1e-6)
    assert abs(km.score(Xh) / float(g["score"]) - 1.0) <= 1e-5
    assert abs(km.score(Xh, sample_weight=wh) / float(g["score_weighted"]) - 1.0) <= 1e-5
    # CUDA tensors in, CUDA tensors out; fit_transform / fit_predict take the weights
    pt = km.predict(torch.from_numpy(Xh).cuda())
    assert pt.is_cuda and np.array_equal(pt.cpu().numpy(), p)
    assert torch.equal(km.transform(torch.from_numpy(Xh[:500]).cuda()).cpu(), torch.from_numpy(t))
    ft = KMeans(n_clusters=K, init=g["init"], n_init=1).fit_transform(X, sample_weight=w)
    assert np.array_equal(ft, km.transform(X))
    assert np.array_equal(KMeans(n_clusters=K, init=g["init"], n_init=1).fit_predict(X, sample_weight=w), km.labels_)


def test_weighted_relocation_vs_sklearn_fixture(golden):
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_weighted_relocate_n2000_k20")
    X, w, _, _ = _problem(g)
    km = KMeans(n_clusters=int(g["K"]), init=g["init"], n_init=1).fit(X, sample_weight=w)
    _fit_checks(km, X, g["labels"], g["centers"], g["n_iter"], g["inertia"])
    assert (km.labels_ == 7).any()


def test_unweighted_relocation_equals_unit_weights_and_restatement(golden):
    """the relocation fixture's problem fitted without weights (centre 7 is empty in the first iteration whatever the weights):
    the same bits as sample_weight = 1, and the numpy restatement's result with unit weights"""
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_weighted_relocate_n2000_k20")
    X, _, _, _ = _problem(g)
    from make_kmeans_weighted import lloyd_reference_weighted
    ones = np.ones(X.shape[0], np.float32)
    km = KMeans(n_clusters=int(g["K"]), init=g["init"], n_init=1).fit(X)
    unit = KMeans(n_clusters=int(g["K"]), init=g["init"], n_init=1).fit(X, sample_weight=ones)
    assert np.array_equal(km.labels_, unit.labels_) and np.array_equal(km.cluster_centers_, unit.cluster_centers_)
    assert km.n_iter_ == unit.n_iter_ and km.inertia_ == unit.inertia_
    labels, centers, n_iter = lloyd_reference_weighted(X, g["init"], ones)
    inertia = ((X.astype(np.float64) - centers.astype(np.float64)[labels]) ** 2).sum()
    _fit_checks(km, X, labels, centers, n_iter, inertia)
    assert (km.labels_ == 7).any()


def _init_problem(golden):
    g = golden("kmeans_weighted_init_n3000_k50")
    X, w, _, _ = _problem(g)
    Xc = X - X.mean(0)
    Xd = torch.from_numpy(Xc).cuda()
    return g, X, w, Xc, Xd


def test_weighted_plusplus_and_random_picks_are_sklearns(golden):
    from gfs3d.kmeans import KMeans
    g, X, w, Xc, Xd = _init_problem(golden)
    K, rs_seed = int(g["K"]), int(g["rs_seed"])
    km = KMeans(n_clusters=K)
    wd = torch.from_numpy(w).cuda()
    got = km._seed_plusplus(Xd, _xt(Xd), np.random.RandomState(rs_seed), w=wd).cpu().numpy()
    same = (got == Xc[g["pp_idx"]]).all(axis=1)
    assert same.all(), f"k-means++ centres differ from sklearn's picks from centre {int(np.argmin(same))} on"
    got = km._seed_random(Xd, np.random.RandomState(rs_seed), X.shape[0], w=wd).cpu().numpy()
    assert np.array_equal(got, Xc[g["random_idx"]])


@pytest.mark.parametrize("init,n_init", [("k-means++", 3), ("random", "auto")])
def test_n_init_keeps_sklearns_run(golden, init, n_init):
    from gfs3d.kmeans import KMeans
    g, X, w, _, _ = _init_problem(golden)
    K, rs_seed = int(g["K"]), int(g["rs_seed"])
    key = "pp" if init == "k-means++" else "random"
    km = KMeans(n_clusters=K, init=init, n_init=n_init, random_state=rs_seed).fit(X, sample_weight=w)
    _fit_checks(km, X, g[key + "_labels"], g[key + "_centers"], g[key + "_n_iter"], g[key + "_inertia"])
    # the single runs, one generator consumed run after run as sklearn's loop does: the same run must win
    rs = np.random.RandomState(rs_seed)
    runs = [KMeans(n_clusters=K, init=init, n_init=1, random_state=rs).fit(X, sample_weight=w) for _ in range(len(g[key + "_inertias"]))]
    inert = np.array([r.inertia_ for r in runs])
    assert np.all(np.abs(inert / g[key + "_inertias"] - 1.0) <= 1e-5)
    best = int(g[key + "_best"])
    assert np.array_equal(runs[best].labels_, km.labels_) and runs[best].inertia_ == km.inertia_


def test_array_init_with_n_init_warns_and_runs_once(golden):
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_weighted_relocate_n2000_k20")
    X, w, _, _ = _problem(g)
    with pytest.warns(RuntimeWarning, match="only one init"):
        km = KMeans(n_clusters=int(g["K"]), init=g["init"], n_init=4).fit(X, sample_weight=w)
    assert np.array_equal(km.labels_, KMeans(n_clusters=int(g["K"]), init=g["init"]).fit(X, sample_weight=w).labels_)


@pytest.mark.parametrize("scale", [1.0, 4.0, 0.125])
def test_unit_and_scaled_weights_are_bit_identical(scale):
    """weights all equal to 1 reproduce the unweighted fit bit for bit; scaling weights by a power of 2 changes nothing"""
    from gfs3d.kmeans import KMeans
    X, rs = _mixture(5000, 192, 60, seed=8)
    w = np.ones(5000, np.float32) if scale == 1.0 else (rs.lognormal(0, 0.75, 5000).astype(np.float32))
    ref = KMeans(n_clusters=60, init="k-means++", random_state=4).fit(X, sample_weight=None if scale == 1.0 else w)
    got = KMeans(n_clusters=60, init="k-means++", random_state=4).fit(X, sample_weight=(w * np.float32(scale)))
    assert np.array_equal(ref.labels_, got.labels_)
    assert np.array_equal(ref.cluster_centers_, got.cluster_centers_)
    assert ref.n_iter_ == got.n_iter_
    assert got.inertia_ == ref.inertia_ * scale
    Xc = torch.from_numpy(X - X.mean(0)).cuda()
    km = KMeans(n_clusters=60)
    wd = torch.from_numpy(w).cuda()
    a = km._seed_plusplus(Xc, _xt(Xc), np.random.RandomState(9), w=None if scale == 1.0 else wd)
    b = km._seed_plusplus(Xc, _xt(Xc), np.random.RandomState(9), w=wd * scale)
    assert torch.equal(a, b)


@pytest.mark.parametrize("n", [253, 5003])
def test_pp_trial_null_weights_equal_unit_weights(n):
    """gfs_kmeans_pp_trial with weights = NULL gives the distances of weights all 1 bit for bit, and their potentials: bit for
    bit within one CTA (256 points); across CTAs the fp64 atomic adds of the CTA sums may land in any order"""
    from gfs3d import ops
    X, rs = _mixture(n, 192, 40, seed=41)
    Xd = torch.from_numpy(X).cuda()
    xt = _xt(Xd)
    xsq = (Xd.double() ** 2).sum(1)
    cand = Xd[torch.from_numpy(rs.choice(n, 8, replace=False)).cuda()].contiguous()
    closest = torch.from_numpy((rs.rand(n) * 400).astype(np.float32)).cuda()
    got = []
    for w in (None, torch.ones(n, device="cuda")):
        m = torch.empty(8, xt.shape[1], device="cuda")
        pots = torch.zeros(8, dtype=torch.float64, device="cuda")
        ops.kmeans_pp_trial(xt, n, xsq, cand, closest, m, pots, weights=w)
        got.append((m[:, :n].clone(), pots))
    assert torch.equal(got[0][0], got[1][0])
    if n <= 256:
        assert torch.equal(got[0][1], got[1][1])
    else:
        assert bool(((got[0][1] - got[1][1]).abs() <= 1e-12 * got[1][1]).all())


def test_weighted_msteps_unit_weights_equal_unweighted_and_repeat():
    from gfs3d import ops
    X, rs = _mixture(20000, 192, 150, seed=21)
    Xd = torch.from_numpy(X).cuda()
    labels = torch.from_numpy(rs.randint(0, 150, 20000).astype(np.int32)).cuda()
    sums, counts = ops.kmeans_accumulate(Xd, labels, 150)
    ws, wsums = ops.kmeans_accumulate_weighted(Xd, labels, torch.ones(20000, device="cuda"), 150)
    assert torch.equal(sums, ws) and torch.equal(wsums, counts.double())
    w = torch.from_numpy(rs.lognormal(0, 1, 20000).astype(np.float32)).cuda()
    a = ops.kmeans_accumulate_weighted(Xd, labels, w, 150)
    b = ops.kmeans_accumulate_weighted(Xd, labels, w, 150)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    C = torch.from_numpy(X[:150].copy()).cuda()
    i1, i2 = ops.kmeans_inertia(Xd, labels, C, w), ops.kmeans_inertia(Xd, labels, C, w)
    assert torch.equal(i1, i2)


def _bounds_check(X, labels, w, K, P):
    """weighted M-step and inertia against fp64, within bounds derived from the kernels' roundings"""
    from gfs3d import ops
    n, D = X.shape
    lab = labels.long()
    sums, wsums = ops.kmeans_accumulate_weighted(X, labels, w, K)
    xw = X.double() * w.double()[:, None]
    ref = torch.zeros(K, D, dtype=torch.float64, device=X.device).index_add_(0, lab, xw)
    absr = torch.zeros(K, D, dtype=torch.float64, device=X.device).index_add_(0, lab, xw.abs())
    wref = torch.zeros(K, dtype=torch.float64, device=X.device).index_add_(0, lab, w.double())
    per = -(-n // P)
    per = -(-per // 32) * 32                          # points one CTA adds in fp32 (one product rounding each)
    bound = (min(per, n) + 2) * U * absr + P * 2.0 ** -52 * absr
    assert bool(((sums - ref).abs() <= bound).all()), float(((sums - ref).abs() / bound.clamp_min(1e-300)).max())
    assert bool(((wsums - wref).abs() <= (n + P) * 2.0 ** -52 * wref).all())
    C = X[torch.randint(0, n, (K,), generator=torch.Generator().manual_seed(n)).to(X.device)].contiguous()
    got = float(ops.kmeans_inertia(X, labels, C, w))
    dref = ((X.double() - C.double()[lab]) ** 2).sum(1)
    iref = float((dref * w.double()).sum())
    ib = ((D // 4 + 6) * U * 1.01 + (n + 1024) * 2.0 ** -52) * iref
    assert abs(got - iref) <= ib, (got, iref, ib)
    got_u = float(ops.kmeans_inertia(X, labels, C))
    assert abs(got_u - float(dref.sum())) <= ((D // 4 + 6) * U * 1.01 + (n + 1024) * 2.0 ** -52) * float(dref.sum())


@pytest.mark.parametrize("n", [1, 31, 6000])
def test_weighted_msteps_and_inertia_within_fp64_bounds(n):
    from gfs3d._lib import lib
    X, rs = _mixture(n, 192, 150, seed=30 + n)
    w = rs.lognormal(0, 0.75, n).astype(np.float32)
    w[rs.rand(n) < 0.1] = 0
    labels = torch.from_numpy(rs.randint(0, 150, n).astype(np.int32)).cuda()
    _bounds_check(torch.from_numpy(X).cuda(), labels, torch.from_numpy(w).cuda(), 150, lib().gfs_kmeans_partials())
    # the numpy restatement that pins the fixtures agrees with fp64 too
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_kmeans_weighted import kmeans_accumulate_weighted_exact
    s, ws = kmeans_accumulate_weighted_exact(X, labels.cpu().numpy(), w, 150)
    assert np.allclose(ws, np.bincount(labels.cpu().numpy(), weights=w.astype(np.float64), minlength=150), rtol=1e-12)


def test_weighted_msteps_and_inertia_within_fp64_bounds_at_4m():
    from gfs3d._lib import lib
    n, D, K = 4 * 1024 * 1024, 192, 150
    g = torch.Generator(device="cuda").manual_seed(5)
    X = torch.randn(n, D, device="cuda", generator=g)
    w = torch.rand(n, device="cuda", generator=g) * 3
    labels = torch.randint(0, K, (n,), device="cuda", generator=g, dtype=torch.int32)
    _bounds_check(X, labels, w, K, lib().gfs_kmeans_partials())


def test_predict_is_the_pinned_e_step_on_both_kernels(golden):
    from gfs3d import ops
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_weighted_n6000_k150")
    X, w, _, _ = _problem(g)
    km = KMeans(n_clusters=int(g["K"]), init=g["init"], n_init=1).fit(X, sample_weight=w)
    Xh, _ = _mixture(3001, 192, 150, seed=77)
    ref = O.kmeans_assign_exact(Xh - km.mean_device_.cpu().numpy(), km.centers_centered_.cpu().numpy())
    saved = ops.ROWSEL_IMPL
    try:
        for impl in ("tc", "fp32"):
            ops.ROWSEL_IMPL = impl
            assert np.array_equal(km.predict(Xh), ref), impl
    finally:
        ops.ROWSEL_IMPL = saved
    assert abs(-km.score(X, sample_weight=w) / km.inertia_ - 1.0) <= 1e-12


def test_integer_weights_match_duplicated_rows_and_zero_weights_match_removed_rows():
    from gfs3d.kmeans import KMeans
    X, rs = _mixture(4000, 192, 40, seed=12)
    init = X[rs.choice(4000, 40, replace=False)].copy()
    c = rs.randint(0, 4, 4000).astype(np.float32)
    c[:40] = np.maximum(c[:40], 1)
    a = KMeans(n_clusters=40, init=init).fit(X, sample_weight=c)
    b = KMeans(n_clusters=40, init=init).fit(np.repeat(X, c.astype(np.int64), axis=0))
    keep = c > 0
    bl = b.labels_[np.cumsum(c.astype(np.int64))[keep] - 1]        # the last copy of each kept row
    assert (a.labels_[keep] == bl).mean() >= 0.999
    assert np.abs(a.cluster_centers_ - b.cluster_centers_).max() <= 1e-4
    z = np.where(keep, 1.0, 0.0).astype(np.float32)
    d = KMeans(n_clusters=40, init=init).fit(X, sample_weight=z)
    e = KMeans(n_clusters=40, init=init).fit(X[keep])
    # the mean-centring stays unweighted (it uses all rows), so agreement is up to rounding, not bits
    assert (d.labels_[keep] == e.labels_).mean() >= 0.999
    assert np.abs(d.cluster_centers_ - e.cluster_centers_).max() <= 1e-4


def test_sharded_fit_on_one_rank_is_bit_identical(golden, tmp_path):
    import torch.distributed as dist
    from gfs3d.kmeans import KMeans
    g, X, w, _, _ = _init_problem(golden)
    K = int(g["K"])
    dist.init_process_group("nccl", init_method=f"file://{tmp_path}/store", rank=0, world_size=1,
                            device_id=torch.device("cuda", torch.cuda.current_device()))
    try:
        for init in ("k-means++", "random"):
            a = KMeans(n_clusters=K, init=init, n_init=2, random_state=3, shard=True).fit(X, sample_weight=w)
            b = KMeans(n_clusters=K, init=init, n_init=2, random_state=3).fit(X, sample_weight=w)
            assert np.array_equal(a.labels_, b.labels_) and np.array_equal(a.cluster_centers_, b.cluster_centers_)
            assert a.n_iter_ == b.n_iter_ and a.inertia_ == b.inertia_
    finally:
        dist.destroy_process_group()


def _worker(rank, world, port, out):
    for p in (ROOT, os.path.join(ROOT, "gfs-3dseg_gws_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from gfs3d.dist import shard_range
    from gfs3d.kmeans import KMeans
    X, rs = _mixture(30000, 192, 100, seed=6)
    w = rs.lognormal(0, 0.75, 30000).astype(np.float32)
    w[rs.rand(30000) < 0.05] = 0
    lo, hi = shard_range(30000, rank, world)
    km = KMeans(n_clusters=100, init="k-means++", random_state=2, shard=True).fit(X[lo:hi], sample_weight=w[lo:hi])
    ref = KMeans(n_clusters=100, init="k-means++", random_state=2).fit(X, sample_weight=w)
    out[rank] = bool(np.array_equal(ref.labels_[lo:hi], km.labels_)
                     and np.abs(ref.cluster_centers_ - km.cluster_centers_).max() <= 1e-6)
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_weighted_fit_on_two_gpus():
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, world, 29900 + os.getpid() % 90, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    assert all(out.get(r) for r in range(world)), dict(out)
