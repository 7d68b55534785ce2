"""GPU suite: k-means E/M kernels vs the pinned-order C oracle (labels bit-exact given identical centroids)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import gfs_oracle as O

pytestmark = pytest.mark.gpu


def _mixture(n, D, K, seed):
    rs = np.random.RandomState(seed)
    cent = rs.randn(K, D).astype(np.float32)
    lab = rs.randint(0, K, size=n)
    return (cent[lab] + 0.35 * rs.randn(n, D)).astype(np.float32), rs


@pytest.mark.parametrize("n,D,K", [(6000, 192, 150), (20000, 192, 180), (4096, 64, 20), (1000, 192, 150), (64, 192, 7)])
def test_assign_bit_exact_and_sums(n, D, K):
    from gfs3d import ops
    X, rs = _mixture(n, D, K, seed=n + K)
    C = X[rs.choice(n, K, replace=False)].copy()
    ref_labels, ref_score = O.kmeans_assign_exact(X, C, return_score=True)
    Kp = (K + 3) // 4 * 4
    ct = np.zeros((D, Kp), np.float32)
    ct[:, :K] = C.T
    xt = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()
    labels, score = ops.kmeans_assign(xt, torch.from_numpy(ct).cuda(), K, want_score=True)
    assert np.array_equal(labels.cpu().numpy(), ref_labels), "labels must be bit-exact given identical fp32 centroids"
    assert np.array_equal(score.cpu().numpy(), ref_score)
    sums, counts = ops.kmeans_accumulate(torch.from_numpy(X).cuda(), labels, K)
    rs_, rc_ = O.kmeans_accumulate_exact(X, ref_labels, K)
    assert np.array_equal(counts.cpu().numpy(), rc_)
    assert np.abs(sums.cpu().numpy() - rs_).max() <= 1e-3 * max(1.0, np.abs(rs_).max())
    # deterministic: same bits on a second run
    sums2, _ = ops.kmeans_accumulate(torch.from_numpy(X).cuda(), labels, K)
    assert torch.equal(sums, sums2)


def test_assign_ties_lowest_index():
    from gfs3d import ops
    xt = torch.zeros(8, 64, device="cuda")
    ct = torch.zeros(8, 8, device="cuda")
    assert int(ops.kmeans_assign(xt, ct, 5).max()) == 0


def _fixture_X(g):
    rs = np.random.RandomState(int(g["seed"]))
    n, D, K = int(g["n"]), int(g["D"]), int(g["K"])
    cent = rs.randn(K, D).astype(np.float32)
    lab = rs.randint(0, K, size=n)
    return (cent[lab] + 0.35 * rs.randn(n, D)).astype(np.float32)


@pytest.mark.parametrize("name", ["kmeans_n6000_k150", "kmeans_n2000_k20"])
def test_kmeans_dropin_vs_sklearn_fixture(golden, name):
    """KMeans(init=<array>).fit(X).labels_ as get_basis.py:210-212 uses it, vs labels produced by sklearn 1.9.0 itself"""
    from gfs3d.kmeans import KMeans
    g = golden(name)
    X = _fixture_X(g)
    km = KMeans(n_clusters=int(g["K"]), init=g["init"], n_init=1).fit(X)
    assert km.labels_.shape == (X.shape[0],) and km.labels_.dtype == np.int32
    assert (km.labels_ == g["labels"]).mean() >= 0.999
    assert np.abs(km.cluster_centers_ - g["centers"]).max() <= 1e-4
    assert km.n_iter_ == int(g["n_iter"])
    # and bit-exact against the pinned-order oracle's Lloyd loop
    o_labels, o_centers, o_it = O.lloyd_reference(X, g["init"])
    assert np.array_equal(km.labels_, o_labels)
    # downstream of the labels: Kmean2Proto + SVD reconstruction (get_basis.py:27-71) reproduces the reference basis
    basis = O.svd_reconstruct(O.kmean_to_proto(X, km.labels_, int(g["K"])))
    assert np.abs(basis - g["basis"]).max() <= 1e-4


def test_kmeans_plusplus_runs_and_is_a_fixed_point():
    from gfs3d.kmeans import KMeans
    X, _ = _mixture(5000, 192, 150, seed=1)
    km = KMeans(n_clusters=150, init="k-means++", random_state=0).fit(X)
    assert len(np.unique(km.labels_)) == 150
    # idempotence: restarting from the converged centres reproduces the labels in one step
    km2 = KMeans(n_clusters=150, init=km.cluster_centers_).fit(X)
    assert (km2.labels_ == km.labels_).mean() >= 0.999
    # size-independent property: every point is assigned to its nearest centre (checked in fp64)
    d = ((X[:500, None, :].astype(np.float64) - km.cluster_centers_[None].astype(np.float64)) ** 2).sum(-1)
    best = d.min(1)
    chosen = d[np.arange(500), km.labels_[:500]]
    assert (chosen <= best + 1e-4 * np.abs(best)).all()


def test_gw_basis_pipeline_end_to_end(golden_sd):
    """get_basis.py:162-222 on synthetic blocks: EdgeConv123 features -> per-class subsample -> GPU k-means -> Kmean2Proto ->
    SVD reconstruction, then the basis drives the GW projection of the model.  Checked against the oracle's numpy pieces."""
    from gfs3d.basis import build_gw_basis, collect_edgeconv_features, kmean_to_proto, svd_reconstruct
    from gfs3d.synthetic import synthetic_blocks
    from model.dgcnn import DGCNN
    enc = DGCNN([[64, 64]] * 3, [512, 256], 9, k=20, return_edgeconvs=True)
    enc.load_state_dict(golden_sd("dgcnn_weights"))
    enc = enc.cuda().eval()
    g = torch.Generator().manual_seed(0)
    blocks = [(synthetic_blocks(4, 512, seed=10 * i), torch.randint(0, 4, (4, 512), generator=g)) for i in range(3)]
    feat = collect_edgeconv_features(enc, blocks, num_classes=4, max_num=1200, rng=np.random.RandomState(1))
    assert feat.shape[1] == 192 and feat.shape[0] <= 3 * 1200 and feat.is_cuda
    basis, km = build_gw_basis(feat, num_cnt=40, random_state=0)
    assert basis.shape == (40, 192) and basis.dtype == np.float32
    X = feat.cpu().numpy()
    assert np.array_equal(kmean_to_proto(X, km.labels_, 40), O.kmean_to_proto(X, km.labels_, 40))
    assert np.abs(svd_reconstruct(O.kmean_to_proto(X, km.labels_, 40)) - O.svd_reconstruct(O.kmean_to_proto(X, km.labels_, 40))).max() < 1e-5
    assert np.linalg.matrix_rank(basis.astype(np.float64), tol=1e-4) < 40          # rank-truncated at 95 % energy


@pytest.mark.parametrize("name", ["kmeanspp_n3000_k50", "kmeanspp_n6000_k150"])
def test_kmeans_plusplus_picks_sklearns_centres(golden, name):
    """KMeans._seed_plusplus (gfs_kmeans_pp_trial + device cumsum/search, sklearn's random-stream order) against the picks of
    sklearn.cluster.kmeans_plusplus itself for a fixed RandomState (tests/golden/make_golden.py:make_kmeanspp): every centre
    must be the same point"""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from gfs3d.kmeans import KMeans
    g = golden(name)
    n, D, K = int(g["n"]), int(g["D"]), int(g["K"])
    rs = np.random.RandomState(int(g["seed"]))
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    X = X - X.mean(0)
    assert abs(float(X.astype(np.float64).sum()) - float(g["x_checksum"])) < 1e-9
    km = KMeans(n_clusters=K, init="k-means++")
    Xd = torch.from_numpy(X).cuda()
    npad = (n + 3) // 4 * 4
    xt = torch.zeros(D, npad, device="cuda")
    xt[:, :n] = Xd.t()
    got = km._seed_plusplus(Xd, xt, np.random.RandomState(int(g["rs_seed"]))).cpu().numpy()
    same = (got == X[g["idx"]]).all(axis=1)
    assert same.all(), f"centres differ from sklearn's picks from centre {int(np.argmin(same))} on"
    o_c, o_idx = O.kmeans_plusplus_ref(X, K, np.random.RandomState(int(g["rs_seed"])))
    assert np.array_equal(o_idx, g["idx"])


def test_kmeans_fit_with_plusplus_init_matches_sklearn_end_to_end(golden):
    """get_basis.py:210 as written -- KMeans(n_clusters, init='k-means++').fit(X).labels_ -- against the labels sklearn 1.9.0
    gave with the same RandomState (tests/golden/make_golden.py:make_kmeans_fit_pp): same seeding picks (pinned above) + same
    Lloyd trajectory => the same labels"""
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_fit_pp_n3000_k50")
    n, D, K = int(g["n"]), int(g["D"]), int(g["K"])
    rs = np.random.RandomState(int(g["seed"]))
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    assert abs(float(X.astype(np.float64).sum()) - float(g["x_checksum"])) < 1e-9
    got = KMeans(n_clusters=K, init="k-means++", random_state=int(g["rs_seed"])).fit(X)
    agree = float((g["labels"] == got.labels_).mean())
    print(f"k-means++ + Lloyd vs sklearn: label agreement {agree:.5f}, iterations {got.n_iter_} vs {int(g['n_iter'])}")
    assert agree >= 0.999


def test_kmeans_pp_trial_matches_a_float64_evaluation():
    from gfs3d import ops
    g = torch.Generator().manual_seed(2)
    n, D, T = 5003, 192, 7
    X = torch.randn(n, D, generator=g)
    npad = (n + 3) // 4 * 4
    xt = torch.zeros(D, npad)
    xt[:, :n] = X.t()
    cand = X[torch.randint(0, n, (T,), generator=g)].contiguous()
    closest = torch.rand(n, generator=g) * 400
    xsq = (X.double() * X.double()).sum(1)
    m = torch.empty(8, npad, device="cuda")
    pots = torch.zeros(8, dtype=torch.float64, device="cuda")
    ops.kmeans_pp_trial(xt.cuda(), n, xsq.cuda(), cand.cuda(), closest.cuda(), m, pots)
    Xd, Cd = X.double(), cand.double()
    d = ((Xd[None] - Cd[:, None]) ** 2).sum(-1)
    ref = torch.minimum(d, closest.double()[None])
    assert float((m[:T, :n].cpu().double() - ref).abs().max()) <= 4e-5          # fp64 accumulation, ONE rounding to fp32 (d ~ 400)
    assert float(((pots[:T].cpu() - ref.sum(1)).abs() / ref.sum(1)).max()) <= 1e-5
    assert float(pots[T:].abs().sum()) == 0.0


@pytest.mark.parametrize("n,D,K,kind", [(6000, 192, 150, "mixture"), (50000, 192, 150, "mixture"), (4096, 64, 20, "mixture"),
                                        (20000, 128, 180, "uniform"), (3000, 192, 150, "duplicate_centres"),
                                        (2048, 192, 7, "zeros"), (10000, 128, 64, "offset")])
def test_tensor_core_assign_returns_the_pinned_labels(n, D, K, kind):
    """gfs_kmeans_assign_tc (bf16 hi/lo tcgen05 product, pinned fp32 re-check of the rows its error bound cannot decide) must
    return the labels of the all-fp32 kernel and of the oracle, bit for bit -- including exact ties (lowest index wins)"""
    from gfs3d import ops
    X, rs = _mixture(n, D, K, seed=n + K)
    if kind == "uniform":
        X = rs.rand(n, D).astype(np.float32)               # no cluster structure: many near-ties
    if kind == "offset":
        X = (X * 0.05 + 20.0).astype(np.float32)           # far from the origin relative to the spread
    if kind == "zeros":
        X[:] = 0
    C = X[rs.choice(n, K, replace=False)].copy()
    if kind == "duplicate_centres":
        C[K // 2:] = C[:K - K // 2]                        # exact ties between a centre and its copy
    n4 = (n + 3) // 4 * 4
    Kp = (K + 3) // 4 * 4
    ct = np.zeros((D, Kp), np.float32)
    ct[:, :K] = C.T
    xt = torch.zeros(D, n4, device="cuda")
    xt[:, :n] = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()
    ctd = torch.from_numpy(ct).cuda()
    ref = ops.kmeans_assign(xt, ctd, K, impl="fp32")
    got = ops.kmeans_assign(xt, ctd, K, impl="tc")
    torch.cuda.synchronize()
    assert torch.equal(ref, got), f"{int((ref != got).sum())} labels differ between the tensor-core and the fp32 kernel"
    assert np.array_equal(got[:n].cpu().numpy(), O.kmeans_assign_exact(X, C))
    rows = ops.kmeans_assign_rows(torch.from_numpy(X).cuda(), ctd, K)            # the row-major (M-step) layout
    assert torch.equal(rows, ref[:n]), "point-major tensor-core path differs"
