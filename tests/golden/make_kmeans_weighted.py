#!/usr/bin/env python
"""Weighted k-means fixtures (tests/golden/kmeans_weighted_*.npz) from scikit-learn 1.9.0, and the numpy restatement of the
weighted path that pins them.

    python tests/golden/make_kmeans_weighted.py        # writes the fixtures + prints restatement-vs-sklearn deltas

The restatement extends oracle/gfs_oracle.py (pinned E-step, unweighted Lloyd loop and k-means++) with sklearn's
`sample_weight` semantics: _k_means_lloyd.pyx:216-218 (M-step), _k_means_common.pyx:_relocate_empty_clusters_dense,
_inertia_dense, and _kmeans.py:_kmeans_plusplus.  X and the weights are regenerated from seeds by the tests; only the .npz
files travel.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import gfs_oracle as O  # noqa: E402


# ----------------------------------------------------------------------------------------
# restatement of sklearn's weighted k-means
# ----------------------------------------------------------------------------------------
def kmeans_accumulate_weighted_exact(X: np.ndarray, labels: np.ndarray, w: np.ndarray, K: int):
    """weighted M-step (sklearn _k_means_lloyd.pyx:216-218): sums of the fp32 products x * w in fp64, ascending point order;
    weight sums in fp64."""
    X = np.ascontiguousarray(X, dtype=np.float32)
    w = np.asarray(w, dtype=np.float32)
    sums = np.zeros((K, X.shape[1]), dtype=np.float64)
    np.add.at(sums, labels, (X * w[:, None]).astype(np.float64))
    wsums = np.zeros(K, dtype=np.float64)
    np.add.at(wsums, labels, w.astype(np.float64))
    return sums, wsums


def lloyd_reference_weighted(X: np.ndarray, init: np.ndarray, sample_weight, max_iter: int = 300, tol: float = 1e-4):
    """oracle.gfs_oracle.lloyd_reference with sklearn's sample_weight: weights cast to float32, mean-centring and tolerance
    unweighted, M-step sums of the fp32 products x * w, a cluster empty when its weight sum is 0, relocation onto the points
    farthest by unweighted distance, moved with their weight.  Returns (labels int32, centers fp32 (un-centred), n_iter)."""
    w = np.asarray(sample_weight, dtype=np.float32)
    X = np.ascontiguousarray(X, dtype=np.float32)
    mean = X.mean(axis=0)
    Xc = X - mean
    centers = np.ascontiguousarray(init, dtype=np.float32) - mean
    K = centers.shape[0]
    tol_abs = float(np.mean(np.var(Xc, axis=0)) * tol)
    labels_old = np.full(X.shape[0], -1, dtype=np.int32)
    strict = False
    it = 0
    for it in range(1, max_iter + 1):
        labels = O.kmeans_assign_exact(Xc, centers)
        sums, wsums = kmeans_accumulate_weighted_exact(Xc, labels, w, K)
        empty = np.where(wsums == 0)[0]
        if len(empty):
            dist = ((Xc - centers[labels]) ** 2).sum(axis=1)
            if dist.max() > 0:
                far = np.argpartition(dist, -len(empty))[: -len(empty) - 1: -1]
                for e, fi in zip(empty, far):
                    old = labels[fi]
                    wx = (Xc[fi] * w[fi]).astype(np.float64)
                    sums[old] -= wx
                    sums[e] = wx
                    wsums[e] = w[fi]
                    wsums[old] -= w[fi]
        new = np.zeros_like(centers)
        for c in range(K):
            if wsums[c] > 0:
                new[c] = (sums[c] / wsums[c]).astype(np.float32)
        shift = float(((new - centers).astype(np.float64) ** 2).sum())
        centers = new
        if np.array_equal(labels, labels_old):
            strict = True
            break
        if shift <= tol_abs:
            break
        labels_old = labels
    if not strict:
        labels = O.kmeans_assign_exact(Xc, centers)
    return labels, centers + mean, it


def kmeans_plusplus_ref_weighted(X, n_clusters, rng, sample_weight):
    """oracle.gfs_oracle.kmeans_plusplus_ref with sklearn's sample_weight: the first centre is choice(n, p=w/sum(w)), the
    potentials are closest @ w and the candidates come from the cumulative sum of w * closest (fp64 here, as in gfs3d.kmeans;
    sklearn's are float32, which is why the fixture generator asserts identical picks).  -> (centres, indices)"""
    X = np.asarray(X, dtype=np.float32)
    n = X.shape[0]
    trials = 2 + int(np.log(n_clusters))
    X64 = X.astype(np.float64)
    xsq = (X64 * X64).sum(1)
    w = np.asarray(sample_weight, dtype=np.float32)
    w64 = w.astype(np.float64)

    def dist(c):
        return np.maximum((xsq[None, :] - 2.0 * (X64[c] @ X64.T) + xsq[c][:, None]).astype(np.float32), 0)

    idx = np.empty(n_clusters, dtype=np.int64)
    idx[0] = int(rng.choice(n, p=w / w.sum()))
    closest = dist(idx[:1])[0]
    pot = (closest.astype(np.float64) * w64).sum()
    for c in range(1, n_clusters):
        rv = rng.uniform(size=trials) * pot
        cand = np.minimum(np.searchsorted(np.cumsum(closest.astype(np.float64) * w64), rv), n - 1)
        d = np.minimum(dist(cand), closest[None, :])
        pots = (d.astype(np.float64) * w64).sum(1)
        best = int(np.argmin(pots))
        pot, closest, idx[c] = pots[best], d[best], cand[best]
    return X[idx], idx


# ----------------------------------------------------------------------------------------
# fixtures
# ----------------------------------------------------------------------------------------
def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez(path, **arrs)
    print(f"  wrote {name}.npz  {os.path.getsize(path) / 1e6:.2f} MB")


def kmeans_weighted_problem(seed, n, D, K):
    """a seeded mixture and its weights (regenerated by the tests): a lognormal spread, ~5 % exact zeros, ~20 % integers 1-4"""
    rs = np.random.RandomState(seed)
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    w = rs.lognormal(0.0, 0.75, n).astype(np.float32)
    ints = rs.rand(n) < 0.2
    w[ints] = rs.randint(1, 5, int(ints.sum())).astype(np.float32)
    w[rs.rand(n) < 0.05] = 0.0
    return X, w, cent, rs


def make_kmeans_weighted():
    """sklearn 1.9.0 with sample_weight: weighted Lloyd from an array init (+ predict / transform / score on held-out rows),
    weighted k-means++ picks, k-means++ with n_init=3, init='random' with n_init='auto' (10 runs), and a relocation case"""
    import sklearn
    from sklearn.cluster import KMeans, kmeans_plusplus
    print(f"kmeans_weighted: sklearn {sklearn.__version__}")

    def runs(X, w, K, init, n_init, rs_seed):
        """the single runs sklearn's n_init loop makes (one RandomState consumed run after run) and the one it keeps"""
        rs = np.random.RandomState(rs_seed)
        inertias, labels = [], []
        for _ in range(n_init):
            km = KMeans(n_clusters=K, init=init, n_init=1, random_state=rs).fit(X, sample_weight=w)
            inertias.append(km.inertia_)
            labels.append(km.labels_)
        best = 0
        for r in range(1, n_init):
            if inertias[r] < inertias[best] and not (np.unique(np.stack([labels[r], labels[best]]), axis=1).shape[1]
                                                     == np.unique(labels[r]).size):
                best = r
        return np.array(inertias), best

    # 1. weighted Lloyd, array init
    n, D, K, seed = 6000, 192, 150, 41
    X, w, cent, rs = kmeans_weighted_problem(seed, n, D, K)
    init = X[rs.choice(n, K, replace=False)].copy()
    Xh = (cent[rs.randint(0, K, 2000)] + 0.35 * rs.randn(2000, D)).astype(np.float32)
    wh = rs.lognormal(0.0, 0.75, 2000).astype(np.float32)
    km = KMeans(n_clusters=K, init=init, n_init=1).fit(X, sample_weight=w)
    o_labels, o_centers, o_it = lloyd_reference_weighted(X, init, w)
    print(f"  lloyd: n_iter={km.n_iter_} restatement n_iter={o_it} label agreement={(o_labels == km.labels_).mean():.6f} "
          f"centres max|diff|={np.abs(o_centers - km.cluster_centers_).max():.3e}")
    assert (o_labels == km.labels_).mean() >= 0.999 and o_it == km.n_iter_
    save("kmeans_weighted_n6000_k150", seed=np.int32(seed), n=np.int32(n), D=np.int32(D), K=np.int32(K), init=init,
         labels=km.labels_.astype(np.int16), centers=km.cluster_centers_.astype(np.float32), n_iter=np.int32(km.n_iter_),
         inertia=np.float64(km.inertia_), predict=km.predict(Xh).astype(np.int16), transform=km.transform(Xh[:500]).astype(np.float32),
         score=np.float64(km.score(Xh)), score_weighted=np.float64(km.score(Xh, sample_weight=wh)),
         x_checksum=np.float64(X.astype(np.float64).sum()), w_checksum=np.float64(w.astype(np.float64).sum()),
         xh_checksum=np.float64(Xh.astype(np.float64).sum()))

    # 2. weighted k-means++ picks (on the centred data KMeans.fit seeds from), 3. k-means++ with n_init=3, 4. init='random'
    n, D, K, seed, rs_seed = 3000, 192, 50, 43, 143
    X, w, _, _ = kmeans_weighted_problem(seed, n, D, K)
    Xc = X - X.mean(0)
    _, idx = kmeans_plusplus(Xc, K, random_state=np.random.RandomState(rs_seed), sample_weight=w)
    _, o_idx = kmeans_plusplus_ref_weighted(Xc, K, np.random.RandomState(rs_seed), w)
    print(f"  k-means++ picks vs restatement: {int(np.cumprod(idx == o_idx).sum())} of {K} identical")
    assert np.array_equal(idx, o_idx), "choose another seed: this draw lands inside sklearn's float32 cumsum rounding"
    ridx = np.random.RandomState(rs_seed).choice(n, size=K, replace=False, p=w / w.sum())
    pp = KMeans(n_clusters=K, init="k-means++", n_init=3, random_state=rs_seed).fit(X, sample_weight=w)
    pp_inertias, pp_best = runs(X, w, K, "k-means++", 3, rs_seed)
    rnd = KMeans(n_clusters=K, init="random", random_state=rs_seed).fit(X, sample_weight=w)
    rnd_inertias, rnd_best = runs(X, w, K, "random", 10, rs_seed)
    # sklearn's inertia is an fp32 sum under OpenMP: the same run can differ in its last bits from one call to the next
    assert abs(pp.inertia_ / pp_inertias[pp_best] - 1) < 1e-5 and abs(rnd.inertia_ / rnd_inertias[rnd_best] - 1) < 1e-5
    print(f"  n_init=3 k-means++: run {pp_best} kept, inertias {np.round(pp_inertias, 1)}")
    print(f"  init='random' (10 runs): run {rnd_best} kept, inertias {np.round(rnd_inertias, 1)}")
    save("kmeans_weighted_init_n3000_k50", seed=np.int32(seed), rs_seed=np.int32(rs_seed), n=np.int32(n), D=np.int32(D),
         K=np.int32(K), pp_idx=idx.astype(np.int32), random_idx=ridx.astype(np.int32),
         pp_labels=pp.labels_.astype(np.int16), pp_centers=pp.cluster_centers_.astype(np.float32), pp_n_iter=np.int32(pp.n_iter_),
         pp_inertia=np.float64(pp.inertia_), pp_inertias=pp_inertias, pp_best=np.int32(pp_best),
         random_labels=rnd.labels_.astype(np.int16), random_centers=rnd.cluster_centers_.astype(np.float32),
         random_n_iter=np.int32(rnd.n_iter_), random_inertia=np.float64(rnd.inertia_), random_inertias=rnd_inertias,
         random_best=np.int32(rnd_best), x_checksum=np.float64(X.astype(np.float64).sum()), w_checksum=np.float64(w.astype(np.float64).sum()))

    # 5. relocation: one initial centre far from every point, so its cluster is empty in the first iteration
    n, D, K, seed = 2000, 64, 20, 47
    X, w, _, rs = kmeans_weighted_problem(seed, n, D, K)
    init = X[rs.choice(n, K, replace=False)].copy()
    init[7] = 50.0
    km = KMeans(n_clusters=K, init=init, n_init=1).fit(X, sample_weight=w)
    o_labels, o_centers, o_it = lloyd_reference_weighted(X, init, w)
    print(f"  relocation: n_iter={km.n_iter_} restatement n_iter={o_it} label agreement={(o_labels == km.labels_).mean():.6f} "
          f"centres max|diff|={np.abs(o_centers - km.cluster_centers_).max():.3e}")
    assert (o_labels == km.labels_).mean() >= 0.999 and o_it == km.n_iter_ and (km.labels_ == 7).any()
    save("kmeans_weighted_relocate_n2000_k20", seed=np.int32(seed), n=np.int32(n), D=np.int32(D), K=np.int32(K), init=init,
         labels=km.labels_.astype(np.int16), centers=km.cluster_centers_.astype(np.float32), n_iter=np.int32(km.n_iter_),
         inertia=np.float64(km.inertia_), x_checksum=np.float64(X.astype(np.float64).sum()))


if __name__ == "__main__":
    make_kmeans_weighted()
