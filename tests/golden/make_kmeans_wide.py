#!/usr/bin/env python
"""k-means fixtures beyond 192 clusters (tests/golden/kmeans_wide.npz) from scikit-learn 1.9.0.

    python tests/golden/make_kmeans_wide.py

X is regenerated from the stored seeds by the tests (tests/test_gpu_wide_dictionary.py:_wide_X); only sklearn's outputs
travel: KMeans(init=<array>) labels / centres / n_iter_ at K = 256 and 512, and the picks of
sklearn.cluster.kmeans_plusplus at K = 256 and 512 (2 + ln K = 8 local trials at 512).
"""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def wide_X(n, D, K, seed):
    """a K-component Gaussian mixture, mean-centred (the data the E-step sees)"""
    rs = np.random.RandomState(seed)
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    return X - X.mean(0)


CASES_FIT = [(6000, 64, 256, 11), (8000, 64, 512, 12)]         # n, D, K, seed
CASES_PP = [(4000, 64, 256, 21, 5), (6000, 64, 512, 22, 7)]     # n, D, K, seed, RandomState seed of the picks


def main():
    import sklearn
    from sklearn.cluster import KMeans, kmeans_plusplus
    assert sklearn.__version__ == "1.9.0", sklearn.__version__
    out = {}
    for n, D, K, seed in CASES_FIT:
        X = wide_X(n, D, K, seed)
        init_idx = np.random.RandomState(seed + 1000).choice(n, K, replace=False)
        km = KMeans(n_clusters=K, init=X[init_idx], n_init=1).fit(X)
        tag = f"fit_k{K}"
        out[tag + "_meta"] = np.array([n, D, K, seed])
        out[tag + "_init_idx"] = init_idx.astype(np.int64)
        out[tag + "_labels"] = km.labels_.astype(np.int32)
        out[tag + "_centers"] = km.cluster_centers_.astype(np.float32)
        out[tag + "_n_iter"] = np.array(km.n_iter_)
        print(tag, "n_iter", km.n_iter_)
    for n, D, K, seed, rs_seed in CASES_PP:
        X = wide_X(n, D, K, seed)
        _, idx = kmeans_plusplus(X, n_clusters=K, random_state=np.random.RandomState(rs_seed))
        tag = f"pp_k{K}"
        out[tag + "_meta"] = np.array([n, D, K, seed, rs_seed])
        out[tag + "_idx"] = idx.astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "kmeans_wide.npz"), **out)


if __name__ == "__main__":
    main()
