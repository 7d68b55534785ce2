"""CPU suite: argument checks of the weighted k-means C entries and of KMeans' sample_weight, without a GPU."""
import ctypes

import numpy as np
import pytest


def test_kmeans_entries_with_weights_reject_bad_arguments_without_gpu():
    from gfs3d._lib import lib
    l = lib()
    buf = (ctypes.c_double * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    err = lambda: l.gfs_last_error_string()
    assert l.gfs_kmeans_accumulate_weighted(p, 10, 8, p, None, 3, p, p, p, p, None) == 1 and b"null pointer" in err()
    assert l.gfs_kmeans_accumulate_weighted(p, 10, 6, p, p, 3, p, p, p, p, None) == 2 and b"D=6" in err()
    assert l.gfs_kmeans_accumulate_weighted(p, 10, 260, p, p, 3, p, p, p, p, None) == 2 and b"D=260" in err()
    assert l.gfs_kmeans_accumulate_weighted(p, 10, 256, p, p, 192, p, p, p, p, None) == 2 and b"shared memory" in err()
    assert l.gfs_kmeans_accumulate_weighted(p, 0, 8, p, p, 3, p, p, p, p, None) == 1 and b"non-positive" in err()
    assert l.gfs_kmeans_pack(p, None, 10, None, 3, 8, p, p, None) == 1 and b"null pointer" in err()
    assert l.gfs_kmeans_pack(p, p, 0, None, 3, 8, p, p, None) == 1 and b"non-positive" in err()
    assert l.gfs_kmeans_update(p, p, 3, 8, 4, p, None, p, None) == 1 and b"null pointer" in err()
    assert l.gfs_kmeans_update(p, p, 5, 8, 4, p, p, p, None) == 1 and b"bad size" in err()
    assert l.gfs_kmeans_pp_trial(p, 12, 10, 8, p, p, 2, None, p, None, p, None) == 1 and b"null pointer" in err()
    assert l.gfs_kmeans_pp_trial(p, 12, 10, 8, p, p, 9, None, p, p, p, None) == 2 and b"T=9" in err()
    assert l.gfs_kmeans_pp_trial(p, 12, 10, 520, p, p, 2, None, p, p, p, None) == 2 and b"D=520" in err()
    assert l.gfs_kmeans_pp_trial(p, 8, 10, 8, p, p, 2, None, p, p, p, None) == 1 and b"non-positive" in err()
    assert l.gfs_kmeans_inertia(p, 10, 8, p, None, 3, None, p, p, None) == 1 and b"null pointer" in err()
    assert l.gfs_kmeans_inertia(p, 10, 10, p, p, 3, None, p, p, None) == 2 and b"D=10" in err()
    assert l.gfs_kmeans_inertia(p, 10, 512, p, p, 3, None, p, p, None) == 2 and b"D=512" in err()
    assert l.gfs_kmeans_inertia(ctypes.c_void_p(p.value + 4), 10, 8, p, p, 3, None, p, p, None) == 1 and b"16-byte" in err()
    assert l.gfs_kmeans_inertia(p, 0, 8, p, p, 3, None, p, p, None) == 1 and b"non-positive" in err()
    assert l.gfs_kmeans_inertia_partials() >= 1


@pytest.mark.parametrize("w,match", [(np.ones(9), "shape"), (np.ones((10, 1)), "shape"),
                                     (np.r_[np.ones(9), np.nan], "finite"), (np.r_[np.ones(9), np.inf], "finite"),
                                     (np.r_[np.ones(9), -1.0], "non-negative"), (np.zeros(10), "positive")])
def test_fit_rejects_bad_weights_before_touching_the_device(w, match):
    import torch
    from gfs3d.kmeans import KMeans
    X = np.random.RandomState(0).randn(10, 8).astype(np.float32)
    for sw in (w, torch.from_numpy(np.asarray(w))):
        with pytest.raises(ValueError, match=match):
            KMeans(n_clusters=3, device="cpu").fit(X, sample_weight=sw)


def test_n_init_resolution_follows_sklearn():
    from gfs3d.kmeans import KMeans
    assert KMeans(n_clusters=3)._n_runs() == 1
    assert KMeans(n_clusters=3, init="random")._n_runs() == 10
    assert KMeans(n_clusters=3, init="random", n_init=4)._n_runs() == 4
    assert KMeans(n_clusters=3, init=np.zeros((3, 8), np.float32))._n_runs() == 1
    with pytest.warns(RuntimeWarning, match="only one init"):
        assert KMeans(n_clusters=3, init=np.zeros((3, 8), np.float32), n_init=5)._n_runs() == 1
    with pytest.raises(ValueError):
        KMeans(n_clusters=3, n_init=0)._n_runs()


def test_weighted_restatement_reproduces_the_sklearn_fixtures(golden):
    """the numpy restatement of tests/golden/make_kmeans_weighted.py (pinned E-step, weighted M-step and relocation, weighted
    k-means++) against the committed sklearn 1.9.0 runs, on the CPU"""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_kmeans_weighted as M
    for name in ("kmeans_weighted_n6000_k150", "kmeans_weighted_relocate_n2000_k20"):
        g = golden(name)
        X, w, _, _ = M.kmeans_weighted_problem(int(g["seed"]), int(g["n"]), int(g["D"]), int(g["K"]))
        assert abs(float(X.astype(np.float64).sum()) - float(g["x_checksum"])) < 1e-9
        labels, centers, it = M.lloyd_reference_weighted(X, g["init"], w)
        assert (labels == g["labels"]).mean() >= 0.999 and it == int(g["n_iter"])
        assert np.abs(centers - g["centers"]).max() <= 1e-4
    g = golden("kmeans_weighted_init_n3000_k50")
    X, w, _, _ = M.kmeans_weighted_problem(int(g["seed"]), int(g["n"]), int(g["D"]), int(g["K"]))
    _, idx = M.kmeans_plusplus_ref_weighted(X - X.mean(0), int(g["K"]), np.random.RandomState(int(g["rs_seed"])), w)
    assert np.array_equal(idx, g["pp_idx"])
    rs = np.random.RandomState(int(g["rs_seed"]))
    assert np.array_equal(rs.choice(X.shape[0], size=int(g["K"]), replace=False, p=w / w.sum()), g["random_idx"])
