"""Dictionaries of 193..512 entries: the panelled tensor-core E-step / GW projection, the centre-split M-step, and the layers
above them (KMeans, the GW model head, the class codings), against the pinned-order C oracle, fp64 and scikit-learn 1.9.0."""
import ctypes
import os
import random
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import gfs_oracle as O
from parity import rel_err, rel_l2

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_kmeans_wide import wide_X  # noqa: E402

gpu = pytest.mark.gpu
RT_BTILE = 192 * 128     # bytes of one 64-channel, 192-entry dictionary tile (csrc/rowsel_tc.cu)


_GW_LIB = None


def _gw_lib():
    """tests/gw_assign_oracle.c, built with the oracle's gcc flags into a temporary directory (the tree may be read-only)"""
    global _GW_LIB
    if _GW_LIB is None:
        import subprocess
        import tempfile
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gw_assign_oracle.c")
        so = os.path.join(tempfile.mkdtemp(prefix="gfs_gw_oracle_"), "libgw_assign_oracle.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-mfma", "-ffp-contract=off", "-o", so, src, "-lm"])
        _GW_LIB = ctypes.CDLL(so)
        _GW_LIB.gw_assign_exact.restype = ctypes.c_int
    return _GW_LIB


def _gw_assign_exact(ec: np.ndarray, gp_l2: np.ndarray) -> np.ndarray:
    """tests/gw_assign_oracle.c -- ec (B, D, N), gp_l2 (G, D) -> (B, N) int32, the pinned fp32 chain of the GW assignment"""
    ec = np.ascontiguousarray(ec, dtype=np.float32)
    gp_l2 = np.ascontiguousarray(gp_l2, dtype=np.float32)
    B, D, N = ec.shape
    out = np.empty((B, N), dtype=np.int32)
    rc = _gw_lib().gw_assign_exact(ec.ctypes.data_as(ctypes.c_void_p), B, D, N, gp_l2.ctypes.data_as(ctypes.c_void_p),
                                   gp_l2.shape[0], out.ctypes.data_as(ctypes.c_void_p))
    assert rc == 0
    return out


def _args():
    return SimpleNamespace(edgeconv_widths=[[64, 64]] * 3, dgcnn_mlp_widths=[512, 256], pc_in_dim=9, dgcnn_k=20,
                           base_widths=[128, 64], output_dim=64, eval_weight=1.2)


# ============================================================== CPU
def test_gw_oracle_is_the_argmax_on_separated_rows():
    rs = np.random.RandomState(3)
    G, D, B, N = 300, 64, 2, 50
    gp = rs.randn(G, D)
    gp /= np.linalg.norm(gp, axis=1, keepdims=True)
    want = rs.randint(0, G, size=(B, N))
    ec = (3.0 * gp[want] + 0.01 * rs.randn(B, N, D)).transpose(0, 2, 1)     # each row next to its own word
    got = _gw_assign_exact(ec, gp)
    ref = np.argmax(np.einsum("bdn,gd->bgn", ec, gp) / np.linalg.norm(ec, axis=1, keepdims=True), axis=1)
    assert np.array_equal(ref, want) and np.array_equal(got, want)


def test_kmeans_limits_raise_before_the_device():
    from gfs3d.kmeans import KMeans
    with pytest.raises(NotImplementedError, match="512"):
        KMeans(n_clusters=513).fit(np.zeros((600, 64), np.float32))
    with pytest.raises(NotImplementedError, match="192"):
        KMeans(n_clusters=256).fit(np.zeros((600, 200), np.float32))


def test_rowsel_workspace_query_learns_the_dictionary_width():
    from gfs3d._lib import lib
    L = lib()
    for rows, D in [(1000, 64), (65536, 192)]:
        assert L.gfs_rowsel_tc_workspace_bytes_kp(rows, D, 192, 1) == L.gfs_rowsel_tc_workspace_bytes(rows, D)
        assert L.gfs_rowsel_tc_workspace_bytes_kp(rows, D, 152, 0) == L.gfs_rowsel_tc_workspace_bytes(rows, D)
    base = 3 * 3 * 2 * RT_BTILE + 512 + 65536 * 4
    assert L.gfs_rowsel_tc_workspace_bytes_kp(65536, 192, 512, 1) == base + 513 * 65536 * 4     # 134 MB at 32 x 2048 x 512
    assert L.gfs_rowsel_tc_workspace_bytes_kp(65536, 192, 512, 0) == base + 16 * 65536
    assert L.gfs_rowsel_tc_workspace_bytes_kp(100, 64, 576, 0) == 0


# ============================================================== E-step
def _assign_tc(X: np.ndarray, C: np.ndarray):
    """labels of gfs_kmeans_assign_tc over the channel-major copy, and the number of re-checked rows"""
    from gfs3d import ops
    from gfs3d._lib import lib
    n, D = X.shape
    K = C.shape[0]
    Kp = (K + 3) // 4 * 4
    ct = np.zeros((D, Kp), np.float32)
    ct[:, :K] = C.T
    xt = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()
    ctd = torch.from_numpy(ct).cuda()
    nbytes = int(lib().gfs_rowsel_tc_workspace_bytes_kp(n, D, Kp, 0))
    ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    cnorm = torch.empty(Kp, device="cuda")
    labels = torch.empty(n, dtype=torch.int32, device="cuda")
    ops._call("gfs_kmeans_assign_tc", 6, ops._ptr(xt), n, n, 0, D, ops._ptr(ctd), K, Kp, ops._ptr(cnorm), ops._ptr(labels),
              ops._ptr(ws), nbytes, ops._stream())
    panels = (Kp + 191) // 192
    off_cnt = panels * (D // 64) * 2 * RT_BTILE + 256
    nre = int(ws[off_cnt:off_cnt + 4].view(torch.int32).item())
    # the public wrapper takes the same path
    assert torch.equal(ops.kmeans_assign(xt, ctd, K), labels)
    return labels.cpu().numpy(), nre


@gpu
@pytest.mark.parametrize("K", [193, 256, 300, 384, 512])
@pytest.mark.parametrize("D", [64, 128, 192])
def test_estep_wide_bit_exact_mixture(K, D):
    X = wide_X(20000, D, K, seed=K + D)
    C = X[np.random.RandomState(K).choice(len(X), K, replace=False)].copy()
    labels, _ = _assign_tc(X, C)
    assert np.array_equal(labels, O.kmeans_assign_exact(X, C))


@gpu
@pytest.mark.parametrize("kind", ["uniform", "zeros", "offset", "dup_across_panels"])
@pytest.mark.parametrize("K", [256, 512])
def test_estep_wide_bit_exact_hard_data(kind, K):
    rs = np.random.RandomState(7)
    D, n = 128, 12000
    if kind == "uniform":
        X = rs.rand(n, D).astype(np.float32)
        C = rs.rand(K, D).astype(np.float32)
    elif kind == "zeros":
        X = np.zeros((n, D), np.float32)
        C = rs.randn(K, D).astype(np.float32)
        C[K - 5] = 0.0                                  # the only centre at distance 0 lives in the last panel
    elif kind == "offset":
        X = (1000.0 + rs.randn(n, D)).astype(np.float32)
        C = (1000.0 + rs.randn(K, D)).astype(np.float32)
    else:
        C = rs.randn(K, D).astype(np.float32)
        C[K - 1] = C[40]                                 # equal centres in the first and the last panel: 40 must win
        C[200] = C[10]
        X = np.concatenate([np.repeat(C[[40, 10, K - 1, 200]], 500, axis=0),
                            (C[rs.randint(0, K, n - 2000)] + 0.3 * rs.randn(n - 2000, D))]).astype(np.float32)
    labels, nre = _assign_tc(X, C)
    ref = O.kmeans_assign_exact(X, C)
    assert np.array_equal(labels, ref)
    if kind == "dup_across_panels":
        assert nre > 0, "exact ties across panels must go through the re-check"
        assert (labels[:500] == 40).all() and (labels[500:1000] == 10).all()
        assert (labels[1000:1500] == 40).all() and (labels[1500:2000] == 10).all()
    if kind == "zeros":
        assert (labels == K - 5).all()


@gpu
def test_estep_wide_point_major_entry():
    from gfs3d import ops
    K, D = 384, 192
    X = wide_X(9000, D, K, seed=5)
    C = X[:K].copy()
    Kp = (K + 3) // 4 * 4
    ct = torch.zeros(D, Kp, device="cuda")
    ct[:, :K] = torch.from_numpy(C.T.copy()).cuda()
    got = ops.kmeans_assign_rows(torch.from_numpy(X).cuda(), ct, K).cpu().numpy()
    assert np.array_equal(got, O.kmeans_assign_exact(X, C))


@gpu
def test_fp32_impl_refuses_wide_dictionaries():
    from gfs3d import ops
    with pytest.raises(RuntimeError):
        ops.kmeans_assign(torch.zeros(64, 256, device="cuda"), torch.zeros(64, 256, device="cuda"), 256, impl="fp32")


# ============================================================== GW projection
def _gw_case(B, N, G, seed, dup=False):
    g = torch.Generator().manual_seed(seed)
    gp = torch.randn(G, 192, generator=g)
    if dup:
        gp[G - 3] = gp[40]                                # the same word in the first and the last panel
    gp_l2 = F.normalize(gp, dim=1)
    ec = torch.randn(B, 192, N, generator=g)
    if dup:
        ec[0, :, :64] = 2.0 * gp_l2[40].unsqueeze(1)      # rows that sit on the duplicated word
    return gp_l2, ec


@gpu
@pytest.mark.parametrize("B,N", [(32, 2048), (3, 384)])
@pytest.mark.parametrize("G", [193, 256, 384, 512])
def test_gw_projection_wide_vs_pinned_chain_and_fp64(B, N, G):
    from gfs3d import ops
    gp_l2, ec = _gw_case(B, N, G, seed=G + N, dup=True)
    Gp = (G + 63) // 64 * 64
    gp_l2t = torch.zeros(192, Gp)
    gp_l2t[:, :G] = gp_l2.t()
    kb0, kblocks = 3, 3 + Gp // 64
    act = ops.new_act(B * N, kblocks, "cuda")
    act.fill_(1.0)                                        # the padding columns must be written as zeros
    assign, cm = ops.gw_project(ec.cuda(), gp_l2t.cuda(), G, cosine_act=act, kb0=kb0, want_cm=True)
    ref = _gw_assign_exact(ec.numpy(), gp_l2.numpy())
    assert np.array_equal(assign.cpu().numpy(), ref)
    assert (assign[0, :64] == 40).all()
    cos = torch.matmul(gp_l2.double().cuda().unsqueeze(0), F.normalize(ec.double().cuda(), dim=1))
    feat = torch.softmax(10 * cos, dim=1)
    assert rel_err(cm.double(), feat) <= 2e-2
    assert float((cm.double().sum(1) - 1).abs().max()) <= 1e-2
    dense = ops.act_to_dense(act, B * N).float()[:, kb0 * 64:(kb0 + Gp // 64) * 64]
    got = dense[:, :G].reshape(B, N, G).permute(0, 2, 1)
    assert rel_err(got.double(), feat) <= 2e-2
    if Gp > G:
        assert float(dense[:, G:].abs().max()) == 0.0


# ============================================================== M-step
@gpu
@pytest.mark.parametrize("n,D,K", [(60000, 192, 512), (40000, 128, 300)])
def test_mstep_centre_split_vs_oracle(n, D, K):
    from gfs3d import ops
    from gfs3d._lib import lib
    X = wide_X(n, D, K, seed=n + K)
    labels = np.random.RandomState(1).randint(0, K, size=n).astype(np.int32)
    labels[: n // 3] = K - 1                              # a crowded centre in the last slice
    Xd, ld = torch.from_numpy(X).cuda(), torch.from_numpy(labels).cuda()
    if (K, D) == (512, 192):
        assert lib().gfs_kmeans_accumulate_ranges(K, D, 0) == lib().gfs_kmeans_partials() // 3
    ws = ops.kmeans_accumulate_workspace(K, D, "cuda")
    assert ws[0].numel() == lib().gfs_kmeans_accumulate_ranges(K, D, 0) * K * D
    sums, counts = ops.kmeans_accumulate(Xd, ld, K, ws=ws)
    rs_, rc_ = O.kmeans_accumulate_exact(X, labels, K)
    assert np.array_equal(counts.cpu().numpy(), rc_)
    assert np.abs(sums.cpu().numpy() - rs_).max() <= 1e-3 * max(1.0, np.abs(rs_).max())
    sums2, counts2 = ops.kmeans_accumulate(Xd, ld, K)
    assert torch.equal(sums, sums2) and torch.equal(counts, counts2)
    wsums_, wsum = ops.kmeans_accumulate_weighted(Xd, ld, torch.ones(n, device="cuda"), K)
    assert torch.equal(wsums_, sums) and torch.equal(wsum, counts.double())


# ============================================================== KMeans against scikit-learn 1.9.0
@gpu
@pytest.mark.parametrize("K", [256, 512])
def test_kmeans_wide_init_array_vs_sklearn(golden, K):
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_wide")
    n, D, K_, seed = (int(v) for v in g[f"fit_k{K}_meta"])
    X = wide_X(n, D, K_, seed)
    km = KMeans(n_clusters=K, init=X[g[f"fit_k{K}_init_idx"]]).fit(X)
    agree = float((km.labels_ == g[f"fit_k{K}_labels"]).mean())
    print(f"K={K}: label agreement {agree:.5f}, n_iter {km.n_iter_} vs {int(g[f'fit_k{K}_n_iter'])}")
    assert agree >= 0.999
    assert np.abs(km.cluster_centers_ - g[f"fit_k{K}_centers"]).max() <= 1e-4
    assert km.n_iter_ == int(g[f"fit_k{K}_n_iter"])
    # unit sample weights: the same labels and centres
    kw = KMeans(n_clusters=K, init=X[g[f"fit_k{K}_init_idx"]]).fit(X, sample_weight=np.ones(n, np.float32))
    assert np.array_equal(kw.labels_, km.labels_) and np.array_equal(kw.cluster_centers_, km.cluster_centers_)


@gpu
@pytest.mark.parametrize("K", [256, 512])
def test_kmeans_plusplus_wide_picks_sklearns_centres(golden, K):
    from gfs3d.kmeans import KMeans
    g = golden("kmeans_wide")
    n, D, K_, seed, rs_seed = (int(v) for v in g[f"pp_k{K}_meta"])
    X = wide_X(n, D, K_, seed)
    Xd = torch.from_numpy(X).cuda()
    xt = torch.zeros(D, (n + 3) // 4 * 4, device="cuda")
    xt[:, :n] = Xd.t()
    got = KMeans(n_clusters=K)._seed_plusplus(Xd, xt, np.random.RandomState(rs_seed)).cpu().numpy()
    same = (got == X[g[f"pp_k{K}_idx"]]).all(axis=1)
    assert same.all(), f"centres differ from sklearn's picks from centre {int(np.argmin(same))} on"


@gpu
@pytest.mark.parametrize("D", [64, 100])
def test_kmeans_wide_fit_predict_transform_score(D):
    """K = 300, with D = 100 padded to 128 zero channels for the E-step: every query runs through the widened entry points"""
    from gfs3d.kmeans import KMeans
    K = 300
    X = wide_X(12000, D, K, seed=D) + 0.5
    km = KMeans(n_clusters=K, init="random", n_init=2, random_state=0).fit(X)
    assert km.cluster_centers_.shape == (K, D)
    Q = X[::7] + 0.01
    Qc = torch.from_numpy(Q).cuda() - km.mean_device_
    ref = O.kmeans_assign_exact(Qc.cpu().numpy(), km.centers_centered_.cpu().numpy())
    assert np.array_equal(km.predict(Q), ref)
    assert np.array_equal(km.predict(X), km.labels_)
    T = km.transform(Q)
    d64 = np.sqrt(((Q[:, None, :].astype(np.float64) - km.cluster_centers_[None].astype(np.float64)) ** 2).sum(-1))
    assert np.abs(T - d64).max() <= 1e-3 * max(1.0, d64.max())
    assert abs(km.score(X) + km.inertia_) <= 1e-6 * km.inertia_


# ============================================================== model, codings, basis
def _wide_model(G, seed):
    from model.capl import mpti_net_Point_GeoAsWeight_v2
    torch.manual_seed(seed)
    gp = torch.randn(G, 192)
    m = mpti_net_Point_GeoAsWeight_v2(classes=13, criterion=torch.nn.CrossEntropyLoss(ignore_index=255), args=_args(),
                                      base_num=7, gp=gp.cuda(), energy=0.9)
    sd = O.randomize_bn_({k: v.detach().clone().cpu() for k, v in m.state_dict().items()}, seed=seed)
    m.load_state_dict(sd, strict=True)
    return m.cuda(), sd, gp


@gpu
@pytest.mark.parametrize("G", [256, 512])
def test_model_eval_with_a_wide_basis_vs_oracle(G):
    m, sd, gp = _wide_model(G, seed=G)
    m.eval()
    x = O.synthetic_blocks(2, 256, seed=G)
    g = torch.Generator().manual_seed(G)
    gened = F.normalize(torch.randn(13, 128, generator=g), dim=1)
    base, novel = (torch.rand(7, G, generator=g) > 0.8).float(), (torch.rand(6, G, generator=g) > 0.8).float()
    with torch.no_grad():
        _, assignment, _ = m._features(x.cuda())
        logits, _, _ = m(x=x.cuda(), eval_model=True, gened_proto=gened.cuda(), base_class_coding=base.cuda(),
                         novel_class_coding=novel.cuda())
    ref, f = O.forward_eval(sd, gp, x, gened, base, novel, 7, 1.2)
    flip = assignment.cpu().long() != f["assignment"]
    if bool(flip.any()):                              # every GW flip is a near-tie of the oracle's two best words
        top2 = torch.topk(f["cos"].double(), 2, dim=1).values
        gap = (top2[:, 0] - top2[:, 1])[flip]
        assert float(gap.max()) <= 1e-2, float(gap.max())
    # a flipped word can change the point's coding weight (1 or eval_weight): compare the logits of the other points
    keep = ~flip.unsqueeze(1).expand_as(ref)
    agree = float((logits.argmax(1).cpu() == ref.argmax(1)).double().mean())
    err = rel_err(logits.cpu()[keep], ref[keep])
    print(f"G={G}: {int(flip.sum())} GW flips, logits rel err {err:.2e} elsewhere, label agreement {agree:.5f}")
    assert err <= 2e-2
    assert agree >= 0.999


@gpu
def test_model_training_step_with_a_wide_basis_vs_oracle(golden, golden_sd):
    from gfs3d import ops
    g = golden("train_s3dis_b4_n128")
    G = 256
    gp = torch.randn(G, 192, generator=torch.Generator().manual_seed(7))
    sd = golden_sd("gfs_s3dis_weights")
    sd["fusion.0.weight"] = 0.05 * torch.randn(128, 192 + G, 1, generator=torch.Generator().manual_seed(8))
    from model.capl import mpti_net_Point_GeoAsWeight_v2
    m = mpti_net_Point_GeoAsWeight_v2(classes=int(g["classes"]), criterion=torch.nn.CrossEntropyLoss(ignore_index=255), args=_args(),
                                      base_num=int(g["base_num"]), gp=gp.cuda(), energy=0.9)
    m.load_state_dict(sd, strict=True)
    m = m.cuda().train()
    m.att_learner.dropout.p = 0.0
    random.seed(99)
    x, y = torch.from_numpy(g["x"]), torch.from_numpy(g["y"]).long()
    _, loss = m(x=x.cuda(), y=y.cuda())
    loss.backward()
    with torch.no_grad():
        outs, _ = m.encoder.forward_train(x.cuda())
        from gfs3d.train_ops import from_cm
        feats = [x.cuda()] + [from_cm(o, x.shape[0], x.shape[2]) for o in outs[:2]]
        idx_list = [ops.knn(f_.contiguous(), 20).cpu() for f_ in feats]
    osd = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v.clone()) for k, v in sd.items()}
    _, o_loss, _ = O.forward_train(osd, gp, x, y, int(g["base_num"]), g["fake_novel"].tolist(), idx_list=idx_list)
    o_loss.backward()
    assert abs(float(loss) - float(o_loss)) <= 2e-4 * abs(float(o_loss))
    worst = max(rel_l2(p.grad.cpu(), osd[n].grad) for n, p in m.named_parameters() if float(osd[n].grad.norm()) >= 1e-5)
    print(f"G={G}: worst relative L2 gradient error {worst:.3e}")
    assert worst <= 2e-2
    assert m.fusion[0].weight.grad.shape == (128, 192 + G, 1)


@gpu
def test_class_codings_at_512_words_equal_one_block_at_a_time():
    from gfs3d.coding import collect_base_class_gp_coding_sum
    m, _, _ = _wide_model(512, seed=3)
    x = O.synthetic_blocks(32, 256, seed=4)
    y = torch.randint(0, 8, (32, 256), generator=torch.Generator().manual_seed(5))
    y[:, :20] = 0
    batched = [(x, y, None)]
    single = [(x[i:i + 1], y[i:i + 1], None) for i in range(32)]
    train_class = list(range(7))
    random.seed(1)
    b_code, b_bg = collect_base_class_gp_coding_sum(m, batched, train_class, 0.9)
    random.seed(1)
    s_code, s_bg = collect_base_class_gp_coding_sum(m, single, train_class, 0.9)
    assert torch.equal(b_code, s_code)
    assert torch.allclose(b_bg, s_bg, rtol=1e-6, atol=1e-7)


@gpu
def test_basis_end_to_end_with_256_words():
    """get_basis.py's compute at num_cnt = 256: EdgeConv features of a few blocks -> k-means++ -> cluster means -> SVD"""
    from gfs3d import basis
    m, _, _ = _wide_model(150, seed=11)
    m.eval()
    blocks = [(O.synthetic_blocks(4, 512, seed=20 + i), torch.randint(0, 4, (4, 512), generator=torch.Generator().manual_seed(i)))
              for i in range(4)]
    feats = basis.collect_edgeconv_features(m.encoder, blocks, num_classes=4, rng=np.random.RandomState(0))
    gw, km = basis.build_gw_basis(feats, 256, random_state=0)
    assert gw.shape == (256, 192) and np.isfinite(gw).all()
    ref = O.kmeans_assign_exact((feats - km.mean_device_).cpu().numpy(), km.centers_centered_.cpu().numpy())
    assert np.array_equal(km.labels_, ref)
