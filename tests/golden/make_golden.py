#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (PYTHONPATH=/root/reference)
on CPU in the build container, and check that oracle/gfs_oracle.py reproduces it.

    python tests/golden/make_golden.py            # writes fixtures + prints oracle-vs-reference deltas

/root/reference does not exist on the GPU box; only the committed .npz files travel.
The reference ships no golden vectors of its own (SURVEY.md section 4): these files ARE the pin.
"""
import argparse
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("GFS_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

from model.capl import mpti_net_Point_GeoAsWeight_v2  # noqa: E402  (reference)
from model.dgcnn import DGCNN, knn as ref_knn  # noqa: E402  (reference)
from oracle import gfs_oracle as O  # noqa: E402

torch.set_num_threads(8)


def ref_args(k=20, eval_weight=1.2):
    return SimpleNamespace(edgeconv_widths=[[64, 64]] * 3, dgcnn_mlp_widths=[512, 256], pc_in_dim=9,
                           dgcnn_k=k, base_widths=[128, 64], output_dim=64, eval_weight=eval_weight)


def np_sd(sd):
    return {k: v.detach().cpu().numpy() for k, v in sd.items()}


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez(path, **arrs)
    print(f"  wrote {name}.npz  {os.path.getsize(path) / 1e6:.2f} MB")


def maxdiff(a, b):
    return float((a - b).abs().max())


def make_dgcnn(name, B, N, k, seed, dup=0.0, subsample=1):
    torch.manual_seed(321)
    m = DGCNN([[64, 64]] * 3, [512, 256], 9, k=k, return_edgeconvs=True).eval()
    sd = O.randomize_bn_({k_: v.clone() for k_, v in m.state_dict().items()}, seed=5)
    m.load_state_dict(sd)
    x = O.synthetic_blocks(B, N, seed=seed, dup_frac=dup)
    with torch.no_grad():
        ecs, out = m(x)
        # reference neighbour indices per layer (inputs: x, ecs[0], ecs[1])
        idx = [ref_knn(t, k) for t in (x, ecs[0], ecs[1])]
        o_ecs, o_out, _ = O.dgcnn_forward(sd, x, k, "", knn="formula")
    d = max(maxdiff(torch.cat(ecs, 1), torch.cat(o_ecs, 1)), maxdiff(out, o_out))
    print(f"{name}: oracle(formula) vs reference max|diff| = {d:.3e}")
    assert d == 0.0, "oracle restatement is not bit-identical to the reference on CPU"
    s = slice(None, None, subsample)
    save(name, x=x.numpy(), k=np.int32(k), subsample=np.int32(subsample),
         ec=torch.cat(ecs, 1)[:, :, s].numpy(), out=out[:, :, s].numpy(),
         idx0=idx[0].numpy().astype(np.int16), idx1=idx[1].numpy().astype(np.int16),
         idx2=idx[2].numpy().astype(np.int16))
    return sd


def make_gfs(name, B, N, classes, base_num, G, seed, wname):
    torch.manual_seed(321)
    args = ref_args()
    gp = torch.randn(G, 192, generator=torch.Generator().manual_seed(7))
    m = mpti_net_Point_GeoAsWeight_v2(classes=classes, criterion=torch.nn.CrossEntropyLoss(ignore_index=255),
                                      args=args, base_num=base_num, gp=gp.clone(), energy=0.9).eval()
    sd = O.randomize_bn_({k_: v.clone() for k_, v in m.state_dict().items()}, seed=6)
    m.load_state_dict(sd)
    x = O.synthetic_blocks(B, N, seed=seed)
    g = torch.Generator().manual_seed(11)
    y = torch.randint(0, classes, (B, N), generator=g)
    gened = torch.nn.functional.normalize(torch.randn(classes, 128, generator=g), dim=1)
    coding = (torch.rand(classes, G, generator=g) < 0.3).float()
    base_c, novel_c = coding[:base_num], coding[base_num:]
    with torch.no_grad():
        pf, sem, oh = m.getFeatures(x)
        logits, gp_acc, gp_nacc = m(x=x, y=y, eval_model=True, gened_proto=gened.unsqueeze(0).repeat(8, 1, 1),
                                    base_class_coding=base_c, novel_class_coding=novel_c)
        fg_feat, fg_gp = m.Get_Fg_Feat(x[:1], (y[:1] == 1).long())
        o_logits, f = O.forward_eval(sd, gp, x, gened, base_c, novel_c, base_num, args.eval_weight)
        o_acc, o_nacc = O.gp_accuracies(coding, f["one_hot_feat"], y, base_num)
        idx = [t.numpy().astype(np.int16) for t in f["idx"]]
    d = max(maxdiff(pf, f["point_feat"]), maxdiff(sem, f["semantic_feat"]), maxdiff(oh, f["one_hot_feat"]),
            maxdiff(logits, o_logits), abs(float(gp_acc) - float(o_acc)), abs(float(gp_nacc) - float(o_nacc)))
    print(f"{name}: oracle vs reference max|diff| = {d:.3e}")
    assert d == 0.0
    save(wname, **np_sd(sd))
    save(name, x=x.numpy(), y=y.numpy().astype(np.int16), gp=gp.numpy(), gened_proto=gened.numpy(),
         base_class_coding=base_c.numpy(), novel_class_coding=novel_c.numpy(),
         classes=np.int32(classes), base_num=np.int32(base_num), eval_weight=np.float32(args.eval_weight),
         point_feat=pf.numpy(), semantic_feat=sem.numpy(), assignment=oh.argmax(1).numpy().astype(np.int16),
         logits=logits.numpy(), gp_acc=np.float32(gp_acc), gp_novel_acc=np.float32(gp_nacc),
         fg_feat=fg_feat.numpy(), fg_gp_sum=fg_gp.sum(0).numpy(),
         idx0=idx[0], idx1=idx[1], idx2=idx[2], feat_level2=f["feat_level2"].numpy())


def make_train(name, B, N, seed, classes=13, base_num=7, G=150, wname="gfs_s3dis_weights", compact=False):
    """one training step of the real reference on CPU (model/capl.py:194-242): loss, predictions, gradients, updated BN
    running statistics.  capl.py:406 hard-codes .cuda(); it is neutralised HERE (not in the reference) by making
    Tensor.cuda the identity for the duration of the call.  Attention dropout is set to p = 0 (SURVEY H5).
    compact=True (the full-size BASELINE.json configs[2] step): inputs are regenerated from the seed by the test
    (O.synthetic_blocks / torch.randint are deterministic), only a subsample of the predictions is stored."""
    import random
    torch.manual_seed(321)
    args = ref_args()
    gp = torch.randn(G, 192, generator=torch.Generator().manual_seed(7))
    m = mpti_net_Point_GeoAsWeight_v2(classes=classes, criterion=torch.nn.CrossEntropyLoss(ignore_index=255), args=args,
                                      base_num=base_num, gp=gp.clone(), energy=0.9)
    sd0 = {k_: v.clone() for k_, v in m.state_dict().items()}
    sd0 = O.randomize_bn_(sd0, seed=6)
    m.load_state_dict(sd0)
    m.train()
    m.att_learner.dropout.p = 0.0
    x = O.synthetic_blocks(B, N, seed=seed)
    y = torch.randint(0, base_num + 1, (B, N), generator=torch.Generator().manual_seed(seed))
    orig_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        random.seed(99)
        pred, loss = m(x=x, y=y)
        loss.backward()
    finally:
        torch.Tensor.cuda = orig_cuda
    # which fake-novel classes did random.sample pick?  replay the same draw
    random.seed(99)
    uy = [int(v) for v in y[B // 2:].unique() if int(v) != 0]
    fake_novel = random.sample(uy, len(uy) // 2)
    # oracle replay (fp32 autograd on the restated formulas)
    sdg = {k_: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k_ else v.clone()) for k_, v in sd0.items()}
    o_pred, o_loss, _ = O.forward_train(sdg, gp, x, y, base_num, fake_novel)
    o_loss.backward()
    grads = {k_: p.grad for k_, p in m.named_parameters()}
    dmax = max(float((grads[k_] - sdg[k_].grad).abs().max()) for k_ in grads if sdg[k_].grad is not None)
    print(f"{name}: loss ref {float(loss):.6f} oracle {float(o_loss):.6f}; max |grad diff| {dmax:.3e}; pred agree "
          f"{float((pred == o_pred).float().mean()):.4f}; fake_novel {fake_novel}")
    assert abs(float(loss) - float(o_loss)) < 1e-6 and dmax < 1e-5
    keep = ["main_proto", "bg_proto", "fusion.0.weight", "fusion.0.bias", "fusion.1.weight", "encoder.edge_convs.0.layer.0.weight",
            "encoder.edge_convs.0.layer.1.weight", "encoder.edge_convs.1.layer.3.weight", "encoder.edge_convs.2.layer.4.bias",
            "encoder.conv.layer.0.weight", "encoder.conv.layer.4.weight", "att_learner.q_map.weight", "att_learner.v_map.weight",
            "base_learner.convs.0.0.weight", "base_learner.convs.1.1.bias"]
    after = m.state_dict()
    inputs = dict(seed=np.int32(seed), B=np.int32(B), N=np.int32(N), G=np.int32(G), pred=pred[:, ::16].numpy().astype(np.int16)) if compact else \
        dict(x=x.numpy(), y=y.numpy().astype(np.int16), gp=gp.numpy(), pred=pred.numpy().astype(np.int16))
    save(name, fake_novel=np.array(fake_novel, np.int32), loss=np.float32(float(loss)),
         base_num=np.int32(base_num), classes=np.int32(classes), **inputs,
         **{"grad." + k_: grads[k_].numpy() for k_ in keep},
         **{"gradnorm." + k_: np.float32(g_.norm()) for k_, g_ in grads.items()},
         **{"after." + k_: after[k_].numpy() for k_ in after if "running" in k_ and ("edge_convs.0" in k_ or "fusion" in k_ or "conv.layer.4" in k_)})
    # weights: identical to the eval fixture's (same seeds), not stored twice
    ref_w = np.load(os.path.join(HERE, wname + ".npz"))
    assert all((ref_w[k_] == sd0[k_].numpy()).all() for k_ in ref_w.files)


def make_kmeans(name, n, D, K, seed):
    """sklearn KMeans driven exactly as get_basis.py:210 does, with an injected init (pins the Lloyd part)."""
    import sklearn
    from sklearn.cluster import KMeans
    rs = np.random.RandomState(seed)
    cent = rs.randn(K, D).astype(np.float32)
    lab = rs.randint(0, K, size=n)
    X = (cent[lab] + 0.35 * rs.randn(n, D)).astype(np.float32)
    init = X[rs.choice(n, K, replace=False)].copy()
    km = KMeans(n_clusters=K, init=init, n_init=1).fit(X)
    o_labels, o_centers, o_it = O.lloyd_reference(X, init)
    agree = float((o_labels == km.labels_).mean())
    print(f"{name}: sklearn {sklearn.__version__} n_iter={km.n_iter_} oracle n_iter={o_it} "
          f"label agreement={agree:.6f} centers max|diff|={np.abs(o_centers - km.cluster_centers_).max():.3e}")
    # Kmean2Proto / compute_svd straight from the reference source (exec of get_basis.py:27-71 only: the module
    # itself cannot be imported here, it needs h5py/transforms3d -- SURVEY.md H6)
    src = open(os.path.join(REF, "get_basis.py")).read().split("\n")
    ns = {"np": np}
    exec("\n".join(src[26:71]), ns)
    proto = ns["Kmean2Proto"](X, km.labels_, K)
    basis = ns["compute_svd"](proto)
    o_basis = O.svd_reconstruct(O.kmean_to_proto(X, km.labels_, K))
    print(f"{name}: svd basis oracle vs reference max|diff| = {np.abs(basis - o_basis).max():.3e}")
    assert np.abs(basis - o_basis).max() == 0.0
    save(name, seed=np.int32(seed), n=np.int32(n), D=np.int32(D), K=np.int32(K), init=init,
         labels=km.labels_.astype(np.int16), centers=km.cluster_centers_.astype(np.float32),
         n_iter=np.int32(km.n_iter_), basis=basis.astype(np.float32),
         x_checksum=np.float64(X.astype(np.float64).sum()))


def kmeanspp_problem(seed, n, D, K):
    """the mean-centred float32 matrix KMeans.fit hands to k-means++ (regenerated from the seed by the tests)"""
    rs = np.random.RandomState(seed)
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    return X - X.mean(0)


def make_kmeanspp(name, n, D, K, seed, rs_seed):
    """sklearn's own k-means++ picks (sklearn.cluster.kmeans_plusplus = _kmeans_plusplus behind get_basis.py:210's
    KMeans(init='k-means++')) for a fixed RandomState: the pin of the seeding."""
    import sklearn
    from sklearn.cluster import kmeans_plusplus
    X = kmeanspp_problem(seed, n, D, K)
    _, idx = kmeans_plusplus(X, K, random_state=np.random.RandomState(rs_seed))
    _, o_idx = O.kmeans_plusplus_ref(X, K, np.random.RandomState(rs_seed))
    same = int(np.cumprod(idx == o_idx).sum())
    print(f"{name}: sklearn {sklearn.__version__} picks vs oracle restatement: {same} of {K} centres identical")
    assert same == K, "choose another seed: this draw lands inside sklearn's float32 cumsum rounding (see oracle docstring)"
    save(name, seed=np.int32(seed), rs_seed=np.int32(rs_seed), n=np.int32(n), D=np.int32(D), K=np.int32(K),
         idx=idx.astype(np.int32), x_checksum=np.float64(X.astype(np.float64).sum()))


def make_kmeans_fit_pp(name, n, D, K, seed, rs_seed):
    """sklearn KMeans(init='k-means++', n_init=1).fit(X) end to end, as get_basis.py:210 drives it: seeding and Lloyd
    iterations together (X regenerated from the seed by the test, not mean-centred: fit centres it itself)"""
    import sklearn
    from sklearn.cluster import KMeans
    rs = np.random.RandomState(seed)
    cent = rs.randn(K, D).astype(np.float32)
    X = (cent[rs.randint(0, K, n)] + 0.35 * rs.randn(n, D)).astype(np.float32)
    km = KMeans(n_clusters=K, init="k-means++", n_init=1, random_state=rs_seed).fit(X)
    print(f"{name}: sklearn {sklearn.__version__} n_iter={km.n_iter_}")
    save(name, seed=np.int32(seed), rs_seed=np.int32(rs_seed), n=np.int32(n), D=np.int32(D), K=np.int32(K),
         labels=km.labels_.astype(np.int16), n_iter=np.int32(km.n_iter_), x_checksum=np.float64(X.astype(np.float64).sum()))


def make_metric(name, seed, scannet):
    """runs/eval.py of the reference (pure numpy/Python, importable as is) on random labels"""
    from runs.eval import evaluate_metric_GFS  # noqa: E402  (reference)
    rng = np.random.default_rng(seed)
    ncls = 21 if scannet else 13
    novel = [ncls - 3, ncls - 2, ncls - 1] if not scannet else [4, 9, 12, 16, 19, 20]
    order = list(rng.permutation(ncls))                       # learning order -> class name index
    gt = [rng.integers(0, ncls, size=(3, 96)) for _ in range(4)]
    pred = [np.where(rng.random(g.shape) < 0.6, g, rng.integers(0, ncls, size=g.shape)) for g in gt]
    log = SimpleNamespace(cprint=lambda *_: None)
    mean_iou, base_iou, novel_iou, hm, ious = evaluate_metric_GFS(log, pred, gt, list(range(ncls)), novel, order, scannet=scannet)
    got = O.evaluate_metric(pred, gt, list(range(ncls)), novel, order, scannet=scannet)
    assert got[:4] == (mean_iou, base_iou, novel_iou, hm) and np.array_equal(got[4], ious), "oracle differs from runs/eval.py"
    print(f"{name}: oracle == reference (mean {mean_iou:.6f} base {base_iou:.6f} novel {novel_iou:.6f} hm {hm:.6f})")
    save(name, gt=np.stack(gt).astype(np.int16), pred=np.stack(pred).astype(np.int16), order=np.array(order, dtype=np.int16),
         novel=np.array(novel, dtype=np.int16), scannet=np.int8(scannet), mean_iou=np.float64(mean_iou),
         base_iou=np.float64(base_iou), novel_iou=np.float64(novel_iou), hm=np.float64(hm), ious=np.asarray(ious, dtype=np.float64))


def _reference_train_functions(names):
    """train.py cannot be imported here (h5py / transforms3d are missing): lift the named functions out of its source"""
    import ast
    import random
    import torch.nn.functional as F
    src = open(os.path.join(REF, "train.py")).read()
    tree = ast.parse(src)
    ns = {"torch": torch, "random": random, "F": F, "np": np}
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            exec(compile(ast.Module(body=[node], type_ignores=[]), "train.py", "exec"), ns)
    return ns


def make_coding(name, seed, G=150, num_base=7, blocks=12, n=256, energy=0.9):
    """train.py:136-241: class codings from the one-hot GW features of a stub model (the model itself is pinned elsewhere)"""
    ns = _reference_train_functions(["post_processing_hard_coding", "collect_base_class_gp_coding_sum",
                                     "collect_new_clsss_gp_coding_sum"])
    rng = np.random.default_rng(seed)
    # geometric words correlate with the class, as in real data (a few dominant words per class + noise)
    labels = [rng.integers(0, num_base + 1, size=n) for _ in range(blocks)]
    assign = [np.where(rng.random(n) < 0.7, (t * 17 + rng.integers(0, 6, size=n)) % G, rng.integers(0, G, size=n)) for t in labels]
    state = {"i": 0}

    class Stub:
        def eval(self):
            return self

        def getFeatures(self, inp):
            a = torch.from_numpy(assign[state["i"]])
            state["i"] += 1
            return None, None, torch.nn.functional.one_hot(a, num_classes=G).transpose(1, 0).float().unsqueeze(0)

    loader = [(torch.zeros(1, 9, n), torch.from_numpy(t).unsqueeze(0), None) for t in labels]
    orig_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self            # the reference calls .cuda(): no driver in this container
    try:
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            coding, bg = ns["collect_base_class_gp_coding_sum"](Stub(), loader, list(range(num_base)), energy)
            novel_feats = {7: [torch.nn.functional.one_hot(torch.from_numpy(rng.integers(0, 40, size=64)), G).float()],
                           9: [torch.nn.functional.one_hot(torch.from_numpy(rng.integers(30, 90, size=50)), G).float(),
                               torch.nn.functional.one_hot(torch.from_numpy(rng.integers(30, 60, size=20)), G).float()]}
            novel_in = {k: [t.clone() for t in v] for k, v in novel_feats.items()}
            novel_coding = ns["collect_new_clsss_gp_coding_sum"](novel_feats, energy)
    finally:
        torch.Tensor.cuda = orig_cuda
    oc, ob, freq = O.class_gw_codings(assign, labels, list(range(num_base)), G, energy)
    assert O.codings_equal_modulo_ties(freq, oc, coding.numpy()), "oracle base-class coding differs from train.py"
    print(f"{name}: oracle coding == reference modulo equal-frequency ties ({int((oc != coding.numpy()).sum())} tied words differ); "
          f"bg coding max diff {float(np.abs(ob - bg.numpy()).max()):.2e}; "
          f"words kept per class {coding.sum(1).int().tolist()}")
    assert float(np.abs(ob - bg.numpy()).max()) <= 1e-7
    save(name, assign=np.stack(assign).astype(np.int16), labels=np.stack(labels).astype(np.int16), G=np.int32(G),
         num_base=np.int32(num_base), energy=np.float64(energy), coding=coding.numpy().astype(np.float32), freq=freq,
         bg_coding=bg.numpy().astype(np.float32), novel_coding=novel_coding.numpy().astype(np.float32),
         novel7=novel_in[7][0].argmax(1).numpy().astype(np.int16), novel9a=novel_in[9][0].argmax(1).numpy().astype(np.int16),
         novel9b=novel_in[9][1].argmax(1).numpy().astype(np.int16))



def make_support_proto(name, seed, wname="gfs_s3dis_weights", shots=2, n=128, energy=0.9):
    """train.py:240-305 (get_new_proto_Geo2SemProto) on the real reference model (CPU), S3DIS-shaped: 7 base + 6 novel"""
    ns = _reference_train_functions(["post_processing_hard_coding", "collect_new_clsss_gp_coding_sum", "get_new_proto_Geo2SemProto"])
    classes, base_num, G = 13, 7, 150
    torch.manual_seed(321)
    gp = torch.randn(G, 192, generator=torch.Generator().manual_seed(7))
    m = mpti_net_Point_GeoAsWeight_v2(classes=classes, criterion=torch.nn.CrossEntropyLoss(ignore_index=255), args=ref_args(),
                                      base_num=base_num, gp=gp, energy=energy)
    sd = dict(np.load(os.path.join(HERE, wname + ".npz")))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.eval()
    novel = list(range(base_num, classes))
    rng = np.random.default_rng(seed)
    xs = O.synthetic_blocks(len(novel) * shots, n, seed=seed)
    masks = (torch.from_numpy(rng.random((len(novel) * shots, n))) < 0.4).long()
    cls_ids = [c for c in novel for _ in range(shots)]
    loader = [(xs[i:i + 1], masks[i:i + 1], torch.tensor([cls_ids[i]])) for i in range(len(cls_ids))]
    ns["args"] = SimpleNamespace(total_classes=classes)
    ns["logger"] = SimpleNamespace(cprint=lambda *_: None)
    orig_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            gened, coding = ns["get_new_proto_Geo2SemProto"](loader, m, base_num=base_num, novel_num=len(novel),
                                                             novel_class_list=novel, energy=energy)
    finally:
        torch.Tensor.cuda = orig_cuda
    # frequencies the codings were cut from (for the tie-aware comparison)
    with torch.no_grad():
        freq = []
        for c in novel:
            h = torch.zeros(G)
            for i, ci in enumerate(cls_ids):
                if ci == c:
                    _, gpf = m.Get_Fg_Feat(x=xs[i:i + 1], y=masks[i:i + 1])
                    h += gpf.sum(0)
            freq.append((h / h.sum()).numpy())
    print(f"{name}: gened_proto {tuple(gened.shape)}, novel coding keeps {coding.sum(1).int().tolist()} words")
    save(name, x=xs.numpy(), mask=masks.numpy().astype(np.int8), cls_id=np.array(cls_ids, dtype=np.int16), gened=gened.numpy(),
         coding=coding.numpy().astype(np.float32), freq=np.stack(freq).astype(np.float32), energy=np.float64(energy),
         base_num=np.int32(base_num))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    todo = a.only.split(",") if a.only else ["dgcnn", "gfs", "kmeans", "kmeanspp", "train", "callers"]
    if "callers" in todo:
        make_metric("metric_s3dis", seed=5, scannet=False)
        make_metric("metric_scannet", seed=6, scannet=True)
        make_coding("coding_s3dis", seed=7)
        make_support_proto("support_proto_s3dis", seed=31)
    if "dgcnn" in todo:
        sd = make_dgcnn("dgcnn_b2_n256", 2, 256, 20, seed=1234)
        save("dgcnn_weights", **np_sd(sd))
        make_dgcnn("dgcnn_dup_b1_n256", 1, 256, 20, seed=77, dup=0.25)
        make_dgcnn("dgcnn_b1_n2048", 1, 2048, 20, seed=1234, subsample=8)       # BASELINE.json configs[0]
        make_dgcnn("dgcnn_b1_n320_k40", 1, 320, 40, seed=99)
    if "gfs" in todo:
        make_gfs("gfs_s3dis_b2_n256", 2, 256, 13, 7, 150, seed=4321, wname="gfs_s3dis_weights")
        make_gfs("gfs_scannet_b2_n128", 2, 128, 21, 15, 180, seed=8765, wname="gfs_scannet_weights")
    if "train" in todo:
        make_train("train_s3dis_b4_n128", 4, 128, seed=2468)
        # BASELINE.json configs[2]: ScanNet-shaped (21 classes, 180 GWs, base_num 15) -- a miniature and the full-size step
        make_train("train_scannet_b4_n128", 4, 128, seed=1357, classes=21, base_num=15, G=180, wname="gfs_scannet_weights")
    if "train_full" in todo:
        make_train("train_scannet_b32_n2048", 32, 2048, seed=97531, classes=21, base_num=15, G=180, wname="gfs_scannet_weights",
                   compact=True)
    if "kmeans" in todo:
        make_kmeans("kmeans_n6000_k150", 6000, 192, 150, seed=99)
        make_kmeans("kmeans_n2000_k20", 2000, 192, 20, seed=3)
    if "kmeanspp" in todo:
        make_kmeanspp("kmeanspp_n3000_k50", 3000, 192, 50, seed=2, rs_seed=102)
        make_kmeanspp("kmeanspp_n6000_k150", 6000, 192, 150, seed=5, rs_seed=105)
        make_kmeans_fit_pp("kmeans_fit_pp_n3000_k50", 3000, 192, 50, seed=2, rs_seed=102)
