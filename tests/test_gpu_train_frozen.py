"""GPU suite, frozen BatchNorm and frozen backbone inside a training model.

torch's rule for every nn.BatchNorm the training path reaches: batch statistics iff `bn.training or bn.running_mean is None`;
otherwise the BN is frozen -- it normalises with its running statistics, leaves its buffers unchanged, and back-propagates
dx = gamma * invstd * g (no batch-statistic terms).  Attention dropout follows its own module's mode.  An encoder in eval mode
with no parameter requiring grad (and an input that needs no gradient) runs through the fused inference kernels.

Checked against fp64 autograd (kernel units, EdgeConvTrain) and against the oracle in fp64 on the CPU with the CUDA path's
neighbour sets pinned (whole model), with the tolerances of test_gpu_train.py."""
import random

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import gfs_oracle as O
from parity import rel_err, rel_l2

pytestmark = pytest.mark.gpu
TOLS = {"f32": 1e-3, "tf32x3": 1e-3}


@pytest.fixture(params=["tf32x3", "f32"])
def train_gemm(request):
    """run the test once per implementation of the training GEMM (gfs3d.ops.TRAIN_GEMM)"""
    from gfs3d import ops
    old, ops.TRAIN_GEMM = ops.TRAIN_GEMM, request.param
    yield request.param
    ops.TRAIN_GEMM = old


@pytest.fixture
def deterministic():
    was_on, was_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    yield
    torch.use_deterministic_algorithms(was_on, warn_only=was_warn)


def _running(C, g):
    return 0.3 * torch.randn(C, generator=g), 0.5 + torch.rand(C, generator=g)


def _clear_of_kink(pre, rm, rv, ga, be, delta=1e-4):
    """move each channel's running mean (in steps of 3 delta) until no pre-BN value `pre` (C, ...) of that channel lies within
    delta of the LeakyReLU kink, x = rm - beta*sigma/gamma: fp32 and fp64 then take the same branch everywhere"""
    rm = rm.clone()
    sig = torch.sqrt(rv.double() + 1e-5)
    for c in range(rm.numel()):
        while bool(((pre[c] - (rm[c].double() - be[c].double() * sig[c] / ga[c].double())).abs() < delta).any()):
            rm[c] += 3 * delta
    return rm


def _quiet_kinks(dy, u):
    """zero dy where u = gamma*xhat + beta is so close to 0 that fp32 and fp64 may take different sides of the activation's kink"""
    return torch.where(u.abs() < 1e-3, torch.zeros_like(dy), dy)


# ------------------------------------------------------------------------------------------------------------------ kernel units
@pytest.mark.parametrize("M,strided", [(3000, False), (3000, True), (70000, False), (70000, True)])
def test_bn_act_bwd_frozen_vs_autograd(M, strided, train_gemm):
    """one-pass frozen backward == fp64 autograd of act(F.batch_norm(training=False)); M >= 65536 takes the split reduction"""
    from gfs3d import ops
    g = torch.Generator().manual_seed(M + strided)
    C, pad = 96, (37 if strided else 0)
    rm, rv = _running(C, g)
    ga, be = 1 + 0.3 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)
    x = torch.randn(C, M, generator=g) * 1.3 + 0.2
    u = ga.double()[:, None] * (x.double() - rm.double()[:, None]) / torch.sqrt(rv.double()[:, None] + 1e-5) + be.double()[:, None]
    dy = _quiet_kinks(torch.randn(C, M, generator=g), u)
    for slope in (0.2, 0.0, 1.0):
        xs, gs, bs = (t.clone().double().requires_grad_(True) for t in (x, ga, be))
        zn = F.batch_norm(xs.t(), rm.double(), rv.double(), gs, bs, False, 0.1, 1e-5).t()
        torch.where(zn > 0, zn, slope * zn).backward(dy.double())
        # rows inside wider buffers: the kernel must honour ldx / lddy
        xb = torch.zeros(C, M + pad, device="cuda")
        db = torch.zeros(C, M + pad, device="cuda")
        xb[:, :M], db[:, :M] = x.cuda(), dy.cuda()
        xc, dc = xb[:, :M], db[:, :M]
        mean, invstd = rm.cuda(), torch.rsqrt(rv.cuda() + 1e-5)
        dx, sg, sgx = ops.bn_act_bwd_frozen(dc, xc, mean, invstd, ga.cuda(), be.cuda(), slope)
        errs = {"dx": rel_err(dx, xs.grad), "sum_g=dbeta": rel_err(sg, bs.grad), "sum_gx=dgamma": rel_err(sgx, gs.grad)}
        print(f"bn_act_bwd_frozen M={M} strided={strided} slope {slope}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
        assert max(errs.values()) <= 1e-5, errs
        again = ops.bn_act_bwd_frozen(dc, xc, mean, invstd, ga.cuda(), be.cuda(), slope)
        assert all(torch.equal(a, b) for a, b in zip((dx, sg, sgx), again))          # fixed-order sums, no atomics


@pytest.mark.parametrize("Mp,k", [(1000, 20), (70000, 20), (64, 40), (3000, 40), (333, 19), (5000, 19)])
def test_bn_act_bwd_argmax_frozen_vs_autograd(Mp, k, train_gemm):
    """frozen BN -> LeakyReLU -> max over k in fp64 autograd; the kernel reads (dy, arg) per point and writes the (64, Mp*k)
    gradient, zero off the arg-max edge.  k = 19 runs the VEC = 1 path, k = 20 / 40 the float4 one"""
    from gfs3d import ops
    g = torch.Generator().manual_seed(Mp * k)
    C = 64
    rm, rv = _running(C, g)
    ga, be = 1 + 0.3 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)
    ga[::7] *= -1                                                  # negative scales: the max is taken after the activation
    Z = torch.randn(C, Mp * k, generator=g)
    dy = torch.randn(C, Mp, generator=g)
    zs, gs, bs = (t.clone().double().requires_grad_(True) for t in (Z, ga, be))
    zn = F.batch_norm(zs.t(), rm.double(), rv.double(), gs, bs, False, 0.1, 1e-5).t()
    a = F.leaky_relu(zn, 0.2).view(C, Mp, k)
    val, arg = a.max(dim=2)
    u = zn.detach().view(C, Mp, k).gather(2, arg[..., None])[..., 0]
    dy = _quiet_kinks(dy, u)
    val.backward(dy.double())
    mean, invstd = rm.cuda(), torch.rsqrt(rv.cuda() + 1e-5)
    argc = arg.to(torch.uint8).cuda()
    dx, sg, sgx = ops.bn_act_bwd_argmax_frozen(dy.cuda(), argc, k, Z.cuda(), mean, invstd, ga.cuda(), be.cuda(), 0.2)
    errs = {"dx": rel_err(dx, zs.grad), "sum_g=dbeta": rel_err(sg, bs.grad), "sum_gx=dgamma": rel_err(sgx, gs.grad)}
    print(f"bn_act_bwd_argmax_frozen Mp={Mp} k={k}: " + " ".join(f"{n} {v:.2e}" for n, v in errs.items()))
    assert max(errs.values()) <= 1e-5, errs
    off = torch.ones(C, Mp, k, dtype=torch.bool)
    off.scatter_(2, arg[..., None], False)
    assert bool((dx.cpu().view(C, Mp, k)[off] == 0).all())
    again = ops.bn_act_bwd_argmax_frozen(dy.cuda(), argc, k, Z.cuda(), mean, invstd, ga.cuda(), be.cuda(), 0.2)
    assert all(torch.equal(p, q) for p, q in zip((dx, sg, sgx), again))


# ------------------------------------------------------------------------------------------------------------------ EdgeConvTrain
@pytest.mark.parametrize("modes", [(False, False), (False, True), (True, False)], ids=["frozen-frozen", "frozen-train", "train-frozen"])
@pytest.mark.parametrize("B,C,N,k", [(2, 9, 128, 20), (1, 64, 256, 20), (3, 64, 100, 7)])
def test_edgeconv_train_with_frozen_bn_vs_autograd(B, C, N, k, modes, train_gemm):
    """test_edgeconv_train_function_vs_autograd with BN1 / BN2 each in its own mode"""
    TOL = TOLS[train_gemm]
    from gfs3d.train_ops import EdgeConvTrain, from_cm, to_cm
    t1, t2 = modes
    g = torch.Generator().manual_seed(B + N)
    x = torch.randn(B, C, N, generator=g) * 0.5
    idx = torch.stack([torch.stack([torch.randperm(N, generator=g)[:k] for _ in range(N)]) for _ in range(B)])
    W1 = torch.randn(64, 2 * C, 1, 1, generator=g) / (2 * C) ** 0.5
    W2 = torch.randn(64, 64, 1, 1, generator=g) / 8
    g1, b1 = 1 + 0.3 * torch.randn(64, generator=g), 0.2 * torch.randn(64, generator=g)
    g2, b2 = 1 + 0.3 * torch.randn(64, generator=g), 0.2 * torch.randn(64, generator=g)
    rm1, rv1 = _running(64, g)
    rm2, rv2 = _running(64, g)
    dy = torch.randn(B, 64, N, generator=g)
    ps = [t.clone().double().requires_grad_(True) for t in (x, W1, g1, b1, W2, g2, b2)]
    e = O.edge_feature(ps[0], idx)
    # a frozen BN's kink position is set by its running statistics: keep every pre-activation at least 1e-4 away from it, so
    # the comparison is not decided by a branch fp32 and fp64 take differently (the batch-statistic BNs are as in test_gpu_train)
    z1 = F.conv2d(e, ps[1])
    if not t1:
        rm1 = _clear_of_kink(z1.detach().transpose(0, 1), rm1, rv1, g1, b1)
    h = F.leaky_relu(F.batch_norm(z1, rm1.double().clone(), rv1.double().clone(), ps[2], ps[3], t1, 0.1, 1e-5), 0.2)
    z2 = F.conv2d(h, ps[4])
    if not t2:
        rm2 = _clear_of_kink(z2.detach().transpose(0, 1), rm2, rv2, g2, b2)
    u2 = F.batch_norm(z2, rm2.double().clone(), rv2.double().clone(), ps[5], ps[6], t2, 0.1, 1e-5)
    a = F.leaky_relu(u2, 0.2)
    top = a.detach().topk(2, dim=-1)
    u_at = u2.detach().gather(-1, top.indices[..., :1])[..., 0]
    # outputs whose max over k is a near-tie, or whose winning edge sits at the kink, get no gradient
    dy = torch.where(top.values[..., 0] - top.values[..., 1] < 1e-4, torch.zeros_like(dy), _quiet_kinks(dy, u_at))
    ref = a.max(dim=-1).values
    ref.backward(dy.double())
    pc = [t.clone().cuda().requires_grad_(True) for t in (x, W1, g1, b1, W2, g2, b2)]
    bufs = [t.cuda() for t in (rm1, rv1, rm2, rv2)]
    saved = [t.clone() for t in bufs]
    y, m1, v1, m2, v2 = EdgeConvTrain.apply(to_cm(pc[0]), idx.int().cuda(), pc[1], pc[2], pc[3], pc[4], pc[5], pc[6], B, N, k,
                                            t1, bufs[0], bufs[1], t2, bufs[2], bufs[3])
    from_cm(y, B, N).backward(dy.cuda())
    assert all(torch.equal(a_, b_) for a_, b_ in zip(bufs, saved))
    if not t1:
        assert torch.equal(m1, bufs[0]) and torch.equal(v1, bufs[1]) and m1.data_ptr() != bufs[0].data_ptr()
    if not t2:
        assert torch.equal(m2, bufs[2]) and torch.equal(v2, bufs[3])
    ey = rel_err(from_cm(y, B, N).detach().cpu(), ref.detach())
    names = ("dx", "dW1", "dg1", "db1", "dW2", "dg2", "db2")
    l2 = {n: rel_l2(got.grad.cpu(), want.grad) for got, want, n in zip(pc, ps, names)}
    mx = {n: rel_err(got.grad.cpu(), want.grad) for got, want, n in zip(pc, ps, names)}
    print(f"EdgeConvTrain[{train_gemm}] BN1 {'train' if t1 else 'frozen'} BN2 {'train' if t2 else 'frozen'}: y {ey:.2e}; rel-L2 "
          + " ".join(f"{n} {v:.2e}" for n, v in l2.items()) + f"; worst max-norm {max(mx.values()):.2e}")
    assert ey <= TOL
    assert max(l2.values()) <= TOL, l2
    assert max(mx.values()) <= 2e-2, mx


# ------------------------------------------------------------------------------------------------------------------ whole model
def _bns(m):
    return {n: mod for n, mod in m.named_modules() if isinstance(mod, nn.modules.batchnorm._BatchNorm)}


def _buffers(m):
    return {n: b.detach().clone() for n, b in m.named_buffers()}


def _step(m, x, y, seed=99):
    random.seed(seed)                                   # generate_fake_proto's random.sample
    pred, loss = m(x=x, y=y)
    loss.backward()
    torch.cuda.synchronize()
    return pred, loss


def _pinned_idx(golden, golden_sd, frozen, x):
    """neighbour sets of the three EdgeConv layers as a fresh model with the same BN modes computes them in training mode"""
    from gfs3d import ops
    from gfs3d.train_ops import from_cm
    from test_gpu_train import _train_model
    m2, _ = _train_model(golden, golden_sd)
    for n, bn in _bns(m2).items():
        bn.train(n not in frozen)
    with torch.no_grad():
        outs, _ = m2.encoder.forward_train(x.cuda())
        feats = [x.cuda()] + [from_cm(o, x.shape[0], x.shape[2]) for o in outs[:2]]
        return [ops.knn(f.contiguous(), 20).cpu() for f in feats]


def _oracle_step(monkeypatch, golden_sd, g, x, y, frozen, idx_list=None, features=None):
    """O.forward_train in fp64 with the BatchNorms named in `frozen` in eval mode (O._bn patched per prefix; a training-mode BN
    updates its own fp64 copy of the running buffers, as nn.BatchNorm does).  features = (ecs, lvl2): the encoder's outputs
    are taken as given.  -> (pred, loss, sd with .grad, updated running buffers)"""
    sd = {k: (v.clone().double().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else
              v.clone().double() if v.dtype.is_floating_point else v.clone()) for k, v in golden_sd("gfs_s3dis_weights").items()}
    run = {}

    def bn(sd_, prefix, x_, training=False):
        if training and prefix not in frozen:
            rm = run.setdefault(prefix + ".running_mean", sd_[prefix + ".running_mean"].clone())
            rv = run.setdefault(prefix + ".running_var", sd_[prefix + ".running_var"].clone())
            return F.batch_norm(x_, rm, rv, sd_[prefix + ".weight"], sd_[prefix + ".bias"], True, 0.1, 1e-5)
        return F.batch_norm(x_, sd_[prefix + ".running_mean"].clone(), sd_[prefix + ".running_var"].clone(), sd_[prefix + ".weight"],
                            sd_[prefix + ".bias"], False, 0.1, 1e-5)

    monkeypatch.setattr(O, "_bn", bn)
    if features is not None:
        ecs, lvl2 = features
        monkeypatch.setattr(O, "dgcnn_forward", lambda *a, **kw: ([e.detach().double().cpu() for e in ecs], lvl2.detach().double().cpu(), []))
    o_pred, o_loss, _ = O.forward_train(sd, torch.from_numpy(g["gp"]).double(), x.double(), y, int(g["base_num"]), g["fake_novel"].tolist(),
                                        idx_list=idx_list)
    o_loss.backward()
    monkeypatch.undo()
    return o_pred, o_loss, sd, run


def _check_against_oracle(m, pred, loss, o_pred, o_loss, sd, names=None):
    """loss and predictions as test_training_step_vs_oracle_with_pinned_graph; every gradient within 2e-2 relative L2 (the
    reference-fixture gate of test_gpu_train.py: one max-over-k near-tie or LeakyReLU-kink decision that fp32 and fp64 take
    differently moves a small tensor such as one BN's gamma gradient by about 1 %), all of them together within 1e-2"""
    names = [n for n, _ in m.named_parameters()] if names is None else names
    params = dict(m.named_parameters())
    worst, checked, got, want = 0.0, 0, [], []
    for n in names:
        if float(sd[n].grad.norm()) < 1e-5:
            continue
        e = rel_l2(params[n].grad.cpu(), sd[n].grad)
        worst, checked = max(worst, e), checked + 1
        got.append(params[n].grad.detach().double().cpu().reshape(-1))
        want.append(sd[n].grad.reshape(-1))
        assert e <= 2e-2, (n, e)
    total = rel_l2(torch.cat(got), torch.cat(want))
    agree = float((pred.cpu() == o_pred).float().mean())
    print(f"loss {float(loss):.6f} vs fp64 oracle {float(o_loss):.6f}; prediction agreement {agree:.4f}; "
          f"worst relative L2 gradient error over {checked} tensors: {worst:.3e}, all together {total:.3e}")
    assert total <= 1e-2
    assert abs(float(loss) - float(o_loss)) <= 2e-4 * abs(float(o_loss))
    assert agree >= 0.99


def _frozen_run(monkeypatch, golden, golden_sd, frozen):
    """one step with the BNs named in `frozen` in eval mode and attention dropout 0.1 in eval mode, checked against the oracle;
    frozen buffers must be bit-identical afterwards, training-mode ones must follow nn.BatchNorm's update"""
    from test_gpu_train import _train_model
    m, g = _train_model(golden, golden_sd)
    m.att_learner.dropout.p = 0.1
    m.att_learner.dropout.eval()
    bns = _bns(m)
    for n, bn in bns.items():
        bn.train(n not in frozen)
    before = _buffers(m)
    x, y = torch.from_numpy(g["x"]), torch.from_numpy(g["y"]).long()
    pred, loss = _step(m, x.cuda(), y.cuda())
    after = _buffers(m)
    idx_list = _pinned_idx(golden, golden_sd, frozen, x)
    o_pred, o_loss, sd, run = _oracle_step(monkeypatch, golden_sd, g, x, y, frozen, idx_list=idx_list)
    _check_against_oracle(m, pred, loss, o_pred, o_loss, sd)
    worst_bn = 0.0
    for n in bns:
        keys = [n + ".running_mean", n + ".running_var", n + ".num_batches_tracked"]
        if n in frozen:
            assert all(torch.equal(before[k], after[k]) for k in keys), n
        else:
            assert int(after[keys[2]]) == int(before[keys[2]]) + 1, n
            worst_bn = max(worst_bn, *(rel_err(after[k].float().cpu(), run[k]) for k in keys[:2]))
    print(f"{len(frozen)} of {len(bns)} BatchNorms frozen; worst running-statistic error of the others: {worst_bn:.3e}")
    assert worst_bn <= 1e-3
    assert all(torch.equal(before[k], after[k]) for k in before if not any(k.startswith(n + ".") for n in bns))


def test_step_with_every_bn_frozen_vs_oracle(monkeypatch, golden, golden_sd, train_gemm):
    from test_gpu_train import _train_model
    m, _ = _train_model(golden, golden_sd)
    _frozen_run(monkeypatch, golden, golden_sd, set(_bns(m)))


@pytest.mark.parametrize("seed", [3, 17])
def test_step_with_a_random_subset_of_bns_frozen_vs_oracle(monkeypatch, golden, golden_sd, train_gemm, seed):
    from test_gpu_train import _train_model
    m, _ = _train_model(golden, golden_sd)
    names = sorted(_bns(m))
    frozen = set(random.Random(seed).sample(names, len(names) // 2))
    print("frozen:", sorted(frozen))
    _frozen_run(monkeypatch, golden, golden_sd, frozen)


def _full_record(m, pred, loss):
    rec = {"loss": loss.detach().clone(), "pred": pred.clone()}
    rec.update({"grad." + n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None})
    rec.update({"buf." + n: b.detach().clone() for n, b in m.named_buffers()})
    return rec


def _assert_same(a, b):
    assert a.keys() == b.keys(), sorted(set(a) ^ set(b))
    bad = [n for n in a if not torch.equal(a[n], b[n])]
    assert not bad, bad


def test_dropout_in_eval_mode_is_no_dropout(golden, golden_sd, train_gemm, deterministic):
    from test_gpu_train import _train_model
    recs = []
    for p, mode in ((0.1, "eval"), (0.0, "train")):
        torch.manual_seed(5)
        m, g = _train_model(golden, golden_sd)
        m.att_learner.dropout.p = p
        m.att_learner.dropout.train(mode == "train")
        pred, loss = _step(m, torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["y"]).long().cuda())
        recs.append(_full_record(m, pred, loss))
    _assert_same(*recs)


def test_frozen_encoder_runs_the_inference_encoder(monkeypatch, golden, golden_sd, train_gemm):
    from test_gpu_train import _train_model
    m, g = _train_model(golden, golden_sd)
    x, y = torch.from_numpy(g["x"]), torch.from_numpy(g["y"]).long()
    xc, yc = x.cuda(), y.cuda()
    # the full step's peak memory, for comparison
    full, _ = _train_model(golden, golden_sd)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    _step(full, xc, yc)
    peak_full = torch.cuda.max_memory_allocated() - base
    del full

    m.encoder.eval()
    m.encoder.requires_grad_(False)
    before = {n: b.clone() for n, b in m.encoder.named_buffers()}
    seen, fused, calls = [], m.encoder.forward_fused, []
    m.encoder.forward_fused = lambda *a, **kw: seen.append(fused(*a, **kw)) or seen[-1]
    m.encoder.forward_train = lambda *a, **kw: calls.append(1)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    pred, loss = _step(m, xc, yc)
    peak_frozen = torch.cuda.max_memory_allocated() - base
    del m.encoder.forward_fused, m.encoder.forward_train
    assert len(seen) == 1 and not calls
    out = seen[0]
    with torch.no_grad():
        ref_ecs, ref_lvl2 = m.encoder(xc)
    assert all(torch.equal(out.ec[:, 64 * i:64 * (i + 1)], r) for i, r in enumerate(ref_ecs))
    assert torch.equal(out.lvl2_cm, ref_lvl2)
    assert all(p.grad is None for p in m.encoder.parameters())
    assert all(torch.equal(before[n], b) for n, b in m.encoder.named_buffers())
    ecs = [out.ec[:, 64 * i:64 * (i + 1)] for i in range(3)]
    o_pred, o_loss, sd, _ = _oracle_step(monkeypatch, golden_sd, g, x, y, set(), features=(ecs, out.lvl2_cm))
    head = [n for n, _ in m.named_parameters() if not n.startswith("encoder.")]
    _check_against_oracle(m, pred, loss, o_pred, o_loss, sd, names=head)
    print(f"peak memory above the inputs: full step {peak_full / 2**20:.1f} MiB, frozen-encoder step {peak_frozen / 2**20:.1f} MiB")
    assert peak_frozen < peak_full


def test_reference_freeze_keeps_the_head_gradients(golden, golden_sd, train_gemm, deterministic):
    """the reference's way (model/capl.py:40-41): encoder in train mode with requires_grad_(False) -- its running statistics
    still update, it gets no .grad, and the head's gradients are those of the full step, bit for bit"""
    from test_gpu_train import _train_model
    recs = []
    for freeze in (False, True):
        m, g = _train_model(golden, golden_sd)
        if freeze:
            m.encoder.requires_grad_(False)
        before = {n: b.clone() for n, b in m.encoder.named_buffers()}
        pred, loss = _step(m, torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["y"]).long().cuda())
        if freeze:
            assert all(p.grad is None for p in m.encoder.parameters())
        for n, b in m.encoder.named_buffers():
            assert not torch.equal(before[n], b), n
        rec = _full_record(m, pred, loss)
        recs.append({k: v for k, v in rec.items() if not k.startswith("grad.encoder.")})
    _assert_same(*recs)


def test_step_with_every_bn_frozen_is_bit_reproducible(golden, golden_sd, train_gemm, deterministic):
    from test_gpu_train import _train_model
    recs = []
    for _ in range(2):
        torch.manual_seed(5)
        m, g = _train_model(golden, golden_sd)
        m.att_learner.dropout.p = 0.1
        for bn in _bns(m).values():
            bn.eval()
        pred, loss = _step(m, torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["y"]).long().cuda())
        recs.append(_full_record(m, pred, loss))
    _assert_same(*recs)


def test_no_state_leaks_from_a_frozen_step(golden, golden_sd, train_gemm, deterministic):
    """a frozen step, then every BN back to train: the next step is bit-identical to a step of an untouched model"""
    from test_gpu_train import _train_model
    recs = []
    for toggle in (True, False):
        m, g = _train_model(golden, golden_sd)
        x, y = torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["y"]).long().cuda()
        if toggle:
            for bn in _bns(m).values():
                bn.eval()
            _step(m, x, y)
            m.zero_grad(set_to_none=True)
            for bn in _bns(m).values():
                bn.train()
        pred, loss = _step(m, x, y)
        recs.append(_full_record(m, pred, loss))
    _assert_same(*recs)
