"""Deterministic training: under torch.use_deterministic_algorithms the backward of the EdgeConv gather (model/dgcnn.py:38-41)
sums every dP row in ascending edge order (gfs_edge_reverse_index + gfs_edge_scatter_bn_ordered) instead of with atomics, so a
seeded training step repeats bit for bit.

The reverse index is compared with torch.sort(stable=True); the ordered scatter's P half with a torch fp32 sum of the kernel's own
per-edge terms in the same order (bit-equal), with the atomic path and with fp64 (derived bounds); EdgeConvTrain and the full
training step are run twice and compared bit for bit; the inference path must not change under the flag.  The last test checks
the argument validation of the two C entries and needs no GPU."""
import ctypes
import random
import warnings

import pytest
import torch

from parity import rel_err, rel_l2

U = 2.0 ** -24          # unit roundoff of fp32

# (B, N, k, graph): "knn" = ops.knn of synthetic_blocks, "rand" = torch.randint (repeated targets within a row), "zero" = all 0
SHAPES = [(32, 2048, 20, "knn"), (2, 8192, 40, "knn"), (3, 100, 7, "rand"), (4, 1000, 64, "rand"), (1, 2048, 20, "zero")]


@pytest.fixture
def deterministic():
    """torch.use_deterministic_algorithms(True, warn_only=True) for the test; the previous strict / warn-only state afterwards"""
    was_on, was_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    yield
    torch.use_deterministic_algorithms(was_on, warn_only=was_warn)


@pytest.fixture(params=["tf32x3", "f32"])
def train_gemm(request):
    from gfs3d import ops
    old, ops.TRAIN_GEMM = ops.TRAIN_GEMM, request.param
    yield request.param
    ops.TRAIN_GEMM = old


def _graph(B, N, k, kind):
    from gfs3d import ops
    from gfs3d.synthetic import synthetic_blocks
    if kind == "knn":
        return ops.knn(synthetic_blocks(B, N, seed=B * N + k).cuda(), k)
    if kind == "zero":
        return torch.zeros(B, N, k, dtype=torch.int32, device="cuda")
    return torch.randint(0, N, (B, N, k), generator=torch.Generator().manual_seed(N + k)).int().cuda()


def _targets(idx, B, N):
    return (idx.long() + torch.arange(B, device=idx.device).view(B, 1, 1) * N).reshape(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,k,kind", SHAPES)
def test_reverse_index_is_the_stable_sort_of_the_targets(B, N, k, kind, deterministic):
    from gfs3d import ops
    idx = _graph(B, N, k, kind)
    tgt = _targets(idx, B, N)
    rev_ptr, rev_edge = ops.edge_reverse_index(idx, B, N)
    want_edge = torch.sort(tgt, stable=True).indices
    deg = torch.bincount(tgt, minlength=B * N)
    want_ptr = torch.cat([deg.new_zeros(1), deg.cumsum(0)])
    print(f"B={B} N={N} k={k} {kind}: max in-degree {int(deg.max())}, targets without edges {int((deg == 0).sum())}")
    assert rev_ptr.dtype == torch.int32 and rev_edge.dtype == torch.int32
    assert torch.equal(rev_ptr.long(), want_ptr)
    assert torch.equal(rev_edge.long(), want_edge)


def _bn_inputs(B, N, k, peaked, seed):
    from gfs3d import ops
    g = torch.Generator().manual_seed(seed)
    E = B * N * k
    H = torch.randn(64, E, generator=g)
    dh1 = torch.randn(64, E, generator=g)
    if peaked:        # log-normal magnitudes over ~5 decades: a few edges dominate each sum
        H = H * torch.exp(1.5 * torch.randn(64, E, generator=g))
        dh1 = dh1 * torch.exp(2.5 * torch.randn(64, E, generator=g))
    ga, be = 1 + 0.3 * torch.randn(64, generator=g), 0.2 * torch.randn(64, generator=g)
    H, dh1, ga, be = H.cuda(), dh1.cuda(), ga.cuda(), be.cuda()
    mean, var = ops.bn_stats(H)
    invstd = torch.rsqrt(var + 1e-5)
    sg, sgx = ops.bn_bwd_sums(dh1, H, mean, invstd, ga, be, 0.2)
    return H, dh1, mean, invstd, ga, be, sg, sgx


def _terms_fp64(H, dh1, mean, invstd, ga, be, sg, sgx, slope=0.2):
    """fp64 BatchNorm / LeakyReLU backward per edge from the kernel's fp32 inputs -> (t64 (E, 64), per-element bound, near-branch mask).
    Kernel: xh = (x - mean) * invstd, u = fma(gamma, xh, beta), g = dy * act'(u), t = (gamma * invstd) * (g - sum_g/E - xh * sum_gx/E),
    every operation rounded once (2^-24 relative): xh carries 2u|xh|, g u|g|, a = sum_g/E u|a|, xh*b 4u|xh b|, the two subtractions
    u each of their running magnitude, gamma*invstd u and the last product u.  To first order the |xh b| term collects 8u, the
    others less: |t - t64| <= 10u |gamma invstd| (|g| + |a| + |xh b|) leaves room for the second-order terms.
    Elements whose pre-activation u is within 1e-5 of its magnitude of the branch point may take the other LeakyReLU branch."""
    E = H.shape[1]
    x, dy = H.double(), dh1.double()
    m, s, g_, b_ = (t.double().view(64, 1) for t in (mean, invstd, ga, be))
    xh = (x - m) * s
    u = g_ * xh + b_
    g = dy * torch.where(u > 0, 1.0, slope)
    a, b = sg.double().view(64, 1) / E, sgx.double().view(64, 1) / E
    t = g_ * s * (g - a - xh * b)
    bound = 10 * U * (g_ * s).abs() * (g.abs() + a.abs() + (xh * b).abs()) + 1e-37
    near = u.abs() <= 1e-5 * ((g_ * xh).abs() + b_.abs())
    return t.t().contiguous(), bound.t().contiguous(), near.t().contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("peaked", [False, True], ids=["gauss", "peaked"])
@pytest.mark.parametrize("B,N,k,kind", SHAPES)
def test_ordered_scatter_sums_in_edge_order(B, N, k, kind, peaked, deterministic):
    from gfs3d import ops
    assert torch.isnan(torch.empty(1024, device="cuda")).all(), "torch must fill uninitialised memory with NaN under the flag"
    idx = _graph(B, N, k, kind)
    M, E = B * N, B * N * k
    H, dh1, mean, invstd, ga, be, sg, sgx = _bn_inputs(B, N, k, peaked, seed=M + k + int(peaked))
    rev_ptr, rev_edge = ops.edge_reverse_index(idx, B, N)
    terms = torch.full((E, 64), float("nan"), device="cuda")
    got = ops.edge_scatter_bn(dh1, H, idx, B, N, k, mean, invstd, ga, be, 0.2, sg, sgx, ordered=True, rev=(rev_ptr, rev_edge),
                              edge_terms=terms)          # dpq comes from torch.empty: NaN-filled under the flag
    atomic = ops.edge_scatter_bn(dh1, H, idx, B, N, k, mean, invstd, ga, be, 0.2, sg, sgx)
    assert not torch.isnan(got).any() and not torch.isnan(terms).any()
    assert torch.equal(got[:, 64:], atomic[:, 64:]), "Q half must be the atomic path's, bit for bit"

    # phase 1: the per-edge terms against fp64
    t64, tb, near = _terms_fp64(H, dh1, mean, invstd, ga, be, sg, sgx)
    del H, dh1
    terr = (terms.double() - t64).abs()
    ok = (terr <= tb) | near
    print(f"terms: worst err/bound {float((terr / tb)[~near].max()):.3f}, near-branch elements {int(near.sum())}")
    assert bool(ok.all()), int((~ok).sum())

    # phase 2: bit-equal to the fp32 sum of the same terms, rank by rank in rev_edge order, from +0.0
    ptr = rev_ptr.long()
    start, deg = ptr[:-1], ptr[1:] - ptr[:-1]
    acc = torch.zeros(M, 64, device="cuda")
    order = torch.argsort(deg, descending=True, stable=True)          # rows with deg > r are a prefix of `order`
    n_above = (M - torch.bincount(deg).cumsum(0)).tolist()            # n_above[r] = #rows with deg > r
    for r in range(int(deg.max())):
        rows = order[: n_above[r]]
        acc[rows] = acc[rows] + terms[rev_edge[start[rows] + r].long()]
    assert torch.equal(got[:, :64], acc), "P half differs from the sequential sum in ascending edge order"

    # against the atomic path and fp64, per element: (d-1) u sum|t| for each order of summation, plus the terms' own bounds
    tgt = _targets(idx, B, N)
    absum = torch.zeros(M, 64, dtype=torch.float64, device="cuda").index_add_(0, tgt, terms.double().abs())
    exact = torch.zeros(M, 64, dtype=torch.float64, device="cuda").index_add_(0, tgt, t64)
    tbsum = torch.zeros(M, 64, dtype=torch.float64, device="cuda").index_add_(0, tgt, torch.where(near, terr, tb))
    dm1 = (deg - 1).clamp_min(0).double().view(M, 1)
    gamma = dm1 * U / (1 - dm1 * U)                                    # gamma_{d-1}: a d-term fp32 sum in any order
    b_atomic = 2 * gamma * absum
    b_exact = gamma * absum + tbsum + 1e-37
    e_atomic = (got[:, :64].double() - atomic[:, :64].double()).abs()
    e_exact = (got[:, :64].double() - exact).abs()
    print(f"P half: worst |ordered - atomic| / bound {float((e_atomic / b_atomic.clamp_min(1e-37)).max()):.3f}, "
          f"worst |ordered - fp64| / bound {float((e_exact / b_exact).max()):.3f}")
    assert bool((e_atomic <= b_atomic).all())
    assert bool((e_exact <= b_exact).all())


def _edgeconv_grads(x, idx, params, dy, B, N, k):
    from gfs3d.train_ops import EdgeConvTrain, from_cm, to_cm
    pc = [t.clone().cuda().requires_grad_(True) for t in (x,) + params]
    y, *_ = EdgeConvTrain.apply(to_cm(pc[0]), idx, *pc[1:], B, N, k)
    from_cm(y, B, N).backward(dy)
    torch.cuda.synchronize()
    return [p.grad for p in pc]


@pytest.mark.gpu
def test_edgeconv_train_backward_is_reproducible(deterministic):
    from gfs3d import ops
    B, C, N, k = 32, 64, 2048, 20
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, C, N, generator=g) * 0.5
    idx = ops.knn(x.cuda(), k)
    params = (torch.randn(64, 2 * C, 1, 1, generator=g) / (2 * C) ** 0.5, 1 + 0.3 * torch.randn(64, generator=g),
              0.2 * torch.randn(64, generator=g), torch.randn(64, 64, 1, 1, generator=g) / 8, 1 + 0.3 * torch.randn(64, generator=g),
              0.2 * torch.randn(64, generator=g))
    dy = torch.randn(B, 64, N, generator=g).cuda()
    names = ("dx", "dW1", "dg1", "db1", "dW2", "dg2", "db2")
    first = _edgeconv_grads(x, idx, params, dy, B, N, k)
    second = _edgeconv_grads(x, idx, params, dy, B, N, k)
    for n, a, b in zip(names, first, second):
        assert torch.equal(a, b), n
    torch.use_deterministic_algorithms(False)
    atomic = _edgeconv_grads(x, idx, params, dy, B, N, k)
    l2 = {n: rel_l2(a, b) for n, a, b in zip(names, first, atomic)}
    mx = {n: rel_err(a, b) for n, a, b in zip(names, first, atomic)}
    print("ordered vs atomic: rel-L2 " + " ".join(f"{n} {v:.1e}" for n, v in l2.items()) + f"; worst max-norm {max(mx.values()):.1e}")
    assert max(l2.values()) <= 1e-3 and max(mx.values()) <= 2e-2      # test_edgeconv_train_function_vs_autograd's tolerances


def _run_steps(golden, golden_sd, steps, drop, seed=5):
    """`steps` Adam steps of a fresh model (as test_gpu_train._train_model builds it) -> everything a step produces, per step"""
    from test_gpu_train import _train_model
    torch.manual_seed(seed)                     # the hashed attention dropout derives its seed from torch.initial_seed()
    m, g = _train_model(golden, golden_sd, "train_scannet_b32_n2048", "gfs_scannet_weights")
    random.seed(seed)                           # generate_fake_proto's random.sample
    m.att_learner.dropout.p = drop
    x, y = torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["y"]).long().cuda()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    out = []
    for _ in range(steps):
        opt.zero_grad(set_to_none=True)
        pred, loss = m(x=x, y=y)
        loss.backward()
        rec = {"loss": loss.detach().clone(), "pred": pred.clone()}
        rec.update({"grad." + n: p.grad.clone() for n, p in m.named_parameters()})
        opt.step()
        rec.update({"state." + n: t.detach().clone() for n, t in m.state_dict().items()})
        out.append(rec)
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
def test_training_steps_are_bit_reproducible(golden, golden_sd, train_gemm, deterministic):
    """two Adam steps of the full GFS model at the ScanNet fixture shape (32 x 2048 points, 21 classes, 180 GWs) with attention
    dropout 0.1, twice from fresh models and the same seeds: every loss, prediction, gradient, parameter and buffer identical"""
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        a = _run_steps(golden, golden_sd, 2, 0.1)
    b = _run_steps(golden, golden_sd, 2, 0.1)
    alerts = sorted({str(w.message).split(" does not have")[0] for w in caught if "deterministic" in str(w.message)})
    print(f"[{train_gemm}] torch's non-determinism alerts during the steps: {alerts}")
    for s, (ra, rb) in enumerate(zip(a, b)):
        assert ra.keys() == rb.keys()
        bad = [n for n in ra if not torch.equal(ra[n], rb[n])]
        assert not bad, f"step {s}: {bad}"
    torch.use_deterministic_algorithms(False)
    c, d = _run_steps(golden, golden_sd, 1, 0.1), _run_steps(golden, golden_sd, 1, 0.1)
    grads = [n for n in c[0] if n.startswith("grad.")]
    diff = sum(int((c[0][n] != d[0][n]).sum()) for n in grads)
    total = sum(c[0][n].numel() for n in grads)
    print(f"[{train_gemm}] flag off, for comparison: {diff} of {total} gradient elements differ between two runs")


@pytest.mark.gpu
def test_deterministic_step_passes_the_reference_fixture_gates(golden, golden_sd, train_gemm, deterministic):
    """the ordered scatter and the flattened loss change bits, not results: test_training_step_vs_reference_fixture's gates hold
    for one step at B = 32 x 2048 with the flag on (dropout 0)"""
    from test_gpu_train import test_training_step_vs_reference_fixture
    test_training_step_vs_reference_fixture(golden, golden_sd, "train_scannet_b32_n2048", "gfs_scannet_weights", train_gemm)


@pytest.mark.gpu
def test_inference_is_unaffected_and_the_flag_selects_the_scatter(golden, golden_sd):
    import os
    from types import SimpleNamespace
    import numpy as np
    from gfs3d import ops
    from gfs3d.synthetic import synthetic_blocks
    from model.capl import mpti_net_Point_GeoAsWeight_v2
    from test_gpu_train import _train_model
    was_on, was_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gfs_s3dis_weights.npz"))
    args = SimpleNamespace(edgeconv_widths=[[64, 64]] * 3, dgcnn_mlp_widths=[512, 256], pc_in_dim=9, dgcnn_k=20,
                           base_widths=[128, 64], output_dim=64, eval_weight=1.2)
    gen = torch.Generator().manual_seed(3)
    gp = torch.randn(150, 192, generator=gen)
    gened = torch.nn.functional.normalize(torch.randn(13, 128, generator=gen), dim=1).cuda()
    coding = (torch.rand(13, 150, generator=gen) < 0.3).float().cuda()
    x = synthetic_blocks(32, 2048, seed=42).cuda()
    try:
        logits = {}
        for on in (True, False):
            torch.use_deterministic_algorithms(on, warn_only=True)
            m = mpti_net_Point_GeoAsWeight_v2(classes=13, args=args, base_num=7, gp=gp.cuda(), energy=0.9)
            m.load_state_dict({k: torch.from_numpy(z[k]) for k in z.files})
            m = m.cuda().eval()
            with torch.no_grad():
                logits[on], _, _ = m(x=x, y=None, eval_model=True, gened_proto=gened, base_class_coding=coding[:7],
                                     novel_class_coding=coding[7:])
        assert not torch.isnan(logits[True]).any()
        assert torch.equal(logits[True], logits[False])
        # one training step each way: which scatter entry points ran
        ran = {}
        for on in (True, False):
            torch.use_deterministic_algorithms(on, warn_only=True)
            m, g = _train_model(golden, golden_sd)
            ops.PROFILE = {}
            _, loss = m(x=torch.from_numpy(g["x"]).cuda(), y=torch.from_numpy(g["y"]).long().cuda())
            loss.backward()
            torch.cuda.synchronize()
            ran[on] = {n: len(v) for n, v in ops.PROFILE.items() if n.startswith(("gfs_edge_scatter", "gfs_edge_reverse"))}
            ops.PROFILE = None
        print(f"scatter entries per step: flag on {ran[True]}, flag off {ran[False]}")
        assert ran[True] == {"gfs_edge_reverse_index": 3, "gfs_edge_scatter_bn_ordered": 3}
        assert ran[False] == {"gfs_edge_scatter_bn": 3}
    finally:
        ops.PROFILE = None
        torch.use_deterministic_algorithms(was_on, warn_only=was_warn)


def test_ordered_entries_validate_their_arguments():
    from gfs3d._lib import lib
    l = lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    rc = l.gfs_edge_reverse_index(None, 1, 128, 20, p, p, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    rc = l.gfs_edge_reverse_index(p, 1, 128, 65, p, p, None)
    assert rc == 2 and b"k=65" in l.gfs_last_error_string()
    rc = l.gfs_edge_reverse_index(p, 1 << 16, 2048, 16, p, p, None)          # E = 2^31
    assert rc == 2 and b"2^31" in l.gfs_last_error_string()
    f = [p] * 4
    rc = l.gfs_edge_scatter_bn_ordered(p, p, p, p, None, 1, 128, 20, *f, 0.2, p, p, p, p, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    rc = l.gfs_edge_scatter_bn_ordered(p, p, p, p, p, 1, 128, 20, *f, 0.2, p, p, None, p, None)
    assert rc == 1 and b"null pointer" in l.gfs_last_error_string()
    rc = l.gfs_edge_scatter_bn_ordered(p, p, p, p, p, 1, 128, 65, *f, 0.2, p, p, p, p, None)
    assert rc == 2 and b"k=65" in l.gfs_last_error_string()
    rc = l.gfs_edge_scatter_bn_ordered(p, p, p, p, p, 1 << 16, 2048, 16, *f, 0.2, p, p, p, p, None)
    assert rc == 2 and b"2^31" in l.gfs_last_error_string()
