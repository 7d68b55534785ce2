"""GPU suite: the training attention, its row softmax and the training GEMMs at the training benchmark's shape, B = 32 blocks
of N = 2048 points (M = 65 536 points, E = 1 310 720 edges at k = 20), with attention dropout on, against fp64.

The training step at this shape runs the attention products as interleaved batches (batch b starts at column b * N of
the (C, M) channel-major tensors), writes row slices of larger tensors (dqkv[128:192] with ldc = M), reduces the EdgeConv
weight gradient over 512 split-K partials, and draws attention dropout from a hash of (seed, global row, column) that the
forward and the backward pass regenerate.  Each case issues the calls of gfs3d/train_ops.py with their arguments and checks

* the result against an fp64 reference computed on the GPU from the kernel's own fp32 inputs, per element, against a
  bound derived from the kernel's arithmetic (written with each helper below);
* sentinels: outputs live in NaN-filled buffers, and everything outside the written window must still be NaN;
* position invariance: a batch computed inside the B = 32 launch equals, bit for bit, the same batch computed alone;
* determinism: split-K results are bit-identical from one run to the next.

Rounding model.  fp32 FFMA / FADD / FMUL and IEEE division round to nearest: unit roundoff U = 2^-24 each.  The tensor
core's accumulation is not specified to round to nearest, so it is charged 2^-23 (one ulp) of the running magnitude per
step.  Bounds are first order; the second-order terms are below 1e-6 of the bound at these sizes.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24       # fp32 unit roundoff, round to nearest
U23 = 2.0 ** -23     # one fp32 ulp of the running magnitude
TINY = 2.0 ** -146   # absolute slack for results that underflow into the subnormal range (a few 2^-149 units)
NAN = float("nan")
B32, N2048 = 32, 2048
BLOCKS = (0, 15, 31)


def _ops():
    from gfs3d import ops
    return ops


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


@pytest.fixture(params=["tf32x3", "f32"])
def train_gemm(request):
    """run the test once per implementation of the training GEMM (gfs3d.ops.TRAIN_GEMM)"""
    ops = _ops()
    old, ops.TRAIN_GEMM = ops.TRAIN_GEMM, request.param
    yield request.param
    ops.TRAIN_GEMM = old


@pytest.fixture(autouse=True)
def _peak_memory():
    torch.cuda.reset_peak_memory_stats()
    yield
    print(f"  peak GPU memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")


# ===================================================== training GEMM =====================================================

def _kper(K, splitk):
    """contraction length of one split-K CTA (gemm_f32.cu:139-140, gemm_tf32.cu:276-277)"""
    if splitk == 1:
        return K
    kper = -(-K // splitk)
    return -(-kper // 32) * 32


def gemm_factor(impl, K, splitk=1):
    """|C - exact| <= gemm_factor * (sum_k |Aop||Bop| + |bias|) per element.

    * f32 (gemm_f32.cu): each CTA accumulates its kper products with one FFMA each (round to nearest), starting from the
      bias or 0: gamma_kper <= kper * U of the magnitude sum.
    * tf32x3 (gemm_tf32.cu): an operand v is held as hi = rna_tf32(v) and lo = rna_tf32(v - hi), |v - hi| <= 2^-11 |v| and
      |lo - (v - hi)| <= 2^-22 |v|; the products hi*hi + hi*lo + lo*hi miss lo*lo and the two lo roundings, together at most
      3 * 2^-22 = 6 * 2^-23 of |a b|.  The tensor core adds the 8 hi*hi products of a k-step (one unit of 2^-23 each) and
      rounds the accumulator once more after each of the two cross-term MMAs of the k-step: 1.25 units per k.
    * the split-K reduction (gemm_*_reduce_kernel) adds the bias and the splitk partials in a fixed order, one fp32 add
      each (splitk * U of their magnitudes); the single-pass epilogue adds the bias once (U).
    """
    kper = min(_kper(K, splitk), K)
    acc = kper * U if impl == "f32" else (1.25 * kper + 6) * U23
    return acc + (splitk + 1) * U


def _view(t, ld, trans, bs, b, rows, cols):
    """(rows, cols) view of batch b of an operand as the GEMM contract addresses it (csrc/gemm_f32.cu:5-7):
    element (i, j) = t[b * bs + (j * ld + i if trans else i * ld + j)]"""
    return torch.as_strided(t, (rows, cols), (1, ld) if trans else (ld, 1), t.storage_offset() + b * bs)


def _at(t, off):
    """a tensor whose data pointer is `off` elements into t's (what the kernel does with a batch stride)"""
    return torch.as_strided(t, (1,), (1,), t.storage_offset() + off)


class Gemm:
    """one ops.gemm_f32 call, kept so that it can be issued again (whole, or one batch alone) and checked against the
    contract C[r, n] (+)= bias[r] + sum_k Aop(k, r) Bop(k, n)"""

    def __init__(self, A, lda, at, B, ldb, bt, R, Ncols, K, C, ldc, ct=False, bias=None, batch=1, a_bs=0, b_bs=0, c_bs=0,
                 splitk=1, accumulate=False, impl=None):
        self.A, self.lda, self.at, self.B, self.ldb, self.bt = A, lda, at, B, ldb, bt
        self.R, self.Ncols, self.K, self.C, self.ldc, self.ct, self.bias = R, Ncols, K, C, ldc, ct, bias
        self.batch, self.a_bs, self.b_bs, self.c_bs = batch, a_bs, b_bs, c_bs
        self.splitk, self.accumulate, self.impl = splitk, accumulate, impl

    def __call__(self, C=None, alone=None):
        C = self.C if C is None else C
        if alone is None:
            _ops().gemm_f32(self.A, self.lda, self.at, self.B, self.ldb, self.bt, self.R, self.Ncols, self.K, C, self.ldc,
                            c_trans=self.ct, bias=self.bias, batch=self.batch, a_bs=self.a_bs, b_bs=self.b_bs, c_bs=self.c_bs,
                            splitk=self.splitk, accumulate=self.accumulate, impl=self.impl)
        else:
            b = alone
            _ops().gemm_f32(_at(self.A, b * self.a_bs), self.lda, self.at, _at(self.B, b * self.b_bs), self.ldb, self.bt, self.R,
                            self.Ncols, self.K, _at(C, b * self.c_bs), self.ldc, c_trans=self.ct, bias=self.bias, batch=1,
                            splitk=self.splitk, accumulate=self.accumulate, impl=self.impl)

    def out(self, b, C=None):
        return _view(self.C if C is None else C, self.ldc, self.ct, self.c_bs, b, self.R, self.Ncols)

    def check(self, tag, batches, before=None):
        """per element against fp64 on the GPU: |C - exact| <= gemm_factor * sum|a||b| (+ one rounding of the accumulate)"""
        impl = self.impl or _ops().TRAIN_GEMM
        f = gemm_factor(impl, self.K, self.splitk) + (U if self.accumulate else 0.0)
        worst = 0.0
        for b in batches:
            Ao = _view(self.A, self.lda, self.at, self.a_bs, b, self.K, self.R).double()
            Bo = _view(self.B, self.ldb, self.bt, self.b_bs, b, self.K, self.Ncols).double()
            exact = Ao.t() @ Bo
            mag = Ao.abs().t() @ Bo.abs()
            del Ao, Bo
            if self.bias is not None:
                exact += self.bias.double()[:, None]
                mag += self.bias.double().abs()[:, None]
            if before is not None:
                exact += before[b]
                mag += before[b].abs()
            ratio = float(((self.out(b).double() - exact).abs() / (f * mag).clamp_min(1e-300)).max())
            worst = max(worst, ratio)
            assert ratio <= 1, f"{tag} [{impl}] batch {b}: |C - fp64| is {ratio:.2f}x the bound {f:.2e} * sum|a||b|"
        print(f"  {tag} [{impl}] K={self.K} splitk={self.splitk}: worst |err| / bound {worst:.3f} (bound {f:.2e} * sum|a||b|)")
        return worst


class Window:
    """an output inside a NaN-filled buffer with `guard` elements on each side, and the record of what was written"""

    def __init__(self, shape, guard):
        n = math.prod(shape)
        self.buf = torch.full((guard + n + guard,), NAN, device="cuda")
        self.mark = torch.zeros(self.buf.numel(), dtype=torch.bool, device="cuda")
        self.t = self.buf[guard:guard + n].view(shape)
        self._mt = self.mark[guard:guard + n].view(shape)

    def written(self, g, tag):
        """record g's output window (every batch) and check that nothing outside the windows written so far changed"""
        mt = _at(self._mt, g.C.storage_offset() - self.t.storage_offset())      # g.C may be a row slice of the window
        for b in range(g.batch):
            g.out(b, mt).fill_(True)
        assert bool(self.buf[~self.mark].isnan().all()), f"{tag}: an element outside the output window was written"
        assert bool(self.buf[self.mark].isfinite().all()), f"{tag}: the output window holds a non-finite element"


def _run(tag, g, win, batches, determinism=False, alone=True):
    """issue g, then: sentinels, position invariance (each checked batch alone, batch = 1), determinism, fp64 bound"""
    g()
    win.written(g, tag)
    if alone and g.batch > 1:
        C1 = torch.full_like(g.C, NAN)
        for b in batches:
            g(C1, alone=b)
            assert torch.equal(g.out(b, C1), g.out(b)), f"{tag}: batch {b} differs when computed alone"
        del C1
    if determinism:
        C2 = torch.full_like(g.C, NAN)
        g(C2)
        assert all(torch.equal(g.out(b, C2), g.out(b)) for b in range(g.batch)), f"{tag}: split-K result differs between two runs"
        del C2
    return g.check(tag, batches)


@pytest.mark.parametrize("B,N", [(B32, N2048), (3, 100)], ids=["b32-n2048", "b3-n100-ragged"])
def test_attention_gemms(B, N, train_gemm):
    """the six batched products of AttentionTrain (train_ops.py:166,170,184-192), with their arguments: interleaved batches
    (a_bs = N with lda = M), outputs written as row slices of dqkv (ldc = M, c_bs = N) and as (B, N, N) matrices"""
    M = B * N
    batches = BLOCKS if B == B32 else tuple(range(B))
    g = _gen(M)
    qkv = torch.randn(192, M, device="cuda", generator=g)
    dy = torch.randn(64, M, device="cuda", generator=g)
    q, kk, v = qkv[0:64], qkv[64:128], qkv[128:192]

    S = Window((B, N, N), guard=4096)
    _run("S = q^T k", Gemm(q, M, False, kk, M, False, N, N, 64, S.t, N, batch=B, a_bs=N, b_bs=N, c_bs=N * N), S, batches)
    del S
    p = torch.rand(B, N, N, device="cuda", generator=g)
    y = Window((64, M), guard=M)
    _run("y = v p^T", Gemm(v, M, True, p, N, True, 64, N, N, y.t, M, batch=B, a_bs=N, b_bs=N * N, c_bs=N), y, batches)
    del y
    dqkv = Window((192, M), guard=M)
    _run("dV -> dqkv[128:192]", Gemm(dy, M, True, p, N, False, 64, N, N, dqkv.t[128:192], M, batch=B, a_bs=N, b_bs=N * N, c_bs=N),
         dqkv, batches)
    del p
    dP = Window((B, N, N), guard=4096)
    _run("dP = dy^T v", Gemm(dy, M, False, v, M, False, N, N, 64, dP.t, N, batch=B, a_bs=N, b_bs=N, c_bs=N * N), dP, batches)
    del dP
    dS = torch.randn(B, N, N, device="cuda", generator=g)
    _run("dQ -> dqkv[0:64]", Gemm(kk, M, True, dS, N, True, 64, N, N, dqkv.t[0:64], M, batch=B, a_bs=N, b_bs=N * N, c_bs=N),
         dqkv, batches)
    _run("dK -> dqkv[64:128]", Gemm(q, M, True, dS, N, False, 64, N, N, dqkv.t[64:128], M, batch=B, a_bs=N, b_bs=N * N, c_bs=N),
         dqkv, batches)


@pytest.mark.parametrize("C", [9, 64])
def test_edgeconv_gemms(C, train_gemm):
    """EdgeConvTrain's three products (train_ops.py:116,145,149) at M = 65 536: pq written transposed (c_trans, ldc = 128),
    the split-K weight gradient dWpq and the data gradient dx; C = 9 (the xyz+rgb+normalised input) has lda = 9, so the
    loaders take their unaligned scalar path"""
    from gfs3d.train_ops import _exact
    ops = _ops()
    M = B32 * N2048
    g = _gen(C)
    x = torch.randn(C, M, device="cuda", generator=g)
    Wpq = torch.randn(128, C, device="cuda", generator=g) / C ** 0.5
    dpq = torch.randn(M, 128, device="cuda", generator=g)
    pq = Window((M, 128), guard=1024)
    _run("pq = (Wpq x)^T", Gemm(Wpq, C, True, x, M, False, 128, M, C, pq.t, 128, ct=True, impl=_exact()), pq, (0,))
    del pq
    dW = Window((128, C), guard=1024)
    sk = ops._splitk(M)
    assert sk == (128 if train_gemm == "tf32x3" else 32)
    _run("dWpq", Gemm(dpq, 128, False, x, M, True, 128, C, M, dW.t, C, splitk=sk, impl=_exact()), dW, (0,), determinism=True)
    dx = Window((C, M), guard=1024)
    _run("dx", Gemm(Wpq, C, False, dpq, 128, True, C, M, 128, dx.t, M, impl=_exact()), dx, (0,))


def _conv_triple(tag, W, x, dz, bias=None):
    """conv_fwd, conv_dgrad and conv_wgrad (ops.py:440-461), each issued with the wrapper's own arguments into a NaN
    window, checked, and compared bit for bit with the wrapper's result"""
    ops = _ops()
    O, I = W.shape
    M = x.shape[1]
    z = Window((O, M), guard=1024)
    _run(f"{tag} conv_fwd", Gemm(W, I, True, x, M, False, O, M, I, z.t, M, bias=bias), z, (0,))
    assert torch.equal(ops.conv_fwd(W, x, bias), z.t)
    del z
    dx = Window((I, M), guard=1024)
    _run(f"{tag} conv_dgrad", Gemm(W, I, False, dz, M, False, I, M, O, dx.t, M), dx, (0,))
    assert torch.equal(ops.conv_dgrad(W, dz), dx.t)
    del dx
    return _conv_wgrad(tag, dz, x)


def _conv_wgrad(tag, dz, x):
    ops = _ops()
    O, M = dz.shape
    I = x.shape[0]
    dW = Window((O, I), guard=1024)
    sk = ops._splitk(M)
    _run(f"{tag} conv_wgrad", Gemm(dz, M, True, x, M, True, O, I, M, dW.t, I, splitk=sk), dW, (0,), determinism=True)
    assert torch.equal(ops.conv_wgrad(dz, x), dW.t)
    return sk


def test_conv_gemms_over_the_edges(train_gemm):
    """EdgeConv's second 1x1 conv at E = 32 * 2048 * 20 edges: Z = W2 h1, dh1 = W2^T dZ, and dW2 = dZ h1^T, a contraction
    over 1 310 720 edges that runs split-K 512.  The weight gradient runs a second time on non-negative operands: there
    sum|a||b| = |sum a b|, so the bound is a few parts in 1e4 of the result and losing one of the 512 partials (1/512 of
    the sum) cannot hide under it."""
    E = B32 * N2048 * 20
    g = _gen(E)
    W2 = torch.randn(64, 64, device="cuda", generator=g) / 8
    h1 = torch.randn(64, E, device="cuda", generator=g)
    dZ = torch.randn(64, E, device="cuda", generator=g)
    assert _conv_triple("E=1310720", W2, h1, dZ) == 512
    _conv_wgrad("E=1310720 non-negative", dZ.abs_(), h1.abs_())


def test_conv_gemms_at_the_mlp_widths(train_gemm):
    """the DGCNN MLP 192 -> 512 -> 256 (ConvBNAct, train_ops.py:41-66) at M = 65 536: forward with bias, data and weight
    gradients"""
    M = B32 * N2048
    g = _gen(M + 1)
    for I, O in ((192, 512), (512, 256)):
        W = torch.randn(O, I, device="cuda", generator=g) / I ** 0.5
        bias = torch.randn(O, device="cuda", generator=g)
        x = torch.randn(I, M, device="cuda", generator=g)
        dz = torch.randn(O, M, device="cuda", generator=g)
        _conv_triple(f"{I}->{O}", W, x, dz, bias)


def test_splitk_with_empty_trailing_splits(train_gemm):
    """K = 262 145 over 512 splits: kper rounds up to 544, so splits 482-511 have no k range and take the nk == 0 epilogue
    (gemm_tf32.cu:199,215), which must contribute exact zeros.  Non-negative operands (see above); ld = K is odd, so the
    loaders take their scalar path"""
    K, sk, R, Nc = 262145, 512, 64, 64
    kper = _kper(K, sk)
    assert kper == 544 and -(-K // kper) == 482, "the shape must leave the trailing 30 splits empty"
    g = _gen(K)
    A = torch.rand(R, K, device="cuda", generator=g)
    Bm = torch.rand(Nc, K, device="cuda", generator=g)
    C = Window((R, Nc), guard=1024)
    _run("empty trailing splits", Gemm(A, K, True, Bm, K, True, R, Nc, K, C.t, Nc, splitk=sk), C, (0,), determinism=True)


def test_splitk_accumulate(train_gemm):
    """accumulate=True (the reduce kernel's *o + acc): C = C_before + A B, into a transposed output with ldc > R"""
    R, Nc, K, sk = 70, 130, 5000, 8
    ldc = R + 3
    g = _gen(K + R)
    A = torch.randn(K, R, device="cuda", generator=g)
    Bm = torch.randn(Nc, K, device="cuda", generator=g)
    C = Window((Nc, ldc), guard=1024)
    gm = Gemm(A, R, False, Bm, K, True, R, Nc, K, C.t, ldc, ct=True, splitk=sk, accumulate=True)
    gm.out(0).copy_(torch.randn(R, Nc, device="cuda", generator=g))
    before = gm.out(0).double().clone()
    C_before = C.t.clone()
    gm()
    C.written(gm, "accumulate")
    again = C_before.clone()
    gm(again)
    assert torch.equal(gm.out(0, again), gm.out(0)), "accumulate: result differs between two runs"
    gm.check("accumulate", (0,), before={0: before})


# ===================================================== row softmax =====================================================

def _softmax_bound(x):
    """per-element bound on |p0 - softmax(x)| for softmax_rows_fwd_kernel (train.cu:491-511), x = s * scale in fp64
    (the kernel's s * scale is exact for scale = 1/8).  One warp per row:
      * d = x - max: one rounding, U |x - max|; expf: 2 ulp = 4 U (CUDA's documented maximum error);
      * sum: each lane adds ceil(n / 32) terms, then 5 butterfly levels: gamma_h with h = ceil(n / 32) + 5, plus the
        p-weighted relative error of its terms;
      * 1 / sum and e * (1 / sum): U each;
      * results below 2^-126 are subnormal: TINY absolute."""
    n = x.shape[1]
    h = -(-n // 32) + 5
    P = torch.softmax(x, dim=1)
    e_rel = U * (x.max(dim=1, keepdim=True).values - x) + 4 * U
    rel = e_rel + h * U + (P * e_rel).sum(dim=1, keepdim=True) + 2 * U
    return P, rel


def _check_fwd(s, scale, p0, tag):
    x = s.double() * scale
    P, rel = _softmax_bound(x)
    bound = P * rel + TINY
    got = p0.double()
    assert bool(got.isfinite().all()), f"{tag}: p0 has a non-finite element"
    ratio = float(((got - P).abs() / bound).max())
    sums = (got.sum(dim=1) - 1).abs()
    sratio = float((sums / bound.sum(dim=1)).max())
    assert ratio <= 1, f"{tag}: |p0 - fp64 softmax| is {ratio:.2f}x the bound"
    assert sratio <= 1, f"{tag}: a row of p0 misses 1 by {sratio:.2f}x the sum of its bounds"
    return max(ratio, sratio)


def _check_bwd(p0, dp, m, scale, ds, tag):
    """ds against fp64 scale * p0 * (dp m - sum p0 dp m) from the kernel's own p0 (softmax_rows_bwd_kernel, train.cu:513-530).
    The dot product sums the terms p0 dp m (two roundings each) per lane and over 5 butterfly levels:
    (h + 2) U sum|p0 dp m|; then dp m (U), the difference (U), and the two products with scale and p0 (U each):
    |ds - ref| <= scale p0 U ((h + 6) A + 4 |dp m|),  A = sum_j |p0 dp m|."""
    n = p0.shape[1]
    h = -(-n // 32) + 5
    P0 = p0.double()
    D = dp.double() if m is None else dp.double() * m.double()
    dot = (P0 * D).sum(dim=1, keepdim=True)
    A = (P0 * D).abs().sum(dim=1, keepdim=True)
    ref = scale * P0 * (D - dot)
    bound = scale * P0 * U * ((h + 6) * A + 4 * D.abs()) + TINY
    got = ds.double()
    assert bool(got.isfinite().all()), f"{tag}: ds has a non-finite element"
    ratio = float(((got - ref).abs() / bound).max())
    assert ratio <= 1, f"{tag}: |ds - fp64| is {ratio:.2f}x the bound"
    return ratio


def _softmax_modes(ops, s, scale, dp, seed, rows_checked, tag, explicit_keep=0.9):
    """every dropout mode on one logit tensor s (B, n, n) or (1, rows, n): none, explicit mask (one row fully dropped),
    hashed at keep 0.9 and 0.5.  Checks p0 / ds against fp64 on rows_checked, p == p0 * mask bit for bit everywhere, and
    hashed ds == explicit-mask ds bit for bit everywhere."""
    rows, n = s.shape[0] * s.shape[1], s.shape[2]
    s2 = s.view(rows, n)
    worst = {}
    p0, p = ops.softmax_rows_fwd(s, scale)
    assert p is p0
    p0_ref = p0
    worst["p0"] = max(_check_fwd(s2[r], scale, p0.view(rows, n)[r], f"{tag} p0 rows {r}") for r in rows_checked)
    ds = ops.softmax_rows_bwd(p0, dp, scale)
    worst["ds none"] = max(_check_bwd(p0.view(rows, n)[r], dp.view(rows, n)[r], None, scale, ds.view(rows, n)[r], f"{tag} ds")
                           for r in rows_checked)
    del ds
    mask = ops.dropout_mask(rows, n, seed ^ 0x5A5A5A5A, explicit_keep, s.device).view_as(s)
    mask.view(rows, n)[rows // 3] = 0                                  # a fully dropped row
    p0m, pm = ops.softmax_rows_fwd(s, scale, mask)
    assert torch.equal(p0m, p0_ref), f"{tag}: p0 depends on the mask"
    assert torch.equal(pm, p0m * mask), f"{tag}: p != p0 * mask (explicit)"
    assert float(pm.view(rows, n)[rows // 3].abs().max()) == 0
    del pm
    dsm = ops.softmax_rows_bwd(p0m, dp, scale, mask)
    assert float(dsm.view(rows, n)[rows // 3].abs().max()) == 0, f"{tag}: a fully dropped row has a non-zero gradient"
    worst["ds explicit"] = max(_check_bwd(p0m.view(rows, n)[r], dp.view(rows, n)[r], mask.view(rows, n)[r], scale,
                                          dsm.view(rows, n)[r], f"{tag} ds explicit") for r in rows_checked + [slice(rows // 3, rows // 3 + 1)])
    del dsm, mask, p0m
    for keep in (0.9, 0.5):
        mask = ops.dropout_mask(rows, n, seed, keep, s.device).view_as(s)
        p0h, ph = ops.softmax_rows_fwd(s, scale, None, seed, keep)
        assert torch.equal(p0h, p0_ref), f"{tag}: p0 depends on the dropout"
        assert torch.equal(ph, p0h * mask), f"{tag}: hashed p != p0 * dropout_mask (keep {keep})"
        del ph
        dsh = ops.softmax_rows_bwd(p0h, dp, scale, None, seed, keep)
        dse = ops.softmax_rows_bwd(p0h, dp, scale, mask)
        assert torch.equal(dsh, dse), f"{tag}: hashed ds != explicit-mask ds (keep {keep}), rows {rows}"
        del dse
        worst[f"ds hashed {keep}"] = max(_check_bwd(p0h.view(rows, n)[r], dp.view(rows, n)[r], mask.view(rows, n)[r], scale,
                                                    dsh.view(rows, n)[r], f"{tag} ds hashed {keep}") for r in rows_checked)
        del dsh, mask, p0h
    print(f"  {tag}: worst |err| / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


@pytest.mark.parametrize("gain", [1.0, 30.0])
def test_softmax_rows_fullshape(gain):
    """rows = 32 * 2048 = 65 536 of n = 2048 (the attention's S at the benchmark shape), Gaussian logits at gain 1 and 30,
    scale 1/8; fp64 checks on the rows of blocks 0, 15 and 31; bit-exact checks on all rows"""
    ops = _ops()
    g = _gen(int(gain))
    s = gain * torch.randn(B32, N2048, N2048, device="cuda", generator=g)
    dp = torch.randn(B32, N2048, N2048, device="cuda", generator=g)
    rows = [slice(b * N2048, (b + 1) * N2048) for b in BLOCKS]
    _softmax_modes(ops, s, 0.125, dp, 0xC0FFEE + int(gain), rows, f"softmax 65536x2048 gain {gain:g}")


@pytest.mark.parametrize("n", [1, 31, 33, 100, 2047])
def test_softmax_rows_ragged(n):
    """ragged row lengths, 1005 rows (not a multiple of the 8 rows of a CTA), in five groups of 201 rows: Gaussian logits at
    gain 1 and 30, peaked rows (one entry 2000 above the rest: every other exponential underflows), constant rows, and rows
    near -1e4"""
    ops = _ops()
    g = _gen(n)
    G = 201
    s = torch.randn(5 * G, n, device="cuda", generator=g)
    s[G:2 * G] *= 30
    s[2 * G:3 * G] = 0.5 * s[2 * G:3 * G]
    s[2 * G + torch.arange(G, device="cuda"), torch.randint(0, n, (G,), device="cuda", generator=g)] = 2000.0
    s[3 * G:4 * G] = 3.7
    s[4 * G:] = -1e4 + 8 * s[4 * G:]
    dp = torch.randn(5 * G, n, device="cuda", generator=g)
    _softmax_modes(ops, s.view(1, 5 * G, n), 0.125, dp.view(1, 5 * G, n), 777 + n, [slice(0, 5 * G)], f"softmax 1005x{n}")


# ===================================================== AttentionTrain =====================================================

def _attention_seed(initial_seed, calls):
    """the dropout seed SelfAttention.forward_train derives (model/attention.py:49)"""
    return (initial_seed * 0x9E3779B1 + calls * 0x85EBCA77) & 0xFFFFFFFF


def _attention_bounds(q, k, v, dy, Mb, scale, impl):
    """Per-element bounds for y and the q / k / v gradients of one block, all fp64 (N, N) on the GPU, first order, from
    the parts above: S = q^T k has |dS| <= ES = g64 sum_c |q||k| (g64 = gemm_factor(impl, 64)); a logit error moves p0_j
    by at most scale (ES_j + max_i ES_i) relative; softmax_rows_fwd adds _softmax_bound, and p = p0 m one more U; so
    |p - P| <= dp = P0 rho m.  y = v p^T and dV = dy p then err <= |v| dp^T + gN |v| (P + dp)^T (gN = gemm_factor(impl, N)).
    dP = dy^T v has EdP = g64 sum_c |dy||v|; ds = scale p0 (D - sum p0 D) with D = dP m gets
      scale (|dp0| |D - dot| + P0 (EdP m + sum_i (dp0_i |D_i| + P0_i m_i EdP_i)) + _check_bwd's rounding bound),
    and dQ = k dS^T, dK = q dS add gN times their magnitude sums."""
    N = q.shape[1]
    h = -(-N // 32) + 5
    g64, gN = gemm_factor(impl, 64), gemm_factor(impl, N)
    ES = g64 * (q.abs().t() @ k.abs())
    x = (q.t() @ k) * scale
    P0, rel = _softmax_bound(x)
    rho = scale * (ES + ES.max(dim=1, keepdim=True).values) + rel + U
    dp0 = P0 * rho + TINY
    del ES, rel, rho, x
    P, dpm = P0 * Mb, dp0 * Mb
    by = v.abs() @ dpm.t() + gN * (v.abs() @ (P + dpm).t())
    bdv = dy.abs() @ dpm + gN * (dy.abs() @ (P + dpm))
    del P, dpm
    EdPm = g64 * (dy.abs().t() @ v.abs()) * Mb
    D = (dy.t() @ v) * Mb
    dot = (P0 * D).sum(dim=1, keepdim=True)
    A = ((P0 + dp0) * (D.abs() + EdPm)).sum(dim=1, keepdim=True)
    EdS = scale * (dp0 * (D - dot).abs() + P0 * (EdPm + (dp0 * D.abs() + P0 * EdPm).sum(dim=1, keepdim=True))
                   + P0 * U * ((h + 6) * A + 4 * (D.abs() + EdPm))) + TINY
    dSmag = (scale * P0 * (D - dot)).abs() + EdS
    bdq = k.abs() @ EdS.t() + gN * (k.abs() @ dSmag.t())
    bdk = q.abs() @ EdS + gN * (q.abs() @ dSmag)
    return by, bdq, bdk, bdv


def _binom_ok(count, n, prob):
    return abs(count - n * prob) <= 6 * math.sqrt(n * prob * (1 - prob))


def test_attention_train_fullshape_hashed_dropout(train_gemm):
    """AttentionTrain at B = 32, N = 2048 with hashed dropout at keep 0.9, the benchmark's training configuration:
    1. forward y and dqkv equal, bit for bit, a run with the explicit mask dropout_mask(B N, N, seed, keep);
    2. blocks 0, 15 and 31 against fp64 autograd of softmax(q^T k / 8) m v^T on the kernel's inputs and mask, per element
       within _attention_bounds;
    3. the mask: the keep fraction of every block, and the agreement between blocks and between seeds s and s + 1, lie
       within 6 sigma of a binomial (the hash takes the global row, so blocks must not share masks)."""
    from gfs3d.train_ops import AttentionTrain
    ops = _ops()
    B, N, keep, scale = B32, N2048, 0.9, 0.125
    M = B * N
    seed = _attention_seed(1234, 1)
    g = _gen(seed)
    qkv = torch.randn(192, M, device="cuda", generator=g)
    dy = torch.randn(64, M, device="cuda", generator=g)

    def run(mask, s, kp):
        t = qkv.clone().requires_grad_(True)
        y = AttentionTrain.apply(t, B, N, scale, mask, s, kp)
        y.backward(dy)
        return y.detach(), t.grad

    yh, gh = run(None, seed, keep)
    mask = ops.dropout_mask(M, N, seed, keep, qkv.device).view(B, N, N)
    ye, ge = run(mask, 0, 1.0)
    assert torch.equal(yh, ye), "hashed-dropout forward differs from the explicit mask it defines"
    assert torch.equal(gh, ge), "hashed-dropout backward differs from the explicit mask it defines"
    del ye, ge

    worst = {}
    for b in BLOCKS:
        cols = slice(b * N, (b + 1) * N)
        t = qkv[:, cols].double().requires_grad_(True)
        q, k, v = t[0:64], t[64:128], t[128:192]
        Mb = mask[b].double()
        P = torch.softmax((q.t() @ k) * scale, dim=1) * Mb
        y = v @ P.t()
        y.backward(dy[:, cols].double())
        bounds = _attention_bounds(q.detach(), k.detach(), v.detach(), dy[:, cols].double(), Mb, scale, train_gemm)
        for name, got, ref, bd in (("y", yh[:, cols], y.detach(), bounds[0]), ("dq", gh[0:64, cols], t.grad[0:64], bounds[1]),
                                   ("dk", gh[64:128, cols], t.grad[64:128], bounds[2]),
                                   ("dv", gh[128:192, cols], t.grad[128:192], bounds[3])):
            err = (got.double() - ref).abs()
            ratio = float((err / bd).max())
            worst[name] = max(worst.get(name, 0.0), ratio)
            assert ratio <= 1, f"block {b} {name}: |err| is {ratio:.2f}x the derived bound"
            worst[name + " bound/max|ref|"] = max(worst.get(name + " bound/max|ref|", 0.0), float(bd.max() / ref.abs().max()))
        del t, q, k, v, P, y, bounds
    print(f"  AttentionTrain[{train_gemm}] B=32 N=2048 keep 0.9: " + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))

    kept = (mask > 0).view(B, N * N).sum(dim=1).tolist()
    for b, c in enumerate(kept):
        assert _binom_ok(c, N * N, keep), f"block {b}: keep fraction {c / (N * N):.5f}, expected {keep} +- 6 sigma"
    agree = keep * keep + (1 - keep) ** 2
    for b0, b1 in ((0, 1), (0, 31), (15, 16)):
        c = int((mask[b0] == mask[b1]).sum())
        assert _binom_ok(c, N * N, agree), f"blocks {b0} and {b1}: mask agreement {c / (N * N):.5f}, expected {agree:.4f}"
    other = ops.dropout_mask(M, N, seed + 1, keep, qkv.device)
    c = int((other.view(B, N, N) == mask).sum())
    assert _binom_ok(c, M * N, agree), f"seeds s and s+1: mask agreement {c / (M * N):.6f}, expected {agree:.4f}"
