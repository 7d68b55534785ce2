"""GPU suite: the persistent tcgen05 kernels past their first round of work items.

gfs_linear_bf16 (linear.cu), gfs_edgeconv_fwd (edgeconv.cu), gfs_attention_fwd (attention.cu) and gfs_gw_project_tc
(rowsel_tc.cu) launch grid = min(work items, SM count) CTAs, and every CTA loops over its items with stride gridDim.x.
From one item to the next a CTA carries mbarrier phases, pipeline-stage and TMEM-accumulator indices, and in linear's
resident mode a weight slice that stays in shared memory.  The shapes here give every CTA at least three items and end
on a partial round (a regime guard asserts this with the device's own SM count), and every case checks

1. position invariance, bit for bit: an item's arithmetic does not depend on which CTA, round, pipeline stage or TMEM
   buffer runs it, so a slice of whole blocks (whole 128-row tiles) computed inside the big launch must equal the same
   slice computed alone, where all its tiles run in the first round.  The slices cover the first, a middle and the last,
   partial round.
2. an fp64 reference computed on the GPU from the kernel's own bf16 operands, on the same slices, against a tolerance
   derived from the kernel's arithmetic (stated with each check).
"""
from collections import Counter

import pytest
import torch
import torch.nn.functional as F

from parity import rel_err

pytestmark = pytest.mark.gpu

U23 = 2.0 ** -23     # one fp32 rounding step, safe for truncating adders (the tensor core's accumulation is not specified RN)
U8 = 2.0 ** -8       # unit roundoff of bf16 (8 significant bits, round to nearest even)


def _ops():
    from gfs3d import ops
    return ops


def _sms():
    """the SM count the launchers size their grids with (sm_count(), csrc/api.cu), read from the device at run time"""
    from gfs3d._lib import lib
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert lib().gfs_device_sm_count() == sms, "the library and torch disagree about the device's SM count"
    return sms


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


class Plan:
    """How a persistent launcher spreads its work.  `per_round` CTAs (or, in linear's resident mode, CTAs per N tile)
    take `work` items round-robin; item i runs on the 128-row tile item_tile[i] in round item_round[i]."""

    def __init__(self, name, items, grid, work, per_round, item_tile, item_round):
        self.name, self.items, self.grid, self.work, self.per_round = name, items, grid, work, per_round
        self.item_tile, self.item_round = item_tile, item_round
        self.rounds = -(-work // per_round)

    def guard(self):
        """the shape must give every CTA at least three items and end on a partial round, on THIS device"""
        hist = Counter(self.item_round)
        print(f"\n{self.name}: {self.items} items, grid {self.grid}, {self.rounds} rounds of {self.per_round}, "
              f"items per round {[hist[r] for r in range(self.rounds)]}")
        assert self.work >= 3 * self.per_round, (
            f"{self.name}: {self.work} items over {self.per_round} per round is fewer than three rounds on this GPU "
            f"({_sms()} SMs): the test would not reach a CTA's later items; enlarge the shape")
        assert self.work % self.per_round != 0, f"{self.name}: the last round is not partial on this GPU"

    def rounds_of_tiles(self, t0, t1):
        return sorted({r for t, r in zip(self.item_tile, self.item_round) if t0 <= t < t1})

    def check_slices(self, tile_ranges):
        """the slices must reach the first round, a middle round and the last, partial round"""
        covered = set()
        for t0, t1 in tile_ranges:
            rs = self.rounds_of_tiles(t0, t1)
            print(f"  slice of tiles [{t0}, {t1}): rounds {rs}")
            covered.update(rs)
        last = self.rounds - 1
        assert 0 in covered and last in covered and any(0 < r < last for r in covered), covered


def _plan_rowwise(name, ntiles, sms):
    """one item per 128-row tile, item i on CTA i % grid in round i // grid"""
    grid = min(ntiles, sms)
    return Plan(name, ntiles, grid, ntiles, grid, list(range(ntiles)), [t // grid for t in range(ntiles)])


def _plan_linear(B, N, K, Nout, sms):
    # gfs_linear_bf16, linear.cu:223-244 (N tile NT, M-tile x N-tile items, grid, resident mode and the grid trim)
    NT = Nout if Nout <= 256 else 256
    while Nout % NT:
        NT -= 32
    n_ntiles = Nout // NT
    n_mtiles = -(-B * N // 128)
    items = n_mtiles * n_ntiles
    grid = min(items, sms)
    kb_count = -(-K // 64)
    resident = kb_count * NT * 128 <= 4 * 32768 and grid >= n_ntiles        # sizeof(LnSmem::W) = 128 KiB
    if resident:
        grid -= grid % n_ntiles
        # a CTA keeps N tile blockIdx % n_ntiles and walks the M tiles blockIdx / n_ntiles + r * (grid / n_ntiles)
        # (linear.cu:46-47): its rounds are counted over the M tiles
        step = grid // n_ntiles
        tiles = [mt for _ in range(n_ntiles) for mt in range(n_mtiles)]
        plan = Plan(f"linear {K}->{Nout} B={B} N={N} resident NT={NT}x{n_ntiles}", items, grid, n_mtiles, step, tiles,
                    [mt // step for mt in tiles])
    else:
        plan = Plan(f"linear {K}->{Nout} B={B} N={N} streaming NT={NT}x{n_ntiles}", items, grid, items, grid,
                    [it // n_ntiles for it in range(items)], [it // grid for it in range(items)])
    plan.resident = resident
    return plan


def _block_slices(B):
    return [(0, 1), (B // 2, B // 2 + 1), (B - 1, B)]


def _act_rows(act, M):
    """(M, kblocks*64) bf16 row-major view of an act matrix"""
    return _ops().act_to_dense(act, M)


def _cm_rows(y, b0, b1):
    """channel-major (B, C, N) fp32 -> (rows of blocks b0..b1, C)"""
    return y[b0:b1].permute(0, 2, 1).reshape(-1, y.shape[1])


# ===================================================== linear =====================================================

_ACT = {0: lambda r: r, 1: lambda r: F.leaky_relu(r, 0.2), 2: F.relu}


def _linear_case(B, N, K, Nout, seed):
    ops = _ops()
    g = _gen(seed)
    x = torch.randn(B, K, N, device="cuda", generator=g)
    w = torch.randn(Nout, K, device="cuda", generator=g) / K ** 0.5
    s = 1 + 0.3 * torch.randn(Nout, device="cuda", generator=g)
    t = 0.2 * torch.randn(Nout, device="cuda", generator=g)
    xa = ops.new_act(B * N, K // 64, "cuda")
    ops.cm_to_act(x, xa, 0)
    del x
    return xa, ops.pack_weight(w, s), t, (w * s[:, None]).bfloat16().double()


def _linear_run(xa, K, wp, t, Nout, act, B, N, with_act):
    ops = _ops()
    y_cm = torch.full((B, Nout, N), float("nan"), device="cuda")
    y_act = ops.new_act(B * N, Nout // 64 + 1, "cuda") if with_act else None
    ops.linear(xa, 0, K // 64, wp, t, Nout, act, B, N, y_act=y_act, y_kb0=1 if with_act else 0, y_cm=y_cm)
    return y_cm, y_act


def _linear_ref_check(xa, wb, t, act, y_rows, r0, r1, tag):
    """fp64 GEMM on the kernel's bf16 operands (act_to_dense of the input, bf16(w * s) as the weights), as in
    test_linear_tcgen05_vs_fp64, with that test's 1e-4 max-norm relative tolerance.  Products of bf16 values are exact,
    so only the fp32 accumulation of K terms remains: at most K * 2^-23 * sum|x||w| per element (6.1e-5 * sum|x||w| at
    K = 512), and for these operands (x ~ N(0, 1), w ~ N(0, 1/K) * s) sum|x||w| is of the order of max|y|."""
    ref = _ACT[act](_act_rows(xa[r0 // 128:-(-r1 // 128)], r1 - r0).double() @ wb.t() + t.double())
    err = rel_err(y_rows, ref)
    print(f"  {tag}: fp64 rel err {err:.2e} (bound 1e-4)")
    assert err <= 1e-4, f"{tag}: tcgen05 GEMM differs from fp64 on identical bf16 operands"


@pytest.mark.parametrize("K,Nout,act", [(192, 512, 1), (512, 256, 1), (384, 128, 2), (256, 480, 0)],
                         ids=["192-512-resident-2nt", "512-256-streaming", "384-128-fusion", "256-480-resident-3nt-trimmed"])
def test_linear_rounds(K, Nout, act):
    B, N = 32, 2048
    plan = _plan_linear(B, N, K, Nout, _sms())
    plan.guard()
    if (K, Nout) == (512, 256):
        assert not plan.resident, "512->256 must exercise the streaming mode"
    else:
        assert plan.resident
    if Nout == 480:
        assert plan.grid < min(plan.items, _sms()), "the grid must be trimmed to a multiple of the 3 N tiles"
    with_act = Nout % 64 == 0            # the launcher allows bf16 act output only for Nout % 64 == 0
    xa, wp, t, wb = _linear_case(B, N, K, Nout, seed=K * 1000 + Nout)
    y_cm, y_act = _linear_run(xa, K, wp, t, Nout, act, B, N, with_act)
    tpb = N // 128
    slices = _block_slices(B)
    plan.check_slices([(b0 * tpb, b1 * tpb) for b0, b1 in slices])
    M = B * N
    if with_act:
        dense = _act_rows(y_act, M)
        assert float(dense[:, :64].abs().max()) == 0, "output block 0 (before y_kb0) was written"
        assert torch.equal(dense[:, 64:], _cm_rows(y_cm, 0, B).bfloat16()), "act output is not bf16(fp32 output)"
    for b0, b1 in slices:
        tag = f"blocks [{b0}, {b1})"
        sub_cm, sub_act = _linear_run(xa[b0 * tpb:b1 * tpb], K, wp, t, Nout, act, b1 - b0, N, with_act)
        assert torch.equal(sub_cm, y_cm[b0:b1]), f"{tag}: fp32 output depends on where the tiles ran"
        if with_act:
            assert torch.equal(sub_act, y_act[b0 * tpb:b1 * tpb]), f"{tag}: bf16 output depends on where the tiles ran"
        _linear_ref_check(xa, wb, t, act, _cm_rows(y_cm, b0, b1), b0 * N, b1 * N, tag)


def test_linear_m_tail_runs_alone_in_the_last_round():
    """B = 1, N = 3 * SMs * 128 + 77 on the single-N-tile 384 -> 128 layer: the 77-row partial M tile is the only item of
    the last round.  Slices are runs of whole tiles (B = 1 has one block)."""
    sms = _sms()
    K, Nout, act = 384, 128, 2
    B, N = 1, 3 * sms * 128 + 77
    plan = _plan_linear(B, N, K, Nout, sms)
    plan.guard()
    assert plan.resident and plan.work % plan.per_round == 1
    xa, wp, t, wb = _linear_case(B, N, K, Nout, seed=77)
    y_cm, y_act = _linear_run(xa, K, wp, t, Nout, act, B, N, True)
    nt = plan.work
    ranges = [(0, 16), (nt // 2, nt // 2 + 16), (nt - 16, nt)]
    plan.check_slices(ranges)
    dense = _act_rows(y_act, N)
    assert float(dense[:, :64].abs().max()) == 0
    assert torch.equal(dense[:, 64:], y_cm[0].t().bfloat16()), "act output is not bf16(fp32 output)"
    # a row's 64 values stay inside its own 128 bytes of the tile (the swizzle permutes 16-byte chunks within the row)
    assert float(y_act[-1].view(-1, 128, 64)[:, 77:].float().abs().max()) == 0, "rows past M of the partial tile were written"
    for t0, t1 in ranges:
        r0, r1 = t0 * 128, min(t1 * 128, N)
        tag = f"tiles [{t0}, {t1}) rows [{r0}, {r1})"
        sub_cm, sub_act = _linear_run(xa[t0:t1], K, wp, t, Nout, act, 1, r1 - r0, True)
        assert torch.equal(sub_cm[0], y_cm[0, :, r0:r1]), f"{tag}: fp32 output depends on where the tiles ran"
        assert torch.equal(sub_act, y_act[t0:t1]), f"{tag}: bf16 output depends on where the tiles ran"
        _linear_ref_check(xa, wb, t, act, y_cm[0, :, r0:r1].t(), r0, r1, tag)


# ===================================================== edgeconv =====================================================

EC_SMEM_FIXED = 4 * 16384 + 8 * 16384 + 8192 + 64 * 4 + (4 + 4 + 4 + 4 + 1) * 8 + 4   # the members of EcSmem, edgeconv.cu:32-39
EC_SMEM_STRUCT = -(-EC_SMEM_FIXED // 8) * 8                                            # sizeof: padded to its 8-byte alignment
# edgeconv.cu:302-304: sizeof(EcSmem) + 1024 (alignment slack) + the [128][k] int32 neighbour tile <= 227 KiB
EC_K_MAX = (227 * 1024 - EC_SMEM_STRUCT - 1024) // (128 * 4)
F32_02 = torch.tensor(0.2, dtype=torch.float32)      # the kernel's 0.2f


def _edgeconv_inputs(B, N, k, seed):
    """bf16 P' - mu rows, fp32 Q' + mu rows (what gfs_edge_pq_f32 produces), block-local neighbour indices with duplicated
    points (identical P' rows) and repeated neighbours (exact ties in the max over k), W2 and BN2"""
    g = _gen(seed)
    M = B * N
    pb = torch.randn(M, 64, device="cuda", generator=g).bfloat16()
    pv = pb.view(B, N, 64)
    pv[:, N // 2:N // 2 + N // 8] = pv[:, :N // 8]                       # points N/2 .. 5N/8 duplicate points 0 .. N/8
    q = 0.5 * torch.randn(M, 64, device="cuda", generator=g)
    idx = torch.randint(0, N, (B, N, k + 1), device="cuda", generator=g, dtype=torch.int32)
    idx[:, ::10, 1] = idx[:, ::10, 0]                                      # a neighbour listed twice
    idx[:, ::7, k - 1] = torch.arange(0, N, 7, device="cuda", dtype=torch.int32)      # the point itself
    w2 = torch.randn(64, 64, device="cuda", generator=g) / 8
    s2 = 1 + 0.3 * torch.randn(64, device="cuda", generator=g)
    t2 = 0.2 * torch.randn(64, device="cuda", generator=g)
    return pb, q, idx, w2, s2, t2


def _edgeconv_run(pb, q, idx, w2p, t2, B, N, k, argmax):
    ops = _ops()
    y = torch.full((B, 64, N), float("nan"), device="cuda")
    act = ops.new_act(B * N, 2, "cuda")
    am = torch.full((B * N, 64), 255, dtype=torch.uint8, device="cuda") if argmax else None
    ops.edgeconv((pb, q), idx, w2p, t2, B, N, k, y_cm=y, y_act=act, y_act_kb=1, argmax=am)
    return y, act, am


def _edgeconv_ref_check(pb, q, idx, W, t2, y, am, b0, b1, N, tag):
    """The A operand rebuilt as the producers build it (edgeconv.cu:143-145): fp32 bf16(P' - mu) + (Q' + mu), LeakyReLU as
    max(v, 0.2f v), rounded to bf16 (pack_bf16x2: RN-even, as torch's .bfloat16()); so A is reproduced bit for bit and
    A . W2s is a sum of 64 exact products.  The tensor core accumulates them in fp32: 64 steps of at most one 2^-23 unit of
    the running sum of magnitudes give |h32 - h64| <= 64 * 2^-23 * sum|a||w|.  The max over k is 1-Lipschitz, so the max
    inherits the largest slot bound; + shift (one fp32 rounding) and LeakyReLU (0.2f != 0.2 and one rounding, 1-Lipschitz)
    add at most 2^-23 * (|max| + |shift|).  The arg-max may pick another slot only where the fp64 values of the two slots
    are within the sum of their bounds."""
    worst = 0.0
    for b in range(b0, b1):
        rows = slice(b * N, (b + 1) * N)
        v = pb[rows].float()[idx[b].long()] + q[rows][:, None, :]                # (N, k, 64) fp32
        a = torch.maximum(v, v * F32_02).bfloat16().double()
        h = a @ W.t()
        eh = 64 * U23 * (a.abs() @ W.abs().t())
        hmax, harg = h.max(dim=1)
        ref = F.leaky_relu(hmax + t2.double(), 0.2)
        bound = eh.max(dim=1).values + U23 * (hmax.abs() + t2.double().abs())
        err = (y[b].t().double() - ref).abs()
        ratio = float((err / bound).max())
        worst = max(worst, ratio)
        assert ratio <= 1, f"{tag} block {b}: |y - fp64| exceeds the fp32 accumulation bound by {ratio:.2f}x"
        if am is not None:
            got = am[rows].long()
            assert int(got.max()) < h.shape[1], f"{tag} block {b}: arg-max slot out of range"
            diff = got != harg
            gap = hmax - h.gather(1, got[:, None]).squeeze(1)
            allowed = eh.gather(1, harg[:, None]).squeeze(1) + eh.gather(1, got[:, None]).squeeze(1)
            assert bool((gap[diff] <= allowed[diff]).all()), \
                f"{tag} block {b}: {int(diff.sum())} arg-max slots differ, some not explained by fp32 near-ties"
    print(f"  {tag}: worst |y - fp64| / bound {worst:.3f}")


@pytest.mark.parametrize("B,N,k,argmax", [(32, 2048, 20, True), (32, 2048, 20, False), (8, 8192, 40, True),
                                          (32, 2048, EC_K_MAX, True), (61, 1000, 20, True)],
                         ids=["b32-n2048-k20-argmax", "b32-n2048-k20", "b8-n8192-k40", "b32-n2048-kmax", "b61-n1000-ragged"])
def test_edgeconv_rounds(B, N, k, argmax):
    ops = _ops()
    M = B * N
    plan = _plan_rowwise(f"edgeconv B={B} N={N} k={k} argmax={argmax}", -(-M // 128), _sms())   # edgeconv.cu:297-301
    plan.guard()
    pb, q, idx_wide, w2, s2, t2 = _edgeconv_inputs(B, N, k, seed=B * 100 + N + k)
    idx = idx_wide[:, :, :k].contiguous()
    w2p = ops.pack_weight(w2, s2)
    W = (w2 * s2[:, None]).bfloat16().double()
    if k == EC_K_MAX:
        assert k < 64, "the shared-memory check must cap k below the k <= 64 limit"
        # idx_wide has k + 1 valid columns, so even a launch that should have been refused reads only valid indices
        with pytest.raises(RuntimeError, match=rf"k={k + 1} needs \d+ bytes of shared memory"):
            _edgeconv_run(pb, q, idx_wide, w2p, t2, B, N, k + 1, argmax)
    y, act, am = _edgeconv_run(pb, q, idx, w2p, t2, B, N, k, argmax)
    assert torch.equal(_act_rows(act, M)[:, 64:], _cm_rows(y, 0, B).bfloat16()), "act output is not bf16(fp32 output)"
    assert float(_act_rows(act, M)[:, :64].abs().max()) == 0
    if argmax:
        y_plain, _, _ = _edgeconv_run(pb, q, idx, w2p, t2, B, N, k, False)
        assert torch.equal(y_plain, y), "the arg-max and plain variants disagree"
    # slices of whole blocks that start on a tile boundary, so that the 128-row tiles map one to one
    step = next(s for s in range(1, B + 1) if (s * N) % 128 == 0)
    if step == 1:
        slices = _block_slices(B)
    else:
        starts = list(range(0, B, step))
        slices = [(0, step), (starts[len(starts) // 2], starts[len(starts) // 2] + step), (starts[-1], B)]
    plan.check_slices([(b0 * N // 128, -(-b1 * N // 128)) for b0, b1 in slices])
    for b0, b1 in slices:
        tag = f"blocks [{b0}, {b1})"
        r0, r1 = b0 * N, b1 * N
        sy, sact, sam = _edgeconv_run(pb[r0:r1], q[r0:r1], idx[b0:b1], w2p, t2, b1 - b0, N, k, argmax)
        assert torch.equal(sy, y[b0:b1]), f"{tag}: fp32 output depends on where the tiles ran"
        assert torch.equal(sact, act[r0 // 128:-(-r1 // 128)]), f"{tag}: bf16 output depends on where the tiles ran"
        if argmax:
            assert torch.equal(sam, am[r0:r1]), f"{tag}: arg-max depends on where the tiles ran"
        _edgeconv_ref_check(pb, q, idx, W, t2, y, am, b0, b1, N, tag)


# ===================================================== attention =====================================================

def _attention_ref_check(dense, kb_q, y_rows, b0, b1, N, scale, tag):
    """fp64 softmax(q^T k * scale) v on the bf16 q, k, v the kernel reads.  Bound, per output element, with A = sum_j P_j |v_j|
    (P the exact probabilities):
      * the kernel's numerator takes the probabilities rounded to bf16 (the A operand of P.V) while its denominator l sums
        them unrounded in fp32: |sum_j (bf16(p_j) - p_j) v_j| / l <= 2^-8 A;
      * a relative perturbation eps of every weight p_j moves the normalised output by at most 2 eps A.  p_j = 2^arg_j with
        arg_j = s_j * scale * log2(e) - m, so an error d in arg_j is a relative error ln2 * d of p_j.  The score's fp32
        accumulation (64 exact products: 64 * 2^-23 * S, S = max_j sum_i |q_i||k_ji|) gives ln2 * log2(e) * scale * that
        = 64 * 2^-23 * scale * S; the fp32 scale constant, the max and the fma add at most 3 * 2^-23 * scale * S the same
        way; ex2.approx (a few ulp; 2^-20 is allowed) enters once for p and once for each of the T tile rescalings;
      * the fp32 sums: 128 products per P.V tile in TMEM, two roundings per tile of the register fold, 128 + T adds of l,
        the reciprocal and the final product: (136 + 3T) * 2^-23 * A;
      * p flushed to zero below 2^-126 (ex2.approx.ftz): at most N * 2^-126 * max|v|."""
    T = N // 128
    c = scale
    worst = 0.0
    for b in range(b0, b1):
        rows = dense[b * N:(b + 1) * N]
        qb, kb, vb = (rows[:, (kb_q + i) * 64:(kb_q + i + 1) * 64].double() for i in range(3))
        for r0 in range(0, N, 2048):                        # query chunks: the N x N fp64 matrices stay small
            qc = qb[r0:r0 + 2048]
            s = qc @ kb.t()
            p = torch.softmax(s * c, dim=1)
            ref = p @ vb
            A = p @ vb.abs()
            sabs = (qc.abs() @ kb.abs().t()).max(dim=1, keepdim=True).values
            eps = (64 + 3) * U23 * c * sabs + (T + 1) * 2.0 ** -20
            bound = (U8 * (1 + eps) + 2.1 * eps + (136 + 3 * T) * U23) * A + N * 2.0 ** -126 * vb.abs().max()
            err = (y_rows[b * N + r0:b * N + r0 + qc.shape[0]].double() - ref).abs()
            ratio = float((err / bound).max())
            worst = max(worst, ratio)
            assert ratio <= 1, f"{tag} block {b}: |y - fp64| exceeds the bf16-probability bound by {ratio:.2f}x"
    print(f"  {tag}: worst |y - fp64| / bound {worst:.3f}")
    return worst


@pytest.mark.parametrize("B,N,gain,kb_q,with_act", [(32, 2048, 1.0, 0, False), (32, 2048, 6.0, 0, False),
                                                    (8, 8192, 1.0, 0, False), (16, 4096, 1.0, 1, True)],
                         ids=["b32-n2048", "b32-n2048-peaked", "b8-n8192", "b16-n4096-kbq1-act"])
def test_attention_rounds(B, N, gain, kb_q, with_act):
    ops = _ops()
    M, T = B * N, N // 128
    # attention.cu:299-305: one item per (block, 128-query tile), items b * T + qt, grid min(items, SMs)
    plan = _plan_rowwise(f"attention B={B} N={N} gain={gain} kb_q={kb_q}", B * T, _sms())
    plan.guard()
    g = _gen(B * N + int(gain))
    kblocks = kb_q + 3 + (1 if kb_q else 0)
    act = ops.new_act(M, kblocks, "cuda")
    x = torch.randn(B, 192, N, device="cuda", generator=g)
    x[:, :128] *= gain                                                    # q and k: gain 6 gives a peaked softmax
    ops.cm_to_act(x, act, kb_q)
    for kb in set(range(kblocks)) - {kb_q, kb_q + 1, kb_q + 2}:           # neighbouring blocks the kernel must not read
        ops.cm_to_act(100 * torch.randn(B, 64, N, device="cuda", generator=g), act, kb)
    del x
    scale = 1.0 / 8.0

    def run(a, nb):
        y = torch.full((nb, 64, N), float("nan"), device="cuda")
        ya = ops.new_act(nb * N, 2, "cuda") if with_act else None
        ops.attention(a, kb_q, nb, N, scale, y_cm=y, y_act=ya, y_kb=1)
        return y, ya

    y, ya = run(act, B)
    if with_act:
        dense_y = _act_rows(ya, M)
        assert float(dense_y[:, :64].abs().max()) == 0
        assert torch.equal(dense_y[:, 64:], _cm_rows(y, 0, B).bfloat16()), "act output is not bf16(fp32 output)"
    slices = _block_slices(B)
    plan.check_slices([(b0 * T, b1 * T) for b0, b1 in slices])
    dense = _act_rows(act, M)
    y_rows = y.permute(0, 2, 1).reshape(M, 64)
    for b0, b1 in slices:
        tag = f"blocks [{b0}, {b1})"
        sy, sya = run(act[b0 * T:b1 * T], b1 - b0)
        assert torch.equal(sy, y[b0:b1]), f"{tag}: fp32 output depends on where the tiles ran"
        if with_act:
            assert torch.equal(sya, ya[b0 * T:b1 * T]), f"{tag}: bf16 output depends on where the tiles ran"
        _attention_ref_check(dense, kb_q, y_rows, b0, b1, N, scale, tag)


# ===================================================== GW projection =====================================================

@pytest.mark.parametrize("G", [150, 180])
def test_gw_project_tc_rounds(G):
    """gfs_gw_project_tc: assignments bit-identical to the all-fp32 kernel (near-ties are re-evaluated with its pinned fp32
    chain); softmax features within 1e-3 of fp64, the tolerance of test_gw_projection_tensor_core_equals_fp32_kernel (the
    bf16 hi/lo split gives fp32-grade cosines, 10 cos is then exponentiated with ex2.approx in fp32)"""
    ops = _ops()
    B, N, D = 32, 2048, 192
    M, T = B * N, N // 128
    plan = _plan_rowwise(f"gw_project_tc B={B} N={N} G={G}", M // 128, _sms())     # rowsel_tc.cu:543-549
    plan.guard()
    g = _gen(G)
    ec = torch.randn(B, D, N, device="cuda", generator=g).abs() * 0.3
    gp = torch.randn(G, D, device="cuda", generator=g)
    Gp = (G + 63) // 64 * 64
    gp_l2t = torch.zeros(D, Gp, device="cuda")
    gp_l2t[:, :G] = F.normalize(gp, dim=1).t()

    def run(e, impl):
        a = ops.new_act(e.shape[0] * N, Gp // 64 + 1, "cuda")
        assign, cm = ops.gw_project(e, gp_l2t, G, cosine_act=a, kb0=1, want_cm=True, impl=impl)
        return assign, cm, a

    assign, cm, cact = run(ec, "tc")
    assign32, _, _ = run(ec, "fp32")
    assert torch.equal(assign, assign32), f"{int((assign != assign32).sum())} assignments differ from the fp32 kernel"
    dense = _act_rows(cact, M)
    assert float(dense[:, :64].abs().max()) == 0 and float(dense[:, 64 + G:].abs().max()) == 0
    assert torch.equal(dense[:, 64:64 + G], _cm_rows(cm, 0, B).bfloat16()), "act output is not bf16(fp32 output)"
    slices = _block_slices(B)
    plan.check_slices([(b0 * T, b1 * T) for b0, b1 in slices])
    gpd = gp_l2t[:, :G].double()
    for b0, b1 in slices:
        tag = f"blocks [{b0}, {b1})"
        sa, scm, sact = run(ec[b0:b1], "tc")
        assert torch.equal(sa, assign[b0:b1]), f"{tag}: assignments depend on where the tiles ran"
        assert torch.equal(scm, cm[b0:b1]), f"{tag}: features depend on where the tiles ran"
        assert torch.equal(sact, cact[b0 * T:b1 * T]), f"{tag}: bf16 features depend on where the tiles ran"
        e = ec[b0:b1].double()
        cos = torch.einsum("dg,bdn->bgn", gpd, e) / e.norm(dim=1, keepdim=True).clamp_min(1e-12)
        ref = torch.softmax(10 * cos, dim=1)
        err = rel_err(cm[b0:b1], ref)
        print(f"  {tag}: features fp64 rel err {err:.2e} (bound 1e-3)")
        assert err <= 1e-3
