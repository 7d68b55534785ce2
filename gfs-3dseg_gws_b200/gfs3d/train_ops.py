"""torch.autograd.Functions of the training path over the C ABI (fp32, channel-major (C, M) tensors).

Reference semantics: model.train() (train.py:614) -- BatchNorm with batch statistics, LeakyReLU(0.2) / ReLU, max over k with
gradient to the arg-max edge, gather backward = scatter-add.  A BatchNorm whose module is in eval mode inside a training model
is frozen, as in torch: it normalises with its running statistics, which it leaves unchanged (see batch_stats).  Every
Function's forward AND backward run in the hand-written kernels of csrc/gemm_f32.cu + csrc/train.cu (+ csrc/knn.cu for the
graph, which is not differentiated, as in the reference where knn returns integer indices)."""
import torch

from . import ops

BN_EPS = 1e-5


def _exact():
    """GEMM implementation for products that feed a cancellation: never the single-pass tf32"""
    return "f32" if ops.TRAIN_GEMM == "f32" else "tf32x3"


def to_cm(x):
    """(B, C, N) -> (C, B*N) contiguous"""
    B, C, N = x.shape
    return x.permute(1, 0, 2).reshape(C, B * N).contiguous()


def from_cm(x, B, N):
    """(C, B*N) -> (B, C, N) contiguous"""
    C = x.shape[0]
    return x.reshape(C, B, N).permute(1, 0, 2).contiguous()


def batch_stats(bn):
    """torch's rule (nn.modules.batchnorm._BatchNorm.forward): a BatchNorm normalises with the statistics of the batch iff it is
    in training mode or keeps no running statistics; otherwise it is frozen"""
    return bn.training or bn.running_mean is None


def _bn_coeffs(z, gamma, beta, running_mean, running_var, training):
    if training:
        return ops.bn_stats_coeffs(z, gamma, beta, BN_EPS)           # mean, var, invstd, scale, shift in one call
    # copies: the Functions return mean / var as outputs, which must not alias the module's buffers
    mean, var = running_mean.detach().float().clone(), running_var.detach().float().clone()
    invstd = torch.rsqrt(var + BN_EPS)
    scale = (gamma * invstd).contiguous()
    shift = (beta - mean * scale).contiguous()
    return mean, var, invstd.contiguous(), scale, shift


class ConvBNAct(torch.autograd.Function):
    """y = act(BN(W x + bias)); x (I, M), W (O, I).  Returns (y, batch_mean, batch_var).
    training=False: BN with the running statistics (returned in place of the batch ones)."""

    @staticmethod
    def forward(ctx, x, W, bias, gamma, beta, running_mean, running_var, slope, training):
        x = x.contiguous()
        Wc = W.detach().contiguous().float()
        z = ops.conv_fwd(Wc, x, None if bias is None else bias.detach().contiguous().float())
        g, b = gamma.detach().contiguous().float(), beta.detach().contiguous().float()
        mean, var, invstd, scale, shift = _bn_coeffs(z, g, b, running_mean, running_var, training)
        y = ops.bn_act_fwd(z, scale, shift, slope)
        ctx.save_for_backward(x, Wc, z, mean, invstd, g, b)
        ctx.slope, ctx.training, ctx.has_bias = slope, training, bias is not None
        ctx.mark_non_differentiable(mean, var)
        return y, mean, var

    @staticmethod
    def backward(ctx, dy, _dm, _dv):
        x, W, z, mean, invstd, g, b = ctx.saved_tensors
        need = ctx.needs_input_grad
        bwd = ops.bn_act_bwd if ctx.training else ops.bn_act_bwd_frozen
        dz, sg, sgx = bwd(dy.contiguous(), z, mean, invstd, g, b, ctx.slope)
        dW = ops.conv_wgrad(dz, x) if need[1] else None
        dx = ops.conv_dgrad(W, dz) if need[0] else None
        dbias = dz.sum(dim=1) if ctx.has_bias and need[2] else None
        return dx, dW, dbias, sgx, sg, None, None, None, None


class ConvOnly(torch.autograd.Function):
    """z = W x (no bias / BN / activation): the q/k/v maps of model/attention.py:25-27"""

    @staticmethod
    def forward(ctx, x, W):
        x = x.contiguous()
        Wc = W.detach().contiguous().float()
        ctx.save_for_backward(x, Wc)
        return ops.conv_fwd(Wc, x)

    @staticmethod
    def backward(ctx, dz):
        x, W = ctx.saved_tensors
        dz = dz.contiguous()
        need = ctx.needs_input_grad
        return (ops.conv_dgrad(W, dz) if need[0] else None), (ops.conv_wgrad(dz, x) if need[1] else None)


class ConvConstW(torch.autograd.Function):
    """z = W x with a constant W (the L2-normalised GW basis, model/capl.py:345-346): data gradient only"""

    @staticmethod
    def forward(ctx, x, W):
        Wc = W.detach().contiguous().float()
        ctx.save_for_backward(Wc)
        return ops.conv_fwd(Wc, x.contiguous())

    @staticmethod
    def backward(ctx, dz):
        (W,) = ctx.saved_tensors
        return ops.conv_dgrad(W, dz.contiguous()), None


class EdgeConvTrain(torch.autograd.Function):
    """One EdgeConv block (model/dgcnn.py:35-41 + :53-58 + :118) in training mode.
    x (C, M) channel-major, idx (B, N, k) int32 -> (y (64, M), mean1, var1, mean2, var2).
    train1 / train2: BN1 / BN2 use batch statistics; False: that BN is frozen and normalises with (rm, rv), its running
    statistics, which are then returned as its mean / var."""

    @staticmethod
    def forward(ctx, x, idx, W1, g1, b1, W2, g2, b2, B, N, k, train1=True, rm1=None, rv1=None, train2=True, rm2=None, rv2=None):
        x = x.contiguous()
        C, M = x.shape
        W1f = W1.detach().float().reshape(64, 2 * C)
        Wa, Wb = W1f[:, :C], W1f[:, C:]
        Wpq = torch.cat([Wa, Wb - Wa], dim=0).contiguous()                          # (128, C): [P | Q] = Wpq x
        pq = torch.empty(M, 128, dtype=torch.float32, device=x.device)
        # fp32-grade products are REQUIRED here (and in the two matching backward GEMMs): H = P[j] + Q[i] is
        # W_a (x_j - x_i) + W_b x_i evaluated as a DIFFERENCE of per-point terms, so an operand rounding of 2^-11 |W_a x| (plain
        # tf32) would be of the order of the neighbour differences themselves
        ops.gemm_f32(Wpq, C, True, x, M, False, 128, M, C, pq, 128, c_trans=True, impl=_exact())   # point-major rows for the gather
        g1f, b1f, g2f, b2f = (t.detach().contiguous().float() for t in (g1, b1, g2, b2))
        if train1:
            # (64, E) pre-BN1 tensor and its batch statistics / BN coefficients in one pass (the tile is summed while on chip)
            H, (m1, v1, is1, sc1, sh1) = ops.edge_gather_stats(pq, idx, B, N, k, g1f, b1f, BN_EPS)
        else:
            H = ops.edge_gather(pq, idx, B, N, k)
            m1, v1, is1, sc1, sh1 = _bn_coeffs(H, g1f, b1f, rm1, rv1, False)
        del pq
        h1 = ops.bn_act_fwd(H, sc1, sh1, 0.2)
        W2f = W2.detach().float().reshape(64, 64).contiguous()
        Z = ops.conv_fwd(W2f, h1)                                                   # (64, E), pre-BN2
        m2, v2, is2, sc2, sh2 = _bn_coeffs(Z, g2f, b2f, rm2, rv2, train2)
        y, arg = ops.bn_act_max_fwd(Z, sc2, sh2, 0.2, M, k)                         # BN2 + LeakyReLU + max over k: one pass over Z
        ctx.save_for_backward(x, idx, Wpq, W2f, H, h1, Z, m1, is1, g1f, b1f, m2, is2, g2f, b2f, arg)
        ctx.dims = (B, N, k, C, M)
        ctx.train = (train1, train2)
        ctx.mark_non_differentiable(m1, v1, m2, v2)
        return y, m1, v1, m2, v2

    @staticmethod
    def backward(ctx, dy, *_):
        x, idx, Wpq, W2f, H, h1, Z, m1, is1, g1, b1, m2, is2, g2, b2, arg = ctx.saved_tensors
        B, N, k, C, M = ctx.dims
        train1, train2 = ctx.train
        need = ctx.needs_input_grad
        # dy lives at the arg-max edge only: BN2's backward reads (dy, arg) directly, the (64, E) sparse gradient is never built
        bwd2 = ops.bn_act_bwd_argmax if train2 else ops.bn_act_bwd_argmax_frozen
        dZ, sg2, sgx2 = bwd2(dy.contiguous(), arg, k, Z, m2, is2, g2, b2, 0.2)
        dW2 = ops.conv_wgrad(dZ, h1).reshape(64, 64, 1, 1) if need[5] else None
        dh1 = ops.conv_dgrad(W2f, dZ)
        del dZ
        # BN1 / LeakyReLU backward is applied inside the scatter while its tile is staged: dH (64, E) is never built
        sg1 = sgx1 = None
        if train1 or need[3] or need[4]:
            sg1, sgx1 = ops.bn_bwd_sums(dh1, H, m1, is1, g1, b1, 0.2)
        dx = dW1 = None
        if need[0] or need[2]:
            if train1:
                ag, agx = sg1, sgx1
            else:
                # frozen BN1: the scatter's apply step gamma*invstd*(g - sum_g/E - xhat*sum_gx/E) is exactly gamma*invstd*g when both
                # sums are zero (g - 0 - xhat*0 == g in fp32), which is the running-statistic backward
                ag = agx = torch.zeros(64, dtype=torch.float32, device=x.device)
            if torch.are_deterministic_algorithms_enabled():
                # reproducible bits: each dP row is summed in ascending edge order instead of by atomics (one (E, 64) buffer of
                # per-edge terms lives until the scatter returns)
                dpq = ops.edge_scatter_bn(dh1, H, idx, B, N, k, m1, is1, g1, b1, 0.2, ag, agx, ordered=True,
                                          rev=ops.edge_reverse_index(idx, B, N))
            else:
                dpq = ops.edge_scatter_bn(dh1, H, idx, B, N, k, m1, is1, g1, b1, 0.2, ag, agx)   # (M, 128): scatter-add over the graph
            del dh1
            if need[2]:
                dWpq = torch.empty(128, C, dtype=torch.float32, device=x.device)
                ops.gemm_f32(dpq, 128, False, x, M, True, 128, C, M, dWpq, C, splitk=ops._splitk(M), impl=_exact())
            if need[0]:
                dx = torch.empty(C, M, dtype=torch.float32, device=x.device)
                ops.gemm_f32(Wpq, C, False, dpq, 128, True, C, M, 128, dx, M, impl=_exact())
            if need[2]:
                dW1 = torch.cat([dWpq[:64] - dWpq[64:], dWpq[64:]], dim=1).reshape(64, 2 * C, 1, 1)
        return (dx, None, dW1, sgx1, sg1, dW2, sgx2, sg2) + (None,) * 9


class AttentionTrain(torch.autograd.Function):
    """model/attention.py:43-46 in training mode: y = dropout(softmax(q^T k * scale)) v^T, per block.
    qkv (192, M) channel-major [q | k | v]; dropout either as an explicit (B, N, N) mask already scaled by 1/(1-p) (tests) or as
    (seed, keep): the kernels derive keep / drop from a hash of (seed, row, column), forward and backward alike, so no mask tensor
    is drawn, stored or read."""

    @staticmethod
    def forward(ctx, qkv, B, N, scale, mask, seed=0, keep=1.0):
        qkv = qkv.contiguous()
        M = qkv.shape[1]
        q, kk, v = qkv[0:64], qkv[64:128], qkv[128:192]
        S = torch.empty(B, N, N, dtype=torch.float32, device=qkv.device)
        ops.gemm_f32(q, M, False, kk, M, False, N, N, 64, S, N, batch=B, a_bs=N, b_bs=N, c_bs=N * N)
        p0, p = ops.softmax_rows_fwd(S, scale, mask, seed, keep if mask is None else 1.0)
        del S
        y = torch.empty(64, M, dtype=torch.float32, device=qkv.device)
        ops.gemm_f32(v, M, True, p, N, True, 64, N, N, y, M, batch=B, a_bs=N, b_bs=N * N, c_bs=N)
        ctx.save_for_backward(qkv, p0, p, mask if mask is not None else torch.empty(0, device=qkv.device))
        ctx.dims = (B, N, scale, mask is not None, seed, keep if mask is None else 1.0)
        return y

    @staticmethod
    def backward(ctx, dy):
        qkv, p0, p, mask = ctx.saved_tensors
        B, N, scale, has_mask, seed, keep = ctx.dims
        M = qkv.shape[1]
        dy = dy.contiguous()
        q, kk, v = qkv[0:64], qkv[64:128], qkv[128:192]
        dqkv = torch.empty_like(qkv)
        # dV[c, key] = sum_q dY[c, q] P[q, key]
        ops.gemm_f32(dy, M, True, p, N, False, 64, N, N, dqkv[128:192], M, batch=B, a_bs=N, b_bs=N * N, c_bs=N)
        # dP[q, key] = sum_c dY[c, q] v[c, key]
        dP = torch.empty(B, N, N, dtype=torch.float32, device=qkv.device)
        ops.gemm_f32(dy, M, False, v, M, False, N, N, 64, dP, N, batch=B, a_bs=N, b_bs=N, c_bs=N * N)
        dS = ops.softmax_rows_bwd(p0, dP, scale, mask if has_mask else None, seed, keep)
        del dP
        # dQ[c, q] = sum_key dS[q, key] k[c, key];   dK[c, key] = sum_q dS[q, key] q[c, q]
        ops.gemm_f32(kk, M, True, dS, N, True, 64, N, N, dqkv[0:64], M, batch=B, a_bs=N, b_bs=N * N, c_bs=N)
        ops.gemm_f32(q, M, True, dS, N, False, 64, N, N, dqkv[64:128], M, batch=B, a_bs=N, b_bs=N * N, c_bs=N)
        return dqkv, None, None, None, None, None, None


class ClassSums(torch.autograd.Function):
    """sums[c, :] = sum of the rows of X (n, D) whose label is c, and the label counts -- the per-class masked sums of
    model/capl.py:398-401 (generate_fake_proto) for ALL classes in one deterministic pass (gfs_kmeans_accumulate: per-CTA fp32
    partials, fp64 reduction in a fixed order) instead of one (mask, multiply, two reductions) chain per class.
    Backward: dX[row] = dSums[label[row]]."""

    @staticmethod
    def forward(ctx, X, labels, K):
        X = X.contiguous()
        labels = labels.to(torch.int32).contiguous()
        sums, counts = ops.kmeans_accumulate(X, labels, K)
        ctx.save_for_backward(labels)
        ctx.mark_non_differentiable(counts)
        return sums.float(), counts

    @staticmethod
    def backward(ctx, dsums, _dcounts):
        (labels,) = ctx.saved_tensors
        return dsums.index_select(0, labels.long()), None, None


def update_running_stats(bn, mean, var, n):
    """nn.BatchNorm semantics: momentum 0.1 (or cumulative when None), unbiased variance for running_var"""
    with torch.no_grad():
        if (bn.momentum is not None and bn.running_mean.is_cuda and bn.running_mean.dtype == torch.float32
                and bn.running_var.dtype == torch.float32 and bn.num_batches_tracked.dtype == torch.int64):
            # one launch for both buffers.  The counter is incremented by torch: that in-place op bumps its version counter,
            # which is what invalidates the folded-weight caches of the inference path (keyed on tensor._version)
            ops.bn_update_running(mean, var, n, bn.momentum, bn.running_mean, bn.running_var, None)
            bn.num_batches_tracked += 1
            return
        bn.num_batches_tracked += 1
        mom = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
        bn.running_mean.mul_(1 - mom).add_(mean.to(bn.running_mean.dtype), alpha=mom)
        bn.running_var.mul_(1 - mom).add_((var * (n / max(n - 1, 1))).to(bn.running_var.dtype), alpha=mom)
