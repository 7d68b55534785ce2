"""Thin torch-facing wrappers over the C ABI: allocate outputs as torch tensors, pass raw device pointers and the
current CUDA stream.  No arithmetic happens here."""
import os
from typing import Optional

import torch

from ._lib import check, lib

ACT_NONE, ACT_LRELU02, ACT_RELU = 0, 1, 2


# ---- launch accounting / optional per-call CUDA-event timing (bench.py's roofline leg) ----
LAUNCHES = 0            # kernels launched through the C ABI since import (each entry point launches a fixed number)
PROFILE_SHAPES = False  # add the GEMM shape to the profile key
PROFILE = None          # set to {} to record (name, start_event, end_event) per call on the current stream


class _StreamArg:
    """placeholder for the stream argument: _call substitutes the current stream OF THE TENSORS' DEVICE"""


_STREAM = _StreamArg()
_SEEN_DEVICES = []      # devices of the tensors whose pointers were taken since the last launch


def _call(name: str, n_kernels: int, *args, tag: str = ""):
    """One C-ABI call.  The launch follows the tensors, not the ambient device: every tensor of the call must live on one
    CUDA device; the library call runs under that device's context and on that device's current stream (a model moved with
    .to('cuda:1') works without torch.cuda.set_device(1), as the reference's torch ops do)."""
    global LAUNCHES
    devs = set(_SEEN_DEVICES)
    _SEEN_DEVICES.clear()
    if len(devs) > 1:
        raise RuntimeError(f"{name}: tensors live on different devices {sorted(str(d) for d in devs)}")
    dev = devs.pop() if devs else torch.device("cuda", torch.cuda.current_device())
    fn = getattr(lib(), name)
    with torch.cuda.device(dev):
        args = tuple(torch.cuda.current_stream(dev).cuda_stream if a is _STREAM else a for a in args)
        if PROFILE is None:
            rc = fn(*args)
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*args)
            e1.record()
            PROFILE.setdefault(name + tag, []).append((e0, e1))
    LAUNCHES += n_kernels
    check(rc, name)


def _ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("gfs3d ops need CUDA tensors: the hot path has no CPU fallback")
    _SEEN_DEVICES.append(t.device)
    return t.data_ptr()


def _stream():
    return _STREAM


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("gfs3d ops need CUDA tensors: the hot path has no CPU fallback")


def act_rows(M: int) -> int:
    return (M + 127) // 128 * 128


def new_act(M: int, kblocks: int, device, zero: bool = True) -> torch.Tensor:
    """bf16 activation matrix in the tiled SWIZZLE_128B layout: [M/128][kblocks] tiles of 16 KiB.  zero=False skips the
    memset when the caller's kernels overwrite every block (padding rows are still zeroed: they must not hold NaN/Inf)."""
    alloc = torch.empty if (not zero and M % 128 == 0) else torch.zeros
    return alloc(act_rows(M) // 128, kblocks, 128 * 64, dtype=torch.bfloat16, device=device)


def act_to_dense(act: torch.Tensor, M: int) -> torch.Tensor:
    """(debug / tests) undo the tiled swizzled layout -> (M, kblocks*64) bf16 row-major"""
    mt, kb, _ = act.shape
    t = act.view(mt, kb, 128, 8, 8)
    r = torch.arange(128, device=act.device).view(128, 1)
    q = torch.arange(8, device=act.device).view(1, 8)
    src = (q ^ (r & 7)).view(1, 1, 128, 8, 1).expand(mt, kb, 128, 8, 8)
    dense = torch.gather(t, 3, src)                       # chunk q of row r lives at position q ^ (r & 7)
    return dense.permute(0, 2, 1, 3, 4).reshape(mt * 128, kb * 64)[:M]


KNN_IMPL = os.environ.get("GFS3D_KNN", "auto")   # "auto" | "tc" | "exact": both are CUDA and return identical bits


def knn_tc_eligible(C: int, N: int, k: int) -> bool:
    return k <= 40 and C <= 64 and N <= 65535 and N % 4 == 0


def knn(x: torch.Tensor, k: int, return_dist: bool = False, impl: Optional[str] = None, ordered: bool = True):
    """x: (B, C, N) fp32 view with unit point stride and channel stride N -> idx (B, N, k) int32

    impl "tc": tensor-core filter + exact finish (gfs_knn_tc_f32); "exact": the all-fp32 kernel (gfs_knn_f32);
    "auto": tc whenever the shape is eligible.  The two produce the same indices and distances bit for bit.
    ordered=False (tc only): the same k neighbours per row in no particular order (gfs_knn_tc_set_f32) -- enough for a
    max over the neighbours, and cheaper: only candidates the error bounds cannot decide get the exact arithmetic."""
    _need_cuda(x)
    B, C, N = x.shape
    assert x.dtype == torch.float32 and x.stride(2) == 1 and x.stride(1) == N, "x must be channel-major"
    impl = impl or KNN_IMPL
    sq = torch.empty(B, N, dtype=torch.float32, device=x.device)
    idx = torch.empty(B, N, k, dtype=torch.int32, device=x.device)
    dist = torch.empty(B, N, k, dtype=torch.float32, device=x.device) if return_dist else None
    if impl == "tc" or (impl == "auto" and knn_tc_eligible(C, N, k)):
        nbytes = int(lib().gfs_knn_tc_workspace_bytes(B, C, N))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            nk = 4 * int(lib().gfs_knn_tc_chains(B, C, N))     # prepare, filter, finish, repair per chain (one or two chains)
        if ordered or return_dist:
            _call("gfs_knn_tc_f32", nk, _ptr(x), x.stride(0), B, C, N, k, _ptr(sq), _ptr(ws), nbytes, _ptr(idx), _ptr(dist),
                  _stream())
        else:
            _call("gfs_knn_tc_set_f32", nk, _ptr(x), x.stride(0), B, C, N, k, _ptr(sq), _ptr(ws), nbytes, _ptr(idx), _stream())
    else:
        _call("gfs_knn_f32", 2, _ptr(x), x.stride(0), B, C, N, k, _ptr(sq), _ptr(idx), _ptr(dist), _stream())
    return (idx, dist) if return_dist else idx


def knn_tc_diag(x: torch.Tensor, k: int):
    """(tests) tc kNN + what its filter saw: returns idx (B,N,k), filter (B,N,Npad) ~ x_i.x_j - |x_j|^2/2, flags (B, ceil(N/64))"""
    _need_cuda(x)
    B, C, N = x.shape
    assert x.dtype == torch.float32 and x.stride(2) == 1 and x.stride(1) == N
    npad = (N + 255) // 256 * 256
    sq = torch.empty(B, N, dtype=torch.float32, device=x.device)
    idx = torch.empty(B, N, k, dtype=torch.int32, device=x.device)
    filt = torch.zeros(B, N, npad, dtype=torch.float32, device=x.device)
    flags = torch.empty(B, (N + 63) // 64, dtype=torch.int32, device=x.device)
    nbytes = int(lib().gfs_knn_tc_workspace_bytes(B, C, N))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    _call("gfs_knn_tc_diag_f32", 4, _ptr(x), x.stride(0), B, C, N, k, _ptr(sq), _ptr(ws), nbytes, _ptr(idx), _ptr(filt),
          _ptr(flags), _stream())
    return idx, filt, flags


def pointwise(x: torch.Tensor, wt: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """x (B,C,N) cm fp32, wt (C,O) fp32 -> (B*N, O) fp32"""
    _need_cuda(x, wt, bias)
    B, C, N = x.shape
    assert x.stride(2) == 1 and x.stride(1) == N and wt.is_contiguous() and wt.shape[0] == C
    O = wt.shape[1]
    out = torch.empty(B * N, O, dtype=torch.float32, device=x.device)
    _call("gfs_pointwise_f32", 1, _ptr(x), x.stride(0), B, C, N, _ptr(wt), _ptr(bias), O, _ptr(out), _stream())
    return out


def edge_pq(x: torch.Tensor, wt: torch.Tensor, bias: Optional[torch.Tensor]):
    """split first EdgeConv conv: x (B,C,N) cm fp32, wt (C,128) = [s1*Wa | s1*(Wb-Wa)]^T, bias (128) ->
    pb (B*N, 64) bf16 = P' - mu,  q (B*N, 64) fp32 = Q' + mu   (what gfs_edgeconv_fwd gathers from)"""
    _need_cuda(x, wt, bias)
    B, C, N = x.shape
    assert x.stride(2) == 1 and x.stride(1) == N and wt.is_contiguous() and wt.shape == (C, 128)
    pb = torch.empty(B * N, 64, dtype=torch.bfloat16, device=x.device)
    q = torch.empty(B * N, 64, dtype=torch.float32, device=x.device)
    _call("gfs_edge_pq_f32", 1, _ptr(x), x.stride(0), B, C, N, _ptr(wt), _ptr(bias), _ptr(pb), _ptr(q), _stream())
    return pb, q


def pack_weight(w: torch.Tensor, row_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """w (R, K) fp32 -> bf16 tiles [ceil(K/64)][R x 64], K-major SWIZZLE_128B, optional per-row scale folded in"""
    _need_cuda(w, row_scale)
    w = w.contiguous().float()
    R, K = w.shape
    kb = (K + 63) // 64
    out = torch.empty(kb, R * 64, dtype=torch.bfloat16, device=w.device)
    rs = None if row_scale is None else row_scale.contiguous().float()
    _call("gfs_pack_weight_bf16", 1, _ptr(w), _ptr(rs), R, K, _ptr(out), _stream())
    return out


def cm_to_act(x: torch.Tensor, act: torch.Tensor, kb0: int):
    _need_cuda(x, act)
    B, C, N = x.shape
    assert x.stride(2) == 1 and x.stride(1) == N
    _call("gfs_cm_to_act", 1, _ptr(x), x.stride(0), B, C, N, _ptr(act), act.shape[1], kb0, _stream())


def edgeconv(pbq, idx, w2_packed, shift2, B, N, k, y_cm=None, y_act=None, y_act_kb=0, y_act2=None, y_act2_kb=0,
             argmax=None):
    """fused EdgeConv given the graph; writes into the provided destinations"""
    pb, q = pbq                     # from edge_pq
    _need_cuda(pb, q, idx, w2_packed, shift2)
    if y_cm is not None:
        assert y_cm.stride(2) == 1 and y_cm.stride(1) == N and y_cm.shape[1] == 64
    _call("gfs_edgeconv_fwd", 1, 
        _ptr(pb), _ptr(q), _ptr(idx), _ptr(w2_packed), _ptr(shift2), B, N, k,
        _ptr(y_cm), 0 if y_cm is None else y_cm.stride(0),
        _ptr(y_act), 0 if y_act is None else y_act.shape[1], y_act_kb,
        _ptr(y_act2), 0 if y_act2 is None else y_act2.shape[1], y_act2_kb,
        _ptr(argmax), _stream())


def linear(x_act: torch.Tensor, x_kb0: int, kb_count: int, w_packed: torch.Tensor, shift: Optional[torch.Tensor],
           nout: int, act: int, B: int, N: int, y_act: Optional[torch.Tensor] = None, y_kb0: int = 0,
           y_cm: Optional[torch.Tensor] = None):
    """Y = act(X . Wp^T + shift) on tcgen05; X / Y bf16 act tiles, optional fp32 channel-major copy of Y"""
    _need_cuda(x_act, w_packed, shift, y_act, y_cm)
    if y_cm is not None:
        assert y_cm.stride(2) == 1 and y_cm.stride(1) == N and y_cm.shape[1] == nout
    _call("gfs_linear_bf16", 1, 
        _ptr(x_act), x_act.shape[1], x_kb0, kb_count, _ptr(w_packed), _ptr(shift), nout, act, B, N,
        _ptr(y_act), 0 if y_act is None else y_act.shape[1], y_kb0,
        _ptr(y_cm), 0 if y_cm is None else y_cm.stride(0), _stream())


def attention(qkv_act: torch.Tensor, kb_q: int, B: int, N: int, scale: float, y_cm: Optional[torch.Tensor] = None,
              y_act: Optional[torch.Tensor] = None, y_kb: int = 0):
    """flash-style softmax(q^T k * scale) v on tcgen05; q/k/v are three 64-column blocks of one bf16 act matrix"""
    _need_cuda(qkv_act, y_cm, y_act)
    if y_cm is not None:
        assert y_cm.stride(2) == 1 and y_cm.stride(1) == N and y_cm.shape[1] == 64
    _call("gfs_attention_fwd", 1, _ptr(qkv_act), qkv_act.shape[1], kb_q, B, N, float(scale), _ptr(y_cm),
          0 if y_cm is None else y_cm.stride(0), _ptr(y_act), 0 if y_act is None else y_act.shape[1], y_kb, _stream())


ROWSEL_IMPL = os.environ.get("GFS3D_ROWSEL", "auto")   # "auto" | "tc" | "fp32": identical assignments / labels
ROWSEL_TC_MAXK = 512      # dictionary width of the tensor-core path (> 192: panelled); the fp32 kernels stop at 192


def gw_project(ec: torch.Tensor, gp_l2t: torch.Tensor, G: int, cosine_act: Optional[torch.Tensor] = None, kb0: int = 0,
               want_cm: bool = False, impl: Optional[str] = None):
    """ec (B, D, N) cm fp32; gp_l2t (D, Gp) -> assignment (B, N) int32 [, cosine_feat (B, G, N) fp32]

    impl "tc": tcgen05 product + pinned fp32 re-check of near-ties (gfs_gw_project_tc); "fp32": the all-fp32 kernel
    (gfs_gw_project, Gp <= 192); "auto": tc whenever the shape is eligible (Gp <= 512).  The assignments are identical."""
    _need_cuda(ec, gp_l2t, cosine_act)
    B, D, N = ec.shape
    assert ec.stride(2) == 1 and ec.stride(1) == N and gp_l2t.is_contiguous() and gp_l2t.shape[0] == D
    Gp = gp_l2t.shape[1]
    assign = torch.empty(B, N, dtype=torch.int32, device=ec.device)
    cm = torch.empty(B, G, N, dtype=torch.float32, device=ec.device) if want_cm else None
    impl = impl or ROWSEL_IMPL
    if impl == "tc" or (impl == "auto" and D % 64 == 0 and D <= 192 and N % 128 == 0 and Gp <= ROWSEL_TC_MAXK and Gp % 64 == 0):
        nbytes = int(lib().gfs_rowsel_tc_workspace_bytes_kp(B * N, D, Gp, 1))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=ec.device)
        _call("gfs_gw_project_tc", 4, _ptr(ec), ec.stride(0), B, D, N, _ptr(gp_l2t), G, Gp, _ptr(cosine_act),
              0 if cosine_act is None else cosine_act.shape[1], kb0, _ptr(cm), _ptr(assign), _ptr(ws), nbytes, _stream())
    else:
        _call("gfs_gw_project", 1, _ptr(ec), ec.stride(0), B, D, N, _ptr(gp_l2t), G, Gp, _ptr(cosine_act),
                                   0 if cosine_act is None else cosine_act.shape[1], kb0, _ptr(cm), _ptr(assign), _stream())
    return assign, cm


def cos_logits(feat: torch.Tensor, proto_l2: torch.Tensor, coding: Optional[torch.Tensor] = None,
               assignment: Optional[torch.Tensor] = None, th: float = 1.0) -> torch.Tensor:
    """feat (B, D, N) cm fp32; proto_l2 (CLS, D) or (B, CLS, D), already L2-normalised -> logits (B, CLS, N)"""
    _need_cuda(feat, proto_l2, coding, assignment)
    B, D, N = feat.shape
    assert feat.stride(2) == 1 and feat.stride(1) == N
    proto_l2 = proto_l2.contiguous().float()
    PB = 1 if proto_l2.dim() == 2 else proto_l2.shape[0]
    CLS = proto_l2.shape[-2]
    out = torch.empty(B, CLS, N, dtype=torch.float32, device=feat.device)
    G = 0
    if coding is not None:
        coding = coding.contiguous().float()
        G = coding.shape[1]
        assert coding.shape[0] == CLS and assignment is not None and assignment.dtype == torch.int32
    _call("gfs_cos_logits", 1, _ptr(feat), feat.stride(0), B, D, N, _ptr(proto_l2), PB, CLS, _ptr(coding), G,
                               _ptr(assignment), float(th), _ptr(out), _stream())
    return out


def refine_proto(pred_proto: torch.Tensor, proto: torch.Tensor, gened: torch.Tensor, base_num: int) -> torch.Tensor:
    """(B, CLS, D) pooled prototypes, (CLS, D) main and generated prototypes -> L2-normalised refined prototypes (B, CLS, D)"""
    _need_cuda(pred_proto, proto, gened)
    B, CLS, D = pred_proto.shape
    pp, q, g = pred_proto.contiguous().float(), proto.contiguous().float(), gened.contiguous().float()
    assert q.shape == (CLS, D) and g.shape == (CLS, D)
    out = torch.empty(B, CLS, D, dtype=torch.float32, device=pp.device)
    _call("gfs_refine_proto", 1, _ptr(pp), _ptr(q), _ptr(g), B, CLS, D, int(base_num), _ptr(out), _stream())
    return out


JOINT_HISTOGRAM_MAXBINS = 12288   # na * nb of one gfs_joint_histogram_i32 call


def joint_histogram(a: torch.Tensor, b: torch.Tensor, na: int, nb: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """counts[x, y] (+)= #{i: a[i] == x and b[i] == y} as int64 (na, nb); labels outside the ranges are skipped.
    a, b: integer CUDA tensors of equal numel (converted to int32 if needed); `out` accumulates across calls."""
    _need_cuda(a, b, out)
    assert a.numel() == b.numel(), "label streams differ in length"
    a32 = a.reshape(-1).to(torch.int32).contiguous()
    b32 = b.reshape(-1).to(torch.int32).contiguous()
    if out is None:
        out = torch.zeros(na, nb, dtype=torch.int64, device=a.device)
    assert out.dtype == torch.int64 and out.shape == (na, nb) and out.is_contiguous()
    if a32.numel() == 0:
        return out
    _call("gfs_joint_histogram_i32", 1, _ptr(a32), _ptr(b32), a32.numel(), na, nb, _ptr(out), _stream())
    return out


def softmax_pool(logits: torch.Tensor, feat: torch.Tensor) -> torch.Tensor:
    """sum_n softmax_n(logits[b,c,:]) * feat[b,:,n] -> (B, CLS, D)"""
    _need_cuda(logits, feat)
    B, CLS, N = logits.shape
    D = feat.shape[1]
    assert logits.is_contiguous() and feat.stride(2) == 1 and feat.stride(1) == N
    dev = feat.device
    stats = torch.empty(B * CLS * 2, dtype=torch.float32, device=dev)
    partial = torch.empty(B * ((N + 63) // 64) * CLS * D, dtype=torch.float32, device=dev)
    out = torch.empty(B, CLS, D, dtype=torch.float32, device=dev)
    _call("gfs_softmax_pool", 3, _ptr(logits), _ptr(feat), feat.stride(0), B, CLS, D, N, _ptr(stats), _ptr(partial),
                                 _ptr(out), _stream())
    return out


def kmeans_pp_trial(xt: torch.Tensor, n: int, xsq: torch.Tensor, cand: torch.Tensor, closest: Optional[torch.Tensor],
                    m_out: torch.Tensor, pots: torch.Tensor, weights: Optional[torch.Tensor] = None):
    """k-means++ step: xt (D, npad) channel-major, xsq (n) fp64, cand (T, D) -> m_out (T, npad) = min(d(x, cand_t), closest),
    pots (T) f64 (+)= sum_i weights[i] * m_out[t, i] (weights (n) fp32, None = 1)"""
    _need_cuda(xt, xsq, cand, closest, m_out, pots, weights)
    D, npad = xt.shape
    T = cand.shape[0]
    assert xt.is_contiguous() and cand.is_contiguous() and cand.shape[1] == D and m_out.is_contiguous() and m_out.shape[1] == npad
    assert m_out.shape[0] >= T and pots.dtype == torch.float64 and pots.numel() >= T and xsq.numel() >= n and xsq.dtype == torch.float64
    assert weights is None or (weights.dtype == torch.float32 and weights.is_contiguous() and weights.numel() >= n)
    _call("gfs_kmeans_pp_trial", 1, _ptr(xt), npad, n, D, _ptr(xsq), _ptr(cand), T, _ptr(closest), _ptr(weights), _ptr(m_out),
          _ptr(pots), _stream())


def kmeans_assign(xt: torch.Tensor, centers_t: torch.Tensor, K: int, want_score: bool = False, impl: Optional[str] = None):
    """xt (D, n) fp32, centers_t (D, Kp) fp32 zero padded -> labels (n) int32

    impl "tc": tcgen05 product + pinned fp32 re-check of near-ties (gfs_kmeans_assign_tc); "fp32": gfs_kmeans_assign;
    "auto": tc when the shape is eligible (Kp <= 512) and no scores are requested; "fp32" and scores stop at Kp = 192.
    The labels are identical."""
    _need_cuda(xt, centers_t)
    D, n = xt.shape
    assert xt.is_contiguous() and centers_t.is_contiguous() and centers_t.shape[0] == D
    Kp = centers_t.shape[1]
    cnorm = torch.empty(Kp, dtype=torch.float32, device=xt.device)
    labels = torch.empty(n, dtype=torch.int32, device=xt.device)
    score = torch.empty(n, dtype=torch.float32, device=xt.device) if want_score else None
    impl = impl or ROWSEL_IMPL
    if (impl == "tc" or (impl == "auto" and D % 64 == 0 and D <= 192 and Kp <= ROWSEL_TC_MAXK)) and not want_score:
        nbytes = int(lib().gfs_rowsel_tc_workspace_bytes_kp(n, D, Kp, 0))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=xt.device)
        _call("gfs_kmeans_assign_tc", 6, _ptr(xt), n, n, 0, D, _ptr(centers_t), K, Kp, _ptr(cnorm), _ptr(labels), _ptr(ws), nbytes, _stream())
    else:
        _call("gfs_kmeans_assign", 2, _ptr(xt), n, D, _ptr(centers_t), K, Kp, _ptr(cnorm), _ptr(labels), _ptr(score), _stream())
    return (labels, score) if want_score else labels


def kmeans_assign_rows(X: torch.Tensor, centers_t: torch.Tensor, K: int) -> torch.Tensor:
    """X (n, D) fp32 ROW-major (the M-step's layout), centers_t (D, Kp) -> labels (n) int32 through gfs_kmeans_assign_tc: a
    128-point tile is one contiguous piece of HBM.  Same labels as kmeans_assign on the transposed copy."""
    _need_cuda(X, centers_t)
    n, D = X.shape
    assert X.is_contiguous() and centers_t.is_contiguous() and centers_t.shape[0] == D
    Kp = centers_t.shape[1]
    cnorm = torch.empty(Kp, dtype=torch.float32, device=X.device)
    labels = torch.empty(n, dtype=torch.int32, device=X.device)
    nbytes = int(lib().gfs_rowsel_tc_workspace_bytes_kp(n, D, Kp, 0))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=X.device)
    _call("gfs_kmeans_assign_tc", 6, _ptr(X), n, D, 1, D, _ptr(centers_t), K, Kp, _ptr(cnorm), _ptr(labels), _ptr(ws), nbytes, _stream())
    return labels


def kmeans_accumulate(X: torch.Tensor, labels: torch.Tensor, K: int, n_valid: Optional[int] = None, sums=None, counts=None, ws=None):
    """X (n, D) fp32 row-major, labels (n) int32 -> sums (K, D) fp64, counts (K) int64 (deterministic).
    sums / counts / ws = (partial, pcount): optional preallocated outputs and workspaces (the Lloyd loop reuses them)"""
    _need_cuda(X, labels)
    n, D = X.shape
    if n_valid is not None:
        n = n_valid
    assert X.is_contiguous() and labels.dtype == torch.int32
    if ws is None:
        ws = kmeans_accumulate_workspace(K, D, X.device)
    partial, pcount = ws
    if sums is None:
        sums = torch.empty(K, D, dtype=torch.float64, device=X.device)
    if counts is None:
        counts = torch.empty(K, dtype=torch.int64, device=X.device)
    assert sums.dtype == torch.float64 and sums.is_contiguous() and counts.dtype == torch.int64
    _call("gfs_kmeans_accumulate", 2, _ptr(X), n, D, _ptr(labels), K, _ptr(partial), _ptr(pcount), _ptr(sums), _ptr(counts),
                                      _stream())
    return sums, counts


def kmeans_accumulate_workspace(K: int, D: int, device):
    """(partial (P*K*D) fp32, pcount (P*K) int32) for the P point ranges of gfs_kmeans_accumulate's grid"""
    P = lib().gfs_kmeans_accumulate_ranges(K, D, 0)
    return (torch.empty(P * K * D, dtype=torch.float32, device=device), torch.empty(P * K, dtype=torch.int32, device=device))


def kmeans_accumulate_weighted(X: torch.Tensor, labels: torch.Tensor, weights: torch.Tensor, K: int, n_valid: Optional[int] = None,
                               sums=None, wsums=None, ws=None):
    """X (n, D) fp32 row-major, labels (n) int32, weights (n) fp32 -> sums (K, D) fp64 of x * w, wsums (K) fp64 of w
    (deterministic; weights of 1 give kmeans_accumulate's sums bit for bit).  ws = (partial, pweight) from
    kmeans_accumulate_weighted_workspace; wsums may be a view of the packed buffer's weight slot."""
    _need_cuda(X, labels, weights)
    n, D = X.shape
    if n_valid is not None:
        n = n_valid
    assert X.is_contiguous() and labels.dtype == torch.int32 and weights.dtype == torch.float32 and weights.is_contiguous()
    assert weights.numel() >= n
    if ws is None:
        ws = kmeans_accumulate_weighted_workspace(K, D, X.device)
    partial, pweight = ws
    if sums is None:
        sums = torch.empty(K, D, dtype=torch.float64, device=X.device)
    if wsums is None:
        wsums = torch.empty(K, dtype=torch.float64, device=X.device)
    assert sums.dtype == torch.float64 and sums.is_contiguous() and wsums.dtype == torch.float64 and wsums.is_contiguous()
    _call("gfs_kmeans_accumulate_weighted", 2, _ptr(X), n, D, _ptr(labels), _ptr(weights), K, _ptr(partial), _ptr(pweight),
          _ptr(sums), _ptr(wsums), _stream())
    return sums, wsums


def kmeans_accumulate_weighted_workspace(K: int, D: int, device):
    P = lib().gfs_kmeans_accumulate_ranges(K, D, 1)
    return (torch.empty(P * K * D, dtype=torch.float32, device=device), torch.empty(P * K, dtype=torch.float64, device=device))


def kmeans_inertia(X: torch.Tensor, labels: torch.Tensor, centers: torch.Tensor, weights: Optional[torch.Tensor] = None,
                   n_valid: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """X (n, D) fp32 row-major, labels (n) int32, centers (K, D) fp32, weights (n) fp32 or None -> (1,) fp64 on the device:
    sum_i w_i |x_i - c_{label_i}|^2 (fp32 distance chain as sklearn's, fp64 sum in a fixed order)"""
    _need_cuda(X, labels, centers, weights)
    n, D = X.shape
    if n_valid is not None:
        n = n_valid
    K = centers.shape[0]
    assert X.is_contiguous() and centers.is_contiguous() and centers.shape[1] == D and labels.dtype == torch.int32
    assert labels.numel() >= n and (weights is None or (weights.dtype == torch.float32 and weights.is_contiguous() and weights.numel() >= n))
    partial = torch.empty(lib().gfs_kmeans_inertia_partials(), dtype=torch.float64, device=X.device)
    if out is None:
        out = torch.empty(1, dtype=torch.float64, device=X.device)
    _call("gfs_kmeans_inertia", 2, _ptr(X), n, D, _ptr(labels), _ptr(centers), K, _ptr(weights), _ptr(partial), _ptr(out), _stream())
    return out


def kmeans_pack(labels, labels_old, n, K, D, packed, scratch, counts=None):
    """packed[-1] = #(labels != labels_old) over the first n; packed[:K*D] are the sums already.  packed[K*D:K*D+K] (the weight
    sums) = counts (K) int64, or, with counts None, the fp64 weight sums kmeans_accumulate_weighted wrote there"""
    _need_cuda(labels, labels_old, counts, packed, scratch)
    assert packed.dtype == torch.float64 and packed.numel() == K * D + K + 1 and scratch.numel() * scratch.element_size() >= 16
    _call("gfs_kmeans_pack", 1, _ptr(labels), _ptr(labels_old), n, _ptr(counts), K, D, _ptr(packed), _ptr(scratch), _stream())


def kmeans_update(packed, centers_old, K, D, Kp, centers_new, ct, result):
    """new centres (K, D) = sums / weight sums, their transpose ct (D, Kp) and result = [changed, shift, empty] from the
    (all-reduced) packed buffer"""
    _need_cuda(packed, centers_old, centers_new, ct, result)
    assert centers_old.is_contiguous() and centers_new.is_contiguous() and ct.is_contiguous() and result.dtype == torch.float64
    _call("gfs_kmeans_update", 1, _ptr(packed), _ptr(centers_old), K, D, Kp, _ptr(centers_new), _ptr(ct), _ptr(result), _stream())


# =====================================================================================================================
# training path: raw wrappers (fp32, channel-major (C, M) 2-D tensors)
# =====================================================================================================================
# the training path's GEMMs (csrc/gemm_tf32.cu, csrc/gemm_f32.cu):
#   "tf32x3" tcgen05 kind::tf32 with hi/lo operand pairs (3 MMAs per k-step): fp32-grade products on the tensor pipe (default)
#   "tf32"   one tf32 product per k-step: 2^-10 relative; fine for a forward pass, too coarse for the backward (branch flips)
#   "f32"    packed-FFMA2 CUDA cores
TRAIN_GEMM = os.environ.get("GFS_TRAIN_GEMM", "tf32x3")


def gemm_f32(A, lda, a_trans, B, ldb, b_trans, R, Ncols, K, C, ldc, c_trans=False, bias=None, batch=1, a_bs=0, b_bs=0, c_bs=0,
             splitk=1, accumulate=False, impl=None):
    _need_cuda(A, B, C, bias)
    impl = impl or TRAIN_GEMM
    if impl not in ("tf32x3", "tf32", "f32"):
        raise ValueError(f"unknown GEMM implementation {impl!r}")
    ws = torch.empty(splitk * R * Ncols, dtype=torch.float32, device=C.device) if splitk > 1 else None
    tag = f"[{R}x{Ncols}x{K} b{batch} t{int(a_trans)}{int(b_trans)}{int(c_trans)} sk{splitk}]" if PROFILE_SHAPES else ""
    head = (_ptr(A), lda, int(a_trans), a_bs, _ptr(B), ldb, int(b_trans), b_bs, _ptr(C), ldc, int(c_trans), c_bs, _ptr(bias), R, Ncols, K,
            batch, splitk, _ptr(ws), int(accumulate))
    if impl == "f32":
        _call("gfs_gemm_f32", 2 if splitk > 1 else 1, *head, _stream(), tag=tag)
    else:
        _call("gfs_gemm_tf32", 2 if splitk > 1 else 1, *head, int(impl == "tf32x3"), _stream(), tag=("x3" if impl == "tf32x3" else "") + tag)
    return C


def _splitk(K):
    """CTAs along the contraction of a weight gradient (K = points or edges).  The tensor-core kernel wants >= 2 waves of CTAs
    on 148 SMs even for the narrow (O, I) outputs, so its chunks are 512 long; the CUDA-core kernel keeps 2048."""
    return int(max(1, min(512, K // (2048 if TRAIN_GEMM == "f32" else 512))))


def conv_fwd(W, x, bias=None):
    """z (O, M) = W (O, I) . x (I, M) [+ bias]"""
    O, I = W.shape
    M = x.shape[1]
    z = torch.empty(O, M, dtype=torch.float32, device=x.device)
    return gemm_f32(W, I, True, x, x.stride(0), False, O, M, I, z, M, bias=bias)


def conv_dgrad(W, dz):
    """dx (I, M) = W^T . dz (O, M)"""
    O, I = W.shape
    M = dz.shape[1]
    dx = torch.empty(I, M, dtype=torch.float32, device=dz.device)
    return gemm_f32(W, I, False, dz, dz.stride(0), False, I, M, O, dx, M)


def conv_wgrad(dz, x):
    """dW (O, I) = dz (O, M) . x (I, M)^T   (contraction over the M points: split-K, fixed-order reduction)"""
    O, M = dz.shape
    I = x.shape[0]
    dW = torch.empty(O, I, dtype=torch.float32, device=x.device)
    return gemm_f32(dz, dz.stride(0), True, x, x.stride(0), True, O, I, M, dW, I, splitk=_splitk(M))


def bn_stats(x):
    C, M = x.shape
    mean = torch.empty(C, dtype=torch.float32, device=x.device)
    var = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = torch.empty(2 * 16 * C, dtype=torch.float64, device=x.device)
    _call("gfs_bn_stats", 2, _ptr(x), x.stride(0), C, M, _ptr(ws), _ptr(mean), _ptr(var), _stream())
    return mean, var


def bn_stats_coeffs(x, gamma, beta, eps):
    """batch statistics of x (C, M) and the affine coefficients the training forward applies: one C call, two launches"""
    C, M = x.shape
    out = torch.empty(5, C, dtype=torch.float32, device=x.device)      # mean | var | invstd | scale | shift
    ws = torch.empty(2 * 16 * C, dtype=torch.float64, device=x.device)
    _call("gfs_bn_stats_coeffs", 2, _ptr(x), x.stride(0), C, M, _ptr(ws), _ptr(gamma), _ptr(beta), float(eps), _ptr(out[0]), _ptr(out[1]),
          _ptr(out[2]), _ptr(out[3]), _ptr(out[4]), _stream())
    return out[0], out[1], out[2], out[3], out[4]


def bn_update_running(mean, var, n, momentum, running_mean, running_var, num_batches_tracked):
    _need_cuda(mean, var, running_mean, running_var, num_batches_tracked)
    assert running_mean.dtype == torch.float32 and running_var.dtype == torch.float32 and running_mean.is_contiguous()
    assert num_batches_tracked is None or num_batches_tracked.dtype == torch.int64
    _call("gfs_bn_update_running", 1, _ptr(mean), _ptr(var), mean.numel(), int(n), float(momentum), _ptr(running_mean), _ptr(running_var),
          _ptr(num_batches_tracked), _stream())


def bn_act_fwd(x, scale, shift, slope, out=None):
    C, M = x.shape
    y = torch.empty(C, M, dtype=torch.float32, device=x.device) if out is None else out
    _call("gfs_bn_act_fwd", 1, _ptr(x), x.stride(0), _ptr(y), y.stride(0), C, M, _ptr(scale), _ptr(shift), float(slope), _stream())
    return y


def bn_act_bwd(dy, x, mean, invstd, gamma, beta, slope):
    C, M = x.shape
    dx = torch.empty(C, M, dtype=torch.float32, device=x.device)
    sg = torch.empty(C, dtype=torch.float32, device=x.device)
    sgx = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = torch.empty(2 * 16 * C, dtype=torch.float64, device=x.device)
    _call("gfs_bn_act_bwd", 3, _ptr(dy), dy.stride(0), _ptr(x), x.stride(0), _ptr(dx), M, C, M, _ptr(mean), _ptr(invstd), _ptr(gamma),
          _ptr(beta), float(slope), _ptr(ws), _ptr(sg), _ptr(sgx), _stream())
    return dx, sg, sgx


def bn_act_bwd_argmax(dy, arg, k, x, mean, invstd, gamma, beta, slope):
    """bn_act_bwd(max_over_k_bwd(dy, arg, k), x, ...) without the (C, Mp*k) gradient in between"""
    C, E = x.shape
    Mp = arg.shape[1]
    assert E == Mp * k and dy.shape == arg.shape
    dx = torch.empty(C, E, dtype=torch.float32, device=x.device)
    sg = torch.empty(C, dtype=torch.float32, device=x.device)
    sgx = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = torch.empty(2 * 16 * C, dtype=torch.float64, device=x.device)
    _call("gfs_bn_act_bwd_argmax", 3, _ptr(dy), dy.stride(0), _ptr(arg), k, _ptr(x), x.stride(0), _ptr(dx), E, C, Mp, _ptr(mean),
          _ptr(invstd), _ptr(gamma), _ptr(beta), float(slope), _ptr(ws), _ptr(sg), _ptr(sgx), _stream())
    return dx, sg, sgx


def bn_act_bwd_frozen(dy, x, mean, invstd, gamma, beta, slope):
    """bn_act_bwd for a BatchNorm that normalises with fixed (running) statistics: dx = gamma * invstd * g, no batch-statistic
    terms; (sum_g, sum_gx) = (dbeta, dgamma).  One pass over dy and x"""
    C, M = x.shape
    dx = torch.empty(C, M, dtype=torch.float32, device=x.device)
    sg = torch.empty(C, dtype=torch.float32, device=x.device)
    sgx = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = torch.empty(2 * 16 * C, dtype=torch.float64, device=x.device)
    _call("gfs_bn_act_bwd_frozen", 2, _ptr(dy), dy.stride(0), _ptr(x), x.stride(0), _ptr(dx), M, C, M, _ptr(mean), _ptr(invstd),
          _ptr(gamma), _ptr(beta), float(slope), _ptr(ws), _ptr(sg), _ptr(sgx), _stream())
    return dx, sg, sgx


def bn_act_bwd_argmax_frozen(dy, arg, k, x, mean, invstd, gamma, beta, slope):
    """bn_act_bwd_frozen(max_over_k_bwd(dy, arg, k), x, ...) without the (C, Mp*k) gradient in between; x is read at the arg-max
    edges only"""
    C, E = x.shape
    Mp = arg.shape[1]
    assert E == Mp * k and dy.shape == arg.shape
    dx = torch.empty(C, E, dtype=torch.float32, device=x.device)
    sg = torch.empty(C, dtype=torch.float32, device=x.device)
    sgx = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = torch.empty(2 * 16 * C, dtype=torch.float64, device=x.device)
    _call("gfs_bn_act_bwd_argmax_frozen", 2, _ptr(dy), dy.stride(0), _ptr(arg), k, _ptr(x), x.stride(0), _ptr(dx), E, C, Mp, _ptr(mean),
          _ptr(invstd), _ptr(gamma), _ptr(beta), float(slope), _ptr(ws), _ptr(sg), _ptr(sgx), _stream())
    return dx, sg, sgx


def bn_act_max_fwd(z, scale, shift, slope, M, k):
    """max over the k slots of act(BN(z)) and its arg-max, one pass over z (C, M*k) -> y (C, M), arg (C, M) uint8"""
    C = z.shape[0]
    assert z.is_contiguous() and z.shape[1] == M * k
    y = torch.empty(C, M, dtype=torch.float32, device=z.device)
    arg = torch.empty(C, M, dtype=torch.uint8, device=z.device)
    _call("gfs_bn_act_max_fwd", 1, _ptr(z), C, M, k, _ptr(scale), _ptr(shift), float(slope), _ptr(y), M, _ptr(arg), _stream())
    return y, arg


def bn_bwd_sums(dy, x, mean, invstd, gamma, beta, slope):
    """(sum_g, sum_gx) = (dbeta, dgamma) of y = act(gamma*xhat + beta) without the apply pass"""
    C, M = x.shape
    sg = torch.empty(C, dtype=torch.float32, device=x.device)
    sgx = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = torch.empty(2 * 16 * C, dtype=torch.float64, device=x.device)
    _call("gfs_bn_bwd_sums", 2, _ptr(dy), dy.stride(0), _ptr(x), x.stride(0), C, M, _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(beta),
          float(slope), _ptr(ws), _ptr(sg), _ptr(sgx), _stream())
    return sg, sgx


def edge_reverse_index(idx, B, N):
    """incoming edges of every target of the graph idx (B, N, k) int32 -> rev_ptr (B*N + 1), rev_edge (B*N*k) int32: the edges of
    target j = b*N + idx[e] are rev_edge[rev_ptr[j]:rev_ptr[j+1]] in ascending edge index (a stable sort of the targets)"""
    _need_cuda(idx)
    k = idx.shape[-1]
    assert idx.dtype == torch.int32 and idx.is_contiguous() and idx.numel() == B * N * k
    rev_ptr = torch.empty(B * N + 1, dtype=torch.int32, device=idx.device)
    rev_edge = torch.empty(B * N * k, dtype=torch.int32, device=idx.device)
    _call("gfs_edge_reverse_index", 1, _ptr(idx), B, N, k, _ptr(rev_ptr), _ptr(rev_edge), _stream())
    return rev_ptr, rev_edge


def edge_scatter_bn(dy, x, idx, B, N, k, mean, invstd, gamma, beta, slope, sg, sgx, ordered=False, rev=None, edge_terms=None):
    """edge_scatter(bn_act_bwd(dy, x, ...).dx) without the (64, E) tensor in between; dy, x (64, E) contiguous.
    ordered=True: the P half is summed per target in ascending edge order (gfs_edge_scatter_bn_ordered), the same bits on every
    run.  rev: the graph's edge_reverse_index (built here if None); edge_terms: optional (E, 64) fp32 buffer for the per-edge terms"""
    assert dy.is_contiguous() and x.is_contiguous() and dy.shape == x.shape and dy.shape[0] == 64
    if not ordered:
        dpq = torch.zeros(B * N, 128, dtype=torch.float32, device=dy.device)
        _call("gfs_edge_scatter_bn", 1, _ptr(dy), _ptr(x), _ptr(idx), B, N, k, _ptr(mean), _ptr(invstd), _ptr(gamma), _ptr(beta),
              float(slope), _ptr(sg), _ptr(sgx), _ptr(dpq), _stream())
        return dpq
    rev_ptr, rev_edge = edge_reverse_index(idx, B, N) if rev is None else rev
    E = B * N * k
    if edge_terms is None:
        edge_terms = torch.empty(E, 64, dtype=torch.float32, device=dy.device)
    assert edge_terms.dtype == torch.float32 and edge_terms.is_contiguous() and edge_terms.shape == (E, 64)
    dpq = torch.empty(B * N, 128, dtype=torch.float32, device=dy.device)
    _call("gfs_edge_scatter_bn_ordered", 2, _ptr(dy), _ptr(x), _ptr(idx), _ptr(rev_ptr), _ptr(rev_edge), B, N, k, _ptr(mean),
          _ptr(invstd), _ptr(gamma), _ptr(beta), float(slope), _ptr(sg), _ptr(sgx), _ptr(edge_terms), _ptr(dpq), _stream())
    return dpq


def edge_gather(pq, idx, B, N, k):
    H = torch.empty(64, B * N * k, dtype=torch.float32, device=pq.device)
    _call("gfs_edge_gather", 1, _ptr(pq), _ptr(idx), B, N, k, _ptr(H), _stream())
    return H


def edge_gather_stats(pq, idx, B, N, k, gamma, beta, eps):
    """edge_gather + bn_stats_coeffs(H) in one pass: -> H (64, E), (mean, var, invstd, scale, shift)"""
    E = B * N * k
    H = torch.empty(64, E, dtype=torch.float32, device=pq.device)
    part = torch.empty(64 * ((E + 127) // 128) * 2, dtype=torch.float64, device=pq.device)      # fp64 (sum, sum of squares) per channel and tile
    out = torch.empty(5, 64, dtype=torch.float32, device=pq.device)
    _call("gfs_edge_gather_stats", 2, _ptr(pq), _ptr(idx), B, N, k, _ptr(H), _ptr(part), _ptr(gamma), _ptr(beta), float(eps),
          _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]), _ptr(out[4]), _stream())
    return H, (out[0], out[1], out[2], out[3], out[4])


def edge_scatter(dH, idx, B, N, k):
    dpq = torch.zeros(B * N, 128, dtype=torch.float32, device=dH.device)
    _call("gfs_edge_scatter", 1, _ptr(dH), _ptr(idx), B, N, k, _ptr(dpq), _stream())
    return dpq


def max_over_k_fwd(a, M, k):
    C = a.shape[0]
    y = torch.empty(C, M, dtype=torch.float32, device=a.device)
    arg = torch.empty(C, M, dtype=torch.uint8, device=a.device)
    _call("gfs_max_over_k_fwd", 1, _ptr(a), C, M, k, _ptr(y), M, _ptr(arg), _stream())
    return y, arg


def max_over_k_bwd(dy, arg, k):
    C, M = arg.shape
    da = torch.empty(C, M * k, dtype=torch.float32, device=dy.device)
    _call("gfs_max_over_k_bwd", 1, _ptr(dy), dy.stride(0), _ptr(arg), C, M, k, _ptr(da), _stream())
    return da


def softmax_rows_fwd(s, scale, mask=None, seed=0, keep=1.0):
    """p0 = softmax(s * scale) per row; p = p0 * dropout factor.  mask: explicit (B, n, n) factors; or mask None and keep < 1: the
    factors come from the counter-based hash of (seed, row, column) that softmax_rows_bwd regenerates (no mask tensor)"""
    rows, n = s.shape[0] * s.shape[1], s.shape[2]
    p0 = torch.empty_like(s)
    p = torch.empty_like(s) if (mask is not None or keep < 1.0) else p0
    _call("gfs_softmax_rows_fwd", 1, _ptr(s), rows, n, float(scale), _ptr(mask), int(seed) & 0xFFFFFFFF, float(keep), _ptr(p0), _ptr(p),
          _stream())
    return p0, p


def dropout_mask(rows, n, seed, keep, device):
    """(tests) the mask the hash of softmax_rows_fwd / _bwd defines: 1/keep or 0"""
    m = torch.empty(rows, n, dtype=torch.float32, device=device)
    _call("gfs_dropout_mask", 1, rows, n, int(seed) & 0xFFFFFFFF, float(keep), _ptr(m), _stream())
    return m


def softmax_rows_bwd(p0, dp, scale, mask=None, seed=0, keep=1.0):
    rows, n = p0.shape[0] * p0.shape[1], p0.shape[2]
    ds = torch.empty_like(p0)
    _call("gfs_softmax_rows_bwd", 1, _ptr(p0), _ptr(dp), _ptr(mask), int(seed) & 0xFFFFFFFF, float(keep), rows, n, float(scale), _ptr(ds),
          _stream())
    return ds
