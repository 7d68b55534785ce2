"""DGCNN EdgeConv backbone -- drop-in for the reference's model/dgcnn.py, computed by the sm_100a kernels.

Public surface kept from the reference (file:line of what each replaces):
  knn(x, k)                         model/dgcnn.py:17-23
  get_edge_feature(x, K, idx)       model/dgcnn.py:26-42   (kept for API parity; the fused path never calls it)
  conv2d / conv1d                   model/dgcnn.py:45-80   (parameter containers with the reference's state-dict keys)
  DGCNN(...).forward(x)             model/dgcnn.py:93-127
  BaseLearner, DGCNNSeg_att         model/dgcnn.py:130-202

Eval-mode forward = per layer: gfs_knn_tc_set_f32 -> gfs_edge_pq_f32 (split conv1) -> gfs_edgeconv_fwd (tcgen05 conv2 + max),
then gfs_linear_bf16 x2 for the 192->512->256 MLP.  There is no PyTorch fallback: on a machine without the CUDA library
the forward raises.
"""
from typing import List, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from gfs3d import ops
from model.attention import SelfAttention

BN_EPS = 1e-5


def knn(x, k):
    """(B, C, N) fp32 -> (B, N, k) int64 neighbour indices, nearest first, ties -> ascending index."""
    return ops.knn(_cm(x), k).long()


def get_edge_feature(x, K=20, idx=None):
    """(B, C, N) -> (B, 2C, N, K) = cat(x_j - x_i, x_i).  Materialises the edge tensor the fused kernels avoid; kept
    only so that code written against the reference API keeps working."""
    B, C, N = x.size()
    if idx is None:
        idx = knn(x, k=K)
    nbr = torch.gather(x, 2, idx.reshape(B, 1, N * K).expand(B, C, N * K)).reshape(B, C, N, K)
    ctr = x.unsqueeze(-1).expand(B, C, N, K)
    return torch.cat((nbr - ctr, ctr), dim=1)


def _cm(x: torch.Tensor) -> torch.Tensor:
    """channel-major fp32 view the kernels accept: unit point stride, channel stride N"""
    if x.dtype != torch.float32:
        x = x.float()
    if x.stride(2) != 1 or x.stride(1) != x.shape[2] or (x.data_ptr() % 16) != 0:
        x = x.contiguous()
    return x


def fold_bn(bn: nn.modules.batchnorm._BatchNorm):
    """eval-mode BatchNorm as y = s*x + t"""
    s = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    t = bn.bias.detach().float() - bn.running_mean.detach().float() * s
    return s, t


class _ConvStack(nn.Module):
    """(Conv 1x1 [, BN] [, LeakyReLU 0.2]) x len(layer_dims), registered as `self.layer` exactly like the reference so
    that checkpoints interchange (keys layer.{0,3,..}.weight, layer.{1,4,..}.{weight,bias,running_*})."""
    conv_cls = None
    bn_cls = None

    def __init__(self, in_feat, layer_dims, batch_norm=True, relu=True, bias=False):
        super().__init__()
        self.layer_dims = layer_dims
        mods = []
        for i, out_dim in enumerate(layer_dims):
            in_dim = in_feat if i == 0 else layer_dims[i - 1]
            mods.append(self.conv_cls(in_dim, out_dim, kernel_size=1, bias=bias))
            if batch_norm:
                mods.append(self.bn_cls(out_dim))
            if relu:
                mods.append(nn.LeakyReLU(0.2))
        self.layer = nn.Sequential(*mods)
        self.fusable = batch_norm and relu and not bias

    def forward(self, x):
        raise RuntimeError(
            f"{type(self).__name__} is a parameter container in the B200 build: it is evaluated inside DGCNN's fused "
            "kernels (no stand-alone PyTorch path is provided)")

    def stages(self):
        """[(conv, bn)] per layer, for the weight folding"""
        m = list(self.layer)
        return [(m[3 * i], m[3 * i + 1]) for i in range(len(self.layer_dims))]


class conv2d(_ConvStack):
    conv_cls = nn.Conv2d
    bn_cls = nn.BatchNorm2d


class conv1d(_ConvStack):
    conv_cls = nn.Conv1d
    bn_cls = nn.BatchNorm1d


class _Folded:
    """device-resident folded / packed weights, rebuilt when any parameter or buffer changes"""

    def __init__(self):
        self.key = None
        self.data = None


def _state_key(module: nn.Module, device):
    return (str(device), module.training) + tuple((id(t), t._version) for t in list(module.parameters()) + list(module.buffers()))


class EncoderOutput:
    """what the fused backbone leaves on the device for the head"""
    __slots__ = ("ec", "cat_act", "lvl2_act", "lvl2_cm", "B", "N")

    def __init__(self, ec, cat_act, lvl2_act, lvl2_cm, B, N):
        self.ec, self.cat_act, self.lvl2_act, self.lvl2_cm, self.B, self.N = ec, cat_act, lvl2_act, lvl2_cm, B, N


class DGCNN(nn.Module):
    """DGCNN with stacked EdgeConv blocks; same constructor and forward contract as model/dgcnn.py:93-127."""

    def __init__(self, edgeconv_widths, mlp_widths, nfeat, k=20, return_edgeconvs=False):
        super(DGCNN, self).__init__()
        self.n_edgeconv = len(edgeconv_widths)
        self.k = k
        self.return_edgeconvs = return_edgeconvs
        self.edge_convs = nn.ModuleList()
        for i in range(self.n_edgeconv):
            in_feat = nfeat * 2 if i == 0 else edgeconv_widths[i - 1][-1] * 2
            self.edge_convs.append(conv2d(in_feat, edgeconv_widths[i]))
        in_dim = sum(w[-1] for w in edgeconv_widths)
        self.conv = conv1d(in_dim, mlp_widths)
        self._edgeconv_widths = [list(w) for w in edgeconv_widths]
        self._mlp_widths = list(mlp_widths)
        self._nfeat = nfeat
        self._folded = _Folded()

    # ------------------------------------------------------------------ weight folding
    def _check_supported(self):
        for w in self._edgeconv_widths:
            if list(w) != [64, 64]:
                raise NotImplementedError(
                    f"edgeconv_widths={self._edgeconv_widths}: the sm_100a EdgeConv kernel is specialised to [64, 64] blocks")
        if self._nfeat > 64:
            raise NotImplementedError(f"nfeat={self._nfeat} > 64 is not built")
        for w in self._mlp_widths:
            if w % 64 != 0:
                raise NotImplementedError(f"dgcnn_mlp_widths={self._mlp_widths}: widths must be multiples of 64")

    def _prepare(self, device):
        key = _state_key(self, device)
        if self._folded.key == key:
            return self._folded.data
        self._check_supported()
        layers = []
        with torch.no_grad():
            for blk in self.edge_convs:
                (c1, b1), (c2, b2) = blk.stages()
                C = c1.weight.shape[1] // 2
                w1 = c1.weight.detach().float().reshape(64, 2 * C)
                s1, t1 = fold_bn(b1)
                wa, wb = w1[:, :C], w1[:, C:]
                wt = torch.cat([s1[:, None] * wa, s1[:, None] * (wb - wa)], dim=0).t().contiguous()   # (C, 128)
                bias = torch.cat([torch.zeros_like(t1), t1]).contiguous()
                s2, t2 = fold_bn(b2)
                w2p = ops.pack_weight(c2.weight.detach().float().reshape(64, 64), s2)
                layers.append((wt, bias, w2p, t2.contiguous()))
            mlp = []
            for conv, bn in self.conv.stages():
                s, t = fold_bn(bn)
                w = conv.weight.detach().float().reshape(conv.weight.shape[0], conv.weight.shape[1])
                mlp.append((ops.pack_weight(w, s), t.contiguous(), w.shape[0], (w.shape[1] + 63) // 64))
        self._folded.key, self._folded.data = key, (layers, mlp)
        return self._folded.data

    # ------------------------------------------------------------------ fused forward
    def forward_fused(self, x, want_lvl2_cm=True, level1_act=None, level1_kb=0) -> EncoderOutput:
        """x (B, nfeat, N) CUDA fp32.  Runs the whole backbone in the sm_100a kernels and returns device buffers:
        ec (B, 64*L, N) fp32, cat_act / lvl2_act bf16 act tiles, lvl2_cm (B, mlp[-1], N) fp32 if requested."""
        if not x.is_cuda:
            raise RuntimeError("DGCNN needs CUDA tensors: the hot path has no CPU fallback")
        if self.training:
            raise RuntimeError("forward_fused is the inference path; training mode goes through forward_train")
        layers, mlp = self._prepare(x.device)
        x = _cm(x)
        B, _, N = x.shape
        M = B * N
        L = self.n_edgeconv
        ec = torch.empty(B, 64 * L, N, dtype=torch.float32, device=x.device)
        cat_act = ops.new_act(M, L, x.device, zero=False)
        xin = x
        for i, (wt, bias, w2p, t2) in enumerate(layers):
            idx = ops.knn(xin, self.k, ordered=False)      # the max over k only needs the neighbour set
            pq = ops.edge_pq(xin, wt, bias)
            y = ec[:, 64 * i:64 * (i + 1), :]
            ops.edgeconv(pq, idx, w2p, t2, B, N, self.k, y_cm=y, y_act=cat_act, y_act_kb=i,
                         y_act2=level1_act if i == 0 else None, y_act2_kb=level1_kb)
            xin = y
        cur, cur_kb = cat_act, L
        lvl2_cm = None
        for j, (wp, shift, nout, kb) in enumerate(mlp):
            last = j == len(mlp) - 1
            nxt = ops.new_act(M, nout // 64, x.device, zero=False)
            if last and want_lvl2_cm:
                lvl2_cm = torch.empty(B, nout, N, dtype=torch.float32, device=x.device)
            ops.linear(cur, 0, kb, wp, shift, nout, ops.ACT_LRELU02, B, N, y_act=nxt, y_cm=lvl2_cm if last else None)
            cur, cur_kb = nxt, nout // 64
        return EncoderOutput(ec, cat_act, cur, lvl2_cm, B, N)

    def forward_train(self, x):
        """training mode (model.train(), train.py:614): batch-statistics BatchNorm, fp32, autograd through the hand-written
        forward/backward kernels of gfs3d/train_ops.py.  Returns channel-major tensors: ([ec_i (64, M)], out (mlp[-1], M)).
        Each BatchNorm follows its own mode: one in eval mode is frozen (running statistics, left unchanged)."""
        from gfs3d.train_ops import ConvBNAct, EdgeConvTrain, batch_stats, from_cm, to_cm, update_running_stats
        if not x.is_cuda:
            raise RuntimeError("DGCNN needs CUDA tensors: the hot path has no CPU fallback")
        self._check_supported()
        x = x.float()
        B, _, N = x.shape
        M = B * N
        cur_bcn, cur_cm = x.detach().contiguous(), to_cm(x)
        outs = []
        for blk in self.edge_convs:
            (c1, b1), (c2, b2) = blk.stages()
            idx = ops.knn(cur_bcn, self.k)                       # integer graph: not differentiated (as in the reference)
            y, m1, v1, m2, v2 = EdgeConvTrain.apply(cur_cm, idx, c1.weight, b1.weight, b1.bias, c2.weight, b2.weight, b2.bias,
                                                    B, N, self.k, batch_stats(b1), b1.running_mean, b1.running_var,
                                                    batch_stats(b2), b2.running_mean, b2.running_var)
            if b1.training:
                update_running_stats(b1, m1, v1, M * self.k)
            if b2.training:
                update_running_stats(b2, m2, v2, M * self.k)
            outs.append(y)
            cur_cm, cur_bcn = y, from_cm(y.detach(), B, N)
        cur = torch.cat(outs, dim=0)
        for conv, bn in self.conv.stages():
            w = conv.weight.reshape(conv.weight.shape[0], conv.weight.shape[1])
            cur, m, v = ConvBNAct.apply(cur, w, None, bn.weight, bn.bias, bn.running_mean, bn.running_var, 0.2, batch_stats(bn))
            if bn.training:
                update_running_stats(bn, m, v, M)
        return outs, cur

    def forward(self, x):
        if self.training:
            from gfs3d.train_ops import from_cm
            B, _, N = x.shape
            outs, cur = self.forward_train(x)
            ecs = [from_cm(o, B, N) for o in outs]
            return (ecs, from_cm(cur, B, N)) if self.return_edgeconvs else (ecs[0], from_cm(cur, B, N))
        out = self.forward_fused(x, want_lvl2_cm=True)
        edgeconv_outputs: List[torch.Tensor] = [out.ec[:, 64 * i:64 * (i + 1), :] for i in range(self.n_edgeconv)]
        if self.return_edgeconvs:
            return edgeconv_outputs, out.lvl2_cm
        return edgeconv_outputs[0], out.lvl2_cm


class BaseLearner(nn.Module):
    """model/dgcnn.py:130-152 -- Conv1d(+bias)+BN stack with ReLU between layers; evaluated by gfs_linear_bf16."""

    def __init__(self, in_channels, params):
        super(BaseLearner, self).__init__()
        self.num_convs = len(params)
        self.convs = nn.ModuleList()
        for i in range(self.num_convs):
            in_dim = in_channels if i == 0 else params[i - 1]
            self.convs.append(nn.Sequential(nn.Conv1d(in_dim, params[i], 1), nn.BatchNorm1d(params[i])))
        self._folded = _Folded()

    def _prepare(self, device):
        key = _state_key(self, device)
        if self._folded.key != key:
            out = []
            with torch.no_grad():
                for seq in self.convs:
                    conv, bn = seq[0], seq[1]
                    if conv.weight.shape[0] % 64 != 0:
                        raise NotImplementedError("BaseLearner widths must be multiples of 64 in the B200 build")
                    s, t = fold_bn(bn)
                    w = conv.weight.detach().float().reshape(conv.weight.shape[0], conv.weight.shape[1])
                    shift = (conv.bias.detach().float() * s + t).contiguous()
                    out.append((ops.pack_weight(w, s), shift, w.shape[0], (w.shape[1] + 63) // 64))
            self._folded.key, self._folded.data = key, out
        return self._folded.data

    def forward_train(self, x_cm):
        """x_cm (in_channels, M) -> (params[-1], M); Conv1d(+bias)+BN with ReLU between layers, batch statistics (running ones for
        a BatchNorm in eval mode)"""
        from gfs3d.train_ops import ConvBNAct, batch_stats, update_running_stats
        M = x_cm.shape[1]
        cur = x_cm
        for i, seq in enumerate(self.convs):
            conv, bn = seq[0], seq[1]
            w = conv.weight.reshape(conv.weight.shape[0], conv.weight.shape[1])
            cur, m, v = ConvBNAct.apply(cur, w, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var,
                                        0.0 if i != self.num_convs - 1 else 1.0, batch_stats(bn))
            if bn.training:
                update_running_stats(bn, m, v, M)
        return cur

    def forward_fused(self, x_act, B, N, y_act=None, y_kb0=0, y_cm=None):
        """x_act: bf16 act tiles of the (B*N, in_channels) input.  Last layer writes y_act / y_cm."""
        if self.training:
            raise RuntimeError("forward_fused is the inference path; training mode goes through forward_train")
        stages = self._prepare(x_act.device)
        cur = x_act
        for i, (wp, shift, nout, kb) in enumerate(stages):
            last = i == len(stages) - 1
            if last:
                ops.linear(cur, 0, kb, wp, shift, nout, ops.ACT_NONE, B, N, y_act=y_act, y_kb0=y_kb0, y_cm=y_cm)
            else:
                nxt = ops.new_act(B * N, nout // 64, x_act.device, zero=False)
                ops.linear(cur, 0, kb, wp, shift, nout, ops.ACT_RELU, B, N, y_act=nxt)
                cur = nxt

    def forward(self, x):
        """(B, C, N) fp32 -> (B, params[-1], N) fp32"""
        if self.training:
            from gfs3d.train_ops import from_cm, to_cm
            return from_cm(self.forward_train(to_cm(x.float())), x.shape[0], x.shape[2])
        x = _cm(x)
        B, C, N = x.shape
        if C % 64 != 0:
            raise NotImplementedError("BaseLearner input width must be a multiple of 64 in the B200 build")
        xa = ops.new_act(B * N, C // 64, x.device, zero=False)
        ops.cm_to_act(x, xa, 0)
        y = torch.empty(B, self.convs[-1][0].weight.shape[0], N, dtype=torch.float32, device=x.device)
        self.forward_fused(xa, B, N, y_cm=y)
        return y


class DGCNNSeg_att(nn.Module):
    """model/dgcnn.py:155-202 (pre-training segmentor with attention); same parameters, fused backbone."""

    def __init__(self, args, num_classes):
        super(DGCNNSeg_att, self).__init__()
        self.encoder = DGCNN(args.edgeconv_widths, args.dgcnn_mlp_widths, args.pc_in_dim, k=args.dgcnn_k)
        self.base_learner = BaseLearner(args.dgcnn_mlp_widths[-1], args.base_widths)
        self.att_learner = SelfAttention(args.dgcnn_mlp_widths[-1], args.output_dim)
        self.feat_dim = args.edgeconv_widths[0][-1] + args.output_dim + args.base_widths[-1]
        self.segmenter = nn.Sequential(
            nn.Conv1d(self.feat_dim, 256, 1, bias=False), nn.BatchNorm1d(256), nn.LeakyReLU(0.2),
            nn.Conv1d(256, 128, 1), nn.BatchNorm1d(128), nn.LeakyReLU(0.2), nn.Dropout(0.3),
            nn.Conv1d(128, num_classes, 1))

    def forward(self, pc, return_feat=False):
        feat_level1, feat_level2 = self.encoder(pc)
        feat_level3 = self.base_learner(feat_level2)
        att_feat = self.att_learner(feat_level2)
        pc_feat = torch.cat((feat_level1, att_feat, feat_level3), dim=1)
        logits = self.segmenter(pc_feat)     # tiny classification tail: outside the hot path (SURVEY.md section 8)
        if return_feat:
            return logits, feat_level1
        return logits
