"""Self-attention block -- drop-in for the reference's model/attention.py:10-48 (SURVEY.md section 8 row a6, "adjacent").

q/k/v 1x1 maps run as ONE fused gfs_linear_bf16 call (256 -> 3*64) whose bf16 output tiles are consumed in place by
gfs_attention_fwd, a flash-style tcgen05 kernel (csrc/attention.cu): the N x N softmax(q^T k / sqrt(d)) matrix is never
materialised.  Eval mode only (dropout is the identity); N must be a multiple of 128.  The training path (forward_train) applies
dropout iff the dropout module itself is in training mode.
"""
import torch
import torch.nn as nn

from gfs3d import ops


class SelfAttention(nn.Module):
    def __init__(self, in_channel, out_channel=None, attn_dropout=0.1):
        super(SelfAttention, self).__init__()
        self.in_channel = in_channel
        self.out_channel = out_channel if out_channel is not None else in_channel
        self.temperature = self.out_channel ** 0.5
        self.q_map = nn.Conv1d(in_channel, self.out_channel, 1, bias=False)
        self.k_map = nn.Conv1d(in_channel, self.out_channel, 1, bias=False)
        self.v_map = nn.Conv1d(in_channel, self.out_channel, 1, bias=False)
        self.dropout = nn.Dropout(attn_dropout)
        self._key = None
        self._wp = None

    def _prepare(self, device):
        ws = (self.q_map.weight, self.k_map.weight, self.v_map.weight)
        key = (str(device),) + tuple((id(w), w._version) for w in ws)
        if self._key != key:
            if self.out_channel % 64 != 0 or self.in_channel % 64 != 0:
                raise NotImplementedError("SelfAttention widths must be multiples of 64 in the B200 build")
            with torch.no_grad():
                w = torch.cat([t.detach().float().reshape(self.out_channel, self.in_channel) for t in ws], dim=0)
                self._wp = ops.pack_weight(w)
            self._key = key
        return self._wp

    def forward_train(self, x_cm, B, N):
        """training mode: x_cm (in_channel, M) -> (64, M); dropout on the attention weights as model/attention.py:45"""
        from gfs3d.train_ops import AttentionTrain, ConvOnly
        w = torch.cat([self.q_map.weight, self.k_map.weight, self.v_map.weight], dim=0).reshape(3 * self.out_channel, self.in_channel)
        qkv = ConvOnly.apply(x_cm, w)
        keep, seed = 1.0, 0
        if self.dropout.training and self.dropout.p > 0:
            # dropout on the attention weights (model/attention.py:45) without a mask tensor: the kernels hash (seed, row, column);
            # the seed advances per call from torch's seed, so torch.manual_seed makes a run repeatable (no host sync)
            keep = 1.0 - self.dropout.p
            self._drop_calls = getattr(self, "_drop_calls", 0) + 1
            seed = (torch.initial_seed() * 0x9E3779B1 + self._drop_calls * 0x85EBCA77) & 0xFFFFFFFF
        return AttentionTrain.apply(qkv, B, N, 1.0 / self.temperature, None, seed, keep)

    def forward_fused(self, x_act, B, N, y_cm=None, y_act=None, y_kb=0):
        """x_act: bf16 act tiles (B*N, in_channel).  Writes y (B, 64, N) fp32 cm and/or one bf16 act block."""
        if self.training:
            raise RuntimeError("forward_fused is the inference path; training mode goes through forward_train")
        if self.out_channel != 64:
            raise NotImplementedError("the tcgen05 attention kernel is built for out_channel = 64")
        wp = self._prepare(x_act.device)
        qkv = ops.new_act(B * N, 3, x_act.device, zero=False)
        ops.linear(x_act, 0, self.in_channel // 64, wp, None, 192, ops.ACT_NONE, B, N, y_act=qkv)
        ops.attention(qkv, 0, B, N, 1.0 / self.temperature, y_cm=y_cm, y_act=y_act, y_kb=y_kb)

    def forward(self, x):
        """(B, in_channel, N) -> (B, out_channel, N)"""
        if self.training:
            from gfs3d.train_ops import from_cm, to_cm
            if self.out_channel != 64:
                raise NotImplementedError("the attention kernels are built for out_channel = 64")
            return from_cm(self.forward_train(to_cm(x.float()), x.shape[0], x.shape[2]), x.shape[0], x.shape[2])
        if x.dtype != torch.float32 or x.stride(2) != 1 or x.stride(1) != x.shape[2]:
            x = x.float().contiguous()
        B, C, N = x.shape
        xa = ops.new_act(B * N, C // 64, x.device, zero=False)
        ops.cm_to_act(x, xa, 0)
        y = torch.empty(B, self.out_channel, N, dtype=torch.float32, device=x.device)
        self.forward_fused(xa, B, N, y_cm=y)
        return y
