"""Geometric-word class codings (train.py:136-241 of the reference) as batched GPU reductions.

The reference runs the training set through the model with batch size 1 and, per block and per class present, sums the
one-hot GW features of the class's points (`torch.unique`, a Python loop over classes, `.item()` syncs).  All of that is a
joint histogram of (label, GW assignment): here any batch size goes through the fused eval path (which already returns
the assignment, so the (B, G, N) one-hot tensor is never built) and `gfs_joint_histogram_i32` accumulates the counts on
the device; one tiny D2H at the end.  Same function names, arguments and return conventions as the reference.
"""
import random

import numpy as np
import torch

from . import ops


def post_processing_hard_coding(coding: torch.Tensor, energy: float) -> torch.Tensor:
    """train.py:136-152: keep the most frequent geometric words until they hold more than `energy` of the mass -> multi-hot.
    In place, like the reference.  The running sum is accumulated sequentially in the tensor's dtype (the reference adds
    0-d tensors one by one); equal frequencies are taken lowest index first (`torch.argsort` leaves that order open)."""
    total = torch.sum(coding)                               # same op on the same device as the reference
    thr = float((energy * total).item())                    # python scalar x tensor: rounded to the tensor's dtype
    c = coding.detach().cpu().numpy()
    order = np.argsort(-c, kind="stable")
    acc = c.dtype.type(0)
    mask = np.zeros(c.shape, dtype=bool)
    for i in order:
        acc = c.dtype.type(acc + c[i])                      # sequential sum in the tensor's dtype
        mask[i] = True
        if float(acc) > thr:
            break
    m = torch.from_numpy(mask).to(coding.device)
    coding[m] = 1
    coding[~m] = 0
    return coding


def label_gw_histogram(assignment: torch.Tensor, labels: torch.Tensor, num_labels: int, G: int, out=None) -> torch.Tensor:
    """H[label, g] (+)= number of points with that label assigned to geometric word g (int64, on the device)"""
    return ops.joint_histogram(labels, assignment, num_labels, G, out=out)


def block_gw_histogram(blk: torch.Tensor, assignment: torch.Tensor, b: int, G: int) -> torch.Tensor:
    """H[i, g] = number of points of block i (blk == i; -1 = not counted) assigned to word g, (b, G) int64.  The histogram
    kernel holds at most 12 288 bins (b * G = 16 384 at 32 blocks of 512 words): the blocks go in groups that fit, each group
    a pass over the labels with its own block range, so the counts are those of one call."""
    per = max(1, ops.JOINT_HISTOGRAM_MAXBINS // G)
    if b <= per:
        return ops.joint_histogram(blk, assignment, b, G)
    H = torch.zeros(b, G, dtype=torch.int64, device=assignment.device)
    for i0 in range(0, b, per):
        nb = min(per, b - i0)
        ops.joint_histogram(blk - i0, assignment, nb, G, out=H[i0:i0 + nb])
    return H


def collect_base_class_gp_coding_sum(model, train_loader, train_class, energy):
    """train.py:156-218.  train_loader yields (input (b, d, n), target (b, n), segment_label) with ANY batch size (the
    reference needs bs = 1).  Returns (base_class_gp_coding (num_base, G) multi-hot, bg_class_coding (G,)) on the device."""
    model.eval()
    G = model.gp.shape[0]
    num_labels = max(train_class) + 2                       # label 0 = background, label cls + 1 = base class cls
    H = None
    bg_class_coding = []
    max_len = 2000
    with torch.no_grad():
        for input, target, _ in train_loader:
            input = input.cuda()
            target = target.cuda()
            _, assignment, _ = model._features(input)       # (b, n) int32: argmax of the GW projection
            b, n = target.shape
            if H is None:
                H = torch.zeros(num_labels, G, dtype=torch.int64, device=input.device)
            label_gw_histogram(assignment, target, num_labels, G, out=H)
            # background: one mean one-hot vector per BLOCK (train.py:186-191) = per-block histogram / count
            blk = torch.arange(b, device=input.device, dtype=torch.int32).unsqueeze(1).expand(b, n)
            blk = torch.where(target == 0, blk, torch.full_like(blk, -1))
            hb = block_gw_histogram(blk, assignment, b, G)
            cnt = hb.sum(dim=1)
            for i in range(b):
                if int(cnt[i]) > 0:
                    bg_class_coding.append(hb[i].float() / cnt[i])
        base_class_gp_coding = []
        counts = H.sum(dim=1)
        for cls in train_class:
            print('processing {}'.format(cls))
            if int(counts[cls + 1]) == 0:
                raise RuntimeError(f"stack expects a non-empty TensorList (no point of base class {cls} in the loader)")
            tmp_feat = H[cls + 1].float() / counts[cls + 1]
            base_class_gp_coding.append(post_processing_hard_coding(tmp_feat, energy=energy))
        base_class_gp_coding = torch.stack(base_class_gp_coding, dim=0)
        if len(bg_class_coding) > max_len:
            bg_class_coding = random.sample(bg_class_coding, max_len)
        bg_class_coding = torch.mean(torch.stack(bg_class_coding, dim=0), dim=0)
    return base_class_gp_coding, bg_class_coding


def collect_new_clsss_gp_coding_sum(new_cls_gp_feat_dict, energy):
    """train.py:221-241: {novel class: [ (m_i, G) one-hot GW features ]} -> (num_new, G) multi-hot codings"""
    new_class_gp_coding = []
    for cls in sorted(new_cls_gp_feat_dict.keys()):
        print('processing {}'.format(cls))
        tmp_feat = torch.sum(torch.cat(new_cls_gp_feat_dict[cls], dim=0), dim=0)
        tmp_feat = tmp_feat / torch.sum(tmp_feat)
        new_class_gp_coding.append(post_processing_hard_coding(tmp_feat, energy=energy))
    return torch.stack(new_class_gp_coding, dim=0)


def get_new_proto_Geo2SemProto(val_supp_loader, model, base_num=16, novel_num=5, novel_class_list=None, train_loader_NoAug=None,
                               base_class_coding=None, energy=None):
    """train.py:240-305: prototypes of the novel classes (mean foreground feature of every support sample, averaged per
    class, eqn. 1) next to the learnt base prototypes, all L2-normalised, plus the novel classes' GW codings.
    val_supp_loader yields (input (b, d, n), target (b, n) binary foreground mask, cls_id (b,)) with ANY batch size (the
    reference needs bs = 1 and calls Get_Fg_Feat per sample).  Per batch: one fused forward, a masked mean of the point
    features and one joint histogram (sample x geometric word) of the foreground points.
    -> (gened_proto (classes, 128) L2-normalised, novel_class_coding (n_novel, G))"""
    model.eval()
    G = model.gp.shape[0]
    with torch.no_grad():
        new_cls_feat_dict = {cls: [] for cls in novel_class_list}
        new_cls_gp_hist = {cls: [] for cls in novel_class_list}
        for input, target, cls_id in val_supp_loader:
            input = input.cuda()
            target = target.cuda()
            point_feat, assignment, _ = model._features(input)               # (b, 128, n), (b, n)
            b, n = target.shape
            fg = (target == 1)
            cnt = fg.sum(dim=1)
            feat = (point_feat * fg.unsqueeze(1)).sum(dim=2) / cnt.unsqueeze(1)      # mean over the foreground points
            blk = torch.arange(b, device=input.device, dtype=torch.int32).unsqueeze(1).expand(b, n)
            hist = block_gw_histogram(torch.where(fg, blk, torch.full_like(blk, -1)), assignment, b, G)
            for i in range(b):
                c = int(cls_id[i])
                new_cls_feat_dict[c].append(feat[i:i + 1])
                new_cls_gp_hist[c].append(hist[i:i + 1].float())                     # = sum of the one-hot GW rows
        gened_proto = torch.zeros_like(model.main_proto, requires_grad=False)
        gened_proto[:base_num, :] = model.main_proto[:base_num, :].detach().clone()
        for cls in novel_class_list:
            gened_proto[cls, :] = torch.mean(torch.cat(new_cls_feat_dict[cls], dim=0), dim=0, keepdim=False)
        gened_proto = torch.nn.functional.normalize(gened_proto, dim=1, p=2)
        novel_class_coding = collect_new_clsss_gp_coding_sum(new_cls_gp_hist, energy=energy)
    return gened_proto, novel_class_coding
