"""Geometric-word GFS model -- drop-in for the reference's model/capl.py, head computed by the sm_100a kernels.

Kept from the reference (file:line):
  mpti_net_Point_GeoAsWeight_v2(classes, criterion, args, base_num, gp, energy)      model/capl.py:21-69
    .getFeatures(x)            -> (point_feat, semantic_feat, one_hot_feat)          :324-362
    .get_pred(x, proto, use_bg_proto)                                                :290-322
    .post_refine_proto_v2(proto, x, point_feat, use_bg_proto)                        :245-287
    .get_gp_weight(gp_classifier, gp_feat, use_bg_weight, gt_label, th)              :92-142
    .forward(x, y, gened_proto, gen_proto, eval_model, ...)                          :144-242
    .Get_Fg_Feat(x, y)                                                               :71-88
    .generate_fake_proto / .post_processing_hard_coding                              :364-433
  BaseLearner                                                                        :435-457
State-dict keys: encoder.*, base_learner.convs.*, att_learner.{q,k,v}_map.weight, main_proto, bg_proto, fusion.{0,1}.*
"""
import random

import torch
import torch.nn.functional as F
from torch import nn

from gfs3d import ops
from model.attention import SelfAttention
from model.dgcnn import DGCNN, BaseLearner, _Folded, _cm, _state_key, fold_bn

manual_seed = 321
torch.manual_seed(manual_seed)
random.seed(manual_seed)


class mpti_net_Point_GeoAsWeight_v2(nn.Module):
    def __init__(self, classes=13, criterion=nn.CrossEntropyLoss(), args=None, base_num=7, gp=None, energy=None):
        super(mpti_net_Point_GeoAsWeight_v2, self).__init__()
        assert classes > 1
        self.criterion = criterion
        self.classes = classes
        self.encoder = DGCNN(args.edgeconv_widths, args.dgcnn_mlp_widths, args.pc_in_dim, k=args.dgcnn_k, return_edgeconvs=True)
        self.base_learner = BaseLearner(args.dgcnn_mlp_widths[-1], args.base_widths)
        self.att_learner = SelfAttention(args.dgcnn_mlp_widths[-1], args.output_dim)
        self.feat_dim = args.edgeconv_widths[0][-1] + args.output_dim + args.base_widths[-1]
        self.gp = gp                       # plain attribute, NOT a buffer (model/capl.py:49-50): it travels as the .pkl
        self.gp.requires_grad = False
        main_dim = 128
        self.main_proto = nn.Parameter(torch.randn((classes, main_dim)))
        self.bg_proto = nn.Parameter(torch.randn((1, main_dim)))
        self.args = args
        self.base_num = base_num
        self.fusion = nn.Sequential(nn.Conv1d(in_channels=self.feat_dim + self.gp.shape[0], out_channels=main_dim, kernel_size=1),
                                    nn.BatchNorm1d(main_dim), nn.LeakyReLU(0.2))
        self.energy = energy
        print('model using energy: {}'.format(self.energy))
        self._folded = _Folded()
        self._warned_eval_grad = False

    # ------------------------------------------------------------------ weight folding for the head
    def _prepare(self, device):
        key = _state_key(self.fusion, device) + (id(self.gp), self.gp._version)
        if self._folded.key != key:
            G = self.gp.shape[0]
            sem = self.feat_dim
            if sem != 192 or self.encoder.n_edgeconv * 64 != self.gp.shape[1] or G > 512:
                raise NotImplementedError(
                    f"head shapes (feat_dim={sem}, GW basis {tuple(self.gp.shape)}) are outside what the sm_100a head is built for "
                    "(feat_dim 192, <=512 geometric words of width 64*n_edgeconv)")
            with torch.no_grad():
                Gp = (G + 63) // 64 * 64
                gp_l2 = F.normalize(self.gp.detach().float().to(device), p=2, dim=1)            # (G, D)
                gp_l2t = torch.zeros(gp_l2.shape[1], Gp, dtype=torch.float32, device=device)
                gp_l2t[:, :G] = gp_l2.t()
                conv, bn = self.fusion[0], self.fusion[1]
                s, t = fold_bn(bn)
                w = conv.weight.detach().float().reshape(conv.weight.shape[0], conv.weight.shape[1])   # (128, G + 192)
                # kernel-side column order: [semantic 192 | cosine G | zero pad]  (reference order: [cosine G | semantic 192])
                wk = torch.zeros(w.shape[0], sem + Gp, dtype=torch.float32, device=device)
                wk[:, :sem] = w[:, G:]
                wk[:, sem:sem + G] = w[:, :G]
                shift = (conv.bias.detach().float() * s + t).contiguous()
                data = dict(G=G, Gp=Gp, gp_l2t=gp_l2t.contiguous(), wp=ops.pack_weight(wk, s), shift=shift,
                            kblocks=(sem + Gp) // 64, nout=w.shape[0])
            self._folded.key, self._folded.data = key, data
        return self._folded.data

    def invalidate_folded(self):
        """drop every folded / packed inference weight of the model.  The caches are keyed on (id, tensor._version) of the
        parameters and buffers, which optimiser steps, load_state_dict and in-place ops bump; edits through ``.data`` (EMA,
        weight surgery) do not -- call this after such an edit."""
        for mod in self.modules():
            f = getattr(mod, "_folded", None)
            if isinstance(f, _Folded):
                f.key = f.data = None
            if hasattr(mod, "_key") and hasattr(mod, "_wp"):
                mod._key = mod._wp = None
        self._mp_key = self._coding_key = None

    # ------------------------------------------------------------------ fused feature extraction
    def _features(self, x, need_semantic=False):
        """-> (point_feat (B,128,N) fp32 cm, assignment (B,N) int32, semantic (B,192,N) fp32 or None)"""
        if self.training:
            return self._features_train(x, need_semantic)
        if not x.is_cuda:
            raise RuntimeError("the GW model needs CUDA tensors: the hot path has no CPU fallback")
        if torch.is_grad_enabled() and not self._warned_eval_grad and any(p.requires_grad for p in self.encoder.parameters()):
            # the fused inference kernels build no autograd graph: with model.eval() and gradients enabled the reference would
            # back-propagate into the backbone (running-stat BatchNorm), this path would silently leave those gradients at zero
            import warnings
            warnings.warn("GFS drop-in: eval-mode features are computed by the fused inference kernels and carry no autograd graph; "
                          "only the prototypes receive gradients. Call under torch.no_grad(), or model.train() to fine-tune the "
                          "backbone.", RuntimeWarning, stacklevel=3)
            self._warned_eval_grad = True
        hd = self._prepare(x.device)
        x = _cm(x)
        B, _, N = x.shape
        M = B * N
        fus_in = ops.new_act(M, hd["kblocks"], x.device, zero=False)                 # [level1 | att | level3 | cosine_feat | pad]
        enc = self.encoder.forward_fused(x, want_lvl2_cm=False, level1_act=fus_in, level1_kb=0)
        semantic = torch.empty(B, 192, N, dtype=torch.float32, device=x.device) if need_semantic else None
        self.att_learner.forward_fused(enc.lvl2_act, B, N, y_act=fus_in, y_kb=1,
                                       y_cm=semantic[:, 64:128, :] if need_semantic else None)
        self.base_learner.forward_fused(enc.lvl2_act, B, N, y_act=fus_in, y_kb0=2,
                                        y_cm=semantic[:, 128:192, :] if need_semantic else None)
        assignment, _ = ops.gw_project(enc.ec, hd["gp_l2t"], hd["G"], cosine_act=fus_in, kb0=3)
        point_feat = torch.empty(B, hd["nout"], N, dtype=torch.float32, device=x.device)
        ops.linear(fus_in, 0, hd["kblocks"], hd["wp"], hd["shift"], hd["nout"], ops.ACT_LRELU02, B, N, y_cm=point_feat)
        if need_semantic:
            semantic[:, 0:64, :].copy_(enc.ec[:, 0:64, :])
        return point_feat, assignment, semantic

    def _features_train(self, x, need_semantic=False):
        """training mode (model/capl.py:324-362 under model.train()): fp32, batch-statistics BatchNorm, differentiable through
        the hand-written training kernels (gfs3d/train_ops.py).  Same return convention as _features.
        A BatchNorm in eval mode is frozen (running statistics, left unchanged).  A frozen encoder -- in eval mode, no parameter
        requiring grad, x not requiring grad -- receives no gradient, so its eval-mode outputs come from the fused inference
        kernels (bit-identical to self.encoder(x) in eval mode): no autograd graph and no per-edge tensors."""
        from gfs3d.train_ops import ConvBNAct, ConvConstW, batch_stats, from_cm, to_cm, update_running_stats
        if not x.is_cuda:
            raise RuntimeError("the GW model needs CUDA tensors: the hot path has no CPU fallback")
        B, _, N = x.shape
        M = B * N
        enc = self.encoder
        if not enc.training and not x.requires_grad and not any(p.requires_grad for p in enc.parameters()):
            out = enc.forward_fused(x, want_lvl2_cm=True)
            ecs, lvl2 = list(to_cm(out.ec).split(64, dim=0)), to_cm(out.lvl2_cm)
        else:
            ecs, lvl2 = enc.forward_train(x)                             # channel-major (64, M) x3, (256, M)
        lvl3 = self.base_learner.forward_train(lvl2)
        att = self.att_learner.forward_train(lvl2, B, N)
        ec = torch.cat(ecs, dim=0)                                       # (192, M)
        semantic = torch.cat([ecs[0], att, lvl3], dim=0)                 # (192, M)
        ec_l2 = ec / ec.norm(dim=0, keepdim=True).clamp_min(1e-12)
        gp_l2 = F.normalize(self.gp.detach().float().to(x.device), p=2, dim=1)
        cos = ConvConstW.apply(ec_l2, gp_l2)                             # (G, M)
        cosine_feat = torch.softmax(10 * cos, dim=0)
        assignment = cosine_feat.argmax(dim=0).reshape(B, N).int()
        conv, bn = self.fusion[0], self.fusion[1]
        w = conv.weight.reshape(conv.weight.shape[0], conv.weight.shape[1])
        pf, m, v = ConvBNAct.apply(torch.cat([cosine_feat, semantic], dim=0), w, conv.bias, bn.weight, bn.bias, bn.running_mean,
                                   bn.running_var, 0.2, batch_stats(bn))
        if bn.training:
            update_running_stats(bn, m, v, M)
        return from_cm(pf, B, N), assignment, (from_cm(semantic, B, N) if need_semantic else None)

    def getFeatures(self, x, segment_label=None):
        """(B, C_in, N) -> point_feat (B,128,N), semantic_feat (B,192,N), one_hot_feat (B,G,N) float 0/1"""
        point_feat, assignment, semantic = self._features(x, need_semantic=True)
        one_hot = F.one_hot(assignment.long(), num_classes=self.gp.shape[0]).transpose(2, 1).float()
        return point_feat, semantic, one_hot

    def Get_Fg_Feat(self, x, y):
        y = y[0]
        point_feat, _, gp_feat = self.getFeatures(x)
        fg_feat = point_feat[0][:, y == 1]
        fg_gp_feat = gp_feat[0][:, y == 1]
        return fg_feat.transpose(1, 0), fg_gp_feat.transpose(1, 0)

    # ------------------------------------------------------------------ logits / prototypes
    def get_pred(self, x, proto, use_bg_proto=False, xn=None):
        """10 * cos(proto, x): x (b, c, n); proto (cls, c) or (b, cls, c); optional bg_proto row first -> (b, cls, n).
        xn: F.normalize(x, dim=1) if the caller already has it (the training forward normalises the point features once)"""
        if proto.dim() == 3:
            if use_bg_proto:
                proto = torch.cat([self.bg_proto.unsqueeze(0).repeat(proto.shape[0], 1, 1), proto], dim=1)
            pn = F.normalize(proto, p=2, dim=-1)
        else:
            if use_bg_proto:
                proto = torch.cat([self.bg_proto, proto], dim=0)
            pn = F.normalize(proto, p=2, dim=1)
        if torch.is_grad_enabled() and (x.requires_grad or pn.requires_grad):
            # training branch: O(B * cls * N) prototype algebra stays in differentiable torch ops (DESIGN.md section 1)
            return torch.matmul(pn if pn.dim() == 3 else pn.unsqueeze(0), xn if xn is not None else F.normalize(x, p=2, dim=1)) * 10
        return ops.cos_logits(_cm(x), pn.detach())

    def _main_proto_l2(self):
        """F.normalize(main_proto) for the eval forward, cached on the parameter's version (three tiny launches per call otherwise)"""
        p = self.main_proto
        key = (id(p), p._version, str(p.device))
        if getattr(self, "_mp_key", None) != key:
            with torch.no_grad():
                self._mp_l2 = F.normalize(p.detach(), p=2, dim=1)
            self._mp_key = key
        return self._mp_l2

    def post_refine_proto_v2(self, proto, x, point_feat, use_bg_proto=False, xn=None):
        """query-adaptive prototype refinement (eqn. 6) -> (b, classes, c)"""
        pred = self.get_pred(x, proto, use_bg_proto, xn=xn)
        if pred.requires_grad or point_feat.requires_grad:
            pred_proto = torch.softmax(pred, dim=2) @ point_feat.permute(0, 2, 1)
        else:
            pred_proto = ops.softmax_pool(pred, _cm(point_feat))
        if use_bg_proto:
            pred_proto = pred_proto[:, 1:, :]
        w = (F.normalize(pred_proto, 2, -1) * F.normalize(proto, 2, -1).unsqueeze(0)).sum(-1, keepdim=True)
        w = w * (w > 0).float()
        return w * pred_proto + (1 - w) * proto.unsqueeze(0)

    def get_gp_weight(self, gp_classifier, gp_feat, use_bg_weight=False, gt_label=None, th=None):
        """(n_cls, k) coding x one-hot (b, k, n) -> weight (b, cls, n) in {1, th} and the two diagnostic accuracies.
        The eval forward does not call this (the weight is applied inside gfs_cos_logits); kept for API parity."""
        assignment = gp_feat.argmax(dim=1)                                   # (b, n)
        score = gp_classifier[:, assignment].permute(1, 0, 2)                # (b, cls, n) == coding @ one_hot
        acc, novel_acc = 0., 0.
        if gt_label is not None and not use_bg_weight:
            per_point = torch.gather(score, 1, gt_label.unsqueeze(1)).squeeze(1)
            acc = per_point.mean()
            novel_mask = gt_label > self.base_num - 1
            novel_acc = per_point[novel_mask].mean() if novel_mask.sum() > 0 else torch.zeros_like(acc)
        elif gt_label is not None and use_bg_weight:
            gt_one_hot = F.one_hot(gt_label, num_classes=score.shape[1] + 1).transpose(2, 1)[:, 1:, :]
            acc = (gt_one_hot * score).sum(dim=1).mean()
        weight = torch.ones_like(score)
        weight[score == 1] = th
        if use_bg_weight:
            weight = torch.cat([torch.ones_like(weight[:, :1]), weight], dim=1)
            gt_mask = F.one_hot(gt_label, num_classes=score.shape[1] + 1).transpose(2, 1)
            weight[gt_mask == 1] = 1
        return weight, acc, novel_acc

    def forward(self, x, y=None, gened_proto=None, gen_proto=False, eval_model=False, target_cls=None, segment_label=None,
                geo2sem_proto=None, base_class_coding=None, novel_class_coding=None, bg_class_coding=None):
        base_num = self.base_num
        if not eval_model:
            return self._forward_train(x, y)
        point_feat, assignment, _ = self._features(x)
        if gened_proto.dim() == 3:
            gened_proto = gened_proto[0]
        with torch.no_grad():
            # post_refine_proto_v2 (eqn. 6), the base/novel prototype update of model/capl.py:117-120 and the normalisation
            # of get_pred as one kernel (gfs_refine_proto) instead of ~25 small tensor ops on (B, classes, 128)
            pred = ops.cos_logits(_cm(point_feat), self._main_proto_l2())          # get_pred(point_feat, main_proto)
            pred_proto = ops.softmax_pool(pred, _cm(point_feat))
            refine_l2 = ops.refine_proto(pred_proto, self.main_proto.detach(), gened_proto, base_num)
            ck = (id(base_class_coding), base_class_coding._version, id(novel_class_coding), novel_class_coding._version)
            if getattr(self, "_coding_key", None) != ck:                           # the codings change once per evaluation, not per batch
                self._coding_cat, self._coding_key = torch.cat([base_class_coding, novel_class_coding], dim=0).float(), ck
                self._coding_refs = (base_class_coding, novel_class_coding)       # keeps the ids of the key alive
            gp_coding = self._coding_cat
            x_pre = ops.cos_logits(point_feat, refine_l2, gp_coding, assignment, float(self.args.eval_weight))
            # diagnostics of model/capl.py:104-114: mean of coding[gt, assignment] over all / novel points
            if y is not None:
                per_point = gp_coding[y.long(), assignment.long()]
                gp_acc = per_point.mean()
                novel = y > base_num - 1
                gp_novel_acc = per_point[novel].mean() if novel.sum() > 0 else torch.zeros_like(gp_acc)
            else:
                gp_acc, gp_novel_acc = 0., 0.
        return x_pre, gp_acc, gp_novel_acc

    def _forward_train(self, x, y):
        """model/capl.py:194-242: episodic base training.  Second half of the batch plays the support set for the fake-novel
        prototypes (eqn. 8), whole batch is the query; loss = 0.5 * (CE(pred with fake protos) + CE(pred with refined protos))."""
        base_num = self.base_num
        point_feat, _, _ = self._features(x)
        fake_num = x.size(0) // 2
        # the L2-normalised point features are needed three times (support prototypes, both logit evaluations): once is enough
        xn = F.normalize(point_feat, p=2, dim=1)
        ori_proto, fake_novel = self.generate_fake_proto(x=point_feat[fake_num:], y=y[fake_num:], main_proto=self.main_proto.clone(),
                                                         xn=xn[fake_num:])
        x_pre_1 = self.get_pred(x=point_feat, proto=ori_proto, use_bg_proto=True, xn=xn)
        loss_ce_1 = self._loss(x_pre_1, y)
        refine_proto = self.post_refine_proto_v2(proto=self.main_proto.clone(), x=point_feat, point_feat=point_feat, use_bg_proto=True, xn=xn)
        post_refine_proto = refine_proto.clone()
        post_refine_proto[:, :base_num] = post_refine_proto[:, :base_num] + ori_proto[:base_num].unsqueeze(0)
        post_refine_proto[:, base_num:] = post_refine_proto[:, base_num:] * 0 + ori_proto[base_num:].unsqueeze(0)
        x_pre_2 = self.get_pred(x=point_feat, proto=post_refine_proto, use_bg_proto=True, xn=xn)
        loss_ce_2 = self._loss(x_pre_2, y)
        return x_pre_2.max(1)[1], 0.5 * loss_ce_2 + 0.5 * loss_ce_1

    def _loss(self, logits, y):
        """self.criterion(logits (b, cls, n), y (b, n)).  torch's CUDA loss for the (b, cls, n) layout (nll_loss2d) adds the
        per-block partial sums with atomics; under torch.use_deterministic_algorithms a CrossEntropyLoss is evaluated on the
        (b*n, cls) view instead, whose reduction runs in a fixed order: the same loss, reproducible to the bit."""
        if (torch.are_deterministic_algorithms_enabled() and logits.is_cuda and isinstance(self.criterion, nn.CrossEntropyLoss)
                and self.criterion.reduction != "none"):
            return self.criterion(logits.transpose(1, 2).reshape(-1, logits.shape[1]), y.reshape(-1))
        return self.criterion(logits, y)

    def generate_fake_proto(self, x, y, main_proto, fake_novel=None, post_processing=False, xn=None):
        """model/capl.py:364-411 (training only): half of the classes present in the support half-batch are declared
        'fake novel'; their classifier rows are replaced by the masked mean of the L2-normalised support features.
        xn: the normalised support features if the caller has them (x / (|x| + 1e-12) and F.normalize agree in fp32 unless
        |x| < 1e-5).  On CUDA the masked sums of ALL classes come from one deterministic segmented-sum kernel
        (gfs3d.train_ops.ClassSums) instead of one mask / multiply / reduce chain per class."""
        tmp_y = y.unsqueeze(1)
        unique_y = list(tmp_y.unique())
        if fake_novel is None:
            if 0 in unique_y:
                unique_y.remove(0)
            novel_num = len(unique_y) // 2
            fake_novel = random.sample(unique_y, novel_num)
        new_proto = main_proto / (torch.norm(main_proto, 2, 1, True) + 1e-12)
        x = xn if xn is not None else x / (torch.norm(x, 2, 1, True) + 1e-12)
        class_sums = None
        if x.is_cuda and len(fake_novel) > 0 and x.shape[1] % 4 == 0:
            from gfs3d.train_ops import ClassSums
            rows = x.permute(0, 2, 1).reshape(-1, x.shape[1])                      # (b*n, c) point-major
            ncls = main_proto.size(0)                                              # labels 0 (background) .. ncls; anything else
            lab = y.reshape(-1)                                                    # (ignore_index 255) goes to a spare bin
            lab = torch.where((lab < 0) | (lab > ncls), torch.full_like(lab, ncls + 1), lab)
            class_sums, class_counts = ClassSums.apply(rows, lab, ncls + 2)
        for fn in fake_novel:
            if class_sums is not None:
                tmp_feat = class_sums[fn.long()] / (class_counts[fn.long()].float() + 1e-12)
            else:
                tmp_mask = (tmp_y == fn).float()
                tmp_feat = (x * tmp_mask).sum(0).sum(-1) / (tmp_mask.sum(0).sum(-1) + 1e-12)
            if post_processing:
                tmp_feat = self.post_processing_hard_coding(tmp_feat)
            fake_vec = torch.zeros(new_proto.size(0), 1, device=new_proto.device)
            fake_vec[fn.long() - 1] = 1
            new_proto = new_proto * (1 - fake_vec) + tmp_feat.unsqueeze(0) * fake_vec
        return new_proto, fake_novel

    def post_processing_hard_coding(self, coding):
        """keep the most frequent geometric words up to `energy` of the mass -> multi-hot (model/capl.py:413-433)"""
        order = torch.argsort(coding, descending=True)
        csum = torch.cumsum(coding[order], dim=0)
        keep = int((csum > self.energy * coding.sum()).nonzero()[0]) + 1 if (csum > self.energy * coding.sum()).any() else len(order)
        mask = torch.zeros_like(coding)
        mask[order[:keep]] = 1
        coding[mask == 1] = 1
        coding[mask == 0] = 0
        return coding
