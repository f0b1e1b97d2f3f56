"""Train-time target layers and losses of the reference on the device (SURVEY A16 / 8f-4).

Host-side mirror of `_AnchorTargetLayer` (lib/model/rpn/anchor_target_layer.py:42-164), `_ProposalTargetLayer`
(lib/model/rpn/proposal_target_layer.py:36-333), the RPN / RCNN losses (stereo_rpn.py:114-140,
stereo_rcnn.py:201-311), the multi-task sum (trainval_net.py:214-219) and `clip_gradient` (net_utils.py:37-49) over
libstereo_b200's kernels (csrc/train_targets.cu, csrc/train_loss.cu).  No host synchronisation anywhere: counts,
sampled indices and losses stay on the device.  Backbone dgrad / wgrad is NOT part of this module.
"""
import ctypes

import numpy as np
import torch

from . import lib as _l
from .ops import check, ptr, stream_ptr, workspace, _f32c

CFG = dict(                                          # lib/model/utils/config.py:55-108,173
    RPN_NEGATIVE_OVERLAP=0.3, RPN_POSITIVE_OVERLAP=0.7, RPN_FG_FRACTION=0.5, RPN_BATCHSIZE=512,
    BATCH_SIZE=512, FG_FRACTION=0.25, FG_THRESH=0.5, BG_THRESH_HI=0.5, BG_THRESH_LO=0.0,
    BBOX_NORMALIZE_MEANS=(0.0, 0.0, 0.0, 0.0), BBOX_NORMALIZE_STDS=(0.1, 0.1, 0.2, 0.2),
    DIM_NORMALIZE_MEANS=(1.6, 1.5, 4.0, 0.0, 0.0), DIM_NORMALIZE_STDS=(0.5, 0.5, 0.5, 0.5, 0.5),
    KPTS_GRID=28,
)


def random_words(shape, device, generator=None):
    """uint32 random words for the samplers (stored as int32 bit patterns: torch has no uint32 arithmetic)"""
    return torch.randint(-2 ** 31, 2 ** 31, shape, dtype=torch.int32, device=device, generator=generator)


def _words(t):
    assert t.dtype == torch.int32 and t.is_contiguous()
    return t


def generate_anchors(feat_shapes, device, ratios=None, scales=None, strides=None):
    """generate_anchors_all_pyramids (generate_anchors.py:157-173) on the device -> [A,4] fp32"""
    from .ops import make_proposal_cfg
    L = _l.load()
    pc = make_proposal_cfg("TRAIN", [list(map(int, s)) for s in feat_shapes], ratios=ratios, scales=scales, strides=strides)
    A = sum(int(h) * int(w) for h, w in feat_shapes) * pc.n_ratios
    out = torch.empty(A, 4, dtype=torch.float32, device=device)
    check(L.sb_generate_anchors(ctypes.byref(pc), A, ptr(out), stream_ptr()), "sb_generate_anchors")
    return out


def anchor_targets(anchors, gt_left, gt_right, gt_merge, im_info, keys, cfg=CFG):
    """_AnchorTargetLayer.forward: anchors [A,4] fp32, gt_* [B,K,5], im_info = (H, W, ...) of image 0 as Python
    numbers, keys [B,A] int32 words -> labels [B,A], targets_left [B,A,4], targets_right [B,A,4], inside_w [B,A],
    outside_w [B,A]"""
    L = _l.load()
    A = anchors.shape[0]
    B, K = gt_left.shape[:2]
    dev = anchors.device
    assert keys.shape == (B, A)
    labels = torch.empty(B, A, dtype=torch.float32, device=dev)
    tl = torch.empty(B, A, 4, dtype=torch.float32, device=dev)
    tr = torch.empty(B, A, 4, dtype=torch.float32, device=dev)
    iw = torch.empty(B, A, dtype=torch.float32, device=dev)
    ow = torch.empty(B, A, dtype=torch.float32, device=dev)
    nbytes = L.sb_anchor_targets_workspace(B, A)
    ws = workspace(nbytes, dev, "anchor_targets")
    num_fg = int(cfg["RPN_FG_FRACTION"] * cfg["RPN_BATCHSIZE"])
    check(L.sb_anchor_targets(ptr(_f32c(anchors)), A, ptr(_f32c(gt_left)), ptr(_f32c(gt_right)), ptr(_f32c(gt_merge)),
                              B, K, int(im_info[0]), int(im_info[1]), ptr(_words(keys)),
                              float(cfg["RPN_NEGATIVE_OVERLAP"]), float(cfg["RPN_POSITIVE_OVERLAP"]),
                              int(cfg["RPN_BATCHSIZE"]), num_fg, ptr(ws), nbytes, ptr(labels), ptr(tl), ptr(tr),
                              ptr(iw), ptr(ow), stream_ptr()), "sb_anchor_targets")
    return labels, tl, tr, iw, ow


def _pt_cfg(cfg):
    c = _l.ProposalTargetCfg()
    c.rois_per_image = int(cfg["BATCH_SIZE"])
    c.fg_rois_per_image = int(np.round(cfg["FG_FRACTION"] * cfg["BATCH_SIZE"]))
    c.fg_thresh, c.bg_thresh_hi, c.bg_thresh_lo = cfg["FG_THRESH"], cfg["BG_THRESH_HI"], cfg["BG_THRESH_LO"]
    c.bbox_means = (ctypes.c_float * 4)(*cfg["BBOX_NORMALIZE_MEANS"])
    c.bbox_stds = (ctypes.c_float * 4)(*cfg["BBOX_NORMALIZE_STDS"])
    c.dim_means = (ctypes.c_float * 5)(*cfg["DIM_NORMALIZE_MEANS"])
    c.dim_stds = (ctypes.c_float * 5)(*cfg["DIM_NORMALIZE_STDS"])
    c.kpts_grid = int(cfg["KPTS_GRID"])
    return c


def proposal_targets(rois_left, rois_right, gt_left, gt_right, gt_dim_orien, gt_kpts, keys, words, cfg=CFG):
    """_ProposalTargetLayer.forward: rois_* [B,R,5], gt_* [B,K,5], gt_dim_orien [B,K,5], gt_kpts [B,K,6],
    keys [B,R+K] / words [B,S] int32 random words -> dict like oracle.train_targets.proposal_target_layer
    (kpts_targets int32, plus status [B])"""
    L = _l.load()
    B, R = rois_left.shape[:2]
    K = gt_left.shape[1]
    S = int(cfg["BATCH_SIZE"])
    dev = rois_left.device
    assert keys.shape == (B, R + K) and words.shape == (B, S)
    f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
    o = dict(rois_left=f(B, S, 5), rois_right=f(B, S, 5), labels=f(B, S), bbox_targets_left=f(B, S, 4),
             bbox_targets_right=f(B, S, 4), dim_orien_targets=f(B, S, 5),
             kpts_targets=torch.empty(B, S, 3, dtype=torch.int32, device=dev), kpts_weight=f(B, S, 3),
             inside_w=f(B, S, 4), outside_w=f(B, S, 4),
             keep_inds=torch.empty(B, S, dtype=torch.int32, device=dev),
             status=torch.empty(B, dtype=torch.int32, device=dev))
    c = _pt_cfg(cfg)
    check(L.sb_proposal_targets(ptr(_f32c(rois_left)), ptr(_f32c(rois_right)), B, R, ptr(_f32c(gt_left)),
                                ptr(_f32c(gt_right)), ptr(_f32c(gt_dim_orien)), ptr(_f32c(gt_kpts)), K,
                                ptr(_words(keys)), ptr(_words(words)), ctypes.byref(c), ptr(o["rois_left"]),
                                ptr(o["rois_right"]), ptr(o["labels"]), ptr(o["bbox_targets_left"]),
                                ptr(o["bbox_targets_right"]), ptr(o["dim_orien_targets"]), ptr(o["kpts_targets"]),
                                ptr(o["kpts_weight"]), ptr(o["inside_w"]), ptr(o["outside_w"]), ptr(o["keep_inds"]),
                                ptr(o["status"]), stream_ptr()), "sb_proposal_targets")
    return o


def rpn_loss(rpn_cls_score, rpn_bbox_pred, labels, targets_left, targets_right, inside_w, outside_w, uncert=None,
             grads=True):
    """stereo_rpn.py:114-140: rpn_cls_score [B,A,2], rpn_bbox_pred [B,A,6] -> losses [2] (cls, box) and, with grads,
    d loss / d rpn_cls_score, d loss / d rpn_bbox_pred (times exp(-uncert[0..1]) if uncert is given)"""
    L = _l.load()
    B, A = labels.shape
    dev = labels.device
    losses = torch.empty(2, dtype=torch.float32, device=dev)
    d_cls = torch.empty_like(rpn_cls_score) if grads else None
    d_box = torch.empty_like(rpn_bbox_pred) if grads else None
    nbytes = L.sb_loss_workspace_bytes()
    ws = workspace(nbytes, dev, "loss")
    check(L.sb_rpn_loss(ptr(_f32c(rpn_cls_score)), ptr(_f32c(rpn_bbox_pred)), ptr(_f32c(labels)),
                        ptr(_f32c(targets_left)), ptr(_f32c(targets_right)), ptr(_f32c(inside_w)),
                        ptr(_f32c(outside_w)), B, A, ptr(uncert) if uncert is not None else None, ptr(ws), nbytes,
                        ptr(losses), ptr(d_cls) if grads else None, ptr(d_box) if grads else None, stream_ptr()),
          "sb_rpn_loss")
    return (losses, d_cls, d_box) if grads else losses


def rcnn_loss(cls_score, bbox_pred, dim_orien_pred, kpts_pred, left_border_pred, right_border_pred, tgt, uncert=None,
              grads=True, kpts_grid=28):
    """stereo_rcnn.py:201-311: predictions of the R = B*S sampled RoIs (bbox_pred [R,6C], dim_orien_pred [R,5C] per
    class), tgt = proposal_targets(...) -> losses [4] (cls, bbox, dim_orien, kpts) and, with grads, the six gradients"""
    L = _l.load()
    R, C = cls_score.shape
    dev = cls_score.device
    losses = torch.empty(4, dtype=torch.float32, device=dev)
    preds = [_f32c(t) for t in (cls_score, bbox_pred, dim_orien_pred, kpts_pred, left_border_pred, right_border_pred)]
    g = [torch.empty_like(t) for t in preds] if grads else [None] * 6
    check(L.sb_rcnn_loss(*[ptr(t) for t in preds], ptr(_f32c(tgt["labels"])), ptr(_f32c(tgt["bbox_targets_left"])),
                         ptr(_f32c(tgt["bbox_targets_right"])), ptr(_f32c(tgt["dim_orien_targets"])),
                         ptr(tgt["kpts_targets"]), ptr(_f32c(tgt["kpts_weight"])), ptr(_f32c(tgt["inside_w"])),
                         ptr(_f32c(tgt["outside_w"])), R, C, kpts_grid, ptr(uncert) if uncert is not None else None,
                         ptr(losses), *[ptr(t) if t is not None else None for t in g], stream_ptr()), "sb_rcnn_loss")
    return (losses, g) if grads else losses


def multitask_loss(losses, uncert):
    """trainval_net.py:214-219: losses [n], uncert [n] -> total [1], d total / d uncert [n]"""
    L = _l.load()
    n = losses.numel()
    total = torch.empty(1, dtype=torch.float32, device=losses.device)
    d_u = torch.empty(n, dtype=torch.float32, device=losses.device)
    check(L.sb_multitask_loss(ptr(_f32c(losses)), ptr(_f32c(uncert)), n, ptr(total), ptr(d_u), stream_ptr()),
          "sb_multitask_loss")
    return total, d_u


def clip_gradient(grads, clip_norm):
    """net_utils.clip_gradient over a list of fp32 gradient tensors, in place -> norm [2] (total norm, factor)"""
    L = _l.load()
    n = len(grads)
    dev = grads[0].device
    assert all(g.dtype == torch.float32 and g.is_contiguous() for g in grads)
    ptrs = (ctypes.c_void_p * n)(*[g.data_ptr() for g in grads])
    counts = (ctypes.c_size_t * n)(*[g.numel() for g in grads])
    nbytes = L.sb_clip_gradient_workspace(n)
    ws = workspace(nbytes, dev, "clip")
    out = torch.empty(2, dtype=torch.float32, device=dev)
    check(L.sb_clip_gradient(ptrs, counts, n, float(clip_norm), ptr(ws), nbytes, ptr(out), stream_ptr()),
          "sb_clip_gradient")
    return out


# ---------------------------------------------------------------------------------------------- box-head training step
# RCNN_top (Conv2d 512->2048 k7 s7 + ReLU + Dropout(0.2), Conv2d 2048->2048 k1 + ReLU + Dropout(0.2); resnet.py:256-263)
# and the three tail linears (resnet.py:282-285), as stereo_rcnn.py:248-257 runs them in training.  fp16 engine only.
# The forward reuses the engine's packed weights and conv kernels; the backward is sb_gemm_tc for the four products,
# SIMT kernels for the tail, the dropout / ReLU masks and the device-chosen fp16 scaling, and the deterministic
# pyramid RoIAlign adjoint into the feature gradients.  Stream ordered, no host reads: graph capturable.
DROPOUT_KEEP_FROM = 858993460          # keep where the uint32 word >= 0.2 * 2^32 (nn.Dropout(p=0.2)), scale 1 / 0.8

BOX_HEAD_PARAMS = ("RCNN_top.0.weight", "RCNN_top.0.bias", "RCNN_top.3.weight", "RCNN_top.3.bias",
                   "RCNN_cls_score.weight", "RCNN_cls_score.bias", "RCNN_bbox_pred.weight", "RCNN_bbox_pred.bias",
                   "RCNN_dim_orien_pred.weight", "RCNN_dim_orien_pred.bias")


def box_head_param_shapes(n_classes=2):
    """the reference's state_dict shapes of the box-head parameters, in BOX_HEAD_PARAMS order"""
    nc = n_classes
    return [(2048, 512, 7, 7), (2048,), (2048, 2048, 1, 1), (2048,), (nc, 2048), (nc,), (6 * nc, 2048), (6 * nc,),
            (5 * nc, 2048), (5 * nc,)]


def _need_fp16(eng):
    if not getattr(eng, "half", False):
        raise NotImplementedError("the box-head training step exists for the fp16 engine (precision='fp16') only")


def _dropout(x, words, out32=None, out16=None):
    L = _l.load()
    R, C = x.shape
    check(L.sb_dropout(ptr(x), ptr(_words(words)), R, C, ptr(out32), ptr(out16), stream_ptr()), "sb_dropout")


def box_head_forward(eng, feats, B, rois_left, rois_right, im_h, drop_words):
    """training forward of the box head (stereo_rcnn.py:248-257).  feats: {"p2".."p5": [2B,H,W,256] fp32 NHWC, left
    images first} as the engine's trunk produces them; rois_* [R,5] (batch index first); drop_words = (w6, w7), two
    int32 [R,2048] random-word tensors (train.random_words) for the dropouts after the two ReLUs of RCNN_top.
    -> ctx: the tensors the forward consumed (pooled fp16, fc6 / fc7 ReLU outputs, fc6 after dropout fp16, fc7 after
    dropout fp32, the words) and its outputs cls_score [R,nc] (logits), bbox_pred [R,6nc], dim_orien_pred [R,5nc]."""
    _need_fp16(eng)
    L = _l.load()
    from . import ops
    mk = ("p2", "p3", "p4", "p5")
    fl, fr = [feats[k][:B] for k in mk], [feats[k][B:] for k in mk]
    R = rois_left.shape[0]
    dev = rois_left.device
    w6, w7 = drop_words
    assert w6.shape == (R, 2048) and w7.shape == (R, 2048)
    pooled = torch.empty(R, 7, 7, 512, dtype=torch.float16, device=dev)
    ops.roi_align_pyramid_nhwc(fl, im_h, rois_left, 7, out=pooled, out_coff=0, half=True)
    ops.roi_align_pyramid_nhwc(fr, im_h, rois_right, 7, out=pooled, out_coff=256, half=True)
    fc6 = eng._conv(pooled.view(R, 1, 1, 7 * 7 * 512), eng.p["RCNN_top.0"], relu=True, tag="top0").view(R, 2048)
    fc6_drop = torch.empty(R, 2048, dtype=torch.float16, device=dev)
    _dropout(fc6, w6, out16=fc6_drop)
    fc7 = eng._conv(fc6_drop.view(R, 1, 1, 2048), eng.p["RCNN_top.3"], relu=True, tag="top3").view(R, 2048)
    fc7_drop = torch.empty(R, 2048, dtype=torch.float32, device=dev)
    _dropout(fc7, w7, out32=fc7_drop)
    nc = eng.n_classes
    cls = torch.empty(R, nc, dtype=torch.float32, device=dev)
    bbox = torch.empty(R, 6 * nc, dtype=torch.float32, device=dev)
    dim = torch.empty(R, 5 * nc, dtype=torch.float32, device=dev)
    check(L.sb_box_tail_logits(ptr(fc7_drop), R, 2048, nc, *[ptr(t) for t in eng.fc], ptr(cls), ptr(bbox), ptr(dim),
                               stream_ptr()), "sb_box_tail_logits")
    return dict(pooled=pooled, fc6=fc6, fc6_drop=fc6_drop, fc7=fc7, fc7_drop=fc7_drop, words6=w6, words7=w7,
                rois_left=rois_left, rois_right=rois_right, im_h=float(im_h), B=B,
                feat_shapes=[tuple(f.shape) for f in fl], cls_score=cls, bbox_pred=bbox, dim_orien_pred=dim)


def _dropout_backward(dy, y, words, db, tag):
    """-> fp16 operand g * 2^e and the device scalar 2^-e (g = dy * mask * 1.25 * ReLU'); db written"""
    L = _l.load()
    R, C = dy.shape
    nbytes = L.sb_dropout_backward_workspace(R, C)
    ws = workspace(nbytes, dy.device, tag)
    g16 = torch.empty(R, C, dtype=torch.float16, device=dy.device)
    inv = torch.empty(1, dtype=torch.float32, device=dy.device)
    check(L.sb_dropout_backward(ptr(dy), ptr(y), ptr(_words(words)), R, C, ptr(db), ptr(g16), ptr(inv), ptr(ws),
                                nbytes, stream_ptr()), "sb_dropout_backward")
    return g16, inv


def box_head_backward(eng, ctx, d_cls_score, d_bbox_pred, d_dim_orien_pred, grads=None, feat_grads=None,
                      stage_events=None):
    """adjoint of box_head_forward.  d_* = d loss / d (cls_score, bbox_pred, dim_orien_pred), e.g. from rcnn_loss.
    grads: optional {name: tensor} in the reference's state_dict shapes (BOX_HEAD_PARAMS; e.g. GradientBuckets views),
    overwritten in place; feat_grads: optional {"left": [4 tensors], "right": [...]} fp32 NHWC [B,H_l,W_l,256].
    stage_events: optional list; a (stage name, recorded CUDA event) pair is appended after each stage (per-stage
    timing of eager runs).  -> (grads, feat_grads)"""
    _need_fp16(eng)
    L = _l.load()
    from . import ops
    R = ctx["pooled"].shape[0]
    dev = ctx["pooled"].device
    nc = eng.n_classes
    if grads is None:
        grads = {n: torch.empty(*s, dtype=torch.float32, device=dev)
                 for n, s in zip(BOX_HEAD_PARAMS, box_head_param_shapes(nc))}
    for n, s in zip(BOX_HEAD_PARAMS, box_head_param_shapes(nc)):
        g = grads[n]
        assert tuple(g.shape) == s and g.dtype == torch.float32 and g.is_contiguous(), n
    def mark(name):
        if stage_events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            stage_events.append((name, ev))
    mark("start")
    # 1. tail: d_fc7 and the tail's weight / bias gradients (fixed-order sums over R)
    d_fc7 = torch.empty(R, 2048, dtype=torch.float32, device=dev)
    wc, _bc, wb, _bb, wd, _bd = eng.fc
    check(L.sb_box_tail_backward(ptr(_f32c(d_cls_score)), ptr(_f32c(d_bbox_pred)), ptr(_f32c(d_dim_orien_pred)),
                                 ptr(ctx["fc7_drop"]), R, 2048, nc, ptr(wc), ptr(wb), ptr(wd), ptr(d_fc7),
                                 ptr(grads["RCNN_cls_score.weight"]), ptr(grads["RCNN_cls_score.bias"]),
                                 ptr(grads["RCNN_bbox_pred.weight"]), ptr(grads["RCNN_bbox_pred.bias"]),
                                 ptr(grads["RCNN_dim_orien_pred.weight"]), ptr(grads["RCNN_dim_orien_pred.bias"]),
                                 stream_ptr()), "sb_box_tail_backward")
    mark("tail backward")
    # 2-3. fc7: mask / scale / convert, dW7 = g7^T fc6_drop, d_fc6 = g7 W7
    g7, inv7 = _dropout_backward(d_fc7, ctx["fc7"], ctx["words7"], grads["RCNN_top.3.bias"], "box_bwd_fc7")
    mark("mask/scale g7")
    ops.gemm(g7, ctx["fc6_drop"], grads["RCNN_top.3.weight"].view(2048, 2048), True, True, alpha=inv7)
    mark("dW7")
    d_fc6 = torch.empty(R, 2048, dtype=torch.float32, device=dev)
    ops.gemm(g7, eng.p["RCNN_top.3"].w16.view(2048, 2048), d_fc6, False, True, alpha=inv7)
    mark("d_fc6")
    # 4-5. fc6: mask / scale / convert, dW6 = g6^T pooled (packed (ph, pw, c) order, then one permute pass into
    # [2048][512][7][7]), d_pooled = g6 W6
    g6, inv6 = _dropout_backward(d_fc6, ctx["fc6"], ctx["words6"], grads["RCNN_top.0.bias"], "box_bwd_fc6")
    mark("mask/scale g6")
    dw6 = workspace(2048 * 25088 * 4, dev, "box_bwd_dw6")[:2048 * 25088 * 4].view(torch.float32).view(2048, 25088)
    ops.gemm(g6, ctx["pooled"].view(R, 25088), dw6, True, True, alpha=inv6)
    mark("dW6")
    check(L.sb_permute_pc_to_cp(ptr(dw6), 2048, 49, 512, ptr(grads["RCNN_top.0.weight"]), stream_ptr()),
          "sb_permute_pc_to_cp")
    mark("dW6 permute")
    d_pooled = torch.empty(R, 7, 7, 512, dtype=torch.float32, device=dev)
    ops.gemm(g6, eng.p["RCNN_top.0"].w16.view(2048, 25088), d_pooled.view(R, 25088), False, True, alpha=inv6)
    mark("d_pooled")
    # 6. into the left / right feature pyramids
    shapes = ctx["feat_shapes"]
    if feat_grads is None:
        feat_grads = {side: [torch.empty(*s, dtype=torch.float32, device=dev) for s in shapes]
                      for side in ("left", "right")}
    ops.roi_align_pyramid_nhwc_backward(d_pooled, ctx["im_h"], ctx["rois_left"], shapes, out_coff=0,
                                        grad_feats=feat_grads["left"])
    ops.roi_align_pyramid_nhwc_backward(d_pooled, ctx["im_h"], ctx["rois_right"], shapes, out_coff=256,
                                        grad_feats=feat_grads["right"])
    mark("RoIAlign backward L + R")
    return grads, feat_grads
