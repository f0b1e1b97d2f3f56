"""Oracles of the box-head training step, shared by the tests (test infrastructure, like oracle/, which it builds on).

* pyramid_roi_feat_backward -- the adjoint of oracle.ops.pyramid_roi_feat.
* box_head_train_fp64 -- torch fp64 autograd of oracle.model.box_head as the reference trains it: dropout after both
  ReLUs of RCNN_top (with given keep masks) and the class logits instead of the softmax (stereo_rcnn.py:248-257).
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import ops as O


def pyramid_roi_feat_backward(grad_pooled, rois, feat_shapes, im_h):
    """adjoint of O.pyramid_roi_feat: grad_pooled [R,C,P,P] -> one NCHW gradient per level (feat_shapes, P2..P5).

    PyramidRoI_Feat (stereo_rcnn.py:110-139) routes each RoI to one level and pools it with RoIAlignAvg
    (modules/roi_align.py:26-29): a (P+1)^2 RoIAlign lattice followed by avg_pool2d(2, stride 1).  Its autograd
    backward spreads each pooled gradient over the four lattice points with weight 1/4 and hands the lattice gradient
    to the RoIAlign backward (roi_align_kernel.cu:94-143) of the RoI's level."""
    rois = np.ascontiguousarray(rois, np.float32)
    grad_pooled = np.asarray(grad_pooled, np.float64)
    lv = O.roi_levels(rois)
    P = grad_pooled.shape[2]
    out = []
    for i, l in enumerate(range(2, 6)):
        idx = np.nonzero(lv == l)[0]
        if idx.size == 0:
            out.append(np.zeros(feat_shapes[i], np.float32))
            continue
        g = grad_pooled[idx] * 0.25
        lat = np.zeros(g.shape[:2] + (P + 1, P + 1), np.float64)
        lat[..., :-1, :-1] += g
        lat[..., :-1, 1:] += g
        lat[..., 1:, :-1] += g
        lat[..., 1:, 1:] += g
        scale = np.float32(feat_shapes[i][2] / float(im_h))          # the forward's per-level scale
        out.append(O.roi_align_backward(lat.astype(np.float32), rois[idx], feat_shapes[i], P + 1, P + 1, scale))
    return out


def keep_mask(words):
    """nn.Dropout(p=0.2) as the device samples it: keep where the uint32 word >= 0.2 * 2^32, scale 1 / 0.8"""
    u = words.to(torch.int64) & 0xFFFFFFFF
    return (u >= 858993460).to(torch.float64) * 1.25


def box_head_train_fp64(pooled_nhwc, sd, mask6, mask7, d_cls, d_bbox, d_dim, relu6=None, relu7=None, device="cpu"):
    """fp64 autograd of the training box head on the given pooled tile [R,7,7,512] (NHWC, as the device saved it) with
    the fp32 parameters of `sd`; the loss is sum(d_cls * cls_score + d_bbox * bbox_pred + d_dim * dim_orien_pred), so
    the gradients are the adjoints of the given incoming gradients.  relu6 / relu7: optional 0/1 masks of the ReLUs
    (where the device's fc6 / fc7 outputs are > 0) -- the adjoint of the forward the device computed: a pre-activation
    within rounding of 0 may take the other side of the ReLU in fp64, and each such flip moves a whole gradient term
    (about 1e-4 of the units flip at fp16 operand rounding, sqrt(1e-4) = 1e-2 relative L2).
    -> ({param name: grad}, d_pooled NHWC)"""
    dd = lambda t: torch.as_tensor(t).to(device=device, dtype=torch.float64)
    x = dd(pooled_nhwc).permute(0, 3, 1, 2).contiguous().requires_grad_()
    names = ("RCNN_top.0.weight", "RCNN_top.0.bias", "RCNN_top.3.weight", "RCNN_top.3.bias", "RCNN_cls_score.weight",
             "RCNN_cls_score.bias", "RCNN_bbox_pred.weight", "RCNN_bbox_pred.bias", "RCNN_dim_orien_pred.weight",
             "RCNN_dim_orien_pred.bias")
    p = {n: dd(sd[n]).requires_grad_() for n in names}
    R = x.shape[0]
    relu = lambda t, m: F.relu(t) if m is None else t * dd(m)
    h = relu(F.conv2d(x, p["RCNN_top.0.weight"], p["RCNN_top.0.bias"], stride=7).view(R, 2048), relu6) * dd(mask6)
    h = relu(F.conv2d(h.view(R, 2048, 1, 1), p["RCNN_top.3.weight"], p["RCNN_top.3.bias"]).view(R, 2048), relu7)
    h = h * dd(mask7)
    cls = F.linear(h, p["RCNN_cls_score.weight"], p["RCNN_cls_score.bias"])
    bbox = F.linear(h, p["RCNN_bbox_pred.weight"], p["RCNN_bbox_pred.bias"])
    dim = F.linear(h, p["RCNN_dim_orien_pred.weight"], p["RCNN_dim_orien_pred.bias"])
    ((cls * dd(d_cls)).sum() + (bbox * dd(d_bbox)).sum() + (dim * dd(d_dim)).sum()).backward()
    return {n: p[n].grad.cpu() for n in names}, x.grad.permute(0, 2, 3, 1).contiguous().cpu()
