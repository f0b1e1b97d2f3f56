"""Torch-tensor front end of the C ABI (device memory + current stream only).

Every function launches hand-written sm_100a kernels from libstereo_b200.so on
torch's current stream; nothing here computes on the host and nothing falls back.
"""
import contextlib
import ctypes
import threading

import numpy as np
import torch

from . import lib as _l
from .lib import ConvDesc, GemmDesc, ProposalCfg, check, ptr, stream_ptr

# constants of lib/model/utils/config.py that the hot path reads (SURVEY section 5)
CFG = dict(
    ANCHOR_RATIOS=[0.5, 1, 2], FPN_ANCHOR_SCALES=[32, 64, 128, 256, 512],
    FPN_FEAT_STRIDES=[4, 8, 16, 32, 64],
    TEST=dict(RPN_PRE_NMS_TOP_N=6000, RPN_POST_NMS_TOP_N=300, RPN_NMS_THRESH=0.7, NMS=0.3),
    TRAIN=dict(RPN_PRE_NMS_TOP_N=12000, RPN_POST_NMS_TOP_N=2000, RPN_NMS_THRESH=0.7),
    POOLING_SIZE=7, KPTS_GRID=28,
)

class WorkspaceOwner(object):
    """Scratch buffers of ONE in-flight unit of work (a pipeline slot, a CUDA graph, a test).

    Kernel workspaces hold live state between the launches of one call sequence (select histograms, NMS masks,
    partial costs), so two sequences that may overlap on the device -- e.g. two CUDA graphs replayed on different
    streams -- must not share them: each owns a WorkspaceOwner and issues its launches inside
    ``with ops.workspace_owner(owner):``.  Buffers are grow-only and a replaced buffer is RETIRED, never freed: a
    CUDA graph captured earlier has its address baked in."""

    def __init__(self):
        self.bufs, self.retired = {}, []

    def get(self, nbytes, device, tag):
        key = (str(device), tag)
        w = self.bufs.get(key)
        if w is None or w.numel() < nbytes:
            if w is not None:
                self.retired.append(w)
            w = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=device)
            self.bufs[key] = w
        return w


_default_owner = WorkspaceOwner()
_tls = threading.local()


@contextlib.contextmanager
def workspace_owner(owner):
    """route every ops.workspace() request of the enclosed launches to `owner`'s private buffers"""
    prev = getattr(_tls, "owner", None)
    _tls.owner = owner
    try:
        yield owner
    finally:
        _tls.owner = prev


def workspace(nbytes, device, tag="default"):
    """grow-only byte workspace per (owner, device, tag); avoids cudaMalloc in steady state.  Without an enclosing
    workspace_owner() the process-wide default owner is used: fine for strictly stream-ordered callers only."""
    owner = getattr(_tls, "owner", None) or _default_owner
    return owner.get(nbytes, device, tag)


def _f32c(t):
    assert t.dtype == torch.float32
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------ NMS ----
def nms_into(keep, dets, num_out, thresh):
    """caller-allocated outputs, as nms.nms_cuda(keep, dets, num_out, thresh) (nms_gpu.py:8-10)"""
    L = _l.load()
    n = dets.shape[0]
    assert dets.dim() == 2 and dets.shape[1] == 5 and keep.dtype == torch.int32 and num_out.dtype == torch.int32
    dets = _f32c(dets)
    nb = L.sb_nms_workspace_bytes(n)
    ws = workspace(nb, dets.device, "nms")
    check(L.sb_nms(ptr(dets), n, float(thresh), ptr(keep), ptr(num_out), ptr(ws), nb, stream_ptr()), "sb_nms")
    return 1


def nms(dets, thresh):
    """-> int32 [K,1] indices kept (ascending), like nms_gpu (lib/model/nms/nms_gpu.py:7-12)"""
    n = dets.shape[0]
    keep = torch.zeros(n, 1, dtype=torch.int32, device=dets.device)
    num_out = torch.zeros(1, dtype=torch.int32, device=dets.device)
    if n == 0:
        return keep
    nms_into(keep, dets, num_out, thresh)
    return keep[:int(num_out[0])]


def nms_mask(dets, thresh):
    L = _l.load()
    n = dets.shape[0]
    cb = (n + 63) // 64
    mask = torch.zeros(n, cb, dtype=torch.int64, device=dets.device)
    check(L.sb_nms_mask(ptr(_f32c(dets)), n, float(thresh), ptr(mask), stream_ptr()), "sb_nms_mask")
    return mask


# -------------------------------------------------------------- RoIAlign ----
def roi_align_forward(ah, aw, scale, features, rois, output):
    """roi_align.roi_align_forward_cuda(ah, aw, scale, features, rois, output) (functions/roi_align.py:24-27)"""
    L = _l.load()
    if rois.dim() != 2 or rois.shape[1] != 5:
        return 0                                   # roi_align_cuda.c:19-22
    N, C, H, W = features.shape
    check(L.sb_roi_align_forward(ptr(_f32c(features)), N, C, H, W, ptr(_f32c(rois)), rois.shape[0],
                                 int(ah), int(aw), float(scale), ptr(output), stream_ptr()), "sb_roi_align_forward")
    return 1


def roi_align_backward(ah, aw, scale, top_grad, rois, bottom_grad):
    L = _l.load()
    if rois.dim() != 2 or rois.shape[1] != 5:
        return 0
    N, C, H, W = bottom_grad.shape
    check(L.sb_roi_align_backward(ptr(_f32c(top_grad)), N, C, H, W, ptr(_f32c(rois)), rois.shape[0],
                                  int(ah), int(aw), float(scale), ptr(bottom_grad), stream_ptr()),
          "sb_roi_align_backward")
    return 1


def roi_align_backward_det(ah, aw, scale, top_grad, rois, bottom_grad):
    """deterministic RoIAlign backward (fixed-point accumulation): overwrites bottom_grad [N,C,H,W]"""
    L = _l.load()
    N, C, H, W = bottom_grad.shape
    nbytes = L.sb_roi_align_backward_det_workspace(N, C, H, W)
    ws = workspace(nbytes, bottom_grad.device, "roi_bwd_det")
    check(L.sb_roi_align_backward_det(ptr(_f32c(top_grad)), N, C, H, W, ptr(_f32c(rois)), rois.shape[0], int(ah),
                                      int(aw), float(scale), ptr(bottom_grad), ptr(ws), nbytes, stream_ptr()),
          "sb_roi_align_backward_det")
    return 1


def roi_align_pyramid_nhwc(feats, im_h, rois, pooled, out=None, out_coff=0, round_tf32=False, half=False):
    """feats: 4 NHWC fp32 tensors (P2..P5); rois [R,5]; -> out [R,pooled,pooled,out_ld] NHWC (fp32, fp32 rounded
    to TF32, or fp16 when half=True)"""
    L = _l.load()
    C = feats[0].shape[3]
    R = rois.shape[0]
    if out is None:
        out = torch.empty(R, pooled, pooled, C, dtype=torch.float16 if half else torch.float32, device=rois.device)
    if half:
        assert out.dtype == torch.float16
        round_tf32 = 2
    fp = (ctypes.c_void_p * 4)(*[f.data_ptr() for f in feats])
    hs = (ctypes.c_int * 4)(*[f.shape[1] for f in feats])
    ws_ = (ctypes.c_int * 4)(*[f.shape[2] for f in feats])
    check(L.sb_roi_align_pyramid_nhwc(fp, hs, ws_, C, float(im_h), ptr(_f32c(rois)), R, pooled, ptr(out),
                                      out.shape[3], out_coff, int(round_tf32), stream_ptr()),
          "sb_roi_align_pyramid_nhwc")
    return out


def roi_align_pyramid_nhwc_backward(top_grad, im_h, rois, feat_shapes, out_coff=0, grad_feats=None):
    """adjoint of roi_align_pyramid_nhwc (deterministic, fixed-point accumulation): top_grad [R,P,P,ld] fp32 read at
    channels [out_coff, out_coff + C); feat_shapes = 4 (N, H_l, W_l, C) of P2..P5 -> grad_feats, 4 fp32 NHWC tensors
    (overwritten; allocated when not given)"""
    L = _l.load()
    assert top_grad.dtype == torch.float32 and top_grad.is_contiguous() and top_grad.dim() == 4
    R, P = top_grad.shape[0], top_grad.shape[1]
    N, C = int(feat_shapes[0][0]), int(feat_shapes[0][3])
    dev = top_grad.device
    if grad_feats is None:
        grad_feats = [torch.empty(*[int(v) for v in s], dtype=torch.float32, device=dev) for s in feat_shapes]
    for g, s in zip(grad_feats, feat_shapes):
        assert g.dtype == torch.float32 and g.is_contiguous() and tuple(g.shape) == tuple(int(v) for v in s)
    hs = (ctypes.c_int * 4)(*[int(s[1]) for s in feat_shapes])
    ws_ = (ctypes.c_int * 4)(*[int(s[2]) for s in feat_shapes])
    gp = (ctypes.c_void_p * 4)(*[g.data_ptr() for g in grad_feats])
    nbytes = L.sb_roi_align_pyramid_nhwc_backward_workspace(N, hs, ws_, C)
    ws = workspace(nbytes, dev, "roi_pyramid_bwd")
    check(L.sb_roi_align_pyramid_nhwc_backward(ptr(top_grad), top_grad.shape[3], int(out_coff), C, float(im_h),
                                               ptr(_f32c(rois)), R, P, N, hs, ws_, gp, ptr(ws), nbytes, stream_ptr()),
          "sb_roi_align_pyramid_nhwc_backward")
    return grad_feats


# ------------------------------------------------------------------ GEMM ----
def gemm(a, b, out, a_mn_major, b_mn_major, alpha=None, bias=None):
    """out[m][n] = alpha * sum_k A(m,k) B(n,k) + bias[n] on the tensor cores (fp16 operands, fp32 accumulation).

    a: fp16 [M, K] (a_mn_major False) or [K, M] (True, A read in place, no transposed copy); b likewise [N, K] or
    [K, N]; out: fp32 [M, N].  Row-pitched views are fine (unit column stride, row strides multiples of 8).  alpha: fp32
    DEVICE tensor of one element or None (1); bias: fp32 [N] or None."""
    L = _l.load()
    assert a.dtype == torch.float16 and b.dtype == torch.float16 and out.dtype == torch.float32
    for t in (a, b, out):
        assert t.is_cuda and t.dim() == 2 and t.stride(1) == 1, "gemm operands are 2-D with unit column stride"
    M, N = out.shape
    K = a.shape[0] if a_mn_major else a.shape[1]
    assert tuple(a.shape) == ((K, M) if a_mn_major else (M, K)), "A shape"
    assert tuple(b.shape) == ((K, N) if b_mn_major else (N, K)), "B shape"
    if alpha is not None:
        assert alpha.dtype == torch.float32 and alpha.numel() == 1 and alpha.is_cuda
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.is_contiguous() and bias.numel() == N
    d = GemmDesc()
    d.a, d.b, d.c = a.data_ptr(), b.data_ptr(), out.data_ptr()
    d.alpha = alpha.data_ptr() if alpha is not None else None
    d.bias = bias.data_ptr() if bias is not None else None
    d.M, d.N, d.K = M, N, K
    d.lda, d.ldb, d.ldc = a.stride(0), b.stride(0), out.stride(0)
    d.a_mn_major, d.b_mn_major = int(bool(a_mn_major)), int(bool(b_mn_major))
    check(L.sb_gemm_tc(ctypes.byref(d), stream_ptr()), "sb_gemm_tc")
    return out


# -------------------------------------------------------- proposal layer ----
def make_proposal_cfg(cfg_key, feat_shapes, ratios=None, scales=None, strides=None, cfg=None):
    cfg = CFG if cfg is None else cfg
    pc = ProposalCfg()
    ratios = cfg["ANCHOR_RATIOS"] if ratios is None else ratios
    scales = cfg["FPN_ANCHOR_SCALES"] if scales is None else scales
    strides = cfg["FPN_FEAT_STRIDES"] if strides is None else strides
    pc.n_levels = len(feat_shapes)
    for i, (h, w) in enumerate(feat_shapes):
        pc.shapes[i][0], pc.shapes[i][1] = int(h), int(w)
        pc.anchor_scales[i], pc.feat_strides[i] = int(scales[i]), int(strides[i])
    pc.n_ratios = len(ratios)
    for i, r in enumerate(ratios):
        pc.ratios[i] = float(r)
    pc.pre_nms_top_n = int(cfg[cfg_key]["RPN_PRE_NMS_TOP_N"])
    pc.post_nms_top_n = int(cfg[cfg_key]["RPN_POST_NMS_TOP_N"])
    pc.nms_thresh = float(cfg[cfg_key]["RPN_NMS_THRESH"])
    return pc


def proposal_layer(cls_prob, bbox_pred_lr, im_info, cfg_key, feat_shapes, pc=None):
    """_ProposalLayer.forward (proposal_layer.py:42-145) -> rois_left, rois_right [B,N,5]"""
    L = _l.load()
    B, A = cls_prob.shape[:2]
    pc = make_proposal_cfg(cfg_key, feat_shapes) if pc is None else pc
    post = pc.post_nms_top_n
    dev = cls_prob.device
    rl = torch.empty(B, post, 5, dtype=torch.float32, device=dev)
    rr = torch.empty(B, post, 5, dtype=torch.float32, device=dev)
    nb = L.sb_proposal_workspace_bytes(B, A, pc.pre_nms_top_n)
    ws = workspace(nb, dev, "proposal")
    check(L.sb_proposal_layer(ptr(_f32c(cls_prob)), ptr(_f32c(bbox_pred_lr)), ptr(_f32c(im_info)), B, A,
                              ctypes.byref(pc), ptr(rl), ptr(rr), ptr(ws), nb, stream_ptr()), "sb_proposal_layer")
    return rl, rr


def rpn_head_epilogue(head, B, P):
    """raw fused head output [B*P, ld] -> cls_prob [B, 3P, 2], bbox_pred [B, 3P, 6]"""
    L = _l.load()
    dev = head.device
    cls_prob = torch.empty(B, 3 * P, 2, dtype=torch.float32, device=dev)
    bbox = torch.empty(B, 3 * P, 6, dtype=torch.float32, device=dev)
    check(L.sb_rpn_head_epilogue(ptr(head), B, P, head.shape[-1], ptr(cls_prob), ptr(bbox), stream_ptr()),
          "sb_rpn_head_epilogue")
    return cls_prob, bbox


# ----------------------------------------------------------- dense_align ----
def calib_vec(p2, p3):
    p2, p3 = np.asarray(p2, np.float64), np.asarray(p3, np.float64)
    return np.array([p2[0, 0], p2[0, 2], p2[1, 2], p2[0, 3] - p3[0, 3]], np.float64)


def dense_align(calib4, scale, im_left, im_right, box_left, keypoints, poses):
    """align_parallel (dense_align.py:240-300) -> solve_status [D], best_dis [D]"""
    L = _l.load()
    iml = _f32c(im_left).reshape(3, *im_left.shape[-2:])
    imr = _f32c(im_right).reshape(3, *im_right.shape[-2:])
    H, W = iml.shape[1:]
    D = box_left.shape[0]
    dev = iml.device
    status = torch.zeros(D, dtype=torch.float32, device=dev)
    best = torch.zeros(D, dtype=torch.float32, device=dev)
    if D == 0:
        return status, best
    nb = L.sb_dense_align_workspace_bytes(H, W, D)
    ws = workspace(nb, dev, "dense_align")
    c4 = (ctypes.c_double * 4)(*[float(v) for v in calib4])
    check(L.sb_dense_align(ptr(iml), ptr(imr), H, W, c4, float(scale), ptr(_f32c(box_left)),
                           ptr(_f32c(keypoints)), ptr(_f32c(poses)), D, ptr(status), ptr(best), ptr(ws), nb,
                           stream_ptr()), "sb_dense_align")
    return status, best


def dense_align_n(calib4, scale, im_left, im_right, boxes_all, keypoints, poses_all, n_dev):
    """align_parallel on device-resident solver outputs: boxes_all [cap,>=4], keypoints [cap,5], poses_all [cap,>=7],
    n_dev int32 [1] (how many rows are live) -> status [cap], best_dis [cap]; rows >= n are left at zero"""
    L = _l.load()
    iml = _f32c(im_left).reshape(3, *im_left.shape[-2:])
    imr = _f32c(im_right).reshape(3, *im_right.shape[-2:])
    H, W = iml.shape[1:]
    cap = boxes_all.shape[0]
    dev = iml.device
    status = torch.zeros(cap, dtype=torch.float32, device=dev)
    best = torch.zeros(cap, dtype=torch.float32, device=dev)
    nb = L.sb_dense_align_workspace_bytes(H, W, cap)
    ws = workspace(nb, dev, "dense_align")
    c4 = (ctypes.c_double * 4)(*[float(v) for v in calib4])
    check(L.sb_dense_align_n(ptr(iml), ptr(imr), H, W, c4, float(scale), ptr(_f32c(boxes_all)), boxes_all.shape[1],
                             ptr(_f32c(keypoints)), ptr(_f32c(poses_all)), poses_all.shape[1], cap, ptr(n_dev),
                             ptr(status), ptr(best), ptr(ws), nb, stream_ptr()), "sb_dense_align_n")
    return status, best


# ------------------------------------------------------------ box solver ----
def _p34(p):
    return (ctypes.c_double * 12)(*[float(v) for v in np.asarray(p, np.float64).reshape(-1)])


def infer_boundary(boxes, keep, num, im_w, col_offset=0):
    """kitti_utils.infer_boundary (kitti_utils.py:398-437) over boxes[keep[:num]] -> left_right [R,2] (kept order)"""
    L = _l.load()
    R = boxes.shape[0]
    out = torch.zeros(R, 2, dtype=torch.float32, device=boxes.device)
    check(L.sb_infer_boundary(ptr(_f32c(boxes)), boxes.shape[1], int(col_offset), ptr(keep), ptr(num), int(im_w),
                              ptr(out), stream_ptr()), "sb_infer_boundary")
    return out


def box_solve(scores, boxes_left, boxes_right, dim_orien, kpts, keep, num, im_hw, p2, p3, cls=1, eval_thresh=0.05,
              inferred=None, cap=None):
    """test_net.py:263-303 on the device: border fix-up + solve_x_y_z_theta_from_kpt per kept detection, solved ones
    appended in order -> boxes_all [cap,5], kpts_all [cap,5], poses_all [cap,8], src_index [cap], n [1] (device)"""
    L = _l.load()
    R, nc = scores.shape
    cap = R if cap is None else int(cap)
    dev = scores.device
    boxes_all = torch.zeros(cap, 5, dtype=torch.float32, device=dev)
    kpts_all = torch.zeros(cap, 5, dtype=torch.float32, device=dev)
    poses_all = torch.zeros(cap, 8, dtype=torch.float32, device=dev)
    src = torch.zeros(cap, dtype=torch.int32, device=dev)
    n = torch.zeros(1, dtype=torch.int32, device=dev)
    check(L.sb_box_solve(ptr(_f32c(scores)), ptr(_f32c(boxes_left)), ptr(_f32c(boxes_right)), ptr(_f32c(dim_orien)),
                         ptr(_f32c(kpts)), ptr(keep), ptr(num), ptr(inferred), nc, int(cls), int(im_hw[0]),
                         int(im_hw[1]), _p34(p2), _p34(p3), float(eval_thresh), cap, ptr(boxes_all), ptr(kpts_all),
                         ptr(poses_all), ptr(src), ptr(n), stream_ptr()), "sb_box_solve")
    return boxes_all, kpts_all, poses_all, src, n


def box_rectify(boxes_all, kpts_all, poses_all, succ, best_dis, n, im_hw, p2, p3):
    """test_net.py:311-325: solve_x_y_theta_from_kpt with the aligned disparity -> final [cap,13] float64
    (valid, score, box_left 4, x, y, z, w, h, l, theta)"""
    L = _l.load()
    cap = boxes_all.shape[0]
    out = torch.zeros(cap, 13, dtype=torch.float64, device=boxes_all.device)
    check(L.sb_box_rectify(ptr(boxes_all), ptr(kpts_all), ptr(poses_all), ptr(succ), ptr(best_dis), ptr(n), cap,
                           int(im_hw[0]), int(im_hw[1]), _p34(p2), _p34(p3), ptr(out), stream_ptr()), "sb_box_rectify")
    return out


def kitti_result_lines(final, t_cam2_cam0_x):
    """kitti_utils.write_detection_results' text (kitti_utils.py:440-460) for the valid rows of box_rectify's output
    (host side: formatting text is not device work)"""
    import math
    lines = []
    for r in final.detach().cpu().numpy():
        if r[0] <= 0:
            continue
        score, box, pos, dim, orien = r[1], r[2:6], r[6:9], r[9:12], r[12]
        alpha = orien - math.pi / 2 + math.atan2(-pos[0], pos[2])
        s = "Car -1 -1 "
        s += "%f %f %f %f %f " % (alpha, box[0], box[1], box[2], box[3])
        s += "%f %f %f %f %f %f %f %f \n" % (dim[1], dim[0], dim[2], pos[0] - t_cam2_cam0_x, pos[1], pos[2], orien - 1.57, score)
        lines.append(s)
    return lines


# ------------------------------------------------------------- layer ops ----
def conv_desc(x, wgt, out, Cin, Cout, kh, kw, stride, pad, Ho, Wo, scale=None, shift=None, residual=None,
              up_src=None, relu=False, in_ld=None, out_coff=0, out_strides=None, out_mode=0, res_biased=False,
              in_biased=False, out16=None, max_ctas=0):
    """x: NHWC [N,H,W,in_ld]; wgt packed [Cout,kh,kw,Cin]; out: any tensor addressed through out_strides
    = (n, h, w) strides in floats (default: dense NHWC of out.shape[-1] channels)."""
    d = ConvDesc()
    N, H, W = x.shape[0], x.shape[1], x.shape[2]
    d.in_, d.wgt = x.data_ptr(), wgt.data_ptr()
    d.out = out.data_ptr() if out is not None else None
    d.out16 = out16.data_ptr() if out16 is not None else None
    d.in_dtype = 1 if x.dtype == torch.float16 else 0
    d.max_ctas = int(max_ctas)
    assert wgt.dtype == x.dtype, "weights and activations of a conv share one operand type"
    d.scale = scale.data_ptr() if scale is not None else None
    d.shift = shift.data_ptr() if shift is not None else None
    d.residual = residual.data_ptr() if residual is not None else None
    d.up_src = up_src.data_ptr() if up_src is not None else None
    d.N, d.H, d.W, d.Cin, d.Cout, d.kh, d.kw = N, H, W, Cin, Cout, kh, kw
    d.stride, d.pad, d.Ho, d.Wo = stride, pad, Ho, Wo
    d.in_ld = x.shape[3] if in_ld is None else in_ld
    d.res_ld = residual.shape[-1] if residual is not None else 0
    d.UH, d.UW = (up_src.shape[1], up_src.shape[2]) if up_src is not None else (0, 0)
    d.relu = 1 if relu else 0
    d.out_coff = out_coff
    d.out_mode, d.res_biased, d.in_biased = int(out_mode), int(bool(res_biased)), int(bool(in_biased))
    if out_strides is None:
        ld = (out if out is not None else out16).shape[-1]
        out_strides = (Ho * Wo * ld, Wo * ld, ld)
    d.out_n_stride, d.out_h_stride, d.out_w_stride = [int(s) for s in out_strides]
    return d


def conv2d(desc, impl="auto"):
    L = _l.load()
    if impl == "auto":
        impl = "tc" if L.sb_conv2d_tc_supported(ctypes.byref(desc)) else "simt"
    if impl == "tc":
        check(L.sb_conv2d_tc(ctypes.byref(desc), stream_ptr()), "sb_conv2d_tc")
    else:
        check(L.sb_conv2d_simt(ctypes.byref(desc), stream_ptr()), "sb_conv2d_simt")
    return impl


def stem_conv(im_nchw, wgt, scale, shift, out_mode=0):
    L = _l.load()
    N, _, H, W = im_nchw.shape
    Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
    out = torch.empty(N, Ho, Wo, 64, dtype=torch.float32, device=im_nchw.device)
    check(L.sb_stem_conv(ptr(_f32c(im_nchw)), N, H, W, ptr(wgt), ptr(scale), ptr(shift), ptr(out), int(out_mode),
                         stream_ptr()), "sb_stem_conv")
    return out


def stem_im2col(im_nchw):
    """-> [N, Ho, Wo, 160] patch matrix of the 7x7/2 stem (147 taps zero-padded to 160)"""
    L = _l.load()
    N, _, H, W = im_nchw.shape
    Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
    out = torch.empty(N, Ho, Wo, 160, dtype=torch.float32, device=im_nchw.device)
    check(L.sb_stem_im2col(ptr(_f32c(im_nchw)), N, H, W, ptr(out), stream_ptr()), "sb_stem_im2col")
    return out


def stem_im2col16(im_nchw):
    """-> fp16 [N, Ho, Wo, 152] patch matrix of the stem (147 taps + 5 zeros; the GEMM's tensor map zero-fills up to
    the 192 columns of its zero-padded weights)"""
    L = _l.load()
    N, _, H, W = im_nchw.shape
    Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
    out = torch.empty(N, Ho, Wo, 152, dtype=torch.float16, device=im_nchw.device)
    check(L.sb_stem_im2col16(ptr(_f32c(im_nchw)), N, H, W, ptr(out), stream_ptr()), "sb_stem_im2col16")
    return out


def pack_stem_w16(weight):
    """[64,3,7,7] stem weights -> fp16 [64,192] in sb_stem_conv_tc's K layout: tap (ci, r, s) at
    k = ci*49 + r*7 + s, zero padded from 147 to three 64-wide K-steps"""
    w = torch.zeros(64, 192, dtype=torch.float32)
    w[:, :147] = weight.detach().float().cpu().reshape(64, 147)
    return w.to(torch.float16)


def stem_conv_tc(im_nchw, w16, scale, shift):
    """stem conv7x7/2 + frozen BN + ReLU as an implicit tensor-core GEMM (patch gather inside the kernel)
    -> fp16 NHWC [N, Ho, Wo, 64]; w16: fp16 [64,192] from pack_stem_w16"""
    L = _l.load()
    N, _, H, W = im_nchw.shape
    Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
    out = torch.empty(N, Ho, Wo, 64, dtype=torch.float16, device=im_nchw.device)
    check(L.sb_stem_conv_tc(ptr(_f32c(im_nchw)), N, H, W, ptr(w16), ptr(scale), ptr(shift), ptr(out), stream_ptr()),
          "sb_stem_conv_tc")
    return out


def maxpool3x3s2_ceil(x):
    L = _l.load()
    N, H, W, C = x.shape

    def osz(v):
        o = (v - 3 + 1) // 2 + 1
        return o - 1 if (o - 1) * 2 >= v else o
    out = torch.empty(N, osz(H), osz(W), C, dtype=x.dtype, device=x.device)
    if x.dtype == torch.float16:
        check(L.sb_maxpool3x3s2_ceil16(ptr(x), N, H, W, C, ptr(out), stream_ptr()), "sb_maxpool3x3s2_ceil16")
    else:
        check(L.sb_maxpool3x3s2_ceil(ptr(x), N, H, W, C, ptr(out), stream_ptr()), "sb_maxpool3x3s2_ceil")
    return out


def subsample2(x):
    """x[:, ::2, ::2, :]; a pure copy, so fp16 tensors go through the same kernel viewed as C/2 fp32 lanes"""
    L = _l.load()
    N, H, W, C = x.shape
    out = torch.empty(N, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C, dtype=x.dtype, device=x.device)
    cw = C // 2 if x.dtype == torch.float16 else C
    check(L.sb_subsample2(ptr(x), N, H, W, cw, ptr(out), stream_ptr()), "sb_subsample2")
    return out


def kpts_tail(x, w, b, want_pred_all=False):
    L = _l.load()
    R, G, _, C = x.shape
    dev = x.device
    kp = torch.empty(R, 4 * G, dtype=torch.float32, device=dev)
    lp = torch.empty(R, G, dtype=torch.float32, device=dev)
    rp = torch.empty(R, G, dtype=torch.float32, device=dev)
    ka = torch.empty(R, 6, G, dtype=torch.float32, device=dev)      # logits; also the staging between the 2 kernels
    check(L.sb_kpts_tail(ptr(x), 1 if x.dtype == torch.float16 else 0, R, G, C, ptr(w), ptr(b), ptr(kp), ptr(lp),
                         ptr(rp), ptr(ka), stream_ptr()),
          "sb_kpts_tail")
    return kp, lp, rp, ka


def box_tail(fc7, w_cls, b_cls, w_box, b_box, w_dim, b_dim, n_classes):
    L = _l.load()
    R, K = fc7.shape
    dev = fc7.device
    cls_prob = torch.empty(R, n_classes, dtype=torch.float32, device=dev)
    bbox = torch.empty(R, 6 * n_classes, dtype=torch.float32, device=dev)
    dim = torch.empty(R, 5 * n_classes, dtype=torch.float32, device=dev)
    check(L.sb_box_tail(ptr(fc7), R, K, n_classes, ptr(w_cls), ptr(b_cls), ptr(w_box), ptr(b_box), ptr(w_dim),
                        ptr(b_dim), ptr(cls_prob), ptr(bbox), ptr(dim), stream_ptr()), "sb_box_tail")
    return cls_prob, bbox, dim


def test_decode(rois_left, rois_right, bbox_pred, dim_orien, kpts_prob, left_prob, right_prob, im_info,
                n_classes=2, grid=28):
    """test_net.py:138-212 -> pred_boxes_left [R,4nc], pred_boxes_right, dim_orien [R,5nc], pred_kpts [R,5]"""
    L = _l.load()
    R = rois_left.shape[0]
    dev = rois_left.device
    pbl = torch.empty(R, 4 * n_classes, dtype=torch.float32, device=dev)
    pbr = torch.empty(R, 4 * n_classes, dtype=torch.float32, device=dev)
    do = torch.empty(R, 5 * n_classes, dtype=torch.float32, device=dev)
    pk = torch.empty(R, 5, dtype=torch.float32, device=dev)
    check(L.sb_test_decode(ptr(_f32c(rois_left)), ptr(_f32c(rois_right)), ptr(_f32c(bbox_pred)),
                           ptr(_f32c(dim_orien)), ptr(_f32c(kpts_prob)), ptr(_f32c(left_prob)),
                           ptr(_f32c(right_prob)), ptr(_f32c(im_info)), R, n_classes, grid, ptr(pbl), ptr(pbr),
                           ptr(do), ptr(pk), stream_ptr()), "sb_test_decode")
    return pbl, pbr, do, pk


def test_decode_record(rois_left, rois_right, cls_prob, bbox_pred, dim_orien, kpts_prob, left_prob, right_prob,
                       im_info, n_classes=2, grid=28, record=None):
    """test_decode + the [R, 14nc+5] detection record of the image (what ranks all-gather), one launch"""
    L = _l.load()
    R = rois_left.shape[0]
    dev = rois_left.device
    pbl = torch.empty(R, 4 * n_classes, dtype=torch.float32, device=dev)
    pbr = torch.empty(R, 4 * n_classes, dtype=torch.float32, device=dev)
    do = torch.empty(R, 5 * n_classes, dtype=torch.float32, device=dev)
    pk = torch.empty(R, 5, dtype=torch.float32, device=dev)
    if record is None:
        record = torch.empty(R, 14 * n_classes + 5, dtype=torch.float32, device=dev)
    check(L.sb_test_decode_record(ptr(_f32c(rois_left)), ptr(_f32c(rois_right)), ptr(_f32c(cls_prob)),
                                  ptr(_f32c(bbox_pred)), ptr(_f32c(dim_orien)), ptr(_f32c(kpts_prob)),
                                  ptr(_f32c(left_prob)), ptr(_f32c(right_prob)), ptr(_f32c(im_info)), R, n_classes,
                                  grid, ptr(pbl), ptr(pbr), ptr(do), ptr(pk), ptr(record), record.shape[-1],
                                  stream_ptr()), "sb_test_decode_record")
    return pbl, pbr, do, pk, record


def class_nms(scores, boxes_left, cls, score_thresh=0.05, nms_thresh=0.3, keep=None, num=None):
    """test_net.py:233-259 on device -> (keep [R] int32 RoI indices in kept order, num [1] int32)"""
    L = _l.load()
    R, nc = scores.shape
    if keep is None:
        keep = torch.empty(R, dtype=torch.int32, device=scores.device)
    if num is None:
        num = torch.empty(1, dtype=torch.int32, device=scores.device)
    check(L.sb_class_nms(ptr(_f32c(scores)), ptr(_f32c(boxes_left)), R, nc, int(cls), float(score_thresh),
                         float(nms_thresh), ptr(keep), ptr(num), stream_ptr()), "sb_class_nms")
    return keep, num


def prep_image(img_u8, scale, rgb_input=False, out=None):
    """prep_im_for_blob (blob.py:44-64) on the device: uint8 [H,W,3] -> fp32 [3,Ho,Wo] (BGR - means, resized)"""
    L = _l.load()
    assert img_u8.dtype == torch.uint8 and img_u8.dim() == 3 and img_u8.shape[2] == 3
    H, W = img_u8.shape[:2]
    ho, wo = ctypes.c_int(), ctypes.c_int()
    check(L.sb_prep_image_size(H, W, float(scale), ctypes.byref(ho), ctypes.byref(wo)), "sb_prep_image_size")
    if out is None:
        out = torch.empty(3, ho.value, wo.value, dtype=torch.float32, device=img_u8.device)
    assert tuple(out.shape) == (3, ho.value, wo.value)
    check(L.sb_prep_image(ptr(img_u8.contiguous()), H, W, float(scale), 1 if rgb_input else 0, ptr(out), stream_ptr()),
          "sb_prep_image")
    return out


def l2_flush(buf):
    L = _l.load()
    check(L.sb_fill(ptr(buf), buf.numel(), 0.0, stream_ptr()), "sb_fill")


def launch_count():
    return int(_l.load().sb_launch_count())


EXACT, ROUND_TF32, BIASED = 0, 1, 2          # sb_conv_desc.out_mode


def round_tf32_(w):
    """in-place round-to-nearest (ties away) of fp32 values to TF32 precision (weights, once at pack time)"""
    b = w.view(torch.int32)
    b.add_(0x1000).bitwise_and_(~0x1FFF)
    return w


def unbias(x):
    """exact fp32 view of a tensor stored pre-biased (out_mode 2); debugging / tests only"""
    return (x.view(torch.int32) - 0x1000).view(torch.float32)
