"""ctypes binding of libstereo_b200.so (the C ABI declared in include/stereo_b200.h).

There is NO fallback: if the shared library is missing or a call fails, this module
raises.  torch is used only for device memory and the current stream.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libstereo_b200.so")

c_int, c_float, c_double, c_void_p, c_size_t = (ctypes.c_int, ctypes.c_float, ctypes.c_double,
                                                ctypes.c_void_p, ctypes.c_size_t)
c_ll = ctypes.c_longlong


class SbError(RuntimeError):
    pass


class ProposalCfg(ctypes.Structure):
    _fields_ = [("n_levels", c_int), ("shapes", (c_int * 2) * 8), ("anchor_scales", c_int * 8),
                ("feat_strides", c_int * 8), ("n_ratios", c_int), ("ratios", c_double * 4),
                ("pre_nms_top_n", c_int), ("post_nms_top_n", c_int), ("nms_thresh", c_float)]


class ConvDesc(ctypes.Structure):
    _fields_ = [("in_", c_void_p), ("wgt", c_void_p), ("scale", c_void_p), ("shift", c_void_p),
                ("residual", c_void_p), ("up_src", c_void_p), ("out", c_void_p),
                ("N", c_int), ("H", c_int), ("W", c_int), ("Cin", c_int), ("Cout", c_int),
                ("kh", c_int), ("kw", c_int), ("stride", c_int), ("pad", c_int), ("Ho", c_int), ("Wo", c_int),
                ("in_ld", c_int), ("res_ld", c_int), ("UH", c_int), ("UW", c_int), ("relu", c_int),
                ("out_coff", c_int), ("out_mode", c_int), ("res_biased", c_int), ("in_biased", c_int),
                ("out_n_stride", c_ll), ("out_h_stride", c_ll), ("out_w_stride", c_ll),
                ("out16", c_void_p), ("in_dtype", c_int), ("max_ctas", c_int)]


class GemmDesc(ctypes.Structure):
    _fields_ = [("a", c_void_p), ("b", c_void_p), ("c", c_void_p), ("alpha", c_void_p), ("bias", c_void_p),
                ("M", c_int), ("N", c_int), ("K", c_int), ("lda", c_int), ("ldb", c_int), ("ldc", c_int),
                ("a_mn_major", c_int), ("b_mn_major", c_int)]


class ProposalTargetCfg(ctypes.Structure):
    _fields_ = [("rois_per_image", c_int), ("fg_rois_per_image", c_int), ("fg_thresh", c_float),
                ("bg_thresh_hi", c_float), ("bg_thresh_lo", c_float), ("bbox_means", c_float * 4),
                ("bbox_stds", c_float * 4), ("dim_means", c_float * 5), ("dim_stds", c_float * 5),
                ("kpts_grid", c_int)]


_SIGS = {
    "sb_version": (c_int, []),
    "sb_device_cc": (c_int, []),
    "sb_launch_count": (ctypes.c_ulonglong, []),
    "sb_nms_workspace_bytes": (c_size_t, [c_int]),
    "sb_nms": (c_int, [c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sb_nms_mask": (c_int, [c_void_p, c_int, c_float, c_void_p, c_void_p]),
    "sb_roi_align_forward": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int,
                                     c_float, c_void_p, c_void_p]),
    "sb_roi_align_backward": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int,
                                      c_float, c_void_p, c_void_p]),
    "sb_roi_align_backward_det_workspace": (c_size_t, [c_int, c_int, c_int, c_int]),
    "sb_roi_align_backward_det": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int,
                                          c_float, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sb_roi_align_pyramid_nhwc": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_int), ctypes.POINTER(c_int),
                                          c_int, c_float, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int,
                                          c_void_p]),
    "sb_roi_align_pyramid_nhwc_backward_workspace": (c_size_t, [c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int),
                                                                 c_int]),
    "sb_roi_align_pyramid_nhwc_backward": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_int, c_int, c_int,
                                                   ctypes.POINTER(c_int), ctypes.POINTER(c_int), ctypes.POINTER(c_void_p),
                                                   c_void_p, c_size_t, c_void_p]),
    "sb_proposal_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "sb_proposal_layer": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, ctypes.POINTER(ProposalCfg),
                                  c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sb_generate_anchors": (c_int, [ctypes.POINTER(ProposalCfg), c_int, c_void_p, c_void_p]),
    "sb_rpn_head_epilogue": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "sb_dense_align_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "sb_dense_align": (c_int, [c_void_p, c_void_p, c_int, c_int, ctypes.POINTER(c_double), c_double,
                               c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_size_t,
                               c_void_p]),
    "sb_dense_align_n": (c_int, [c_void_p, c_void_p, c_int, c_int, ctypes.POINTER(c_double), c_double, c_void_p, c_int,
                                 c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                 c_void_p]),
    "sb_infer_boundary": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "sb_box_solve": (c_int, [c_void_p] * 8 + [c_int, c_int, c_int, c_int, ctypes.POINTER(c_double),
                             ctypes.POINTER(c_double), c_float, c_int] + [c_void_p] * 5 + [c_void_p]),
    "sb_box_rectify": (c_int, [c_void_p] * 6 + [c_int, c_int, c_int, ctypes.POINTER(c_double),
                               ctypes.POINTER(c_double), c_void_p, c_void_p]),
    "sb_conv2d_simt": (c_int, [ctypes.POINTER(ConvDesc), c_void_p]),
    "sb_conv2d_tc": (c_int, [ctypes.POINTER(ConvDesc), c_void_p]),
    "sb_conv2d_tc_supported": (c_int, [ctypes.POINTER(ConvDesc)]),
    "sb_gemm_tc": (c_int, [ctypes.POINTER(GemmDesc), c_void_p]),
    "sb_conv_trace_bytes": (c_size_t, [c_int]),
    "sb_conv_trace": (c_int, [c_void_p, c_int]),
    "sb_conv_trace_count": (c_int, []),
    "sb_conv_trace_info": (c_int, [c_int, ctypes.POINTER(c_int)]),
    "sb_stem_conv": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "sb_stem_im2col": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sb_stem_conv_tc": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sb_stem_im2col16": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sb_maxpool3x3s2_ceil16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sb_maxpool3x3s2_ceil": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sb_subsample2": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sb_kpts_tail": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_void_p]),
    "sb_box_tail": (c_int, [c_void_p, c_int, c_int, c_int] + [c_void_p] * 9 + [c_void_p]),
    "sb_test_decode": (c_int, [c_void_p] * 8 + [c_int, c_int, c_int] + [c_void_p] * 4 + [c_void_p]),
    "sb_test_decode_record": (c_int, [c_void_p] * 9 + [c_int, c_int, c_int] + [c_void_p] * 5 + [c_int, c_void_p]),
    "sb_class_nms": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p]),
    "sb_prep_image_size": (c_int, [c_int, c_int, c_double, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "sb_prep_image": (c_int, [c_void_p, c_int, c_int, c_double, c_int, c_void_p, c_void_p]),
    "sb_fill": (c_int, [c_void_p, c_size_t, c_float, c_void_p]),
    "sb_peer_mailbox_bytes": (c_size_t, [c_int, c_int, c_int]),
    "sb_peer_alloc": (c_int, [c_size_t, ctypes.POINTER(c_void_p)]),
    "sb_peer_free": (c_int, [c_void_p]),
    "sb_ipc_export": (c_int, [c_void_p, c_void_p]),
    "sb_ipc_import": (c_int, [c_void_p, ctypes.POINTER(c_void_p)]),
    "sb_ipc_close": (c_int, [c_void_p]),
    "sb_peer_put_record": (c_int, [c_void_p, ctypes.POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "sb_peer_wait_records": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_double, c_void_p]),
    # train-time target layers and losses (A16)
    "sb_anchor_targets_workspace": (c_size_t, [c_int, c_int]),
    "sb_anchor_targets": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                  c_float, c_float, c_int, c_int, c_void_p, c_size_t] + [c_void_p] * 5 + [c_void_p]),
    "sb_proposal_targets": (c_int, [c_void_p, c_void_p, c_int, c_int] + [c_void_p] * 4 + [c_int, c_void_p, c_void_p,
                                    ctypes.POINTER(ProposalTargetCfg)] + [c_void_p] * 12 + [c_void_p]),
    "sb_loss_workspace_bytes": (c_size_t, []),
    "sb_rpn_loss": (c_int, [c_void_p] * 7 + [c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p,
                            c_void_p]),
    "sb_rcnn_loss": (c_int, [c_void_p] * 14 + [c_int, c_int, c_int] + [c_void_p] * 8 + [c_void_p]),
    "sb_multitask_loss": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "sb_dropout": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "sb_box_tail_logits": (c_int, [c_void_p, c_int, c_int, c_int] + [c_void_p] * 9 + [c_void_p]),
    "sb_box_tail_backward": (c_int, [c_void_p] * 4 + [c_int, c_int, c_int] + [c_void_p] * 10 + [c_void_p]),
    "sb_dropout_backward_workspace": (c_size_t, [c_int, c_int]),
    "sb_dropout_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_size_t, c_void_p]),
    "sb_permute_pc_to_cp": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sb_clip_gradient_workspace": (c_size_t, [c_int]),
    "sb_clip_gradient": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_size_t), c_int, c_float, c_void_p, c_size_t,
                                 c_void_p, c_void_p]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def load():
    """load the shared library; raises if it has not been built (no CPU fallback exists)"""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise SbError("libstereo_b200.so not built: run `python -m stereo_rcnn_b200.build` "
                          "(there is no CPU or PyTorch fallback for the hot path)")
        lib = ctypes.CDLL(SO_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        raise SbError("%s failed with code %d" % (what, rc))


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """device pointer of a contiguous CUDA tensor (None -> NULL)"""
    if t is None:
        return c_void_p(0)
    assert t.is_cuda and t.is_contiguous(), "stereo_b200 ops take contiguous CUDA tensors"
    return c_void_p(t.data_ptr())
