"""CPU: the oracle of the pyramid RoIAlign backward (tests/box_head_oracle.py: the adjoint of
oracle.ops.pyramid_roi_feat, composed from its level routing, the reference-semantics RoIAlign backward per level and
the adjoint of the 2x2 average) and the ABI layout of sb_gemm_desc.  The GPU kernels are checked against this
composition in test_gpu_box_head_backward.py."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from box_head_oracle import pyramid_roi_feat_backward
from oracle import ops as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def pyramid_case(B, seed, im_h=128, im_w=160, R=40, C=8):
    """features of a 4-level pyramid (strides 4..32) and RoIs that land on every level, touch or cross the image
    borders, and include degenerate (zero / negative extent) boxes"""
    rs = np.random.RandomState(seed)
    shapes = [(B, C, int(np.ceil(im_h / s)), int(np.ceil(im_w / s))) for s in (4, 8, 16, 32)]
    feats = [rs.randn(*s).astype(np.float32) for s in shapes]
    sizes = np.concatenate([rs.uniform(8, 45, R // 4), rs.uniform(60, 130, R // 4), rs.uniform(150, 360, R // 4),
                            rs.uniform(380, 700, R - 3 * (R // 4))])
    cx, cy = rs.uniform(-10, im_w + 10, R), rs.uniform(-10, im_h + 10, R)
    asp = rs.uniform(0.5, 2.0, R)
    w, h = sizes * np.sqrt(asp), sizes / np.sqrt(asp)
    rois = np.stack([rs.randint(0, B, R).astype(np.float64), cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1)
    rois[0, 1:] = [0, 0, im_w - 1, im_h - 1]                         # the whole image
    rois[1, 1:] = [im_w - 20, im_h - 20, im_w - 1, im_h - 1]         # the bottom-right border
    rois[2, 1:] = [30, 40, 30, 40]                                   # a point
    rois[3, 1:] = [50, 60, 45, 52]                                   # negative extent
    rois = rois.astype(np.float32)
    return feats, shapes, rois


@pytest.mark.parametrize("B,seed", [(1, 0), (2, 1), (2, 7)])
def test_pyramid_backward_oracle_is_the_adjoint(B, seed):
    feats, shapes, rois = pyramid_case(B, seed)
    lv = O.roi_levels(rois)
    assert set(lv.tolist()) == {2, 3, 4, 5}
    im_h, P = 128, 7
    G = np.random.RandomState(seed + 100).randn(rois.shape[0], shapes[0][1], P, P)
    fwd = O.pyramid_roi_feat(feats, rois, im_h, P).astype(np.float64)
    back = pyramid_roi_feat_backward(G, rois, shapes, im_h)
    lhs = float(np.sum(fwd * G))
    rhs = float(sum(np.sum(f.astype(np.float64) * b) for f, b in zip(feats, back)))
    scale = float(np.sum(np.abs(fwd * G)))
    # both oracle kernels round their outputs (and the backward its contributions) to fp32; beyond that the identity
    # is exact, so the defect is a few fp32 ulps of the terms
    assert abs(lhs - rhs) <= 1e-6 * scale, (lhs, rhs, scale)
    # every level received gradient
    assert all(np.abs(b).sum() > 0 for b in back)


def test_gemm_desc_layout_against_the_header_compiled_as_c(tmp_path):
    from stereo_rcnn_b200.lib import GemmDesc
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "stereo_b200.h"', "int main(void) {",
             'printf("size %zu\\n", sizeof(sb_gemm_desc));']
    for f in GemmDesc._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(sb_gemm_desc, %s));' % (f[0], f[0]))
    lines += ["return 0;", "}"]
    src = tmp_path / "gemm_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "gemm_layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o",
                           str(exe)])
    got = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["size"]) == ctypes.sizeof(GemmDesc)
    for f in GemmDesc._fields_:
        assert int(got[f[0]]) == getattr(GemmDesc, f[0]).offset, f[0]


def test_new_entry_points_are_bound():
    from stereo_rcnn_b200 import lib as L
    for name in ("sb_gemm_tc", "sb_roi_align_pyramid_nhwc_backward", "sb_roi_align_pyramid_nhwc_backward_workspace"):
        assert name in L.EXPORTS
