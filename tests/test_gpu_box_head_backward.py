"""GPU: the two building blocks of the box-head backward -- the tcgen05 GEMM that reads its operands in their stored
(K-major or M/N-major) layout, and the deterministic adjoint of the fused pyramid RoIAlign."""
import ctypes

import numpy as np
import pytest
import torch

from stereo_rcnn_b200 import lib as _l
from stereo_rcnn_b200 import ops as G
from box_head_oracle import pyramid_roi_feat_backward
from test_box_head_backward_oracle import pyramid_case

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


# ------------------------------------------------------------------------------------------------------------- GEMM
def padded(rows, cols, g):
    """fp16 [rows, cols] view whose row pitch is cols rounded up to 8 (the GEMM's alignment rule)"""
    return torch.randn(rows, (cols + 7) // 8 * 8, generator=g, device="cuda").half()[:, :cols]


def operands(M, N, K, a_mn, b_mn, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    a = padded(*((K, M) if a_mn else (M, K)), g)
    b = padded(*((K, N) if b_mn else (N, K)), g)
    return a, b


def reference(a, b, a_mn, b_mn):
    A = a.double().t() if a_mn else a.double()          # [M, K]
    Bt = b.double() if b_mn else b.double().t()          # [K, N]
    return A @ Bt


SHAPES = [(1024, 25088, 2048), (2048, 25088, 1024), (1000, 200, 136), (77, 2048, 1024), (1, 8, 1), (130, 72, 65)]


@pytest.mark.parametrize("a_mn", [False, True])
@pytest.mark.parametrize("b_mn", [False, True])
@pytest.mark.parametrize("M,N,K", SHAPES)
def test_gemm_layouts_vs_fp64(M, N, K, a_mn, b_mn):
    a, b = operands(M, N, K, a_mn, b_mn, seed=M + N + K)
    out = torch.full((M, N), float("nan"), device="cuda")       # every element must be written
    G.gemm(a, b, out, a_mn, b_mn)
    ref = reference(a, b, a_mn, b_mn)
    err = (torch.linalg.norm(out.double() - ref) / torch.linalg.norm(ref)).item()
    # the operands are exact fp16 values and their products exact in fp32: the only error is fp32 accumulation order
    assert err <= 2e-5, err
    again = torch.empty_like(out)
    G.gemm(a, b, again, a_mn, b_mn)
    torch.cuda.synchronize()
    assert torch.equal(out, again), "C must be bit-identical from run to run"


@pytest.mark.parametrize("a_mn,b_mn", [(True, True), (False, True), (True, False)])
def test_gemm_device_alpha_bias_and_pitched_views(a_mn, b_mn):
    M, N, K = 300, 260, 200
    a_full, b_full = operands(M + 16, N + 24, K + 8, a_mn, b_mn, seed=5)
    # row-pitched views: leading dimensions larger than the matrix
    a = a_full[:K, :M] if a_mn else a_full[:M, :K]
    b = b_full[:K, :N] if b_mn else b_full[:N, :K]
    out_full = torch.zeros(M, N + 12, device="cuda")             # row pitch 272: a multiple of 8
    out = out_full[:, :N]
    alpha = torch.tensor([2.0 ** -20], device="cuda")
    bias = torch.randn(N, device="cuda")
    G.gemm(a, b, out, a_mn, b_mn, alpha=alpha, bias=bias)
    ref = reference(a, b, a_mn, b_mn) * 2.0 ** -20 + bias.double()
    assert rel_l2(out.cpu(), ref.cpu()) <= 2e-5
    assert torch.count_nonzero(out_full[:, N:]) == 0, "columns past N are not written"


def test_gemm_bias_with_a_partial_column_quad():
    M, N, K = 64, 6, 32
    a, b = operands(M, N, K, True, True, seed=9)
    bias = torch.randn(N, device="cuda")
    out = torch.empty(M, 8, device="cuda")[:, :N]
    G.gemm(a, b, out, True, True, bias=bias)
    ref = reference(a, b, True, True) + bias.double()
    assert rel_l2(out.cpu(), ref.cpu()) <= 2e-5


def test_gemm_rejects_bad_arguments():
    L = _l.load()
    a = torch.zeros(64, 64, dtype=torch.float16, device="cuda")
    c = torch.zeros(64, 64, device="cuda")
    d = _l.GemmDesc()
    d.a, d.b, d.c = a.data_ptr(), a.data_ptr(), c.data_ptr()
    d.M = d.N = d.K = 64
    d.lda = d.ldb = d.ldc = 64
    assert L.sb_gemm_tc(ctypes.byref(d), _l.stream_ptr()) == 0
    for field, v in (("lda", 60), ("ldc", 12), ("M", 0), ("K", 0), ("ldb", 32)):
        bad = _l.GemmDesc.from_buffer_copy(d)
        setattr(bad, field, v)
        assert L.sb_gemm_tc(ctypes.byref(bad), _l.stream_ptr()) == -22, field
    bad = _l.GemmDesc.from_buffer_copy(d)
    bad.a = a.data_ptr() + 2                                   # not 16-byte aligned
    assert L.sb_gemm_tc(ctypes.byref(bad), _l.stream_ptr()) == -22
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------ pyramid RoIAlign backward
def nhwc(x):
    return torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 3, 1))).cuda()


def gpu_case(B, seed, C=256, R=60, ld=None, coff=0):
    feats, shapes, rois = pyramid_case(B, seed, R=R, C=C)
    P = 7
    ld = C if ld is None else ld
    top = torch.from_numpy(np.random.RandomState(seed + 1).randn(rois.shape[0], P, P, ld).astype(np.float32)).cuda()
    nshapes = [(s[0], s[2], s[3], s[1]) for s in shapes]
    return feats, shapes, nshapes, rois, top, P


@pytest.mark.parametrize("B,seed", [(1, 3), (2, 4)])
def test_pyramid_backward_is_the_adjoint_of_the_gpu_forward(B, seed):
    feats, shapes, nshapes, rois, top, P = gpu_case(B, seed)
    im_h = 128
    fg = [nhwc(f) for f in feats]
    rc = torch.from_numpy(rois).cuda()
    fwd = G.roi_align_pyramid_nhwc(fg, im_h, rc, P)                      # exact fp32 output mode
    back = G.roi_align_pyramid_nhwc_backward(top, im_h, rc, nshapes)
    lhs = torch.sum(fwd.double() * top.double()).item()
    rhs = sum(torch.sum(f.double() * g.double()).item() for f, g in zip(fg, back))
    scale = torch.sum((fwd.double() * top.double()).abs()).item()
    assert abs(lhs - rhs) <= 1e-5 * scale, (lhs, rhs, scale)


@pytest.mark.parametrize("B,seed,ld,coff", [(1, 5, 256, 0), (2, 6, 512, 256), (2, 8, 512, 0)])
def test_pyramid_backward_vs_oracle(B, seed, ld, coff):
    C = 256
    feats, shapes, nshapes, rois, top, P = gpu_case(B, seed, C=C, ld=ld, coff=coff)
    back = G.roi_align_pyramid_nhwc_backward(top, 128, torch.from_numpy(rois).cuda(), nshapes, out_coff=coff)
    gp = top[..., coff:coff + C].permute(0, 3, 1, 2).cpu().numpy()      # [R, C, P, P]
    ref = pyramid_roi_feat_backward(gp, rois, shapes, 128)
    for lvl, (g, r) in enumerate(zip(back, ref)):
        err = rel_l2(g.permute(0, 3, 1, 2).cpu().numpy(), r)
        assert err <= 1e-4, (lvl, err)


def test_pyramid_backward_is_independent_of_roi_order_and_overwrites():
    feats, shapes, nshapes, rois, top, P = gpu_case(2, 11, R=200)
    rc = torch.from_numpy(rois).cuda()
    first = [torch.full(tuple(s), 7.0, device="cuda") for s in nshapes]          # garbage: must be overwritten
    G.roi_align_pyramid_nhwc_backward(top, 128, rc, nshapes, grad_feats=first)
    perm = torch.from_numpy(np.random.RandomState(0).permutation(rois.shape[0])).cuda()
    second = G.roi_align_pyramid_nhwc_backward(top[perm].contiguous(), 128, rc[perm].contiguous(), nshapes)
    again = G.roi_align_pyramid_nhwc_backward(top, 128, rc, nshapes)
    torch.cuda.synchronize()
    for a, b, c in zip(first, second, again):
        assert torch.equal(a, b) and torch.equal(a, c)


def test_pyramid_backward_without_rois_writes_zeros():
    _, _, nshapes, rois, top, P = gpu_case(1, 12, C=8)
    grads = [torch.full(tuple(s), 3.0, device="cuda") for s in nshapes]
    G.roi_align_pyramid_nhwc_backward(top[:0], 128, torch.from_numpy(rois[:0]).cuda(), nshapes, grad_feats=grads)
    torch.cuda.synchronize()
    assert all(torch.count_nonzero(g) == 0 for g in grads)


def test_pyramid_backward_skips_rois_outside_the_batch():
    """a RoI whose batch index is not an image of the batch contributes nothing (and writes nowhere)"""
    feats, shapes, nshapes, rois, top, P = gpu_case(2, 13, C=64, R=40)
    bad = rois[:6].copy()
    bad[:3, 0], bad[3:, 0] = 2, -1                                   # N = 2: indices 2 and -1 are outside
    rc = torch.from_numpy(rois).cuda()
    rc_bad = torch.from_numpy(np.concatenate([rois, bad])).cuda()
    top_bad = torch.cat([top, torch.randn(6, P, P, top.shape[3], device="cuda")]).contiguous()
    want = G.roi_align_pyramid_nhwc_backward(top, 128, rc, nshapes)
    got = G.roi_align_pyramid_nhwc_backward(top_bad, 128, rc_bad, nshapes)
    torch.cuda.synchronize()
    for a, b in zip(got, want):
        # the fixed-point quantum follows max|top_grad|, so compare to fp32 rounding rather than bit for bit
        assert rel_l2(a.cpu(), b.cpu()) <= 1e-6
