"""GPU parity tests: hand-written sm_100a operators (through the C ABI) vs the CPU oracle, the
committed goldens, and the outputs of the reference's own CUDA kernels compiled unmodified
(tests/golden/ref_kernels.npz, minted by `make_golden.py ref_kernels`)."""
import os

import numpy as np
import pytest
import torch

from oracle import ops as O
from stereo_rcnn_b200 import ops as G
from stereo_rcnn_b200.synth import DEMO_P2, DEMO_P3, gen_rois, synth_pair

pytestmark = pytest.mark.gpu


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def rand_dets(n, seed, size=600.0, wh=120.0):
    rs = np.random.RandomState(seed)
    xy = rs.rand(n, 2) * size
    w = rs.rand(n, 2) * wh + 1
    sc = np.sort(rs.rand(n))[::-1]
    d = np.concatenate([xy, xy + w, sc[:, None]], 1).astype(np.float32)
    if n > 10:
        d[5, :4] = d[2, :4]            # exact duplicates
        d[7, :4] = d[2, :4]
    return d


@pytest.fixture(scope="module")
def ref_kernels(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_kernels.npz"))


# ------------------------------------------------------------------------ NMS
@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 300, 1000, 6000, 12000])
@pytest.mark.parametrize("thresh", [0.7, 0.3])
def test_nms_bit_exact_vs_oracle(n, thresh):
    d = rand_dets(n, n)
    keep = G.nms(cu(d), thresh).cpu().numpy().reshape(-1)
    np.testing.assert_array_equal(keep, O.nms(d, thresh))


def test_nms_empty_and_module_api():
    from stereo_rcnn_b200.model.nms.nms_wrapper import nms
    assert nms(torch.zeros(0, 5).cuda(), 0.5) == []
    d = rand_dets(500, 3)
    k = nms(cu(d), 0.7)
    assert k.dtype == torch.int32 and k.dim() == 2 and k.shape[1] == 1
    np.testing.assert_array_equal(k.cpu().numpy().reshape(-1), O.nms(d, 0.7))
    with pytest.raises(NotImplementedError):
        nms(cu(d), 0.7, force_cpu=True)


def test_nms_mask_upper_triangle_bits():
    d = rand_dets(777, 9, size=200)
    m = G.nms_mask(cu(d), 0.5).cpu().numpy().view(np.uint64)
    ref = O.nms_mask(d, 0.5)
    cb = ref.shape[1]
    for i in range(0, 777, 13):
        np.testing.assert_array_equal(m[i, i // 64:], ref[i, i // 64:])
        assert not m[i, :i // 64].any() or cb == 1


NMS_REF_CASES = [(6000, 1), (1234, 2), (64, 3)]          # (boxes, seed of rand_dets), IoU 0.7


def test_nms_vs_reference_cuda_kernel(ref_kernels):
    """keep lists of nms_cuda_compute of the reference (nms_cuda_kernel.cu:87-161), compiled unmodified"""
    for n, seed in NMS_REF_CASES:
        d = rand_dets(n, seed)
        ref_keep = ref_kernels["nms_keep_%d_%d" % (n, seed)]
        np.testing.assert_array_equal(ref_keep, O.nms(d, 0.7))              # pins the oracle
        np.testing.assert_array_equal(G.nms(cu(d), 0.7).cpu().numpy().reshape(-1), ref_keep)


# ------------------------------------------------------------------- RoIAlign
def rand_rois(R, H, W, scale, seed, batch=1):
    rs = np.random.RandomState(seed)
    x1 = rs.rand(R) * W / scale * 0.9
    y1 = rs.rand(R) * H / scale * 0.9
    w = rs.rand(R) * W / scale * 0.5 + 1
    h = rs.rand(R) * H / scale * 0.5 + 1
    b = rs.randint(0, batch, R)
    r = np.stack([b, x1, y1, np.minimum(x1 + w, W / scale - 1), np.minimum(y1 + h, H / scale - 1)], 1)
    r[0] = [0, 0, 0, 0, 0]                               # the zero-padded proposal row (Q11)
    r[1] = [0, 0, 0, W / scale - 1, H / scale - 1]       # touches the extrapolation band (Q16)
    return r.astype(np.float32)


@pytest.mark.parametrize("lat", [8, 15])
def test_roi_align_forward_vs_oracle(lat):
    rs = np.random.RandomState(0)
    feat = rs.randn(2, 48, 38, 125).astype(np.float32)
    rois = rand_rois(77, 38, 125, 38 / 600.0, 1, batch=2)
    scale = np.float32(38 / 600.0)
    out = torch.zeros(77, 48, lat, lat, device="cuda")
    assert G.roi_align_forward(lat, lat, scale, cu(feat), cu(rois), out) == 1
    ref = O.roi_align_forward(feat, rois, lat, lat, scale)
    np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=1e-6, atol=1e-6)
    assert (out.cpu().numpy() == ref).mean() > 0.999


def roi_align_ref_inputs():
    """feature map [1,32,40,60], 50 RoIs at spatial scale 0.25 and the top gradient [50,32,8,8] of the comparison with
    the reference's RoIAlign kernels"""
    rs = np.random.RandomState(5)
    feat = rs.randn(1, 32, 40, 60).astype(np.float32)
    rois = rand_rois(50, 40, 60, 0.25, 2)
    top = rs.randn(50, 32, 8, 8).astype(np.float32)
    return feat, rois, top


def test_roi_align_vs_reference_cuda_kernel(ref_kernels):
    """ROIAlignForwardLaucher / ROIAlignBackwardLaucher of the reference (roi_align_kernel.cu), compiled unmodified.
    The golden holds their outputs at a fixed sample of positions (every output of the two edge-case RoIs 0 and 1
    included) and their sums over the whole output; ours and the oracle's full outputs are compared to each other."""
    g = ref_kernels
    feat, rois, top = roi_align_ref_inputs()
    np.testing.assert_array_equal(rois, g["roi_rois"])
    f, r = cu(feat), cu(rois)
    out = torch.zeros(50, 32, 8, 8, device="cuda")
    G.roi_align_forward(8, 8, 0.25, f, r, out)
    out = out.cpu().numpy()
    ora = O.roi_align_forward(feat, rois, 8, 8, np.float32(0.25))
    idx, ref = g["roi_fwd_idx"], g["roi_fwd"]
    np.testing.assert_allclose(ora.reshape(-1)[idx], ref, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(out.reshape(-1)[idx], ref, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(out, ora, rtol=1e-6, atol=1e-6)
    _check_sums(out, g["roi_fwd_sums"], 1e-6)
    # backward
    gr = torch.zeros(1, 32, 40, 60, device="cuda")
    G.roi_align_backward(8, 8, 0.25, cu(top), r, gr)
    gr = gr.cpu().numpy()
    idx, ref = g["roi_bwd_idx"], g["roi_bwd"]
    np.testing.assert_allclose(gr.reshape(-1)[idx], ref, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(gr, O.roi_align_backward(top, rois, feat.shape, 8, 8, np.float32(0.25)),
                               rtol=1e-4, atol=1e-4)
    _check_sums(gr, g["roi_bwd_sums"], 1e-4)


def _check_sums(a, ref_sums, tol):
    """(sum, sum of magnitudes) of `a` against the reference's: the bound elementwise |a - ref| <= tol + tol * |ref|
    implies for both sums"""
    got = [a.sum(dtype=np.float64), np.abs(a).sum(dtype=np.float64)]
    np.testing.assert_allclose(got, ref_sums, rtol=0, atol=tol * (a.size + ref_sums[1]))


def test_roi_align_backward_vs_oracle_and_autograd_module():
    from stereo_rcnn_b200.model.roi_align.modules.roi_align import RoIAlignAvg
    rs = np.random.RandomState(7)
    feat = rs.randn(1, 16, 19, 63).astype(np.float32)
    rois = rand_rois(20, 19, 63, 19 / 600.0, 3)
    scale = np.float32(19 / 600.0)
    top = rs.randn(20, 16, 8, 8).astype(np.float32)
    g = torch.zeros(1, 16, 19, 63, device="cuda")
    G.roi_align_backward(8, 8, scale, cu(top), cu(rois), g)
    np.testing.assert_allclose(g.cpu().numpy(), O.roi_align_backward(top, rois, feat.shape, 8, 8, scale),
                               rtol=1e-4, atol=1e-4)
    f = cu(feat).requires_grad_(True)
    y = RoIAlignAvg(7, 7, 1 / 16.0)(f, cu(rois), float(scale))
    np.testing.assert_allclose(y.detach().cpu().numpy(), O.roi_align_avg(feat, rois, 7, 7, scale), rtol=1e-5,
                               atol=1e-5)
    y.sum().backward()
    assert f.grad is not None and torch.isfinite(f.grad).all()


def test_roi_align_backward_deterministic_fixed_point():
    """sb_roi_align_backward_det: same gradient as the atomic kernel / the oracle, but bit-identical run to run and
    under any permutation of the RoIs (integer accumulation), also with heavily overlapping RoIs and a wide range"""
    rs = np.random.RandomState(9)
    feat_shape = (2, 24, 19, 63)
    scale = np.float32(19 / 600.0)
    rois = np.concatenate([rand_rois(60, 19, 63, 19 / 600.0, 5)] * 3)          # every pixel hit many times
    rois[:, 0] = rs.randint(0, 2, rois.shape[0])
    top = (rs.randn(rois.shape[0], 24, 8, 8) * np.exp(rs.uniform(-8, 8, (rois.shape[0], 1, 1, 1)))).astype(np.float32)
    ref = np.zeros(feat_shape, np.float64)
    for n in range(2):
        sel = rois[:, 0] == n
        r = rois[sel].copy()
        r[:, 0] = 0
        ref[n] = O.roi_align_backward(top[sel], r, (1,) + feat_shape[1:], 8, 8, scale)[0]
    g = torch.full(feat_shape, 7.0, device="cuda")                               # overwritten, not accumulated
    G.roi_align_backward_det(8, 8, scale, cu(top), cu(rois), g)
    amax = np.abs(ref).max()
    assert np.abs(g.cpu().numpy() - ref).max() <= 2e-5 * amax        # the oracle itself sums in fp32
    perm = rs.permutation(rois.shape[0])
    g2 = torch.empty(feat_shape, device="cuda")
    G.roi_align_backward_det(8, 8, scale, cu(top[perm]), cu(rois[perm]), g2)
    assert torch.equal(g, g2)
    for _ in range(3):
        G.roi_align_backward_det(8, 8, scale, cu(top), cu(rois), g2)
        assert torch.equal(g, g2)
    G.roi_align_backward_det(8, 8, scale, cu(np.zeros_like(top)), cu(rois), g2)
    assert float(g2.abs().max()) == 0.0


@pytest.mark.parametrize("pooled", [7, 14])
def test_roi_align_pyramid_nhwc_vs_oracle(pooled):
    rs = np.random.RandomState(11)
    shapes = [(150, 497), (75, 249), (38, 125), (19, 63)]
    C = 64
    feats = [rs.randn(1, C, h, w).astype(np.float32) for h, w in shapes]
    R = 120
    x1 = rs.rand(R) * 1500
    y1 = rs.rand(R) * 400
    side = np.exp(rs.uniform(np.log(8), np.log(900), R))
    rois = np.stack([np.zeros(R), x1, y1, np.minimum(x1 + side * rs.uniform(0.5, 2, R), 1986),
                     np.minimum(y1 + side, 599)], 1).astype(np.float32)
    rois[0] = 0
    ref = O.pyramid_roi_feat(feats, rois, 600.0, pooled)             # R,C,p,p
    assert len(set(O.roi_levels(rois).tolist())) == 4
    fd = [cu(f.transpose(0, 2, 3, 1)) for f in feats]
    out = G.roi_align_pyramid_nhwc(fd, 600.0, cu(rois), pooled).cpu().numpy().transpose(0, 3, 1, 2)
    np.testing.assert_allclose(out, ref, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------- proposal layer
def test_proposal_layer_golden_bit_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "proposal_small.npz"))
    shapes = g["shapes"].tolist()
    rl, rr = G.proposal_layer(cu(g["cls_prob"]), cu(g["bbox_pred"]), cu(g["im_info"]), "TEST", shapes)
    ol, orr = O.proposal_layer(g["cls_prob"], g["bbox_pred"], g["im_info"], "TEST", shapes)
    np.testing.assert_array_equal(rl.cpu().numpy(), ol)
    np.testing.assert_array_equal(rr.cpu().numpy(), orr)
    # and against the reference's own output (differs from the oracle only by torch.exp vs sb_expf ulps)
    np.testing.assert_allclose(rl.cpu().numpy(), g["rois_left"], rtol=1e-6, atol=2e-4)


@pytest.mark.parametrize("cfg_key", ["TEST", "TRAIN"])
def test_proposal_layer_full_size_with_ties_bit_exact(cfg_key):
    shapes = [[150, 497], [75, 249], [38, 125], [19, 63], [10, 32]]
    A = 3 * sum(h * w for h, w in shapes)
    rs = np.random.RandomState(21)
    B = 2
    prob = rs.rand(B, A, 2).astype(np.float32)
    prob[0, ::5, 1] = 1.0                     # saturated scores: > pre_nms_top_n exact ties at the top
    prob[1, :, 1] = np.round(prob[1, :, 1] * 64) / 64     # heavy quantisation: ties straddle the cut
    bbox = (rs.randn(B, A, 6) * 0.5).astype(np.float32)
    info = np.array([[600, 1987, 1.6]] * B, np.float32)
    rl, rr = G.proposal_layer(cu(prob), cu(bbox), cu(info), cfg_key, shapes)
    ol, orr = O.proposal_layer(prob, bbox, info, cfg_key, shapes)
    np.testing.assert_array_equal(rl.cpu().numpy(), ol)
    np.testing.assert_array_equal(rr.cpu().numpy(), orr)


def test_proposal_layer_module_api():
    from stereo_rcnn_b200.model.rpn.proposal_layer import _ProposalLayer
    shapes = [[20, 32], [10, 16], [5, 8], [3, 4], [2, 2]]
    A = 3 * sum(h * w for h, w in shapes)
    rs = np.random.RandomState(2)
    prob = rs.rand(1, A, 2).astype(np.float32)
    bbox = (rs.randn(1, A, 6) * 0.2).astype(np.float32)
    info = np.array([[80, 128, 1.0]], np.float32)
    layer = _ProposalLayer(16, [0.5, 1, 2])
    rl, rr = layer((cu(prob), cu(bbox), cu(info), "TEST", shapes))
    ol, orr = O.proposal_layer(prob, bbox, info, "TEST", shapes)
    np.testing.assert_array_equal(rl.cpu().numpy(), ol)
    np.testing.assert_array_equal(rr.cpu().numpy(), orr)


def test_rpn_head_epilogue_channel_pairing():
    rs = np.random.RandomState(4)
    P = 1000
    head = (rs.randn(1, P, 32) * 2).astype(np.float32)
    cp, bp = G.rpn_head_epilogue(cu(head), 1, P)
    c = head[0, :, :6].astype(np.float64)
    e = np.exp(c)
    # Q7: score(a) = prob channel 2a+1 of the (c, c+3)-paired softmax
    s0 = e[:, 1] / (e[:, 1] + e[:, 4]); s1 = e[:, 3] / (e[:, 0] + e[:, 3]); s2 = e[:, 5] / (e[:, 2] + e[:, 5])
    sc = cp.cpu().numpy().reshape(P, 3, 2)[:, :, 1]
    np.testing.assert_allclose(sc, np.stack([s0, s1, s2], 1), rtol=1e-5, atol=1e-7)
    np.testing.assert_array_equal(bp.cpu().numpy().reshape(P, 18), head[0, :, 6:24])


# ---------------------------------------------------------------- dense_align
def test_dense_align_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "dense_align.npz"))
    left, right = synth_pair(int(g["H"]), int(g["W"]), int(g["seed"]), int(g["shift"]))
    c4 = G.calib_vec(g["p2"], g["p3"])
    st, dis = G.dense_align(c4, float(g["scale"]), cu(left), cu(right), cu(g["box_left"]), cu(g["keypoints"]),
                            cu(g["poses"]))
    np.testing.assert_array_equal(st.cpu().numpy(), g["status"])
    _check_dense(dis.cpu().numpy(), left, right, c4, float(g["scale"]), g["box_left"], g["keypoints"], g["poses"],
                 ref_dis=g["best_dis"])


def _check_dense(dis, left, right, c4, scale, b, k, p, ref_dis=None):
    """exact argmin agreement except on photometric near-ties (fp32 sum order), judged on the oracle's costs"""
    st_o, dis_o, dg = O.dense_align(c4, scale, left, right, b, k, p, diagnostics=True)
    if ref_dis is not None:
        np.testing.assert_allclose(dis_o, ref_dis, rtol=1e-6)
    same = np.abs(dis - dis_o) <= 1e-5 * np.abs(dis_o)
    assert same.mean() >= 0.97, same.mean()
    for i in np.nonzero(~same)[0]:
        cf = dg["cost_fine"][i]
        cc = dg["cost_coarse"][i]
        srt = np.sort(cf)
        src = np.sort(cc)
        near = (srt[1] - srt[0]) < 1e-4 * srt[0] or (src[1] - src[0]) < 1e-4 * src[0]
        assert near, (i, dis[i], dis_o[i])


@pytest.mark.parametrize("D", [1, 128])
def test_dense_align_sweep_vs_oracle(D):
    left, right = synth_pair(600, 1987, 3, 40)
    b, k, p = gen_rois(D, seed=5)
    c4 = G.calib_vec(DEMO_P2, DEMO_P3)
    scale = float(np.float32(1.6))
    st, dis = G.dense_align(c4, scale, cu(left), cu(right), cu(b), cu(k), cu(p))
    st_o, _ = O.dense_align(c4, scale, left, right, b, k, p)
    np.testing.assert_array_equal(st.cpu().numpy(), st_o)
    _check_dense(dis.cpu().numpy(), left, right, c4, scale, b, k, p)


def test_dense_align_no_valid_pixel_early_out_and_module_api():
    from stereo_rcnn_b200.model.dense_align.dense_align import align_parallel

    class Calib:
        p2 = np.array([[100., 0, 100, 4], [0, 100., 60, 0], [0, 0, 1, 0]])
        p3 = np.array([[100., 0, 100, -50], [0, 100., 60, 0], [0, 0, 1, 0]])
    left, right = synth_pair(120, 200, 5, 4)
    b = np.array([[5, 5, 30, 30], [6, 6, 28, 33]], np.float32)
    k = np.array([[17, 1, .9, 5, 30], [17, 1, .9, 6, 28]], np.float32)
    p = np.array([[30., 1.6, 20., 1.6, 1.5, 3.9, 0.3], [-30., 1.6, 25., 1.6, 1.5, 3.9, 1.0]], np.float32)
    st, dis = align_parallel(Calib, 1.0, cu(left)[None], cu(right)[None], cu(b), cu(k), cu(p))
    st_o, dis_o = O.dense_align(O.calib_vec(Calib.p2, Calib.p3), 1.0, left, right, b, k, p)
    assert st_o.sum() == 0
    np.testing.assert_array_equal(st.cpu().numpy(), st_o)
    np.testing.assert_array_equal(dis.cpu().numpy(), dis_o)          # dis_init, bit-exact
    st, dis = align_parallel(Calib, 1.0, cu(left)[None], cu(right)[None], cu(b[:0]), cu(k[:0]), cu(p[:0]))
    assert st.numel() == 0 and dis.numel() == 0


def test_class_nms_vs_oracle():
    rs = np.random.RandomState(8)
    R = 300
    scores = rs.rand(R, 2).astype(np.float32)
    scores[::7, 1] = 0.01                                  # below eval_thresh
    scores[5, 1] = scores[9, 1]                            # a tie
    xy = rs.rand(R, 2) * 300
    wh = rs.rand(R, 2) * 150 + 10
    boxes = np.zeros((R, 8), np.float32)
    boxes[:, 4:6], boxes[:, 6:8] = xy, xy + wh
    keep, num = G.class_nms(cu(scores), cu(boxes), 1, 0.05, 0.3)
    ref = O.per_class_nms(scores, boxes, 1, 0.05, 0.3)
    assert int(num[0]) == ref.size
    np.testing.assert_array_equal(keep[:ref.size].cpu().numpy(), ref)
    keep, num = G.class_nms(cu(scores * 0), cu(boxes), 1, 0.05, 0.3)
    assert int(num[0]) == 0


# Golden tests against the reference's own script lines (green on B200 since round 1).
def test_test_decode_vs_reference_script_golden(golden_dir):
    """sb_test_decode against the golden minted by executing test_net.py's own decode lines (tests/golden/
    make_golden.py (6)): index-valued columns exact, boxes to the exp-ulp level (torch.exp vs sb_expf)"""
    g = np.load(os.path.join(golden_dir, "test_decode.npz"))
    pbl, pbr, do, pk = G.test_decode(cu(g["rois_left"][0]), cu(g["rois_right"][0]), cu(g["bbox_pred"][0]),
                                     cu(g["bbox_pred_dim"][0]), cu(g["kpts_prob"]), cu(g["left_prob"]),
                                     cu(g["right_prob"]), cu(g["im_info"][0]))
    ref = O.test_decode(g["rois_left"][0], g["rois_right"][0], g["cls_prob"][0], g["bbox_pred"][0],
                        g["bbox_pred_dim"][0], g["kpts_prob"], g["left_prob"], g["right_prob"], g["im_info"][0])
    for a, b in zip((pbl, pbr, do, pk), ref[1:]):
        np.testing.assert_array_equal(a.cpu().numpy(), b)                      # bit-exact against the oracle
    np.testing.assert_allclose(pbl.cpu().numpy(), g["pred_boxes_left"], rtol=0, atol=2e-4)
    np.testing.assert_allclose(pbr.cpu().numpy(), g["pred_boxes_right"], rtol=0, atol=2e-4)
    np.testing.assert_array_equal(do.cpu().numpy(), g["dim_orien"])
    np.testing.assert_array_equal(pk.cpu().numpy(), g["pred_kpts"])


def test_class_nms_vs_reference_script_golden(golden_dir):
    """sb_class_nms against the golden minted by executing test_net.py:234-259 on the decode golden"""
    g = np.load(os.path.join(golden_dir, "class_nms.npz"))
    keep, num = G.class_nms(cu(g["scores"]), cu(g["pred_boxes_left"]), int(g["cls"]), float(g["score_thresh"]),
                            float(g["nms_thresh"]))
    assert int(num[0]) == g["kept_rois"].size
    np.testing.assert_array_equal(keep[:g["kept_rois"].size].cpu().numpy(), g["kept_rois"])


def test_proposal_layer_train_golden_bit_exact(golden_dir):
    """TRAIN configuration (12000 / 2000 / IoU 0.7; here pre_nms_top_n exceeds the 10 236 anchors of the small
    pyramid, so every anchor is a candidate) against the oracle (bit-exact) and the reference's own output"""
    g = np.load(os.path.join(golden_dir, "proposal_train.npz"))
    shapes = g["shapes"].tolist()
    rl, rr = G.proposal_layer(cu(g["cls_prob"]), cu(g["bbox_pred"]), cu(g["im_info"]), "TRAIN", shapes)
    ol, orr = O.proposal_layer(g["cls_prob"], g["bbox_pred"], g["im_info"], "TRAIN", shapes)
    np.testing.assert_array_equal(rl.cpu().numpy(), ol)
    np.testing.assert_array_equal(rr.cpu().numpy(), orr)
    np.testing.assert_allclose(rl.cpu().numpy(), g["rois_left"], rtol=1e-6, atol=2e-4)
    np.testing.assert_allclose(rr.cpu().numpy(), g["rois_right"], rtol=1e-6, atol=2e-4)
