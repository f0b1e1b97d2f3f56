"""Mint golden vectors from the REFERENCE's own Python (run in the build container only).

    python tests/golden/make_golden.py

Imports the reference from /root/reference through oracle/ref_shim.py (runtime
shims only, nothing copied), runs it on seeded inputs and stores small
input/output fixtures as ``tests/golden/*.npz``.  The GPU box has no
/root/reference; tests there only read the committed fixtures.
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
torch.set_num_threads(1)

from oracle import model, ops, ref_shim  # noqa: E402
from stereo_rcnn_b200.synth import synth_pair, gen_rois  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def demo_goldens():
    """(8) input pipeline and (9) the reference forward on a crop of the reference's own demo pair.

    demo/left.png|right.png (375x1242) are read where they lie; only small uint8 crops are stored.  The blob is made
    by the reference's own recipe (demo.py:106-120 / blob.py:44-64: BGR - PIXEL_MEANS, cv2.resize fx=fy=scale,
    INTER_LINEAR) with the cv2 of this image, then fed to the reference's `_StereoRCNN.forward` with our seeded weights."""
    import cv2
    ref = ref_shim.load()
    cfg = ref.cfg
    left = cv2.imread(os.path.join(ref_shim.REF, "demo/left.png"))        # BGR uint8 (= imread(...)[:,:,::-1])
    right = cv2.imread(os.path.join(ref_shim.REF, "demo/right.png"))
    assert left.shape == (375, 1242, 3)

    def blob(im, scale):
        f = im.astype(np.float32, copy=True)
        f -= cfg.PIXEL_MEANS
        f = cv2.resize(f, None, None, fx=scale, fy=scale, interpolation=cv2.INTER_LINEAR)
        return np.ascontiguousarray(f.transpose(2, 0, 1))
    # (8) prep_im_for_blob on a 64x96 crop at the demo scale 1.6 and at a KITTI-like non-dyadic scale
    c8 = left[170:234, 560:656].copy()
    np.savez_compressed(os.path.join(HERE, "prep_image.npz"), crop_bgr=c8, scale_a=1.6, blob_a=blob(c8, 1.6),
                        scale_b=600.0 / 370.0, blob_b=blob(c8, 600.0 / 370.0), cv2_version=cv2.__version__)
    # (9) forward on a 192x320 crop of the demo pair (cars + road), scale 1.6 -> 307x512
    y0, x0 = 150, 480
    cl, cr = left[y0:y0 + 192, x0:x0 + 320].copy(), right[y0:y0 + 192, x0:x0 + 320].copy()
    scale = 1.6
    bl, br = blob(cl, scale), blob(cr, scale)
    sd = model.make_state_dict(3)
    m = ref_shim.build_reference_model(sd)
    info = torch.tensor([[float(bl.shape[1]), float(bl.shape[2]), scale]])
    d = torch.zeros(1)
    with torch.no_grad():
        outs = m(torch.from_numpy(bl)[None], torch.from_numpy(br)[None], info, d, d, d, d, d, d)
    names = ["rois_left", "rois_right", "cls_prob", "bbox_pred", "dim_orien_pred", "kpts_prob",
             "left_border_prob", "right_border_prob"]
    gold = {n: o.numpy() for n, o in zip(names, outs[:8])}
    np.savez_compressed(os.path.join(HERE, "forward_demo.npz"), crop_left_bgr=cl, crop_right_bgr=cr, scale=scale,
                        crop_origin=np.array([y0, x0]), weight_seed=3, blob_checksum=np.array([bl.sum(dtype=np.float64),
                        br.sum(dtype=np.float64)]), **gold)
    print("demo goldens written")


def solver_goldens():
    """(10) the reference's own box solvers / infer_boundary / result writer (box_estimator.py, kitti_utils.py), executed
    from the files where they lie with two runtime patches (py2 implicit import, `scipy.array` removed from scipy)."""
    import math as m
    import tempfile
    import types
    src = open(os.path.join(ref_shim.REF, "lib/model/utils/box_estimator.py")).read()
    src = src.replace("import kitti_utils as utils", "utils = None").replace("scipy.array", "np.array")
    be = types.ModuleType("box_estimator")
    exec(compile(src, "box_estimator.py", "exec"), be.__dict__)
    ku = types.ModuleType("kitti_utils")
    exec(compile(open(os.path.join(ref_shim.REF, "lib/model/utils/kitti_utils.py")).read(), "kitti_utils.py", "exec"), ku.__dict__)
    calib = ref_shim.demo_calib()
    P2, P3 = calib.p2, calib.p3
    f32 = np.float32
    b, k, p = gen_rois(64, seed=7, p2=P2)
    rs = np.random.RandomState(1)
    rows = dict(alpha=[], dim=[], box_left=[], box_right=[], kpts=[], status=[], state=[], disparity=[], state_rect=[], z_rect=[])
    shape = (375, 1242, 3)
    for i in range(64):
        x, y, z, w, h, l, th = [float(v) for v in p[i]]
        bl = (P2[0, 3] - P3[0, 3]) / P2[0, 0]
        disp = P2[0, 0] * bl / z
        box_l = b[i].astype(np.float64)
        if i % 8 == 7:          # a truncated detection (left border)
            box_l[0] = 5.0
        box_r = box_l.copy()
        box_r[[0, 2]] -= disp
        box_r += rs.randn(4) * 0.5
        kt = int(rs.randint(0, 4))
        vw, vl = [(-w, -l), (-w, l), (w, l), (w, -l)][kt]
        X = x + np.cos(th) * vw / 2 + np.sin(th) * vl / 2
        Z = z - np.sin(th) * vw / 2 + np.cos(th) * vl / 2
        kp = np.array([P2[0, 0] * X / Z + P2[0, 2], kt, 0.9, box_l[0], box_l[2]])
        alpha = th - m.pi / 2 + m.atan2(-x, z) + rs.randn() * 0.05
        dim = np.array([w, h, l]) + rs.randn(3) * 0.05
        # everything reaches the solvers as float32 tensor elements in test_net.py
        box_l, box_r, kp, dim, alpha = [np.asarray(v, f32).astype(np.float64) for v in (box_l, box_r, kp, dim, alpha)]
        st, s = be.solve_x_y_z_theta_from_kpt(shape, calib, float(alpha), dim, box_l, box_r, kp)
        s = np.zeros(4) if np.isscalar(s) else np.asarray(s, np.float64)
        disp2 = float(f32(disp + rs.randn() * 0.3))
        s3, z3 = be.solve_x_y_theta_from_kpt(shape, calib, float(alpha), dim, box_l, disp2, kp)
        for key, v in (("alpha", alpha), ("dim", dim), ("box_left", box_l), ("box_right", box_r), ("kpts", kp),
                       ("status", st), ("state", s), ("disparity", disp2), ("state_rect", np.asarray(s3)), ("z_rect", z3)):
            rows[key].append(v)
    # infer_boundary on overlapping detections (kept order)
    rs = np.random.RandomState(4)
    x1 = rs.rand(24) * 1000
    y1 = rs.rand(24) * 200
    ib_boxes = np.stack([x1, y1, np.minimum(x1 + 30 + rs.rand(24) * 300, 1241), np.minimum(y1 + 30 + rs.rand(24) * 140, 374),
                         rs.rand(24)], 1).astype(f32)
    ib = ku.infer_boundary(shape, ib_boxes)
    # write_detection_results
    tmp = tempfile.mkdtemp()
    calib.t_cam2_cam0 = np.array([(P2[0, 3] - 0.0) / P2[0, 0], 0.0, 0.0])
    ku.write_detection_results(tmp, "000001", calib, rows["box_left"][0], np.array([1.5, 1.6, 20.25]),
                               np.array([1.6, 1.5, 3.9]), 0.3, 0.87)
    line = open(os.path.join(tmp, "data", "000001.txt")).read()
    np.savez_compressed(os.path.join(HERE, "box_solver.npz"), p2=P2, p3=P3, im_shape=np.array(shape),
                        **{k_: np.array(v) for k_, v in rows.items()}, ib_boxes=ib_boxes, ib_left_right=ib,
                        t_cam2_cam0_x=calib.t_cam2_cam0[0], kitti_line=np.array(line),
                        kitti_args=np.array([1.5, 1.6, 20.25, 1.6, 1.5, 3.9, 0.3, 0.87]))
    print("solver goldens written")


def train_goldens():
    """(11) train-time target layers (A16): the reference's OWN `_AnchorTargetLayer` / `_ProposalTargetLayer` /
    `_smooth_l1_loss` run on CPU (oracle/ref_shim.load_train: text patches only) with numpy's global stream seeded as
    trainval_net.py does (np.random.seed(cfg.RNG_SEED) = 3).  Inputs come from stereo_rcnn_b200.synth generators
    (recorded by their arguments; the arrays are stored too, the fixture is self-contained)."""
    from stereo_rcnn_b200 import synth
    ref = ref_shim.load_train()
    cfg = ref.cfg
    t = torch.from_numpy
    out = {}
    H, W = 160, 256
    feat_shapes = [[int(np.ceil(H / s)), int(np.ceil(W / s))] for s in (4, 8, 16, 32, 64)]
    out["feat_shapes"] = np.asarray(feat_shapes)
    for case, (B, batchsize, seed) in {"a": (2, 512, 0), "b": (3, 32, 5)}.items():
        gl, gr, gm, dim, kp, nb = synth.synth_train_gt(B, 30, H, W, seed)
        im_info = np.array([[H, W, 1.6]] * B, np.float32)
        cfg.TRAIN.RPN_BATCHSIZE = batchsize
        layer = ref.anchor_target_layer._AnchorTargetLayer(1, cfg.ANCHOR_RATIOS)
        np.random.seed(3)
        res = layer((torch.zeros(B, 2, 1, 1), t(gl), t(gr), t(gm), t(im_info), t(nb), feat_shapes))
        cfg.TRAIN.RPN_BATCHSIZE = 512
        out.update({"at_%s_gt_left" % case: gl, "at_%s_gt_right" % case: gr, "at_%s_gt_merge" % case: gm,
                    "at_%s_im_info" % case: im_info, "at_%s_rpn_batchsize" % case: batchsize})
        for nm, r in zip(("labels", "targets_left", "targets_right", "inside_w", "outside_w"), res):
            out["at_%s_%s" % (case, nm)] = r.numpy()
        lab = res[0].numpy()
        print("anchor targets", case, "fg", (lab == 1).sum(1), "bg", (lab == 0).sum(1))
    names = ("rois_left", "rois_right", "labels", "bbox_targets_left", "bbox_targets_right", "dim_orien_targets",
             "kpts_targets", "kpts_weight", "inside_w", "outside_w")
    for case, (B, R, near, seed) in {"a": (2, 200, 0.34, 1), "b": (2, 700, 0.6, 2)}.items():
        gl, gr, gm, dim, kp, nb = synth.synth_train_gt(B, 30, H, W, seed)
        rl, rr = synth.synth_train_rois(gl, R, H, W, seed + 100, near_gt=near)
        layer = ref.proposal_target_layer._ProposalTargetLayer(2)
        np.random.seed(3)
        res = layer(t(rl), t(rr), t(gl), t(gr), t(dim), t(kp), t(nb))
        out.update({"pt_%s_in_rois_left" % case: rl, "pt_%s_in_rois_right" % case: rr, "pt_%s_gt_left" % case: gl,
                    "pt_%s_gt_right" % case: gr, "pt_%s_gt_dim_orien" % case: dim, "pt_%s_gt_kpts" % case: kp})
        for nm, r in zip(names, res):
            out["pt_%s_%s" % (case, nm)] = r.numpy()
        print("proposal targets", case, "fg", (res[2].numpy() > 0).sum(1))
    g = torch.Generator().manual_seed(0)
    pred, tgt = torch.randn(3, 40, 6, generator=g), torch.randn(3, 40, 6, generator=g) * 0.5
    iw = (torch.rand(3, 40, 6, generator=g) > 0.5).float()
    ow = torch.rand(3, 40, 6, generator=g)
    out.update(sl1_pred=pred.numpy(), sl1_target=tgt.numpy(), sl1_inside=iw.numpy(), sl1_outside=ow.numpy(),
               sl1_sigma3=float(ref.net_utils._smooth_l1_loss(pred, tgt, iw, ow, sigma=3, dim=[1])),
               sl1_plain=float(ref.net_utils._smooth_l1_loss(pred[0], tgt[0])))
    np.savez_compressed(os.path.join(HERE, "train_targets.npz"), **out)


def ref_kernel_goldens(out_dir=HERE):
    """(12) outputs of the reference's own CUDA kernels (nms_cuda_compute, ROIAlignForwardLaucher,
    ROIAlignBackwardLaucher), compiled unmodified for sm_100a by oracle/build.py build_ref(), on the seeded inputs of
    tests/test_gpu_ops.py.  Needs a GPU and oracle/_ref/libref_ops.so:

        python tests/golden/make_golden.py ref_kernels [OUT_DIR]

    The RoIAlign outputs are stored at a fixed seeded sample of positions (plus every output of the edge-case RoIs 0
    and 1) and as (sum, sum of magnitudes) over the whole array, which keeps the fixture small."""
    import ctypes
    from oracle import build as ob
    sys.path.insert(0, os.path.join(HERE, ".."))
    from test_gpu_ops import NMS_REF_CASES, rand_dets, roi_align_ref_inputs
    so = ob.build_ref()
    assert so is not None, "oracle/_ref/libref_ops.so not built (needs the reference's sources)"
    lib = ctypes.CDLL(so)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    out = {}
    for n, seed in NMS_REF_CASES:
        d = torch.from_numpy(rand_dets(n, seed)).cuda()
        keep = torch.zeros(n, dtype=torch.int32, device="cuda")
        num = torch.zeros(1, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        lib.nms_cuda_compute(p(keep), p(num), p(d), n, 5, ctypes.c_float(0.7))
        torch.cuda.synchronize()
        out["nms_keep_%d_%d" % (n, seed)] = keep[:int(num[0])].cpu().numpy()
    feat, rois, top = roi_align_ref_inputs()
    f, r, t = (torch.from_numpy(a).cuda() for a in (feat, rois, top))
    R, C, H, W, P = rois.shape[0], feat.shape[1], feat.shape[2], feat.shape[3], 8
    fwd = torch.zeros(R, C, P, P, device="cuda")
    bwd = torch.zeros(1, C, H, W, device="cuda")
    torch.cuda.synchronize()
    lib.ROIAlignForwardLaucher(p(f), ctypes.c_float(0.25), R, H, W, C, P, P, p(r), p(fwd), ctypes.c_void_p(0))
    lib.ROIAlignBackwardLaucher(p(t), ctypes.c_float(0.25), 1, R, H, W, C, P, P, p(r), p(bwd), ctypes.c_void_p(0))
    torch.cuda.synchronize()
    fwd, bwd = fwd.cpu().numpy().reshape(-1), bwd.cpu().numpy().reshape(-1)
    rs = np.random.RandomState(12)
    edge = 2 * C * P * P                                 # RoI 0 (all zero) and RoI 1 (extrapolation band)
    fidx = np.concatenate([np.arange(edge), np.sort(rs.choice(np.arange(edge, fwd.size), 4096, replace=False))])
    bidx = np.sort(rs.choice(bwd.size, 8192, replace=False))
    sums = lambda a: np.array([a.sum(dtype=np.float64), np.abs(a).sum(dtype=np.float64)])
    out.update(roi_rois=rois, roi_fwd_idx=fidx.astype(np.int32), roi_fwd=fwd[fidx], roi_fwd_sums=sums(fwd),
               roi_bwd_idx=bidx.astype(np.int32), roi_bwd=bwd[bidx], roi_bwd_sums=sums(bwd))
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "ref_kernels.npz"), **out)
    print({k: v.shape for k, v in out.items()})


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "demo":
        return demo_goldens()
    if len(sys.argv) > 1 and sys.argv[1] == "solver":
        return solver_goldens()
    if len(sys.argv) > 1 and sys.argv[1] == "ref_kernels":
        return ref_kernel_goldens(*sys.argv[2:3])
    ref = ref_shim.load()
    cfg = ref.cfg
    calib = ref_shim.demo_calib()

    # ---- (1) anchors + decode/clip --------------------------------------------------
    shapes = [[150, 497], [75, 249], [38, 125], [19, 63], [10, 32]]
    a = ref.generate_anchors.generate_anchors_all_pyramids(
        np.array(cfg.FPN_ANCHOR_SCALES), cfg.ANCHOR_RATIOS, shapes,
        np.array(cfg.FPN_FEAT_STRIDES), cfg.FPN_ANCHOR_STRIDE)
    sel = np.random.RandomState(0).choice(a.shape[0], 4096, replace=False)
    sel.sort()
    deltas = (np.random.RandomState(1).randn(4096, 4) * 0.4).astype(np.float32)
    an32 = torch.from_numpy(a[sel].astype(np.float32)).view(1, -1, 4)
    dec = ref.bbox_transform.bbox_transform_inv(an32, torch.from_numpy(deltas).view(1, -1, 4), 1)
    dec = ref.bbox_transform.clip_boxes(dec, torch.tensor([[600., 1987., 1.6]]), 1)[0].numpy()
    np.savez_compressed(os.path.join(HERE, "anchors_decode.npz"), shapes=np.array(shapes),
                        n_anchors=a.shape[0], sel=sel, anchors_sel=a[sel],
                        anchors_sum=a.sum(0), anchors_abs_sum=np.abs(a).sum(0),
                        deltas=deltas, decoded=dec)

    # ---- (2) proposal layer on synthetic RPN outputs (small pyramid) ----------------
    pshapes = [[40, 64], [20, 32], [10, 16], [5, 8], [3, 4]]
    A = 3 * sum(h * w for h, w in pshapes)
    rs = np.random.RandomState(7)
    prob = rs.rand(1, A, 2).astype(np.float32)
    # no forced score ties here: the reference leaves tie order to torch.sort (unspecified),
    # so a golden can only pin tie-free inputs; the tie rule is covered by oracle-level tests.
    bbox = (rs.randn(1, A, 6) * 0.3).astype(np.float32)
    info = np.array([[160., 256., 1.0]], np.float32)
    layer = ref.proposal_layer._ProposalLayer(cfg.FEAT_STRIDE[0], cfg.ANCHOR_RATIOS)
    rl, rr = layer((torch.from_numpy(prob), torch.from_numpy(bbox), torch.from_numpy(info), "TEST", pshapes))
    np.savez_compressed(os.path.join(HERE, "proposal_small.npz"), shapes=np.array(pshapes), cls_prob=prob,
                        bbox_pred=bbox, im_info=info, rois_left=rl.numpy(), rois_right=rr.numpy())

    # ---- (3) dense_align ------------------------------------------------------------
    H, W = 600, 1987
    left, right = synth_pair(H, W, seed=3, shift=40)
    b, k, p = gen_rois(24, seed=3, p2=calib.p2)
    scale = float(np.float32(1.6))
    st, dis = ref.dense_align.align_parallel(calib, scale, torch.from_numpy(left)[None],
                                             torch.from_numpy(right)[None], torch.from_numpy(b),
                                             torch.from_numpy(k), torch.from_numpy(p))
    s2 = scale * 2
    uvz, wgt = ref.dense_align.sample(calib, s2, 2 * H, 2 * W, torch.from_numpy(b) * s2,
                                      torch.from_numpy(p), (torch.from_numpy(k) * s2)[:, 3:5])
    np.savez_compressed(os.path.join(HERE, "dense_align.npz"), H=H, W=W, seed=3, shift=40,
                        p2=calib.p2, p3=calib.p3, scale=scale, box_left=b, keypoints=k, poses=p,
                        status=st.numpy(), best_dis=dis.numpy(), npix=wgt.sum(1).numpy().astype(np.int32),
                        uvz_head=uvz.numpy()[:, :64].copy())

    # ---- (4) full forward on a small pair -------------------------------------------
    sd = model.make_state_dict(3)
    m = ref_shim.build_reference_model(sd)
    H, W = 160, 256
    left, right = synth_pair(H, W, seed=11, shift=7)
    iml, imr = torch.from_numpy(left)[None], torch.from_numpy(right)[None]
    info = torch.tensor([[H, W, 1.0]])
    d = torch.zeros(1)
    with torch.no_grad():
        outs = m(iml, imr, info, d, d, d, d, d, d)
    names = ["rois_left", "rois_right", "cls_prob", "bbox_pred", "dim_orien_pred", "kpts_prob",
             "left_border_prob", "right_border_prob"]
    gold = {n: o.numpy() for n, o in zip(names, outs[:8])}
    np.savez_compressed(os.path.join(HERE, "forward_small.npz"), H=H, W=W, seed=11, shift=7,
                        weight_seed=3, **gold)
    # ---- (5) proposal layer, TRAIN configuration (12000 / 2000, NMS 0.7) ----------------
    rs = np.random.RandomState(17)
    prob = rs.rand(1, A, 2).astype(np.float32)
    bbox = (rs.randn(1, A, 6) * 0.3).astype(np.float32)
    info = np.array([[160., 256., 1.0]], np.float32)
    layer = ref.proposal_layer._ProposalLayer(cfg.FEAT_STRIDE[0], cfg.ANCHOR_RATIOS)
    rl, rr = layer((torch.from_numpy(prob), torch.from_numpy(bbox), torch.from_numpy(info), "TRAIN", pshapes))
    np.savez_compressed(os.path.join(HERE, "proposal_train.npz"), shapes=np.array(pshapes), cls_prob=prob,
                        bbox_pred=bbox, im_info=info, rois_left=rl.numpy(), rois_right=rr.numpy())

    # ---- (6) test-time decode: the reference's own script lines (test_net.py:138-212) -----
    # executed from the file where it lies -- nothing is copied -- on synthetic head outputs
    R = 96
    rs = np.random.RandomState(23)
    x1 = rs.rand(R) * 1500
    y1 = rs.rand(R) * 400
    rois_l = np.stack([np.zeros(R), x1, y1, x1 + 8 + rs.rand(R) * 400, y1 + 8 + rs.rand(R) * 180], 1).astype(np.float32)
    rois_r = rois_l.copy()
    rois_r[:, [1, 3]] -= (rs.rand(R, 1) * 60).astype(np.float32)

    def softmax(z):
        e = np.exp(z - z.max(1, keepdims=True))
        return (e / e.sum(1, keepdims=True)).astype(np.float32)
    inp = dict(rois_left=rois_l[None], rois_right=rois_r[None], cls_prob=softmax(rs.randn(R, 2))[None],
               bbox_pred=(rs.randn(1, R, 12) * 0.8).astype(np.float32),
               bbox_pred_dim=rs.randn(1, R, 10).astype(np.float32),
               kpts_prob=softmax(rs.randn(R, 4 * cfg.KPTS_GRID) * 2), left_prob=softmax(rs.randn(R, cfg.KPTS_GRID) * 2),
               right_prob=softmax(rs.randn(R, cfg.KPTS_GRID) * 2), im_info=np.array([[600., 1987., 1.6]], np.float32))
    import time as _time
    import types
    src = open(os.path.join(ref_shim.REF, "test_net.py")).read().split("\n")
    lo = next(i for i, l in enumerate(src) if l.strip() == "scores = cls_prob.data")
    hi = next(i for i, l in enumerate(src) if l.strip() == "dim_orien = dim_orien.squeeze()")
    block = "\n".join(l[4:] if l.startswith("    ") else l for l in src[lo:hi + 1])
    ns = {k: torch.from_numpy(v) for k, v in inp.items()}
    ns.update(torch=torch, cfg=cfg, time=_time, imdb=types.SimpleNamespace(_classes=("__background__", "Car")),
              bbox_transform_inv=ref.bbox_transform.bbox_transform_inv, clip_boxes=ref.bbox_transform.clip_boxes,
              kpts_transform_inv=ref.bbox_transform.kpts_transform_inv,
              border_transform_inv=ref.bbox_transform.border_transform_inv)
    exec(compile(block, "test_net.py[%d:%d]" % (lo + 1, hi + 1), "exec"), ns)
    np.savez_compressed(os.path.join(HERE, "test_decode.npz"), ref_lines=np.array([lo + 1, hi + 1]),
                        scores=ns["scores"].numpy(), pred_boxes_left=ns["pred_boxes_left"].numpy(),
                        pred_boxes_right=ns["pred_boxes_right"].numpy(), pred_kpts=ns["pred_kpts"].numpy(),
                        dim_orien=ns["dim_orien"].numpy(), **inp)

    # ---- (7) per-class NMS: the reference's own script lines (test_net.py:234-259) on the decode outputs of (6) ----
    # threshold / sort / gather are the reference's statements; `nms` is ref_shim's stand-in for the cffi extension
    # (the C restatement of nms_cuda_kernel.cu, itself pinned to the compiled reference kernel on the GPU box)
    lo2 = next(i for i, l in enumerate(src) if l.strip().startswith("inds = torch.nonzero(scores[:,j] > eval_thresh)"))
    hi2 = next(i for i, l in enumerate(src) if i > lo2 and l.strip() == "cls_kpts = cls_kpts[keep]")
    body = [l for l in src[lo2:hi2 + 1] if l.strip() and not l.strip().startswith("#")]
    ind0 = len(body[0]) - len(body[0].lstrip())
    ind1 = len(body[2]) - len(body[2].lstrip())          # body of the `if inds.numel() > 0:` block
    block2 = "\n".join((l[ind1:] if (len(l) - len(l.lstrip())) >= ind1 else l[ind0:]) for l in body
                       if not l.strip().startswith("if inds.numel()"))
    ns2 = dict(torch=torch, cfg=cfg, j=1, eval_thresh=0.05, nms=sys.modules["model.nms.nms_wrapper"].nms, scores=ns["scores"],
               pred_boxes_left=ns["pred_boxes_left"], pred_boxes_right=ns["pred_boxes_right"],
               dim_orien=ns["dim_orien"], pred_kpts=ns["pred_kpts"])
    exec(compile(block2, "test_net.py[%d:%d]" % (lo2 + 1, hi2 + 1), "exec"), ns2)
    kept_rois = ns2["inds"][ns2["order"]][ns2["keep"]].numpy().astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "class_nms.npz"), ref_lines=np.array([lo2 + 1, hi2 + 1]),
                        scores=ns["scores"].numpy(), pred_boxes_left=ns["pred_boxes_left"].numpy(), cls=1,
                        score_thresh=0.05, nms_thresh=float(cfg.TEST.NMS), kept_rois=kept_rois,
                        cls_dets_left=ns2["cls_dets_left"].numpy(), cls_kpts=ns2["cls_kpts"].numpy())
    demo_goldens()
    solver_goldens()
    train_goldens()
    print("goldens written to", HERE)


if __name__ == "__main__":
    main()
