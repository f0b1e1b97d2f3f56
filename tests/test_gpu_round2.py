"""GPU parity tests added in round 2 (all through the C ABI):

* the composed forward at the BENCHMARKED configuration (600x1987 pair, default fp16-operand mode) against the
  CPU oracle, per tensor, with the errors printed;
* the reference's own (un-normalised) random initialisation in the tf32 mode;
* a crop of the reference's demo pair through the device input pipeline (prep_im_for_blob) and the forward, against
  the reference's own forward (tests/golden/forward_demo.npz);
* several pipeline slots in flight at once (private workspaces) against one-at-a-time results;
* the record-emitting decode, and the record all-gather over peer memory (needs >= 2 GPUs).
"""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import model as OM
from oracle import ops as O
from stereo_rcnn_b200 import engine as E
from stereo_rcnn_b200 import ops as G
from stereo_rcnn_b200 import parallel as P
from stereo_rcnn_b200 import pipeline as PL
from stereo_rcnn_b200.synth import (DEMO_P2, DEMO_P3, gen_rois, make_reference_init_state_dict, make_state_dict,
                                    synth_pair)

pytestmark = pytest.mark.gpu


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def l2_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


# The stated bar of the tensor-core modes (DESIGN.md section 2): operands carry an 11-bit significand (fp16 / TF32 --
# tcgen05 has no fp32 kind), so per tensor the RELATIVE L2 error is held below 1e-3 (measured 2e-4 ... 7e-4) and the
# max-norm relative error below 1.5e-3 (measured up to ~1.2e-3: the largest of 10^5..10^8 element errors sits at
# 4-5 sigma).  Both are printed per tensor; bench.py reports the same table in its `parity` key.
L2_BAR, MAX_BAR = 1.0e-3, 1.5e-3
# Probability tensors (softmax outputs in [0, 1]) are held to the same relative L2 bar and to an ABSOLUTE deviation of
# 3e-3: a logit error of relative 5e-4 on a logit of magnitude 10 moves a probability by up to 0.25 * 5e-3, so their
# max-norm is set by how peaked the distribution is, not by the kernels (measured up to 2.2e-3 on the real demo crop).
PROB_ABS_BAR = 3.0e-3
PROBS = ("rpn_cls_prob", "cls_prob", "kpts_prob", "left_border_prob", "right_border_prob")


def check(name, got, ref, report, l2_bar=L2_BAR, max_bar=MAX_BAR):
    l2, mx = l2_err(got, ref), rel_err(got, ref)
    if name.split(" ")[0] in PROBS:
        ab = float(np.abs(np.asarray(got, np.float64) - np.asarray(ref, np.float64)).max())
        report.append("%-18s l2 %.2e  max-norm %.2e  max abs %.2e (probabilities)" % (name, l2, mx, ab))
        return l2 < l2_bar and ab < PROB_ABS_BAR
    report.append("%-18s l2 %.2e  max-norm %.2e" % (name, l2, mx))
    return l2 < l2_bar and mx < max_bar


def compare_forward(eng, o, iml, imr, info, overlap_min):
    """GPU forward vs oracle tensors `o` of the same pair; heads on the oracle's RoIs (identical inputs)"""
    r = eng.forward(iml.cuda(), imr.cuda(), info.cuda(), keep_features=True)
    torch.cuda.synchronize()
    rep, bad = [], []
    for k in ("c2", "c3", "c4", "c5", "p5", "p4", "p3", "p2", "p6"):
        got = r["feats"][k].float().permute(0, 3, 1, 2).cpu().numpy()
        for side, s in (("left", 0), ("right", 1)):
            if not check("%s/%s" % (k, side), got[s:s + 1], o[side][k].numpy(), rep):
                bad.append(k + side)
    for k in ("rpn_cls_prob", "rpn_bbox_pred"):
        if not check(k, r[k].cpu().numpy(), o[k].numpy(), rep):
            bad.append(k)
    # proposal layer on the ORACLE's RPN tensors: bit-exact indices and boxes at this size
    rl, rr = G.proposal_layer(o["rpn_cls_prob"].cuda(), o["rpn_bbox_pred"].cuda(), info.cuda(), "TEST", o["rpn_shapes"])
    np.testing.assert_array_equal(rl.cpu().numpy(), o["rois_left"].numpy())
    np.testing.assert_array_equal(rr.cpu().numpy(), o["rois_right"].numpy())
    h = eng.heads(r["feats_raw"], 1, rl.view(-1, 5), rr.view(-1, 5), float(iml.shape[2]))
    torch.cuda.synchronize()
    for k in ("pooled_box", "pooled_kpts"):
        if not check(k, h[k].float().permute(0, 3, 1, 2).cpu().numpy(), o[k].numpy(), rep):
            bad.append(k)
    for k in ("fc7", "cls_prob", "bbox_pred", "dim_orien_pred", "kpts_pred_all", "kpts_prob", "left_border_prob",
              "right_border_prob"):
        if not check(k, h[k].cpu().numpy().reshape(o[k].shape), o[k].numpy(), rep):
            bad.append(k)
    a = {tuple(np.round(x, 1)) for x in r["rois_left"][0].cpu().numpy()}
    b = {tuple(np.round(x, 1)) for x in o["rois_left"][0].numpy()}
    frac = len(a & b) / float(len(b))
    rep.append("end-to-end proposal set overlap %.3f (floor %.2f)" % (frac, overlap_min))
    print("\n".join(rep))
    assert not bad, bad
    assert frac >= overlap_min
    return r, h


def test_forward_full_config_fp16_vs_oracle():
    """BASELINE.json configs[1]: the 600x1987 pair of the bench, default fp16-operand mode, every stage"""
    H, W = 600, 1987
    left, right = synth_pair(H, W, seed=3, shift=48)                 # bench.py make_inputs(rank 0)
    sd = make_state_dict(3)
    iml, imr = torch.from_numpy(left)[None], torch.from_numpy(right)[None]
    info = torch.tensor([[float(H), float(W), 1.6]])
    o = OM.forward(sd, iml, imr, info)
    eng = E.StereoRCNNEngine(sd, "cuda", precision="fp16")
    assert eng.precision == "fp16"
    compare_forward(eng, o, iml, imr, info, overlap_min=FULL_OVERLAP_MIN)


# measured end-to-end proposal-set overlaps (GPU proposals from GPU RPN scores vs the oracle's; greedy NMS amplifies
# 1e-3 score perturbations) minus a margin -- see DESIGN.md section 2 for the measured values
# measured on B200 (round 2): 0.840 at 600x1987, 0.743 on the demo crop
FULL_OVERLAP_MIN = float(os.environ.get("SB_FULL_OVERLAP_MIN", "0.78"))
DEMO_OVERLAP_MIN = float(os.environ.get("SB_DEMO_OVERLAP_MIN", "0.68"))


def test_reference_init_tf32_trunk_fpn_rpn():
    """the reference's own un-normalised init (resnet.py:123-129, stereo_rcnn.py:47-85): activations reach ~1e6 by
    C4, which fp16 cannot hold -- the tf32 mode (fp32 storage) runs them.  Without normalisation nothing damps the
    operand-rounding noise of the ~100 layers: measured relative L2 0.8e-3 ... 1.25e-3 and max-norm up to 2.1e-3 (about
    twice the variance-preserving weights'), so this weight set is held to 2e-3 / 3e-3; the exact-fp32 SIMT path is the
    yardstick below.  With these weights the RPN deltas overflow exp() in the reference itself, so the comparison
    stops at the RPN tensors."""
    H, W = 160, 256
    left, right = synth_pair(H, W, 11, 7)
    sd = make_reference_init_state_dict(3)
    iml, imr = torch.from_numpy(left)[None], torch.from_numpy(right)[None]
    info = torch.tensor([[float(H), float(W), 1.0]])
    o = OM.forward(sd, iml, imr, info, stop_after="rpn")
    assert float(o["left"]["c4"].abs().max()) > 1e5                 # really un-normalised
    eng = E.StereoRCNNEngine(sd, "cuda", precision="tf32")
    feats = eng.trunk_fpn(torch.cat((iml, imr), 0).cuda())
    cls_prob, bbox, shapes = eng.rpn(feats, 1)
    torch.cuda.synchronize()
    rep, bad = [], []
    for k in ("c2", "c3", "c4", "c5", "p5", "p4", "p3", "p2", "p6"):
        v = feats[k]
        if k[0] == "c":
            v = G.unbias(v)
        got = v.permute(0, 3, 1, 2).cpu().numpy()
        if not check(k + "/left", got[0:1], o["left"][k].numpy(), rep, 2e-3, 3e-3):
            bad.append(k)
        if not check(k + "/right", got[1:2], o["right"][k].numpy(), rep, 2e-3, 3e-3):
            bad.append(k)
    if not check("rpn_bbox_pred", bbox.cpu().numpy(), o["rpn_bbox_pred"].numpy(), rep, 2e-3, 3e-3):
        bad.append("rpn_bbox_pred")
    # saturated probabilities: compare as absolute values (they are exactly 0 or 1 almost everywhere)
    d = np.abs(cls_prob.cpu().numpy() - o["rpn_cls_prob"].numpy())
    rep.append("rpn_cls_prob       mean abs diff %.2e, fraction differing by > 1e-3: %.4f" % (d.mean(), (d > 1e-3).mean()))
    print("\n".join(rep))
    assert not bad, bad
    assert (d > 1e-3).mean() < 0.01
    # exact-fp32 yardstick on the same weights: the SIMT path reproduces the oracle to fp32 rounding
    eng = E.StereoRCNNEngine(sd, "cuda", conv_impl="simt")
    feats = eng.trunk_fpn(torch.cat((iml, imr), 0).cuda())
    torch.cuda.synchronize()
    for k in ("c3", "c5", "p2"):
        got = feats[k].permute(0, 3, 1, 2).cpu().numpy()
        assert l2_err(got[0:1], o["left"][k].numpy()) < 2e-5, k


def test_prep_image_kernel_vs_oracle_and_cv2_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "prep_image.npz"))
    crop = torch.from_numpy(g["crop_bgr"]).cuda()
    for tag in ("a", "b"):
        sc = float(g["scale_" + tag])
        got = G.prep_image(crop, sc).cpu().numpy()
        np.testing.assert_array_equal(got, O.prep_image(g["crop_bgr"], sc))       # same operation order: bit-exact
        np.testing.assert_allclose(got, g["blob_" + tag], rtol=0, atol=6.2e-5)   # cv2 itself: <= 2 ulp
    rgb = torch.from_numpy(np.ascontiguousarray(g["crop_bgr"][:, :, ::-1])).cuda()
    np.testing.assert_array_equal(G.prep_image(rgb, 1.6, rgb_input=True).cpu().numpy(), O.prep_image(g["crop_bgr"], 1.6))
    # full KITTI frame size
    im = np.random.RandomState(3).randint(0, 256, (375, 1242, 3)).astype(np.uint8)
    got = G.prep_image(torch.from_numpy(im).cuda(), 1.6)
    assert tuple(got.shape) == (3, 600, 1987)
    np.testing.assert_array_equal(got.cpu().numpy(), O.prep_image(im, 1.6))


def test_demo_pair_crop_forward_vs_reference_golden(golden_dir):
    """a crop of the reference's demo/left.png|right.png: device input pipeline -> forward; features against the
    oracle, head outputs on the reference's RoIs against the reference's OWN forward (golden)"""
    g = np.load(os.path.join(golden_dir, "forward_demo.npz"))
    sc = float(g["scale"])
    bl = G.prep_image(torch.from_numpy(g["crop_left_bgr"]).cuda(), sc)
    br = G.prep_image(torch.from_numpy(g["crop_right_bgr"]).cuda(), sc)
    torch.cuda.synchronize()
    np.testing.assert_allclose([float(bl.double().sum()), float(br.double().sum())], g["blob_checksum"], rtol=1e-6)
    sd = make_state_dict(int(g["weight_seed"]))
    iml, imr = bl[None].cpu(), br[None].cpu()
    info = torch.tensor([[float(bl.shape[1]), float(bl.shape[2]), sc]])
    o = OM.forward(sd, iml, imr, info)
    eng = E.StereoRCNNEngine(sd, "cuda")
    r, _h = compare_forward(eng, o, iml, imr, info, overlap_min=DEMO_OVERLAP_MIN)
    # heads on the REFERENCE's RoIs vs the reference's outputs
    rl, rr = torch.from_numpy(g["rois_left"]).cuda(), torch.from_numpy(g["rois_right"]).cuda()
    h = eng.heads(r["feats_raw"], 1, rl.view(-1, 5), rr.view(-1, 5), float(bl.shape[1]))
    torch.cuda.synchronize()
    rep, bad = [], []
    for k in ("cls_prob", "bbox_pred", "dim_orien_pred", "kpts_prob", "left_border_prob", "right_border_prob"):
        if not check(k + " (ref)", h[k].cpu().numpy().reshape(g[k].shape), g[k], rep):
            bad.append(k)
    print("\n".join(rep))
    assert not bad, bad


def test_decode_record_kernel():
    rs = np.random.RandomState(5)
    R = 300
    x1 = rs.rand(R) * 1000
    y1 = rs.rand(R) * 300
    rl = np.stack([np.zeros(R), x1, y1, x1 + rs.rand(R) * 300 + 5, y1 + rs.rand(R) * 200 + 5], 1).astype(np.float32)
    rr = rl.copy()
    rr[:, [1, 3]] -= 20

    def sm(z):
        e = np.exp(z - z.max(1, keepdims=True))
        return (e / e.sum(1, keepdims=True)).astype(np.float32)
    cls, bp, dp = sm(rs.randn(R, 2)), (rs.randn(R, 12) * 0.8).astype(np.float32), rs.randn(R, 10).astype(np.float32)
    kp, lp, rp = sm(rs.randn(R, 112)), sm(rs.randn(R, 28)), sm(rs.randn(R, 28))
    info = np.array([600, 1987, 1.6], np.float32)
    c = lambda a: torch.from_numpy(a).cuda()
    base = G.test_decode(c(rl), c(rr), c(bp), c(dp), c(kp), c(lp), c(rp), c(info))
    pbl, pbr, do, pk, rec = G.test_decode_record(c(rl), c(rr), c(cls), c(bp), c(dp), c(kp), c(lp), c(rp), c(info))
    for a, b in zip(base, (pbl, pbr, do, pk)):
        assert torch.equal(a, b)
    assert torch.equal(rec, P.detection_record(c(cls), pbl, pbr, do, pk))
    assert rec.shape == (R, P.REC_COLS)


def test_slots_in_flight_keep_private_workspaces():
    """Three pipeline slots with DIFFERENT pairs replayed concurrently on their own streams (the bench's throughput
    schedule) must each reproduce what the same slot gives when it runs alone: the proposal / NMS / dense_align
    workspaces hold live state between launches and are private to a slot (ops.WorkspaceOwner)."""
    H, W = 192, 416
    sd = make_state_dict(3)
    dev = torch.device("cuda")
    pipe = PL.StereoPipeline(sd, dev, throughput=True, scale=1.0)
    calib4 = G.calib_vec(DEMO_P2 / np.array([[3.], [3.], [1.]]), DEMO_P3 / np.array([[3.], [3.], [1.]]))
    slots = []
    for i in range(3):
        left, right = synth_pair(H, W, seed=20 + i, shift=6 + i)
        b, k, p = gen_rois(8, seed=5 + i)
        b = b / 3.0
        k[:, [0, 3, 4]] /= 3.0
        rois3d = tuple(torch.from_numpy(x).cuda() for x in (b, k, p))
        slots.append(PL.GraphSlot(pipe, torch.from_numpy(left)[None].cuda(), torch.from_numpy(right)[None].cuda(),
                                  calib4, rois3d))
    alone = []
    for s in slots:                      # one at a time
        rec, keep, nkeep, st, dis = s.run()
        torch.cuda.synchronize()
        alone.append((rec.clone(), keep.clone(), nkeep.clone(), st[0].clone(), dis[0].clone()))
    assert not torch.equal(alone[0][0], alone[1][0])            # the pairs really differ
    for rep in range(8):                 # all in flight, interleaved
        for s in slots:
            with torch.cuda.stream(s.stream):
                s.run()
        torch.cuda.synchronize()
        for s, ref in zip(slots, alone):
            rec, keep, nkeep, st, dis = s.outputs
            assert torch.equal(rec, ref[0]), "record differs with slots in flight (rep %d)" % rep
            n = int(ref[2][0])
            assert int(nkeep[0]) == n and torch.equal(keep[0, :n], ref[1][0, :n])
            assert torch.equal(st[0], ref[3]) and torch.equal(dis[0], ref[4])
    # growing a workspace never frees the old one (a captured graph keeps its address)
    own = G.WorkspaceOwner()
    with G.workspace_owner(own):
        w1 = G.workspace(1024, dev, "t")
        p1 = w1.data_ptr()
        w2 = G.workspace(1 << 20, dev, "t")
    assert w2.data_ptr() != p1 and any(t.data_ptr() == p1 for t in own.retired)


def test_pipeline_batch_of_pairs_matches_single_pairs():
    """B pairs in one step (M-batched launches) give, per pair, the batch-1 result: every stage is per image or per
    RoI (frozen BN), so only tile shapes differ -- proposals identical, records to rounding"""
    H, W = 160, 320
    sd = make_state_dict(3)
    dev = torch.device("cuda")
    pipe = PL.StereoPipeline(sd, dev, throughput=True, scale=1.0)
    calib4 = G.calib_vec(DEMO_P2 / np.array([[3.], [3.], [1.]]), DEMO_P3 / np.array([[3.], [3.], [1.]]))
    ims, rois = [], []
    for i in range(3):
        left, right = synth_pair(H, W, seed=30 + i, shift=5 + i)
        b, k, p = gen_rois(6, seed=9 + i)
        b = b / 3.0
        k[:, [0, 3, 4]] /= 3.0
        ims.append((torch.from_numpy(left)[None].cuda(), torch.from_numpy(right)[None].cuda()))
        rois.append(tuple(torch.from_numpy(x).cuda() for x in (b, k, p)))
    singles = [pipe.step(l, r, calib4, ro) for (l, r), ro in zip(ims, rois)]
    torch.cuda.synchronize()
    recB, keepB, nB, stB, disB = pipe.step(torch.cat([l for l, _ in ims]), torch.cat([r for _, r in ims]), calib4, rois)
    torch.cuda.synchronize()
    for i, (rec, keep, nk, st, dis) in enumerate(singles):
        assert rel_err(recB[i].cpu(), rec[0].cpu()) < 1e-5
        assert int(nB[i]) == int(nk[0]) and torch.equal(keepB[i, :int(nk[0])], keep[0, :int(nk[0])])
        assert torch.equal(stB[i], st[0]) and torch.equal(disB[i], dis[0])


# ------------------------------------------------------------------ multi-GPU (needs >= 2 devices)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, mode, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        gat = P.RecordGather(world, rank, dev, dist, n_slots=2, mode=mode)
        ok = True
        for step in range(6):
            for slot in range(2):
                g = torch.Generator().manual_seed(1000 * step + 10 * slot + rank)
                rec = torch.rand(P.REC_ROIS, P.REC_COLS, generator=g).to(dev)
                out = gat(slot, rec)
                torch.cuda.synchronize()
                for r in range(world):
                    g2 = torch.Generator().manual_seed(1000 * step + 10 * slot + r)
                    ok &= bool(torch.equal(out[r].cpu(), torch.rand(P.REC_ROIS, P.REC_COLS, generator=g2)))
        gat.check()
        if mode == "peer":      # pipelined exchange (lag 1): a call returns the slot's PREVIOUS step, drain() the last one
            gl = P.RecordGather(world, rank, dev, dist, n_slots=2, mode="peer", lag=1)
            mk = lambda step, slot, r: torch.full((P.REC_ROIS, P.REC_COLS), float(1000 * step + 10 * slot + r))
            for step in range(7):
                for slot in range(2):
                    out = gl(slot, mk(step, slot, rank).to(dev)).clone()
                    torch.cuda.synchronize()
                    if step > 0:
                        for r in range(world):
                            ok &= bool(torch.equal(out[r].cpu(), mk(step - 1, slot, r)))
            for slot in range(2):
                out = gl.drain(slot).clone()
                torch.cuda.synchronize()
                for r in range(world):
                    ok &= bool(torch.equal(out[r].cpu(), mk(6, slot, r)))
            gl.check()
        # shard equivalence: N ranks x 1 pair == 1 rank computing the same pairs (bit for bit)
        sd = make_state_dict(3)
        pipe = PL.StereoPipeline(sd, dev, throughput=True, scale=1.0)
        calib4 = G.calib_vec(DEMO_P2 / np.array([[3.], [3.], [1.]]), DEMO_P3 / np.array([[3.], [3.], [1.]]))

        def one(seed):
            left, right = synth_pair(128, 256, seed=seed, shift=5)
            b, k, p = gen_rois(4, seed=seed)
            b = b / 3.0
            k[:, [0, 3, 4]] /= 3.0
            ro = tuple(torch.from_numpy(x).to(dev) for x in (b, k, p))
            return pipe.step(torch.from_numpy(left)[None].to(dev), torch.from_numpy(right)[None].to(dev), calib4, ro)[0][0]
        mine = one(40 + rank)
        allrec = gat(0, mine).clone()
        torch.cuda.synchronize()
        if rank == 0:
            for r in range(world):
                ok &= bool(torch.equal(allrec[r], one(40 + r)))
        q.put((rank, gat.mode, ok, gat.describe()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_record_gather_and_shard_equivalence_on_hardware(mode):
    """world = 2..N GPUs of the box: the gathered records are every rank's records (both exchange paths), and the
    N-GPU result equals the 1-GPU result on the same pairs"""
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, world, port, mode, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    print(res[0][3])
    for rank, m, ok, _d in res:
        assert ok, "rank %d: gathered records differ" % rank
        assert m == mode, "requested %s, ran %s" % (mode, res[0][3])


# ------------------------------------------------------------------ 8f-1: box solvers on the device
def test_box_solver_device_chain_vs_oracle(golden_dir):
    """infer_boundary -> border fix-up -> solve_x_y_z_theta -> (dense_align) -> solve_x_y_theta on the device against
    the oracle's restatement of the reference: indices / boundaries exact, solver end points stationary for the
    reference's own gradient (tests/test_box_solver.py explains why end points are not compared digit by digit)"""
    from oracle import box_solver as BS
    g = np.load(os.path.join(golden_dir, "box_solver.npz"))
    shape = tuple(int(v) for v in g["im_shape"])
    n = len(g["alpha"])
    R, nc = 80, 2
    rs = np.random.RandomState(11)
    scores = np.zeros((R, nc), np.float32)
    pbl, pbr = np.zeros((R, 8), np.float32), np.zeros((R, 8), np.float32)
    do, pk = np.zeros((R, 10), np.float32), np.zeros((R, 5), np.float32)
    rows = rs.permutation(R)[:n]                      # detections scattered over the RoI rows
    sc = np.sort(rs.rand(n).astype(np.float32) * 0.9 + 0.06)[::-1]
    for j, r in enumerate(rows):
        scores[r, 1] = sc[j]
        pbl[r, 4:8], pbr[r, 4:8] = g["box_left"][j], g["box_right"][j]
        do[r, 5:8] = g["dim"][j]
        do[r, 8], do[r, 9] = np.sin(g["alpha"][j]), np.cos(g["alpha"][j])
        pk[r] = g["kpts"][j]
    keep = np.zeros(R, np.int32)
    keep[:n] = rows                                   # kept order = score order
    c = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    keep_d, num_d = c(keep), c(np.array([n], np.int32))
    inf = G.infer_boundary(c(pbl), keep_d, num_d, shape[1], col_offset=4)
    inf_ref = BS.infer_boundary(shape, pbl[rows, 4:8])
    np.testing.assert_array_equal(inf[:n].cpu().numpy(), inf_ref)
    boxes_all, kpts_all, poses_all, src, nd = G.box_solve(c(scores), c(pbl), c(pbr), c(do), c(pk), keep_d, num_d, shape[:2],
                                                         g["p2"], g["p3"], inferred=inf)
    torch.cuda.synchronize()
    ns = int(nd[0])
    src = src[:ns].cpu().numpy()
    poses = poses_all[:ns].cpu().numpy().astype(np.float64)
    kall = kpts_all[:ns].cpu().numpy()
    # every solved detection, in kept order; unsolved ones are exactly the reference's status-0 rules
    pos = {int(r): j for j, r in enumerate(rows)}
    last = -1
    for q in range(ns):
        j = pos[int(src[q])]
        assert j > last
        last = j
        kp = pk[rows[j]].copy()
        if kp[4] - kp[3] < np.float32(0.5) * (inf_ref[j, 1] - inf_ref[j, 0]):
            kp[3:5] = inf_ref[j]
        np.testing.assert_array_equal(kall[q], kp)
        alpha = float(np.arctan2(np.float64(do[rows[j], 8]), np.float64(do[rows[j], 9])))
        pb = BS.Problem(shape, g["p2"], g["p3"], alpha, do[rows[j], 5:8].astype(np.float64), pbl[rows[j], 4:8].astype(np.float64),
                        pbr[rows[j], 4:8].astype(np.float64), kp.astype(np.float64))
        s = poses[q, [0, 1, 2, 6]]
        assert np.abs(pb.gradient(s)).max() < 1e-5, (q, pb.gradient(s))       # fp32-rounded end point of an fp64 solve
        assert poses[q, 2] <= 100
    assert ns >= n // 2
    # rectification with synthetic aligned disparities
    succ = torch.ones(R, device="cuda")
    dis = torch.zeros(R, device="cuda")
    dis[:ns] = c(np.array([g["disparity"][pos[int(r)]] for r in src], np.float32))
    final = G.box_rectify(boxes_all, kpts_all, poses_all, succ, dis, nd, shape[:2], g["p2"], g["p3"]).cpu().numpy()
    for q in range(ns):
        j = pos[int(src[q])]
        assert final[q, 0] == 1
        f = g["p2"][0, 0]
        z = f * ((g["p2"][0, 3] - g["p3"][0, 3]) / f) / float(np.float32(g["disparity"][j]))
        assert abs(final[q, 8] - z) < 1e-9 * z
        pr = BS.Problem(shape, g["p2"], g["p3"], float(poses_all[q, 7]), poses[q, 3:6], boxes_all[q, :4].cpu().numpy().astype(np.float64),
                        None, kall[q].astype(np.float64), z_fixed=z)
        assert np.abs(pr.gradient(final[q, [6, 7, 12]])).max() < 1e-8
    assert (final[ns:, 0] == 0).all()
    lines = G.kitti_result_lines(torch.from_numpy(final), float(g["t_cam2_cam0_x"]))
    assert len(lines) == ns and lines[0].startswith("Car -1 -1 ")


def test_pipeline_with_device_solver_runs_sync_free():
    """the whole test_net.py per-image path incl. the solver stage, captured into a CUDA graph (proves there is no
    host synchronisation anywhere) and replayed: identical results"""
    H, W = 192, 416
    sd = make_state_dict(3)
    dev = torch.device("cuda")
    pipe = PL.StereoPipeline(sd, dev, scale=1.0)
    left, right = synth_pair(H, W, seed=21, shift=6)
    iml, imr = torch.from_numpy(left)[None].cuda(), torch.from_numpy(right)[None].cuda()
    p2, p3 = DEMO_P2 / np.array([[3.], [3.], [1.]]), DEMO_P3 / np.array([[3.], [3.], [1.]])
    own = G.WorkspaceOwner()
    with G.workspace_owner(own):
        eager = pipe.step_with_solver(iml, imr, p2, p3, (H, W))
        torch.cuda.synchronize()
        runner = E.GraphRunner(lambda a, b: pipe.step_with_solver(a, b, p2, p3, (H, W)), [iml, imr])
    out = runner()
    torch.cuda.synchronize()
    for k in ("record", "n_solved", "poses_all", "status", "best_dis", "final"):
        assert torch.equal(out[k], eager[k]), k
    assert int(out["nkeep"][0]) >= int(out["n_solved"][0]) >= 0
