"""GPU: the box-head training step (train.box_head_forward / box_head_backward) against torch fp64 autograd of the
same head with the same dropout masks on the tensors the device forward consumed, its device-side fp16 scaling at
extreme gradient magnitudes, and its capture in one CUDA graph together with the target layer and the loss."""
import numpy as np
import pytest
import torch

from box_head_oracle import box_head_train_fp64, keep_mask, pyramid_roi_feat_backward
from stereo_rcnn_b200 import engine, synth
from stereo_rcnn_b200 import train as G
from stereo_rcnn_b200.parallel import GradientBuckets

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def pyramid_shapes(H, W):
    """P2..P5 of an H x W input (stem 7x7/2, max-pool 3x3/2 ceil, stride-2 stages)"""
    def pool(v):
        o = (v - 3 + 1) // 2 + 1
        return o - 1 if (o - 1) * 2 >= v else o
    h, w = pool((H - 1) // 2 + 1), pool((W - 1) // 2 + 1)
    out = []
    for _ in range(4):
        out.append((h, w))
        h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    return out


@pytest.fixture(scope="module")
def setup():
    sd = synth.make_state_dict(3)
    eng = engine.StereoRCNNEngine(sd, DEV)              # fp16 engine (default precision)
    return sd, eng


def make_case(H, W, B, seed):
    """features of both images (random, [2B,H_l,W_l,256]), sampled RoIs from the device proposal target layer"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    feats = {k: torch.randn(2 * B, h, w, 256, generator=g, device=DEV) * 0.5
             for k, (h, w) in zip(("p2", "p3", "p4", "p5"), pyramid_shapes(H, W))}
    gl, gr, _gm, dim, kp, _nb = synth.synth_train_gt(B, 30, H, W, seed)
    rl, rr = synth.synth_train_rois(gl, 2000, H, W, seed + 100)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    words = lambda shape, s: cu(np.random.RandomState(s).randint(0, 2 ** 32, shape, dtype=np.uint64)
                                .astype(np.uint32).view(np.int32))
    inputs = [cu(rl), cu(rr), cu(gl), cu(gr), cu(dim), cu(kp), words((B, 2030), seed + 1), words((B, 512), seed + 2)]
    tgt = G.proposal_targets(*inputs)
    R = B * 512
    drop = (words((R, 2048), seed + 3), words((R, 2048), seed + 4))
    return feats, inputs, tgt, drop


def incoming(R, nc, seed, scale):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(R, n, generator=g, device=DEV) * (scale / R) for n in (nc, 6 * nc, 5 * nc)]


def check_against_fp64(sd, eng, feats, tgt, drop, B, H, d_in):
    R = B * 512
    rl, rr = tgt["rois_left"].view(R, 5), tgt["rois_right"].view(R, 5)
    ctx = G.box_head_forward(eng, feats, B, rl, rr, float(H), drop)
    grads, fg = G.box_head_backward(eng, ctx, *d_in)
    torch.cuda.synchronize()
    # the oracle takes the device's ReLU decisions: the backward must be the adjoint of the forward that was computed
    ref, d_pooled = box_head_train_fp64(ctx["pooled"].cpu(), sd, keep_mask(drop[0].cpu()), keep_mask(drop[1].cpu()),
                                        *[t.cpu() for t in d_in], relu6=(ctx["fc6"] > 0).cpu(),
                                        relu7=(ctx["fc7"] > 0).cpu())
    errs = {}
    for n, r in ref.items():
        got = grads[n].cpu()
        assert torch.isfinite(got).all(), n
        errs[n] = rel_l2(got, r)
    # parameter gradients: both GEMM operands carry fp16 rounding (11-bit significands) -> 2e-3.  The bias gradients of
    # the tail and of fc7 are fixed-order fp32 sums of gradients that never pass an fp16 operand -> 1e-5.  The fc6 bias
    # sums d_fc6, which comes out of the fp16 product g7 W7: it carries that product's rounding -> 2e-3.
    for n, e in errs.items():
        tight = n.endswith(".bias") and n != "RCNN_top.0.bias"
        assert e <= (1e-5 if tight else 2e-3), (n, e, errs)
    nchw = [(B, 256, f.shape[1], f.shape[2]) for f in (feats[k][:B] for k in ("p2", "p3", "p4", "p5"))]
    for side, rois, sl in (("left", rl, slice(0, 256)), ("right", rr, slice(256, 512))):
        want = pyramid_roi_feat_backward(d_pooled[..., sl].permute(0, 3, 1, 2).numpy(), rois.cpu().numpy(), nchw, H)
        for lvl, (gg, w) in enumerate(zip(fg[side], want)):
            got = gg.permute(0, 3, 1, 2).cpu().numpy()
            assert np.isfinite(got).all()
            if np.abs(w).sum() > 0:
                e = rel_l2(got, w)
                assert e <= 2e-3, (side, lvl, e)
    return errs


@pytest.mark.parametrize("scale", [1.0, 2.0 ** -24, 2.0 ** 8])
def test_box_head_gradients_vs_fp64_autograd_160x256(setup, scale):
    """fast size; the scales show the device-chosen fp16 scaling: neither flushing nor overflowing"""
    sd, eng = setup
    H, W, B = 160, 256, 1
    feats, _inputs, tgt, drop = make_case(H, W, B, 0)
    check_against_fp64(sd, eng, feats, tgt, drop, B, H, incoming(B * 512, eng.n_classes, 1, scale))


def test_box_head_gradients_vs_fp64_autograd_600x1987_r1024(setup):
    sd, eng = setup
    H, W, B = 600, 1987, 2
    feats, _inputs, tgt, drop = make_case(H, W, B, 5)
    assert tgt["status"].cpu().tolist() == [0, 0]
    check_against_fp64(sd, eng, feats, tgt, drop, B, H, incoming(B * 512, eng.n_classes, 2, 1.0))


def test_training_step_in_one_graph_bit_identical_buckets_and_clip(setup):
    """proposal_targets -> box_head_forward -> rcnn_loss -> box_head_backward captured once; two replays give the same
    bits; gradients written into GradientBuckets views equal the returned ones; clip() equals train.clip_gradient"""
    sd, eng = setup
    H, W, B = 160, 256, 2
    feats, inputs, _tgt, drop = make_case(H, W, B, 9)
    R, nc = B * 512, eng.n_classes
    gd = 28
    zeros = [torch.zeros(R, 4 * gd, device=DEV), torch.zeros(R, gd, device=DEV), torch.zeros(R, gd, device=DEV)]
    buckets = GradientBuckets(G.box_head_param_shapes(nc), DEV)
    views = dict(zip(G.BOX_HEAD_PARAMS, buckets.grads))

    def step(*inp):
        tgt = G.proposal_targets(*inp)
        ctx = G.box_head_forward(eng, feats, B, tgt["rois_left"].view(R, 5), tgt["rois_right"].view(R, 5), float(H),
                                 drop)
        losses, g = G.rcnn_loss(ctx["cls_score"], ctx["bbox_pred"], ctx["dim_orien_pred"], *zeros, tgt)
        grads, fg = G.box_head_backward(eng, ctx, g[0], g[1], g[2])
        G.box_head_backward(eng, ctx, g[0], g[1], g[2], grads=views)
        return losses, grads, fg

    runner = engine.GraphRunner(step, inputs)
    losses, grads, fg = runner()
    torch.cuda.synchronize()
    first = {n: t.clone() for n, t in grads.items()}
    first_f = [t.clone() for side in ("left", "right") for t in fg[side]]
    first_v = {n: t.clone() for n, t in views.items()}
    runner()
    torch.cuda.synchronize()
    assert torch.isfinite(losses).all()
    for n in G.BOX_HEAD_PARAMS:
        assert torch.equal(first[n], grads[n]), n
        assert torch.equal(first_v[n], grads[n]), n                     # bucket views == returned gradients
        assert float(grads[n].abs().max()) > 0, n
    for a, b in zip(first_f, [t for side in ("left", "right") for t in fg[side]]):
        assert torch.equal(a, b)
    clones = [t.clone() for t in buckets.grads]
    want = G.clip_gradient(clones, 1e-4)
    got = buckets.clip(1e-4)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    for a, b in zip(buckets.grads, clones):
        assert torch.equal(a, b)


def test_tf32_engine_raises(setup):
    sd, _eng = setup
    eng32 = engine.StereoRCNNEngine(sd, DEV, precision="tf32")
    with pytest.raises(NotImplementedError):
        G.box_head_forward(eng32, {}, 1, None, None, 160.0, (None, None))
    with pytest.raises(NotImplementedError):
        G.box_head_backward(eng32, {}, None, None, None)
