"""Box-head training step on the B200: proposal targets -> box_head_forward -> rcnn_loss -> box_head_backward replayed
as one CUDA graph at the benchmarked 600x1987 pair (B = 2 / R = 1024 and B = 1 / R = 512), with per-stage CUDA-event
times of eager runs; then its building blocks: the four GEMMs of the fc6 / fc7 backward (resnet.py:256-263 RCNN_top:
a 7x7 conv over the pooled 7x7 tile = a 25088 -> 2048 linear, then a 1x1 2048 -> 2048) through sb_gemm_tc with the
operands in their stored layouts, against torch.matmul (cuBLAS, fp16 operands, fp32 output where torch offers it) on
the same shapes and layouts in the same call, and the deterministic pyramid RoIAlign backward (both halves of the
pooled [R,7,7,512] gradient) at the benchmarked 600x1987 pair.

    python tools/box_head_backward_bench.py [--reps 20] [--out DIR]

Prints one JSON line (and writes it to DIR/box_head_backward_bench.json when --out is given).  Timing: CUDA events
around `reps` back-to-back launches after a warm-up of every shape; the operands of dW6 / d_pooled (51 + 103 MB) and
the fixed-point workspace of the RoIAlign backward (306 MB at B = 2) exceed the 126 MB L2.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from stereo_rcnn_b200 import ops  # noqa: E402

IM_H, IM_W = 600, 1987
K6, CO = 512 * 7 * 7, 2048            # fc6: 25088 -> 2048 (packed (ph, pw, c) order), fc7: 2048 -> 2048


def gpu_info():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                                     "-i", "0"], text=True).strip().split(",")
        info["power_limit"], info["max_sm_clock"] = q[0].strip(), q[1].strip()
    except (OSError, subprocess.CalledProcessError) as e:
        info["power_limit"] = info["max_sm_clock"] = "unavailable (%s)" % type(e).__name__
    return info


def time_us(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) * 1e3 / reps


def gemm_cases(R, dev):
    g = torch.Generator(device=dev).manual_seed(R)
    h = lambda *s: (torch.randn(*s, generator=g, device=dev) * 0.1).half()
    g6, g7 = h(R, CO), h(R, CO)                    # fp16 gradients w.r.t. the fc6 / fc7 outputs (after mask / scale)
    pooled, fc6 = h(R, K6), h(R, CO)               # saved forward activations
    w6, w7 = h(CO, K6), h(CO, CO)                  # packed weights [Cout][K]
    return [
        # name, A, B, a_mn, b_mn, M, N, K   (C[m][n] = sum_k A(m,k) B(n,k))
        ("dW6 = g6^T pooled", g6, pooled, True, True, CO, K6, R),
        ("d_pooled = g6 W6", g6, w6, False, True, R, K6, CO),
        ("dW7 = g7^T fc6", g7, fc6, True, True, CO, CO, R),
        ("d_fc6 = g7 W7", g7, w7, False, True, R, CO, CO),
    ]


def bench_gemms(R, reps, dev):
    rows = []
    for name, a, b, a_mn, b_mn, M, N, K in gemm_cases(R, dev):
        out = torch.empty(M, N, device=dev)
        ours = lambda: ops.gemm(a, b, out, a_mn, b_mn)
        ta = a.t() if a_mn else a                  # [M, K] view
        tb = b if b_mn else b.t()                  # [K, N] view
        ref_out = torch.empty(M, N, device=dev)
        # cuBLAS on the same operands in the same layouts (the transposes are views, no copies)
        fn, mode = (lambda: torch.mm(ta, tb, out_dtype=torch.float32, out=ref_out)), "fp16 in, fp32 out"
        try:
            fn()
        except (TypeError, RuntimeError):
            fn, mode = (lambda: torch.mm(ta, tb)), "fp16 in, fp16 out"
        ours()
        torch.cuda.synchronize()
        ref = torch.mm(ta.double(), tb.double()) if M * N * K <= 1 << 36 else None
        err = float((torch.linalg.norm(out.double() - ref) / torch.linalg.norm(ref)).item()) if ref is not None else None
        t_ours, t_cublas = time_us(ours, reps), time_us(fn, reps)
        flop = 2.0 * M * N * K
        rows.append(dict(stage=name, M=M, N=N, K=K, a_mn_major=a_mn, b_mn_major=b_mn, us=round(t_ours, 1),
                         tflops=round(flop / t_ours * 1e-6, 1), cublas_us=round(t_cublas, 1),
                         cublas_tflops=round(flop / t_cublas * 1e-6, 1), cublas_mode=mode,
                         ours_over_cublas_time=round(t_ours / t_cublas, 3), rel_l2_vs_fp64=err))
        del out, ref_out, ref
    return rows


def pyramid_shapes(B, C=256):
    """NHWC shapes of P2..P5 for the IM_H x IM_W input: stem conv 7x7/2 pad 3, max-pool 3x3/2 (ceil), then the
    stride-2 stages"""
    def pool(v):
        o = (v - 3 + 1) // 2 + 1
        return o - 1 if (o - 1) * 2 >= v else o
    h, w = pool((IM_H - 1) // 2 + 1), pool((IM_W - 1) // 2 + 1)
    out = []
    for _ in range(4):
        out.append((B, h, w, C))
        h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    return out


def bench_roi_backward(B, R, reps, dev):
    rs = np.random.RandomState(B)
    sizes = np.exp(rs.uniform(np.log(16), np.log(600), R))
    asp = rs.uniform(0.5, 2.0, R)
    w, hh = sizes * np.sqrt(asp), sizes / np.sqrt(asp)
    cx, cy = rs.uniform(0, IM_W, R), rs.uniform(0, IM_H, R)
    rois = np.stack([rs.randint(0, B, R), np.clip(cx - w / 2, 0, IM_W - 1), np.clip(cy - hh / 2, 0, IM_H - 1),
                     np.clip(cx + w / 2, 0, IM_W - 1), np.clip(cy + hh / 2, 0, IM_H - 1)], 1).astype(np.float32)
    rois_t = torch.from_numpy(rois).to(dev)
    top = torch.randn(R, 7, 7, 512, device=dev) * 1e-3           # pooled gradient [R,7,7,512]: L half | R half
    shapes = pyramid_shapes(B)
    gl = [torch.empty(*s, device=dev) for s in shapes]
    gr = [torch.empty(*s, device=dev) for s in shapes]

    def run():
        ops.roi_align_pyramid_nhwc_backward(top, IM_H, rois_t, shapes, out_coff=0, grad_feats=gl)
        ops.roi_align_pyramid_nhwc_backward(top, IM_H, rois_t, shapes, out_coff=256, grad_feats=gr)
    t = time_us(run, reps)
    feat = sum(int(np.prod(s)) for s in shapes)
    # compulsory traffic of the two calls: the pooled gradient read once, the fp32 feature gradients written once.
    # The fixed-point accumulators add 2 x 8 B per feature element (zeroing, conversion) plus the atomics' traffic.
    nbytes = R * 49 * 512 * 4 + 2 * feat * 4
    ws_bytes = 2 * feat * (8 + 8)
    return dict(stage="pyramid RoIAlign backward (L + R)", B=B, R=R, us=round(t, 1), compulsory_bytes=nbytes,
                gbps=round(nbytes / t * 1e-3, 1), fixed_point_workspace_bytes=ws_bytes)


def bench_step(eng, B, reps, dev):
    """the box-head training step at the benchmarked pair: proposal targets of 2000 proposals per image ->
    box_head_forward -> rcnn_loss -> box_head_backward, replayed as one CUDA graph; per-stage times from CUDA events
    in eager runs"""
    from stereo_rcnn_b200 import engine, synth, train
    R, nc, gd = B * 512, eng.n_classes, 28
    g = torch.Generator(device=dev).manual_seed(B)
    shapes = pyramid_shapes(2 * B)
    feats = {k: torch.randn(*s, generator=g, device=dev) * 0.5 for k, s in zip(("p2", "p3", "p4", "p5"), shapes)}
    gl, gr, _gm, dim, kp, _nb = synth.synth_train_gt(B, 30, IM_H, IM_W, B)
    rl, rr = synth.synth_train_rois(gl, 2000, IM_H, IM_W, B + 100)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    inputs = [cu(rl), cu(rr), cu(gl), cu(gr), cu(dim), cu(kp), train.random_words((B, 2030), dev, g),
              train.random_words((B, 512), dev, g)]
    drop = (train.random_words((R, 2048), dev, g), train.random_words((R, 2048), dev, g))
    zeros = [torch.zeros(R, 4 * gd, device=dev), torch.zeros(R, gd, device=dev), torch.zeros(R, gd, device=dev)]

    def step(*inp, events=None):
        mark = (lambda n: events.append((n, torch.cuda.Event(enable_timing=True))) or events[-1][1].record()) \
            if events is not None else (lambda n: None)
        mark("start")
        tgt = train.proposal_targets(*inp)
        mark("proposal_targets")
        ctx = train.box_head_forward(eng, feats, B, tgt["rois_left"].view(R, 5), tgt["rois_right"].view(R, 5),
                                     float(IM_H), drop)
        mark("box_head_forward")
        _losses, gr_ = train.rcnn_loss(ctx["cls_score"], ctx["bbox_pred"], ctx["dim_orien_pred"], *zeros, tgt)
        mark("rcnn_loss")
        bev = [] if events is not None else None
        out = train.box_head_backward(eng, ctx, gr_[0], gr_[1], gr_[2], stage_events=bev)
        if events is not None:
            events.extend(bev[1:])
        return out

    runner = engine.GraphRunner(step, inputs)
    t_graph = time_us(runner, reps)
    stages = {}
    for _ in range(3):
        ev = []
        step(*inputs, events=ev)
        torch.cuda.synchronize()
        for (n0, e0), (n1, e1) in zip(ev[:-1], ev[1:]):
            stages.setdefault(n1, []).append(e0.elapsed_time(e1) * 1e3)
    flops = {"dW7": 2.0 * CO * CO * R, "d_fc6": 2.0 * R * CO * CO, "dW6": 2.0 * CO * K6 * R, "d_pooled": 2.0 * R * K6 * CO}
    rows = []
    for n, ts in stages.items():
        t = float(np.median(ts))
        row = dict(stage=n, us=round(t, 1))
        if n in flops:
            row.update(flop=flops[n], tflops=round(flops[n] / t * 1e-6, 1))
        rows.append(row)
    return dict(B=B, R=R, graph_replay_us=round(t_graph, 1), stages_eager=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("box_head_backward_bench needs a GPU")
    dev = torch.device("cuda", 0)
    res = dict(bench="box_head_backward", gpu=gpu_info(), configs=[])
    from stereo_rcnn_b200 import engine, synth
    eng = engine.StereoRCNNEngine(synth.make_state_dict(3), dev)          # fp16 engine, synthetic weights
    for B, R in ((2, 1024), (1, 512)):
        res["configs"].append(dict(B=B, R=R, step=bench_step(eng, B, args.reps, dev),
                                   gemm=bench_gemms(R, args.reps, dev),
                                   roi_align_backward=bench_roi_backward(B, R, args.reps, dev)))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "box_head_backward_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
