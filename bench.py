#!/usr/bin/env python
"""bench.py -- stereo pairs/sec of the Stereo R-CNN hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our sm_100a path
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU port of the reference path

Workload (config[1] of BASELINE.json): batch-1 inference, one synthetic KITTI-shape stereo pair
per GPU per step (1242x375 resized by 1.6 -> 2 x [1,3,600,1987] fp32), full pipeline:
trunk+FPN (L and R), stereo RPN, proposal layer, RoIAlign, box + keypoint heads, test-time decode,
per-class NMS, and dense_align on D=32 synthetic poses (the scipy solver that produces poses in the
reference is a CPU stage outside the kernels, SURVEY 8d config 2).  N>1: one process per GPU, one
pair per rank per step (weak scaling), one NCCL all-gather of the fixed-size detection records.

One JSON line on stdout (rank 0).  `value` = pairs/s with inputs resident in HBM; `e2e` = the same
through the public forward with pinned-host inputs (H2D inside the timed region) and a D2H read of
the detection record.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H_NET, W_NET, SCALE = 600, 1987, 1.6
D_ALIGN = 32
N_ROIS = 300
REC_COLS = 2 + 8 + 8 + 10 + 5        # scores, boxes L/R, dim_orien, kpts  (per RoI)

# algorithmic MACs per *pair* at test (SURVEY 8 header / BASELINE.md 3), for the roofline line
TC_GMACS_PER_PAIR = 2 * (15.88 + 22.64 + 123.58 + 17.89 + 66.99 + 117.37) + 2.45 + 16.7 + 223.9
# (the 2 x 2.81 GMAC stem GEMM is executed on the tensor cores too but not counted as algorithmic work here)
CONV_DRAM_BYTES_PER_STEP = 5.655e9     # profiles/r02c_conv_dram.md (fp16-operand default, 213 conv launches of one forward)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                f = [x.strip() for x in out.stdout.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons}


# ----------------------------------------------------------------------------------------------
def make_inputs(rank, j=0):
    """pair j of rank `rank` (seeded; j > 0 only with --microbatch)"""
    from stereo_rcnn_b200.synth import DEMO_P2, DEMO_P3, gen_rois, synth_pair
    seed = 3 + rank + 1000 * j
    left, right = synth_pair(H_NET, W_NET, seed=seed, shift=48)
    b, k, p = gen_rois(D_ALIGN, seed=seed)
    return left, right, (b, k, p), (DEMO_P2, DEMO_P3)


SCALE32 = float(np.float32(SCALE))
H_CAM, W_CAM = 375, 1242


def make_frames(rank, j=0):
    """a synthetic uint8 KITTI-shape camera pair [375,1242,3] BGR (what demo.py / test_net.py read from disk): the e2e
    path ships these to the GPU and runs prep_im_for_blob (blob.py:44-64) there -> 2 x [3,600,1987] fp32"""
    from stereo_rcnn_b200.synth import synth_pair
    left, right = synth_pair(H_CAM, W_CAM, seed=3 + rank + 1000 * j, shift=30)
    f = lambda a: np.ascontiguousarray(np.clip(np.rint(a.transpose(1, 2, 0) + 110.0), 0, 255).astype(np.uint8))
    return f(left), f(right)


def run_ours(args):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        # N ranks synthesise and pack the same weights on the host at start-up: do not let each of them spawn one
        # CPU thread per core (has no effect on the timed, GPU-side region)
        torch.set_num_threads(max(1, min(8, (os.cpu_count() or 8) // world)))
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from stereo_rcnn_b200 import ops, parallel, pipeline
    from stereo_rcnn_b200.synth import make_state_dict
    MB = max(1, args.microbatch)          # pairs per step of one in-flight slot (batched through every launch)
    pairs = [make_inputs(rank, j) for j in range(MB)]
    P2, P3 = pairs[0][3]
    calib4 = ops.calib_vec(P2, P3)
    host_l = torch.from_numpy(np.stack([q[0] for q in pairs])).pin_memory()      # [MB,3,H,W]
    host_r = torch.from_numpy(np.stack([q[1] for q in pairs])).pin_memory()
    iml, imr = host_l.to(dev), host_r.to(dev)
    rois3d = [tuple(torch.from_numpy(x).to(dev) for x in q[2]) for q in pairs]
    frames = [make_frames(rank, j) for j in range(MB)]
    host_l8 = torch.from_numpy(np.stack([f[0] for f in frames])).pin_memory()     # [MB,375,1242,3] uint8
    host_r8 = torch.from_numpy(np.stack([f[1] for f in frames])).pin_memory()
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)      # 256 MB > 126 MB L2
    n_inflight = max(1, args.inflight)
    use_graph = os.environ.get("SB_GRAPH", "1") != "0"
    if not use_graph:
        n_inflight = 1
    sd = make_state_dict(3)
    # the public end-to-end API of the package (stereo_rcnn_b200.pipeline): StereoPipeline.step is the call a user
    # makes, GraphSlot is one in-flight step (own stream, fixed inputs, private workspaces, CUDA graph)
    pipe_lat = pipeline.StereoPipeline(sd, dev, scale=SCALE)             # one pair at a time: lowest latency
    pipe = pipeline.StereoPipeline(sd, dev, throughput=True, scale=SCALE) if (n_inflight > 1 or MB > 1) else pipe_lat
    copy_stream = torch.cuda.Stream(device=dev)
    # peer mode (opt-in) runs the exchange pipelined (lag 1): a step puts its record and collects the previous step's, so
    # no rank waits for a slower peer's current step; the last step of every slot is drained inside the timed region
    gather = parallel.RecordGather(world, rank, dev, dist, n_slots=n_inflight + 1, mode=args.gather,
                                   rec_shape=(MB * N_ROIS, REC_COLS), lag=args.gather_lag)

    class Slot(pipeline.GraphSlot):
        """a GraphSlot plus the bench's host side: the pinned-host staging of the next H2D and the host landing
        buffers of the slot's results.  `mb` pairs per step (batched through every launch)."""

        def __init__(self, pipe, own_stream, index, gather, mb):
            self.mb, self.gather, self.index = mb, gather, index
            self.h_l, self.h_r = host_l[:mb], host_r[:mb]
            super().__init__(pipe, iml[:mb], imr[:mb], calib4, rois3d[:mb], own_stream=own_stream, use_graph=use_graph)
            self.host_rec = torch.empty(world, mb * N_ROIS, REC_COLS).pin_memory()
            self.host_dis = torch.empty(mb, D_ALIGN).pin_memory()
            self.staging = [(torch.empty_like(self.iml), torch.empty_like(self.imr)) for _ in range(1 if own_stream else 2)]
            self.ready = [torch.cuda.Event() for _ in self.staging]
            self.freed = [torch.cuda.Event() for _ in self.staging]
            for ev in self.freed:
                ev.record()
            self.k, self.primed = 0, False
            # e2e: uint8 camera frames -> staging (H2D) -> prep_im_for_blob on the device, straight into the graph's inputs
            self.h_l8, self.h_r8 = host_l8[:mb], host_r8[:mb]
            self.staging8 = [(torch.empty_like(self.h_l8, device=dev), torch.empty_like(self.h_r8, device=dev))
                             for _ in self.staging]
            self.ready8 = [torch.cuda.Event() for _ in self.staging]
            self.freed8 = [torch.cuda.Event() for _ in self.staging]
            for ev in self.freed8:
                ev.record()
            self.k8, self.primed8 = 0, False

        def prefetch8(self, j):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(self.freed8[j])
                self.staging8[j][0].copy_(self.h_l8, non_blocking=True)
                self.staging8[j][1].copy_(self.h_r8, non_blocking=True)
                self.ready8[j].record(copy_stream)

        def build_e2e_graph(self):
            """the whole end-to-end step of this slot as ONE CUDA graph: H2D of the uint8 frames from pinned host memory,
            prep_im_for_blob on the device, the pipeline step, D2H of the disparities (and of the record when there is
            no exchange).  A user writes the next frames into the pinned buffers and replays."""
            from stereo_rcnn_b200.engine import GraphRunner
            l8, r8 = self.staging8[0]

            def fn(l8_, r8_):
                l8_.copy_(self.h_l8, non_blocking=True)
                r8_.copy_(self.h_r8, non_blocking=True)
                for b_ in range(self.mb):
                    ops.prep_image(l8_[b_], SCALE, out=self.iml[b_])
                    ops.prep_image(r8_[b_], SCALE, out=self.imr[b_])
                out = self.pipe.step(self.iml, self.imr, calib4, self.rois3d)
                for b_ in range(self.mb):
                    self.host_dis[b_].copy_(out[4][b_], non_blocking=True)
                if world == 1:
                    self.host_rec.copy_(out[0].view(1, -1, REC_COLS), non_blocking=True)
                return out
            with ops.workspace_owner(self.ws):
                self.e2e_runner = GraphRunner(fn, [l8, r8])

        def step_e2e(self):
            if use_graph and getattr(self, "e2e_runner", None) is not None:
                rec, keep, nkeep, st, dis = self.e2e_runner()
                if world > 1:
                    g = self.gather(self.index, rec.view(-1, REC_COLS))
                    self.host_rec.copy_(g, non_blocking=True)
                return rec, dis
            return self.step_e2e_eager()

        def step_e2e_eager(self):
            """the call a user of demo.py / test_net.py makes: uint8 camera frames on the host in, records out.  H2D
            of the next frames (2 x 1.4 MB per pair, pinned host -> staging, copy stream) overlaps compute;
            prep_im_for_blob runs on the device and writes the graph's fixed inputs; every step moves its own frames in
            and its records out inside the timed region"""
            nst = len(self.staging8)
            j = self.k8 % nst
            if not self.primed8:
                self.prefetch8(j)
                self.primed8 = True
            cur = torch.cuda.current_stream()
            cur.wait_event(self.ready8[j])
            for b_ in range(self.mb):
                ops.prep_image(self.staging8[j][0][b_], SCALE, out=self.iml[b_])
                ops.prep_image(self.staging8[j][1][b_], SCALE, out=self.imr[b_])
            self.freed8[j].record(cur)
            self.prefetch8((self.k8 + 1) % nst)
            self.k8 += 1
            rec, keep, nkeep, st, dis = self.run()
            g = self.gather(self.index, rec.view(-1, REC_COLS))
            self.host_rec.copy_(g, non_blocking=True)
            for b_ in range(self.mb):
                self.host_dis[b_].copy_(dis[b_], non_blocking=True)
            return g, dis

        def prefetch(self, j):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(self.freed[j])
                self.staging[j][0].copy_(self.h_l, non_blocking=True)
                self.staging[j][1].copy_(self.h_r, non_blocking=True)
                self.ready[j].record(copy_stream)

        def step_resident(self):
            rec, keep, nkeep, st, dis = self.run()
            return self.gather(self.index, rec.view(-1, REC_COLS)), dis

        def step_e2e_blob(self):
            """round 1's end-to-end definition: PRE-RESIZED fp32 blobs on the host (28.6 MB per pair) -> H2D -> forward.
            H2D of this slot's next pair(s) (pinned host -> staging, copy stream) overlaps compute; every step
            still moves its own 28.6 MB per pair in and its records out inside the timed region"""
            if use_graph:
                nst = len(self.staging)
                j = self.k % nst
                if not self.primed:
                    self.prefetch(j)
                    self.primed = True
                cur = torch.cuda.current_stream()
                cur.wait_event(self.ready[j])
                self.load(*self.staging[j])              # device-to-device into the graph's fixed inputs
                self.freed[j].record(cur)
                self.prefetch((self.k + 1) % nst)         # the next pair's H2D runs under this compute
                self.k += 1
            else:
                self.load(self.h_l, self.h_r)
            rec, keep, nkeep, st, dis = self.run()
            g = self.gather(self.index, rec.view(-1, REC_COLS))
            self.host_rec.copy_(g, non_blocking=True)
            for j in range(self.mb):
                self.host_dis[j].copy_(dis[j], non_blocking=True)
            return g, dis

    # the latency slot always runs ONE pair at a time (batch 1, the reference's test configuration)
    gather_lat = gather if MB == 1 else parallel.RecordGather(world, rank, dev, dist, n_slots=1, mode=args.gather,
                                                              lag=args.gather_lag)
    pipelined = n_inflight > 1 or MB > 1
    lat_slot = Slot(pipe_lat, False, n_inflight if (pipelined and MB == 1) else 0, gather_lat, 1)
    slots = [Slot(pipe, True, i, gather, MB) for i in range(n_inflight)] if pipelined else [lat_slot]
    host_rec, host_dis = slots[0].host_rec, slots[0].host_dis

    def timed(fn, steps, warmup, drain=None):
        """one pair in flight: every step bracketed by its own events, L2 flushed (untimed) between steps"""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for s, e in ev:
            ops.l2_flush(flush)          # untimed, between iterations
            s.record()
            fn()
            if drain is not None:
                drain()                  # pipelined exchange: the step is complete when its records have been collected
            e.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        return parallel.max_over_ranks(sum(s.elapsed_time(e) for s, e in ev), dev, world, dist)

    def timed_pipelined(method, steps, warmup):
        """n_inflight independent pairs in flight, each on its own stream (a pair's proposal / NMS stages leave most
        SMs idle; the other pair's convolutions fill them).  One event pair around all K steps; no L2 flush is
        needed or possible between overlapping steps: every step streams ~5.9 GB through the 126 MB L2."""
        main = torch.cuda.current_stream()

        def issue(k):
            sl = slots[k % n_inflight]
            with torch.cuda.stream(sl.stream):
                getattr(sl, method)()
        for k in range(warmup):
            issue(k)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ops.l2_flush(flush)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(main)
        for sl in slots:
            sl.stream.wait_event(s)
        for k in range(steps):
            issue(k)
        for sl in slots:                     # pipelined exchange: collect the last step's records of every slot
            with torch.cuda.stream(sl.stream):
                g_ = sl.gather.drain(sl.index)
                if g_ is not None and method != "step_resident":
                    sl.host_rec.copy_(g_, non_blocking=True)
        for sl in slots:
            main.wait_stream(sl.stream)
        main.wait_stream(copy_stream)
        e.record(main)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        return parallel.max_over_ranks(s.elapsed_time(e), dev, world, dist)

    sampler = ClockSampler(local)
    sampler.start()
    l0 = ops.launch_count()
    pipe.step(iml, imr, calib4, rois3d)                 # one eager step (MB pairs) only to count our kernel launches
    launches = ops.launch_count() - l0
    W = max(args.warmup, 3)
    single = None
    dumped = None
    if not pipelined:
        dr = lambda: slots[0].gather.drain(slots[0].index)
        total_ms = timed(slots[0].step_resident, args.steps, W, dr)
        if args.dump_outputs:
            dumped = host_outputs(slots[0].outputs)
        e2e_blob_ms = timed(slots[0].step_e2e_blob, args.steps, 1, dr)
        if use_graph:
            slots[0].build_e2e_graph()
        e2e_ms = timed(slots[0].step_e2e, args.steps, 1, dr)
    else:
        one_ms = timed(lat_slot.step_resident, args.steps, W, lambda: lat_slot.gather.drain(lat_slot.index))    # one pair in flight, reported beside the headline
        single = {"inflight": 1, "ms_per_step": round(one_ms / args.steps, 3),
                  "value": round(world * args.steps / (one_ms / 1e3), 3), "unit": "pairs/s",
                  "schedule": "latency: left/right chains, RPN levels and box head forked onto a second stream",
                  "l2": "256 MB flush between timed iterations"}
        total_ms = timed_pipelined("step_resident", args.steps, W + n_inflight)
        if args.dump_outputs:
            dumped = host_outputs(slots[(args.steps - 1) % n_inflight].outputs)     # the slot of the last step
        e2e_blob_ms = timed_pipelined("step_e2e_blob", args.steps, W + n_inflight)
        if use_graph:
            for sl in slots:
                sl.build_e2e_graph()
        e2e_ms = timed_pipelined("step_e2e", args.steps, W + n_inflight)
        # leave the synthetic fp32 pair in the slots' inputs again (the e2e legs overwrote them with the camera frames)
        for sl in slots:
            with torch.cuda.stream(sl.stream):
                sl.load(iml[:sl.mb], imr[:sl.mb])
                sl.run()
    # the exchange step alone (records already packed): device time of one gather per step, max over ranks
    gather_ms = None
    if world > 1:
        rec0 = slots[0].outputs[0].view(-1, REC_COLS)
        gather_ms = timed(lambda: gather(slots[0].index, rec0), args.steps, W, lambda: gather.drain(slots[0].index)) / args.steps
        gather.check()
    # every in-flight slot must have produced the result of the one-pair-at-a-time run on the same input: the
    # schedules differ only in tile widths / stream forks, proposals are index-exact and records agree to rounding
    torch.cuda.synchronize()
    checks = []
    for sl in slots:
        for j in range(sl.mb):
            if j == 0:
                ref_rec = lat_slot.outputs[0][0]
            else:       # pair j alone through the batch-1 pipeline
                ref_rec = pipe_lat.step(iml[j:j + 1], imr[j:j + 1], calib4, rois3d[j:j + 1])[0][0]
                torch.cuda.synchronize()
            checks.append(float((sl.outputs[0][j] - ref_rec).abs().max() / ref_rec.abs().max()))
    sampler.stop_flag = True
    ms_per_step = total_ms / args.steps
    value = world * args.steps * MB / (total_ms / 1e3)
    e2e_value = world * args.steps * MB / (e2e_ms / 1e3)
    e2e_blob_value = world * args.steps * MB / (e2e_blob_ms / 1e3)

    # ---- roofline of the dominant kernel (tcgen05 implicit-GEMM conv), timed live with CUDA events ----
    roof = None
    cpu_base = None
    parity = None
    if rank == 0:
        pk = peaks()
        conv_ms, conv_classes = conv_time_per_step(pipe, iml[:1], imr[:1])
        tflops = 2 * TC_GMACS_PER_PAIR * 1e9 / (conv_ms / 1e3) / 1e12
        half = pipe.eng.half
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel (tcgen05 kind::%s implicit GEMM, all conv/FC launches of one step)" % ("f16" if half else "tf32"),
                "achieved": round(tflops, 2), "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": round(tflops / pk["bf16_tflops_sustained"], 4),
                # dram__bytes_read+write summed over the conv launches of one step, ncu capture of this same
                # command (profiles/); algorithmic FLOPs per step = 2 * 0.978 TMAC
                "traffic": CONV_DRAM_BYTES_PER_STEP if half else None,
                "traffic_unit": "bytes per step (all conv launches)",
                "peak_source": pk["src"] + " cuBLAS bf16 sustained" + ("" if half else " (kind::tf32 issues at half that rate)"),
                # conv_ms_serialized: all conv launches back to back on ONE stream (no other pair to fill idle SMs);
                # in the pipelined step the same FLOPs retire within ms_per_step, hence the in-step lower bound
                "conv_ms_serialized": round(conv_ms, 3),
                # each class issued alone back to back; compare tflops with `peak` and algorithmic_tb_per_s with hbm_peak
                "by_class": conv_classes, "hbm_peak_tb_per_s": round(pk["hbm_gbs"] / 1e3, 3),
                "achieved_in_step_lower_bound": round(2 * TC_GMACS_PER_PAIR * MB * 1e9 / (ms_per_step / 1e3) / 1e12, 2)}
        if world == 1 and not args.no_cpu_baseline:
            cpu_base, parity = cpu_baseline_sample(pipe_lat)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    out = {
        "metric": "stereo pairs/sec (1242x375)", "value": round(value, 3), "unit": "pairs/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": pipe.eng.precision + (" operands (tcgen05 kind::f16), fp32 accumulate, fp32 residual stream/outputs" if pipe.eng.half else " (fp32 storage, kind::tf32, fp32 accumulate)"),
        "data": "synthetic",
        "config": {"workload": "configs[1]: batch-1 inference per GPU, synthetic KITTI-shape pair 2x[1,3,600,1987], "
                               "full pipeline incl. dense_align (D=%d synthetic poses)" % D_ALIGN,
                   "weights": "seeded variance-preserving random init (stereo_rcnn_b200.synth.make_state_dict(3))",
                   "l2": ("256 MB flush between timed iterations" if not pipelined else
                          "inputs larger than L2: every step reads ~0.4 GB of weights and streams ~5.9 GB of activations "
                          "through the 126 MB L2; steps of the %d in-flight pairs overlap, so no flush between them "
                          "(single_stream: flushed)" % n_inflight),
                   "inflight": n_inflight, "microbatch": MB, "pairs_per_step": MB, "schedule": ("throughput: %d independent steps in flight (%d pair(s) per step, batched "
                   "through every launch), one stream + CUDA graph + private workspaces each, no intra-pair forks" % (n_inflight, MB))
                   if pipelined else "latency (one pair in flight)",
                   "api": "stereo_rcnn_b200.pipeline.StereoPipeline.step via pipeline.GraphSlot",
                   "cuda_graph": use_graph, "parallelism": "dp%d (1 pair/rank)" % world,
                   "gather": gather.describe()},
        # e2e: the repo's public call with HOST inputs as demo.py / test_net.py have them -- uint8 camera frames; the
        # input pipeline (prep_im_for_blob) runs on the device.  e2e_fp32_blob: round 1's definition (pre-resized fp32
        # blobs on the host, 10x the H2D bytes), kept for continuity.
        "e2e": {"value": round(e2e_value, 3), "unit": "pairs/s",
                "h2d_bytes_per_step": int(slots[0].h_l8.numel() * 2),
                "d2h_bytes_per_step": int(host_rec.numel() * 4 + host_dis.numel() * 4),
                "input": "uint8 %dx%dx3 frames (pinned host) -> H2D -> sb_prep_image on the device -> %dx%d fp32; the whole "
                         "step incl. both copies is one CUDA graph per slot" % (H_CAM, W_CAM, H_NET, W_NET)},
        "e2e_fp32_blob": {"value": round(e2e_blob_value, 3), "unit": "pairs/s",
                          "h2d_bytes_per_step": int(slots[0].h_l.numel() * 4 * 2),
                          "d2h_bytes_per_step": int(host_rec.numel() * 4 + host_dis.numel() * 4)},
        "gpu_launches": int(launches) * args.steps,
        "inflight_vs_single_max_rel_diff": [round(c, 9) for c in checks],
        "clocks": sampler.summary(), "roofline": roof,
    }
    if gather_ms is not None:
        out["gather_ms_per_step"] = round(gather_ms, 4)
    if single is not None:
        out["single_stream"] = single
    if cpu_base is not None:
        out["cpu_baseline"] = cpu_base
    if parity is not None:
        out["parity"] = parity
    print(json.dumps(out))


def host_outputs(outputs):
    """what StereoPipeline.step returned -- (record, keep, nkeep, status, best_dis) of MB pairs -- as host float32 /
    float64 arrays.  Entries of `keep` past `nkeep` are left unwritten by the NMS kernel and are set to -1 here."""
    rec, keep, nkeep, st, dis = outputs
    torch.cuda.synchronize()
    nkeep = nkeep.cpu().numpy()
    keep = keep.cpu().numpy().astype(np.float64)
    for b, n in enumerate(nkeep):
        keep[b, n:] = -1
    return {"record": rec.float().cpu().numpy(), "keep": keep, "nkeep": nkeep.astype(np.float64),
            "status": torch.stack(st).float().cpu().numpy(), "best_dis": torch.stack(dis).float().cpu().numpy()}


def conv_time_per_step(pipe, iml, imr):
    """CUDA-event duration of all tcgen05 conv launches of one forward, issued back to back on the launching stream
    (nothing else in between).  The descriptors (and their tensors, kept alive) are recorded during one forward and
    then re-launched in a tight ctypes loop, so that the host is faster than the kernels and the event pair brackets
    GPU time only."""
    import ctypes
    from stereo_rcnn_b200 import lib
    eng = pipe.eng
    eng.record = []
    eng.forward(iml, imr, pipe.im_info(1, iml.shape[2], iml.shape[3]))
    rec, eng.record = eng.record, None
    L = lib.load()
    st = lib.stream_ptr()
    tc = [(d, keep) for d, impl, keep in rec if impl == "tc"]

    def seq_ms(descs):
        """one event pair around a back-to-back sequence (PDL overlap as in the real step), best of 3"""
        best = None
        for _ in range(3):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for d in descs:
                L.sb_conv2d_tc(ctypes.byref(d), st)
            e.record()
            torch.cuda.synchronize()
            t = s.elapsed_time(e)
            best = t if best is None else min(best, t)
        return best

    total = seq_ms([d for d, _k in tc])
    # the same launches by what bounds them: big-M 3x3 convs (tensor pipe), big-M 1x1 convs with the residual
    # epilogue (HBM: fp16 in + fp32 residual in + fp32 out + fp16 twin out), everything else (small M: layers 3-4,
    # FC heads, 1x1 convs without residual -- L2 fill / latency)
    classes = {"tensor: 3x3 convs, M >= 30000 px": [], "hbm: 1x1 + residual, M >= 30000 px": [], "other (small M / plain 1x1)": []}
    for d, _k in tc:
        M = d.N * d.Ho * d.Wo
        key = ("tensor: 3x3 convs, M >= 30000 px" if d.kh == 3 and M >= 30000 else
               "hbm: 1x1 + residual, M >= 30000 px" if d.residual and M >= 30000 else "other (small M / plain 1x1)")
        classes[key].append(d)
    by_class = []
    for key, ds in classes.items():
        if not ds:
            continue
        ms = seq_ms(ds)
        fl = sum(2.0 * d.N * d.Ho * d.Wo * d.Cout * d.kh * d.kw * d.Cin for d in ds)
        by = sum(d.N * d.Ho * d.Wo * (d.Cin * (2 if d.in_dtype == 1 else 4) + d.Cout *
                                      ((4 if d.out else 0) + (2 if d.out16 else 0) + (4 if d.residual else 0))) for d in ds)
        by_class.append({"class": key, "launches": len(ds), "ms": round(ms, 3), "tflops": round(fl / ms / 1e9, 1),
                         "algorithmic_tb_per_s": round(by / ms / 1e9, 2)})
    return total, by_class

# ----------------------------------------------------------------------------------------------
def _cpu_threads():
    n = os.cpu_count() or 1
    import torch.nn.functional as F
    x, w = torch.randn(2, 256, 38, 125), torch.randn(256, 256, 3, 3)     # a layer-3 sized conv (11 GFLOP)
    best, best_t = 1, None
    for nt in sorted({1, max(1, n // 2), n}):
        torch.set_num_threads(nt)
        F.conv2d(x, w, padding=1)
        t = time.time()
        for _ in range(2):
            F.conv2d(x, w, padding=1)
        t = time.time() - t
        if best_t is None or t < best_t:
            best, best_t = nt, t
    torch.set_num_threads(best)
    os.environ["OMP_NUM_THREADS"] = str(best)
    return best


def cpu_port_step(sd, left, right, crop_w, rois3d, calib, want_outputs=False):
    """one pass of the hot path on the CPU port of the reference (oracle): forward + decode + NMS + dense_align
    on a width-`crop_w` crop of the pair; returns seconds (and the oracle's tensors if asked)"""
    from oracle import model as OM
    from oracle import ops as O
    iml = torch.from_numpy(left[:, :, :crop_w].copy())[None]
    imr = torch.from_numpy(right[:, :, :crop_w].copy())[None]
    info = torch.tensor([[float(H_NET), float(crop_w), SCALE]])
    t = time.time()
    o = OM.forward(sd, iml, imr, info)
    dec = O.test_decode(o["rois_left"][0].numpy(), o["rois_right"][0].numpy(), o["cls_prob"].numpy(),
                        o["bbox_pred"].numpy(), o["dim_orien_pred"].numpy(), o["kpts_prob"].numpy(),
                        o["left_border_prob"].numpy(), o["right_border_prob"].numpy(), info[0].numpy())
    O.per_class_nms(dec[0], dec[1], 1)
    b, k, p = rois3d
    O.dense_align(calib, SCALE32, left, right, b, k, p)
    sec = time.time() - t
    return (sec, o, (iml, imr, info)) if want_outputs else sec


def parity_report(eng, o, iml, imr, info):
    """the GPU forward against the oracle's tensors of the SAME pair at the benchmarked size and dtype: per tensor
    (relative L2 error, max-norm relative error).  Heads are evaluated on the oracle's RoIs (identical inputs); the
    end-to-end proposal overlap says how many of the oracle's 300 proposals the GPU's own RPN scores reproduce."""
    from stereo_rcnn_b200 import ops

    def err(a, b_):
        a, b_ = np.asarray(a, np.float64), np.asarray(b_, np.float64)
        return [float("%.3g" % (np.linalg.norm(a - b_) / max(np.linalg.norm(b_), 1e-30))),
                float("%.3g" % (np.abs(a - b_).max() / max(np.abs(b_).max(), 1e-30)))]
    dev = eng.device
    r = eng.forward(iml.to(dev), imr.to(dev), info.to(dev), keep_features=True)
    torch.cuda.synchronize()
    rep = {}
    for k in ("c2", "c3", "c4", "c5", "p2", "p3", "p4", "p5", "p6"):
        got = r["feats"][k].float().permute(0, 3, 1, 2).cpu().numpy()
        el, er = err(got[0:1], o["left"][k].numpy()), err(got[1:2], o["right"][k].numpy())
        rep[k] = [max(el[0], er[0]), max(el[1], er[1])]
    for k in ("rpn_cls_prob", "rpn_bbox_pred"):
        rep[k] = err(r[k].cpu().numpy(), o[k].numpy())
    a = {tuple(np.round(x, 1)) for x in r["rois_left"][0].cpu().numpy()}
    b_ = {tuple(np.round(x, 1)) for x in o["rois_left"][0].numpy()}
    rl, rr = ops.proposal_layer(o["rpn_cls_prob"].to(dev), o["rpn_bbox_pred"].to(dev), info.to(dev), "TEST", o["rpn_shapes"])
    exact = bool(np.array_equal(rl.cpu().numpy(), o["rois_left"].numpy()) and
                 np.array_equal(rr.cpu().numpy(), o["rois_right"].numpy()))
    h = eng.heads(r["feats_raw"], 1, rl.view(-1, 5), rr.view(-1, 5), float(iml.shape[2]))
    torch.cuda.synchronize()
    for k in ("pooled_box", "pooled_kpts"):
        rep[k] = err(h[k].float().permute(0, 3, 1, 2).cpu().numpy(), o[k].numpy())
    for k in ("fc7", "cls_prob", "bbox_pred", "dim_orien_pred", "kpts_prob", "left_border_prob", "right_border_prob"):
        rep[k] = err(h[k].cpu().numpy().reshape(o[k].shape), o[k].numpy())
    return {"vs": "CPU oracle (fp32) on the same pair, %dx%d, dtype %s" % (iml.shape[2], iml.shape[3], eng.precision),
            "format": "[relative L2, max-norm relative] per tensor",
            "tensors": rep, "worst_l2": max(v[0] for v in rep.values()), "worst_max_norm": max(v[1] for v in rep.values()),
            "proposals_bit_exact_on_identical_inputs": exact,
            "end_to_end_proposal_overlap": round(len(a & b_) / float(len(b_)), 4)}


def pick_crop(threads):
    """bound one CPU step to ~<= 8 s: probe the conv rate, then pick the crop width"""
    import torch.nn.functional as F
    x, w = torch.randn(1, 256, 38, 125), torch.randn(256, 256, 3, 3)
    F.conv2d(x, w, padding=1)
    t = time.time()
    for _ in range(3):
        F.conv2d(x, w, padding=1)
    rate = 3 * 2 * 38 * 125 * 256 * 256 * 9 / (time.time() - t)        # FLOP/s
    fixed = 2 * (16.7 + 223.9) * 1e9 / rate                            # RoI heads: 300 RoIs whatever the crop
    scal = 2 * (TC_GMACS_PER_PAIR - 16.7 - 223.9 + 5.6) * 1e9 / rate   # trunk + FPN + RPN scale with the pixels
    for frac, wcrop in ((1.0, W_NET), (0.5, 993), (0.25, 497), (0.125, 248)):
        if fixed + scal * frac <= 10.0 or wcrop == 248:
            return wcrop, frac


def cpu_baseline_sample(pipe=None, passes=3):
    """reported CPU baseline (kind "port": the oracle, all host threads): 1 warm-up + `passes` timed passes, mean;
    the oracle's tensors of the last pass double as the parity reference for the GPU forward (same pair, same size)"""
    from oracle import ops as O
    from stereo_rcnn_b200.synth import make_state_dict
    threads = _cpu_threads()
    left, right, rois3d, (P2, P3) = make_inputs(0)
    wcrop, frac = pick_crop(threads)
    sd = make_state_dict(3)
    calib = O.calib_vec(P2, P3)
    cpu_port_step(sd, left, right, wcrop, rois3d, calib)
    secs = []
    for _ in range(passes):
        sec, o, ins = cpu_port_step(sd, left, right, wcrop, rois3d, calib, want_outputs=True)
        secs.append(sec)
    sec = sum(secs) / len(secs)
    base = {"value": round((wcrop / W_NET) / sec, 5), "unit": "pairs/s", "cores": threads, "kind": "port",
            "sample": "mean of %d passes (after 1 warm-up; min %.2f s, max %.2f s) of the oracle (CPU port of the reference "
                      "forward + decode + NMS + dense_align D=%d) on a 600x%d crop of the pair (%.3f of the pixels), scaled "
                      "to full pairs" % (passes, min(secs), max(secs), D_ALIGN, wcrop, wcrop / W_NET)}
    parity = parity_report(pipe.eng, o, *ins) if pipe is not None else None
    return base, parity


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from oracle import ops as O
    from stereo_rcnn_b200.synth import make_state_dict
    threads = _cpu_threads()
    left, right, rois3d, (P2, P3) = make_inputs(0)
    wcrop, frac = pick_crop(threads)
    sd = make_state_dict(3)
    calib = O.calib_vec(P2, P3)
    for _ in range(min(args.warmup, 1)):
        cpu_port_step(sd, left, right, wcrop, rois3d, calib)
    tot = 0.0
    steps = args.steps
    for _ in range(steps):
        tot += cpu_port_step(sd, left, right, wcrop, rois3d, calib)
    value = steps * (wcrop / W_NET) / tot
    sample = ("oracle (CPU port of the reference path: torch-CPU fp32 forward + C decode/NMS/RoIAlign/dense_align), "
              "600x%d crop per step (%.3f of a pair), %d timed steps" % (wcrop, wcrop / W_NET, steps))
    out = {"impl": "reference", "metric": "stereo pairs/sec (1242x375)", "value": round(value, 5), "unit": "pairs/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)), "steps": steps, "warmup": min(args.warmup, 1),
           "ms_per_step": round(1e3 * tot / steps, 1), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
           "config": {"workload": "configs[1] on host cores (reference CPU path; the reference's CUDA ops cannot be "
                                  "built on this stack: torch.utils.ffi/THC are gone)", "parallelism": "cpu"},
           "cpu_baseline": {"value": round(value, 5), "unit": "pairs/s", "cores": threads, "kind": "port",
                            "sample": sample},
           "e2e": {"value": round(value, 5), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", default=None, choices=[None, "peer", "nccl"],
                    help="record exchange at N>1: ncclAllGather on per-slot communicators (default, measured faster) or "
                         "own kernels over NVLink peer memory")
    ap.add_argument("--microbatch", type=int, default=int(os.environ.get("SB_MICROBATCH", "1")),
                    help="pairs per step of one in-flight slot, batched through every launch (M-batching)")
    ap.add_argument("--gather-lag", type=int, default=int(os.environ.get("SB_GATHER_LAG", "1")), choices=[0, 1],
                    help="peer exchange: 1 = pipelined (a step collects the previous step's records), 0 = same step")
    ap.add_argument("--inflight", type=int, default=int(os.environ.get("SB_INFLIGHT", "3")),
                    help="independent pairs in flight per GPU (each batch-1, own stream + CUDA graph)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline path returned in its last step (record, "
                         "keep, nkeep, status, best_dis of rank 0) as DIR/<name>.npy; the inputs are seeded, so two "
                         "builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
