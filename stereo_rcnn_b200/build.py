"""Build libstereo_b200.so (all hand-written sm_100a kernels + the C ABI) in-tree with nvcc.

    python -m stereo_rcnn_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libstereo_b200.so")
SOURCES = ["misc.cu", "nms.cu", "proposal.cu", "roi_align.cu", "dense_align.cu", "conv_simt.cu", "conv_tc.cu", "peer.cu", "box_solver.cu",
           "train_targets.cu", "train_loss.cu", "train_backward.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
         "-Xcompiler", "-Wall", "-Xcompiler", "-Wno-unused-function"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "stereo_b200.h"))
    objdir = os.path.join(HERE, "_obj")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            cmd = ["nvcc", "-c", src, "-o", obj] + ARCH + FLAGS + (["-Xptxas", "-v"] if verbose else [])
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("---- %s ----\n%s\n" % (s, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(SO, objs):
        subprocess.check_call(["nvcc", "-shared", "-o", SO] + objs + ARCH + ["-lcudart", "-lcuda"])
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
