"""Builds libfetalb200.so (hand-written CUDA for sm_100a + the C ABI) in-tree with nvcc.

Usage:  python fetal-mri-segmentation_b200/build.py [--force]
The .so lands next to this file's `fetal_net/` package (git-ignored, but it travels to the GPU box).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "fetal_net", "libfetalb200.so")
SOURCES = ["api.cu", "bandwidth.cu", "conv_simt.cu", "conv_tc.cu", "conv_march.cu", "conv_wgrad_march.cu", "comm.cu", "sampler.cu", "conv_first_tc.cu", "postprocess.cu", "tta.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr"]


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(HERE, "..", "include", "fetal_b200.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return OUT
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("---- nvcc %s ----\n%s\n" % (src, out))
        failed = failed or p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [NVCC, "-shared", "-o", OUT] + objs + ["-lcudart", "-ldl"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
