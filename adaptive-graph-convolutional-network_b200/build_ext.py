"""Builds libagcn_sm100.so (the C-ABI CUDA library, sm_100a only) in-tree with nvcc.

    python adaptive-graph-convolutional-network_b200/build_ext.py [--force]

nvcc cross-compiles without a GPU; the built .so sits next to this file (git-ignored, but it
travels to the GPU box with the snapshot).
"""
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = sorted(glob.glob(os.path.join(HERE, "csrc", "*.cu")))
HDR = sorted(glob.glob(os.path.join(HERE, "csrc", "*.cuh"))) + [os.path.join(ROOT, "include", "agcn_sgcll.h")]
OUT = os.path.join(HERE, "libagcn_sm100.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"),
]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(f) > t for f in SRC + HDR + [os.path.abspath(__file__)])


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SRC:  # one nvcc per translation unit, in parallel
        obj = os.path.join(HERE, "build", os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc] + [f for f in NVCC_FLAGS if f != "-shared"] + ["-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, out))
    cmd = [nvcc, "-shared", "-o", OUT] + objs
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
