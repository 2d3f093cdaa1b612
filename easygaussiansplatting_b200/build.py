"""Builds libgsplat_b200.so (the C-ABI of include/gsplat_b200.h) for sm_100a with nvcc.

In-tree on purpose: the .so travels with the repository snapshot to the GPU box, and the
driver records which in-tree .so files the test/bench processes loaded.

    python -m easygaussiansplatting_b200.build [--force] [--verbose]
"""
import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# A/B builds (benchmarks only): GSB_VARIANT=name + GSB_EXTRA_NVCC_FLAGS="-DX=1 ..." produce
# libgsplat_b200_<name>.so next to the default library; _lib.py loads it when GSB_LIB points at it.
VARIANT = os.environ.get("GSB_VARIANT", "")
OBJ = os.path.join(HERE, "_obj" + ("_" + VARIANT if VARIANT else ""))
LIB = os.path.join(HERE, "libgsplat_b200%s.so" % ("_" + VARIANT if VARIANT else ""))
SOURCES = ["api.cu", "pergaussian.cu", "fused.cu", "binning.cu", "raster_bwd.cu",
           "raster_fwd3.cu", "raster_bwd4.cu", "loss.cu", "smallbmm.cu", "density.cu", "comm.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr",
         "-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"]
EXTRA = os.environ.get("GSB_EXTRA_NVCC_FLAGS", "").split()


def _deps_mtime():
    m = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def _compile(src, verbose):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    cmd = [NVCC] + FLAGS[:-2] + EXTRA + FLAGS[-2:] + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(obj + ".log", "w") as f:
        f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr[-4000:]))
    if verbose:
        print(r.stderr)
    return obj


def build(force=False, verbose=False):
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _deps_mtime():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-lcudart", "-ccbin", FLAGS[-1]]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stderr[-4000:])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
