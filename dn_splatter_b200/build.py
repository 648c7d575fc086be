"""Builds libdnr_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension machinery).

    python -m dn_splatter_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libdnr_b200.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "--extended-lambda"]
# name -> extra flags.  project / image_ops: no FMA contraction (bit-exact integer outputs vs the oracle).
SOURCES = {
    "project.cu": ["-fmad=false"],
    "image_ops.cu": ["-fmad=false"],
    "binning.cu": [],
    "raster.cu": [],
    "misc.cu": [],
    "ssim.cu": [],
    "adam.cu": ["-fmad=false"],
    "knn.cu": ["-fmad=false"],
    "density.cu": ["-fmad=false"],
    "tsdf.cu": ["-fmad=false"],
}


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libdnr_b200.so cannot be built (no CPU fallback exists)")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = nvcc_path()
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "loss_common.cuh"), os.path.join(CSRC, "mc_tables.cuh"), os.path.join(HERE, "..", "include", "dnr.h"), os.path.abspath(__file__)]
    objs = []
    for src, extra in SOURCES.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc, *ARCH, *COMMON, *extra, "-c", s, "-o", o]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), flush=True)
            subprocess.run(cmd, check=True)
    if force or _stale(LIB, objs):
        cmd = [nvcc, *ARCH, "-shared", "-o", LIB, *objs]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
