"""Build libmisob200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

The shared object is git-ignored but travels to the GPU box with the gpurun snapshot.
`-fmad=false` is deliberate: the reference's CPU kernels round every product and sum
separately, and the parity-critical code relies on that; kernels that want FMAs call fmaf().
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libmisob200.so")
STAMP = os.path.join(HERE, ".libmisob200.stamp")
SOURCES = ["api.cu", "nms.cu", "roi_align.cu", "roi_align_tma.cu", "boxops.cu", "rpn.cu", "detpost.cu", "crop.cu", "mosaic.cu", "seam.cu", "train.cu", "paste.cu", "morph.cu", "png.cu", "jpeg.cu", "transform.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "--shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest() -> str:
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + [os.path.join(INCLUDE, "misob200.h")]
    for f in files:
        path = f if os.path.isabs(f) else os.path.join(CSRC, f)
        with open(path, "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    h.update(" ".join(NVCC_FLAGS + SOURCES).encode())
    return h.hexdigest()


def is_current() -> bool:
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as fh:
        return fh.read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and is_current():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-o", LIB, *srcs]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libmisob200.so")
    with open(STAMP, "w") as fh:
        fh.write(_digest())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
