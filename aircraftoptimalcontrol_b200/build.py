"""Compile libacoc.so in-tree for sm_100a:  python -m aircraftoptimalcontrol_b200.build [--force]

nvcc cross-compiles without a GPU.  -fmad=false because every fused multiply-add in the library is written
explicitly (csrc/acoc_math.cuh explains why); -lineinfo so that ncu's source page maps to the .cuh files.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "acoc_api.cu")
DEPS = [SRC, os.path.join(HERE, "csrc", "acoc_kernels.cuh"), os.path.join(HERE, "csrc", "acoc_math.cuh"), os.path.join(HERE, "csrc", "acoc_tma.cuh"),
        os.path.join(HERE, "..", "include", "acoc.h")]
OUT = os.path.join(HERE, "libacoc.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS):
        return OUT
    cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT, SRC]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
