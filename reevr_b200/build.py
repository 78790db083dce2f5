"""Builds reevr_b200/libb200conv.so (the C-ABI shared library) with nvcc for sm_100a, in-tree."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libb200conv.so")
SOURCES = ["engine.cu", "irshape.cu"]
DEPS = ["engine.cu", "irshape.cu", "kernels.cuh", "kernels_stream.cuh", "kernels_fft512.cuh", "kernels_rt.cuh", "kernels_chain.cuh", "kernels_tc.cuh", "kernels_tfft.cuh",
        os.path.join("..", "..", "include", "b200conv.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared",
    "--use_fast_math" if os.environ.get("B200CONV_FAST_MATH") else "-fmad=true",
]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found")
    return p


def stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    cmd = [nvcc_path(), *NVCC_FLAGS, "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + out.stdout + out.stderr)
    if verbose:
        print(out.stdout + out.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
