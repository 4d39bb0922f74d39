"""In-tree build of the CUDA library (``csrc/libste_ukf.so``) with nvcc for sm_100a.

The shared object is git-ignored but travels with the working tree to the GPU box; nothing is
JIT-compiled at import time.  ``python -m ship_track_estimators_b200.build`` rebuilds it.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.environ.get("STE_UKF_LIB") or os.path.join(CSRC, "libste_ukf.so")  # env override: developer A/B builds
SOURCES = ["ste_ukf.cu", "ste_text.cu"]
HEADERS = ["ste_fastmath.cuh", "ste_math.cuh", "ste_filter.cuh", "ste_tracks.cuh", "ste_generic.cuh", "ste_ingest.cuh", "ste_text.cuh",
           os.path.join("..", "..", "include", "ste_ukf.h")]

NVCC_FLAGS = [
    "-O3",
    "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    # No implicit a*b+c -> fma contraction: every FMA in the kernels is written as fma().  Contraction
    # choices depend on the surrounding code, so with them the same per-track function inlined into
    # different kernels (forward / fused / single-step predict) rounds differently; without them all
    # entry points agree bit for bit.  Costs < 1 % (59 of 2 762 FP64 instructions were implicit).
    "-fmad=false",
    "-Xcompiler", "-fPIC",
    "-shared",
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; cannot build libste_ukf.so")
    return exe


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > built for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile ``libste_ukf.so`` if missing or older than its sources; returns its path."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc(), *NVCC_FLAGS, *os.environ.get("STE_EXTRA_NVCC_FLAGS", "").split()]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    tmp = LIB_PATH + ".tmp"
    cmd += ["-o", tmp, *[os.path.join(CSRC, s) for s in SOURCES]]
    proc = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    os.replace(tmp, LIB_PATH)
    if verbose:
        print(proc.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
