"""Builds libthetarrt.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

The .so is git-ignored but travels to the GPU box with the repo snapshot.
nvcc cross-compiles without a GPU, so this runs in the build container too.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libthetarrt.so")
SOURCES = ["thetarrt.cu"]
HEADERS = ["trrt_device.cuh", "trrt_los.cuh", "trrt_bike.cuh", "trrt_lane.cuh", "trrt_rrt.cuh", "trrt_mission.cuh", "trrt_rng.cuh", "trrt_libm.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "--std=c++17",
    "-fmad=false",                       # parity: no implicit multiply-add contraction on the device
    "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off",
    "-shared",
]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found")
    return p


def needs_build() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(HERE, "..", "include", "thetarrt.h"))
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, extra_flags=()) -> str:
    if not force and not needs_build():
        return SO
    cmd = [nvcc_path(), *NVCC_FLAGS, *extra_flags, "-o", SO] + [os.path.join(CSRC, f) for f in SOURCES]
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    build(force=True, verbose=True, extra_flags=tuple(sys.argv[1:]))
