"""ctypes front-end of oracle/legacy_normals.c, the sequential restatement of the device's seeded normal streams.

TEST INFRASTRUCTURE ONLY -- imported by tests/; the product package theta_rrt_b200 never imports this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "legacy_normals.c")
_SO = os.path.join(_HERE, "liblegacy_normals.so")
_DEPS = (_SRC, os.path.join(_HERE, "..", "theta_rrt_b200", "csrc", "trrt_libm.h"))
# the flags of oracle/Makefile: no contraction, so the host build of trrt_libm.h computes what the device build does
CFLAGS = ["-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-Wall", "-Wextra"]
_lib = None

c_dp = C.POINTER(C.c_double)


def build(force: bool = False) -> str:
    if force or not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(d) for d in _DEPS):
        subprocess.check_call(["gcc", *CFLAGS, "-shared", "-o", _SO, _SRC, "-lm"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.orc_init_genrand.argtypes = [C.c_uint32, C.c_void_p]
        _lib.orc_legacy_normals.argtypes = [C.c_uint32, C.c_int64, C.c_void_p, C.c_void_p]
        _lib.orc_tl_log_dd_array.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    return _lib


def init_genrand(seed):
    key = np.zeros(624, np.uint32)
    lib().orc_init_genrand(int(seed), key.ctypes.data)
    return key


def standard_normal(seed, n, stats=None):
    """RandomState(seed).standard_normal(n).  `stats` (int64 [3], accumulated): logs evaluated, undecided logs taken from
    libm, decided logs that differ from libm's log."""
    out = np.empty(int(n), np.float64)
    st = np.zeros(3, np.int64) if stats is None else stats
    lib().orc_legacy_normals(int(seed), int(n), out.ctypes.data, st.ctypes.data)
    return out


def log_dd(x):
    """tl_log_dd over an array: (hi, lo, decided)."""
    x = np.ascontiguousarray(x, np.float64)
    hi, lo, dec = np.empty_like(x), np.empty_like(x), np.empty(x.shape, np.uint8)
    lib().orc_tl_log_dd_array(x.ctypes.data, x.size, hi.ctypes.data, lo.ctypes.data, dec.ctypes.data)
    return hi, lo, dec.astype(bool)
