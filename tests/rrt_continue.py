"""The C parity oracle's RRT loop continued from a given tree and iteration (tests/rrt_continue.c).

TEST INFRASTRUCTURE ONLY -- used by tests/test_tree_repair.py.  The library is compiled on first use, with the oracle's
compiler flags (oracle/Makefile), into a temporary directory keyed by the sources, so the tree stays untouched.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import re
import subprocess
import tempfile

import numpy as np

from oracle.c_oracle import Params, _grid, _p, c_dp, c_i32p, c_i64p, c_u8p

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "rrt_continue.c"), os.path.join(_ROOT, "oracle", "trrt_oracle.c"),
            os.path.join(_ROOT, "theta_rrt_b200", "csrc", "trrt_libm.h"), os.path.join(_ROOT, "oracle", "Makefile")]
_lib = None


def _cflags():
    mk = open(os.path.join(_ROOT, "oracle", "Makefile")).read()
    return re.search(r"^CFLAGS \?= (.*)$", mk, flags=re.M).group(1).split()


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for s in _SOURCES:
            h.update(open(s, "rb").read())
        so = os.path.join(tempfile.gettempdir(), f"trrt_rrt_continue_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(so))
            os.close(fd)
            subprocess.check_call(["gcc", *_cflags(), "-shared", "-o", tmp, _SOURCES[0], "-lm"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.trc_rrt_continue.restype = C.c_int
        L.trc_rrt_continue.argtypes = [c_u8p, C.c_int, C.c_int, C.POINTER(Params), C.c_int, c_dp, c_i32p, c_dp,
                                       c_dp, c_dp, c_dp, c_i32p, c_dp, c_i32p, c_i32p, c_u8p, C.c_int32, C.c_int32,
                                       c_i32p, c_i32p, c_i32p, c_u8p, C.c_int64, c_i64p]
        _lib = L
    return _lib


def rrt_continue(free, goal, sxy, sth, tree, it0, K, params=None):
    """The rrt loop continued on image `free` from tree = dict(x, y, theta, parent, u) of n >= 1 rows, no solution, next
    iteration it0 (samples it0 .. K-2 of sxy int32 [K-1, 2] / sth [K-1] are consumed), capacity K.  Returns the dict of
    oracle.c_oracle.rrt; it_near / it_new / it_code cover iterations >= it0 (-1 / -1 / 255 before), los and n_los the
    continuation's lineofsight calls."""
    P = params or Params()
    g, H, W = _grid(free)
    sxy = np.ascontiguousarray(sxy, np.int32).reshape(-1, 2)
    sth = np.ascontiguousarray(sth, np.float64)
    assert len(sth) >= K - 1
    n0 = len(tree["x"])
    assert 1 <= n0 <= K and 0 <= it0 <= K - 1
    gl = np.array([goal[0][0], goal[0][1], goal[1]], np.float64)
    nx, ny, nth = np.zeros(K), np.zeros(K), np.zeros(K)
    parent = np.full(K, -1, np.int32)
    u = np.full((K, 5), np.nan)
    nx[:n0], ny[:n0], nth[:n0], parent[:n0], u[:n0] = tree["x"], tree["y"], tree["theta"], tree["parent"], tree["u"]
    it_near = np.full(max(K - 1, 1), -1, np.int32)
    it_new = np.full(max(K - 1, 1), -1, np.int32)
    it_code = np.full(max(K - 1, 1), 255, np.uint8)
    n_nodes, sol, iters = C.c_int32(0), C.c_int32(-1), C.c_int32(0)
    los_cap = 2 * K + 8
    los = np.zeros(los_cap, np.uint8)
    n_los = C.c_int64(0)
    status = lib().trc_rrt_continue(_p(g, c_u8p), H, W, C.byref(P), K, _p(gl, c_dp), _p(sxy, c_i32p), _p(sth, c_dp),
                                    _p(nx, c_dp), _p(ny, c_dp), _p(nth, c_dp), _p(parent, c_i32p), _p(u, c_dp),
                                    _p(it_near, c_i32p), _p(it_new, c_i32p), _p(it_code, c_u8p), n0, int(it0),
                                    C.byref(n_nodes), C.byref(sol), C.byref(iters), _p(los, c_u8p), los_cap,
                                    C.byref(n_los))
    n = n_nodes.value
    return dict(status=status, n_nodes=n, sol=sol.value, iters=iters.value, x=nx[:n], y=ny[:n], theta=nth[:n],
                parent=parent[:n], u=u[:n], it_near=it_near[:K - 1], it_new=it_new[:K - 1], it_code=it_code[:K - 1],
                los=los[:n_los.value].astype(bool), n_los=n_los.value)
