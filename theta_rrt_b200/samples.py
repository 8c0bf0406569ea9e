"""Sample streams: rrt.rand_conf (rrt.py:53-68) restated in vectorised form.

The reference draws, every loop iteration and before any rejection test
(rrt.py:144), two normals for xy around the goal (std = xystdv * image dims),
clips them to the image and truncates to int, then one normal for the heading
(std = anglestdv) wrapped by standardangle.  The draws do not depend on the
tree, so the whole stream of a query can be generated up front and handed to
the device ("injected stream").  With numpy's legacy generator the sequence of
`normal(loc, scale, 2)` / `normal(loc, scale, 1)` calls consumes exactly the
gaussians of one `standard_normal(3*n)` call, and loc + scale*z is the same
arithmetic, so the stream is bit-identical to calling rand_conf n times.
"""
from __future__ import annotations

import numpy as np


def standardangle(a):
    """rrt.standardangle (rrt.py:9-14) for scalars or arrays (same repeated +-360 steps)."""
    a = np.array(a, dtype=np.float64, copy=True)
    while True:
        hi = a > 180
        if not hi.any():
            break
        a[hi] = a[hi] - 360
    while True:
        lo = a <= -180
        if not lo.any():
            break
        a[lo] = a[lo] + 360
    return a if a.ndim else float(a)


def stream_from_normals(z, goal, shape, xystdv=0.4, anglestdv=100):
    """z: float64 [n,3] standard normals in draw order -> (xy int32 [n,2], theta float64 [n])."""
    (gx, gy), gth = goal
    H, W = shape
    z = np.asarray(z, dtype=np.float64).reshape(-1, 3)
    x = gx + (xystdv * H) * z[:, 0]
    y = gy + (xystdv * W) * z[:, 1]
    x = np.clip(x, 0, H - 1)
    y = np.clip(y, 0, W - 1)
    xy = np.stack([x, y], axis=1).astype(np.int64).astype(np.int32)  # int(): toward zero (values are >= 0)
    th = standardangle(float(standardangle(gth)) + anglestdv * z[:, 2])
    return xy, np.ascontiguousarray(th, dtype=np.float64)


def make_stream(goal, n, seed, shape, xystdv=0.4, anglestdv=100):
    """Stream of n samples equal to `np.random.seed(seed); [rand_conf(goal) for _ in range(n)]`."""
    z = np.random.RandomState(seed).standard_normal(3 * n)
    return stream_from_normals(z, goal, shape, xystdv, anglestdv)


def make_streams(goals, n, seeds, shape, xystdv=0.4, anglestdv=100):
    """make_stream for many queries: goals [q, 3] = (x, y, theta), seed int(seeds[q]) for query q.
    Returns (xy int32 [q, n, 2], theta float64 [q, n])."""
    goals = np.asarray(goals, dtype=np.float64).reshape(-1, 3)
    xy = np.empty((len(goals), n, 2), np.int32)
    th = np.empty((len(goals), n), np.float64)
    for q, g in enumerate(goals):
        xy[q], th[q] = make_stream(((g[0], g[1]), g[2]), n, int(seeds[q]), shape, xystdv, anglestdv)
    return xy, th


def draw_stream_global(goal, n, shape, xystdv=0.4, anglestdv=100):
    """Same, but consuming numpy's GLOBAL legacy generator like the reference does."""
    z = np.random.standard_normal(3 * n)
    return stream_from_normals(z, goal, shape, xystdv, anglestdv)
