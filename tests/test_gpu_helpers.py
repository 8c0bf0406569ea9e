"""GPU parity of the drop-in helper callables (SURVEY 8b): the pixel LISTS of search.getCircle / getArc / bresenham in the
reference's own order, search.getneighbors, rrt.bike_clear / front_of_bike_clear / anglediff and the search.drawpath
rasterisation -- against the golden circle sets generated from the unmodified reference and against the C oracle."""
import builtins
import json
import os

import numpy as np
import pytest

from tests import util
from tests.util import O, planner_for  # noqa: F401  (O is a fixture)

pytestmark = pytest.mark.gpu


def as_tuples(a):
    return [tuple(map(int, p)) for p in a]


def test_getcircle_pixel_sets_golden_and_oracle_order(O, maps):
    """circle_kat.json holds sorted pixel SETS from the reference; the oracle gives the list order (with duplicates)."""
    p = planner_for(maps["map1"])
    kat = json.load(open(os.path.join(util.GOLDEN, "circle_kat.json")))
    rows = [[0, 0, 0, 0, 0, c["center"][0], c["center"][1], c["r"], 2] for c in kat]
    got = p.arc_pixels(rows)
    for c, g in zip(kat, got):
        assert sorted(set(as_tuples(g))) == [tuple(q) for q in c["pixels"]], (c["center"], c["r"])
        assert as_tuples(g) == O.getcircle((100, 100), c["center"], c["r"]), (c["center"], c["r"])
    # every radius 0..300 around a few centres, centres outside the image, huge radii
    rng = np.random.default_rng(11)
    rows = [[0, 0, 0, 0, 0, cx, cy, float(r), 2] for r in range(0, 301, 1) for cx, cy in ((50.5, 49.2), (-3.7, 12.0), (99.9, 99.9))]
    rows += [[0, 0, 0, 0, 0, 50 + rr * np.cos(a), 50 + rr * np.sin(a), rr + d, 2]
             for rr in (150.3, 1000.7, 41014.2) for a in rng.uniform(0, 6.28, 6) for d in (-20.0, 0.0, 35.5)]
    got = p.arc_pixels(rows, cap=64)  # small first buffer: the retry with a larger one is exercised too
    for v, g in zip(rows, got):
        assert as_tuples(g) == O.getcircle((100, 100), (v[5], v[6]), v[7]), v


def test_getarc_pixel_lists_vs_oracle(O, maps):
    free = maps["map1"]
    rng = np.random.default_rng(5)
    rows = []
    for i in range(1500):
        ox, oy = rng.uniform(0, 100, 2)
        o = O.steer((ox, oy), rng.uniform(-180, 180), rng.integers(0, 100, 2), rng.uniform(-180, 180))
        rows.append([ox, oy, o["x"], o["y"], o["steer"], o["icc"][0], o["icc"][1], o["rad"], float(o["straight"])])
    for i in range(200):
        r = float(rng.choice([150.3, 1000.7, 41014.2]))
        ang = rng.uniform(0, 2 * np.pi)
        cx, cy = 50 + (r + rng.uniform(-40, 40)) * np.cos(ang), 50 + (r + rng.uniform(-40, 40)) * np.sin(ang)
        rows.append([rng.uniform(0, 100), rng.uniform(0, 100), rng.uniform(0, 100), rng.uniform(0, 100),
                     float(rng.choice([-65, 65, 10.5])), cx, cy, r, 0.0])
    p = planner_for(free)
    got = p.arc_pixels(np.array(rows))
    n_curved = 0
    for v, g in zip(rows, got):
        u = (v[4], None if v[8] else (v[5], v[6]), None if v[8] else v[7], 1.0)
        assert as_tuples(g) == O.getarc(free.shape, v[0:2], v[2:4], u), v
        n_curved += (not v[8]) and len(g) > 0
    assert n_curved > 500


def test_bresenham_lists(O, maps):
    p = planner_for(maps["map1"])
    rng = np.random.default_rng(2)
    seg = rng.integers(-20, 140, size=(500, 4))
    seg[:20, 2:] = seg[:20, :2]  # zero length
    seg[20:40, 3] = seg[20:40, 1]  # horizontal
    seg[40:60, 2] = seg[40:60, 0]  # vertical
    rows = [[a, b, c, d, 0, 0, 0, 0, 1] for a, b, c, d in seg]
    for s, g in zip(seg, p.arc_pixels(rows)):
        assert as_tuples(g) == O.bresenham(s[:2], s[2:]), s


def test_clearance_and_anglediff_vs_oracle(O, maps):
    free = maps["map1"]
    p = planner_for(free)
    rng = np.random.default_rng(8)
    nodes = np.stack([rng.uniform(-5, 105, 3000), rng.uniform(-5, 105, 3000), rng.uniform(-180, 180, 3000)], 1)
    nodes[:50, :2] = np.floor(nodes[:50, :2])
    nodes[:10, 2] = 0.0
    got = p.clearance(nodes).cpu().numpy().astype(bool)
    for v, g in zip(nodes, got):
        for k, L in enumerate((5.0, 10.0)):  # bikelength, bikelength * frontclearance (rrt.py:208-222)
            r = O.rotz(v[2], (L, 0.0))
            assert g[k] == O.lineofsight(free, (int(v[0]), int(v[1])), (int(r[0] + v[0]), int(r[1] + v[1]))), (v, k)
    pairs = rng.uniform(-400, 400, size=(4000, 2))
    pairs[:5] = [[0, 0], [180, -180], [10, 190], [-179.999, 179.999], [90, 90]]
    d = p.anglediff(pairs).cpu().numpy()
    ref = np.array([O.anglediff(a, b) for a, b in pairs])
    assert np.array_equal(d.view(np.int64), ref.view(np.int64))


def test_dropin_helper_callables(O, maps):
    """The module-level callables a script written against the reference uses (SURVEY 8b)."""
    from theta_rrt_b200 import rrt as R, search as S
    free = maps["map1"]
    builtins.imarray = free
    kat = json.load(open(os.path.join(util.GOLDEN, "circle_kat.json")))
    for c in kat[:6]:
        assert sorted(set(S.getCircle(c["center"], c["r"]))) == [tuple(q) for q in c["pixels"]]
    assert S.bresenham((3, 4), (40, 17)) == O.bresenham((3, 4), (40, 17))
    u = (-65.0, np.array([20.3, 30.1]), 2.331538290774993, 9.0)
    begin = (20.3 + 2.331538290774993, 30.1)
    land = (20.3, 30.1 - 2.331538290774993)
    assert S.getArc(begin, land, u) == O.getarc(free.shape, begin, land, (u[0], tuple(u[1]), u[2], u[3]))
    assert S.getArc((3, 4), (40, 17), (0, None, None, 1)) == O.bresenham((3, 4), (40, 17))
    # getneighbors: `node - delta` in itertools.product order, valid and free only (search.py:184-194)
    for node in ((5, 5), (0, 0), (99, 99), (50, 0), (43, 39)):
        want = []
        for dx in (-1, 0, 1):
            for dy in (-1, 0, 1):
                if (dx, dy) != (0, 0):
                    x, y = node[0] - dx, node[1] - dy
                    if 0 <= x < 100 and 0 <= y < 100 and free[y, x]:
                        want.append((x, y))
        assert S.getneighbors(node) == want
    path = [(5, 5), (43, 39), (46, 41), (90, 50)]
    assert S.pathpixels(path) == [q for a, b in zip(path, path[1:]) for q in O.bresenham(a, b)]
    assert S.pathpixels([]) == [] and S.pathpixels(path + [None]) == S.pathpixels(path)
    node = ((20.5, 20.25), 33.0)
    r5, r10 = O.rotz(33.0, (5.0, 0.0)), O.rotz(33.0, (10.0, 0.0))
    assert R.bike_clear(node) == O.lineofsight(free, (20, 20), (int(r5[0] + 20.5), int(r5[1] + 20.25)))
    assert R.front_of_bike_clear(node) == O.lineofsight(free, (20, 20), (int(r10[0] + 20.5), int(r10[1] + 20.25)))
    assert R.anglediff(10.0, 350.0) == O.anglediff(10.0, 350.0)
    del builtins.imarray


def test_device_libm_against_glibc_without_the_shared_header():
    """The oracle shares csrc/trrt_libm.h with the device code, so a bug in that header would be invisible to the bitwise
    CUDA-vs-oracle tests.  Here the DEVICE's sin / cos / atan2 (through rrt.anglediff's quaternion evaluation, rrt.py:108-115)
    are compared with numpy / glibc, which know nothing of that header: same formula, 1e-12 degrees."""
    from theta_rrt_b200 import OccupancyGrid, Planner
    p = Planner(OccupancyGrid(np.ones((8, 8), bool)))
    rng = np.random.default_rng(21)
    a = np.concatenate([rng.uniform(-720, 720, size=(200000, 2)), rng.uniform(-1e-6, 1e-6, size=(1000, 2)),
                        np.array([[0, 180], [180, 0], [90, -90], [-90, 90], [179.999999, -179.999999], [45, 45 + 1e-9]])])
    got = p.anglediff(a).cpu().numpy()
    h1, h2 = np.deg2rad(a[:, 0]) / 2, np.deg2rad(a[:, 1]) / 2
    s1, c1, s2, c2 = np.sin(h1), np.cos(h1), np.sin(h2), np.cos(h2)
    qz, qw = c1 * s2 - c2 * s1, c1 * c2 + s1 * s2          # q1^-1 * q2 about z
    n = np.hypot(qz, qw)
    ang = 2 * np.arctan2(qz / n, qw / n)
    ang = np.where(ang < -np.pi, ang + 2 * np.pi, np.where(ang > np.pi, ang - 2 * np.pi, ang))
    ref = np.rad2deg(ang)
    d = np.abs(got - ref)
    d = np.minimum(d, np.abs(d - 360))                     # +180 and -180 are the same angle
    assert d.max() < 1e-12, d.max()


def test_int16_sample_coordinates_equal_int32(maps):
    """trrt_rrt_args.sample_xy_i16: the same trees from int16 sample pairs (half the host-to-device bytes of that array)."""
    import torch
    from theta_rrt_b200 import samples
    free = maps["map2"]  # 300 x 300: coordinates above 255
    nq, K = 12, 301
    starts, goals = util.random_queries(free, nq, 31)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 900 + q, free.shape)
    assert sxy.max() > 255
    p = planner_for(free, tol_xy=0.0)
    a = p.rrt(starts, goals, sxy, sth, K=K, logs=True).host()
    for lanes, schedule in ((32, 0), (8, 0), (16, 1)):
        b = p.rrt(starts, goals, torch.from_numpy(sxy.astype(np.int16)), sth, K=K, logs=True, lanes=lanes, schedule=schedule).host()
        for k in ("n_nodes", "it_near", "it_code", "status", "iters"):
            assert np.array_equal(a[k], b[k]), (k, lanes, schedule)
        for q in range(nq):
            n = int(a["n_nodes"][q])  # rows beyond n_nodes are not written
            assert np.array_equal(a["parent"][q, :n], b["parent"][q, :n])
            assert np.array_equal(a["node_x"][q, :n].view(np.int64), b["node_x"][q, :n].view(np.int64))


def test_theta_memory_budget_cuts_the_slots_not_the_results(O, maps):
    """Planner.theta(mem_budget=...): fewer concurrent searches, same answers; a budget below one slot is refused."""
    from theta_rrt_b200 import _lib
    free = maps["map1"]
    p = planner_for(free)
    rng = np.random.default_rng(4)
    cells = np.argwhere(free)
    a, b = cells[rng.integers(len(cells), size=200)], cells[rng.integers(len(cells), size=200)]
    sg = np.stack([a[:, 1], a[:, 0], b[:, 1], b[:, 0]], 1).astype(np.int32)
    full = p.theta(sg, path_cap=64)
    per_slot = (100 * 100 + int(full.extra["heap_cap"])) * 16
    small = p.theta(sg, path_cap=64, mem_budget=5 * per_slot + 256)
    assert small.extra["n_slots"] == 5 < full.extra["n_slots"]
    for k in ("path_len", "expanded", "status", "cost", "path"):
        assert np.array_equal(full.host()[k], small.host()[k]), k
    with pytest.raises(_lib.TrrtError):
        p.theta(sg, mem_budget=per_slot // 2)


def test_astar_batch_returns_long_paths_whole(O, maps):
    """search.astar_batch: paths longer than the first pass's capacity are fetched by a second pass (A* mode: 86-node path)."""
    from theta_rrt_b200 import search as S
    builtins.imarray = maps["map1"]
    builtins.THETASTAR = False
    try:
        q = [[5, 5, 90, 50], [2, 97, 97, 2], [5, 5, 6, 6]]
        h = S.astar_batch(q, path_cap=16)
        for i, (sx, sy, gx, gy) in enumerate(q):
            o = O.astar(maps["map1"], (sx, sy), (gx, gy), thetastar=False)
            n = int(h["path_len"][i])
            assert n == len(o["path"]) and [tuple(v) for v in h["path"][i, :n].tolist()] == o["path"], i
        assert h["path"].shape[1] >= 86
    finally:
        builtins.THETASTAR = True
        del builtins.imarray
