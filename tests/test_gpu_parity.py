"""GPU parity tests: every kernel, called through the C ABI (theta_rrt_b200.Planner ->
libthetarrt.so), against the CPU oracle (oracle/trrt_oracle.c) on the same seeded inputs,
and against the golden fixtures generated from the unmodified reference.

Bars: bit-exact for integer / byte / index outputs (LOS booleans, nearest indices,
parent arrays, iteration codes, Theta* paths and expansion counts); fp64 outputs of the
CUDA path are compared BITWISE with the oracle (both use the deterministic libm of
trrt_libm.h and no contraction), and within 1e-9 relative with the reference goldens.
"""
import numpy as np
import pytest

from tests import util
from tests.util import O, bits_equal, planner_for  # noqa: F401  (O is a fixture)

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ grid + LOS
def test_los_golden(maps):
    z = np.load(util.GOLDEN + "/los_kat.npz")
    for name in ("map1", "map2"):
        p = planner_for(maps[name])
        out = p.los(z[name + "_seg"]).cpu().numpy().astype(bool)
        assert np.array_equal(out, z[name + "_los"]), name


@pytest.mark.parametrize("layout", ["tiles", "rows"])
@pytest.mark.parametrize("n,seed", [(64, 1), (257, 2), (1000, 3)])
def test_los_vs_oracle_random(O, n, seed, layout):
    free = util.synthetic_map(n, 0.12, 4, seed)
    rng = np.random.default_rng(seed)
    seg = rng.integers(-5, n + 5, size=(20000, 4)).astype(np.int32)
    seg[:2000, 2:] = seg[:2000, :2] + rng.integers(-40, 41, size=(2000, 2))
    seg[2000:2100, 2:] = seg[2000:2100, :2]  # zero length
    p = planner_for(free)
    got = p.los(seg, layout=layout).cpu().numpy().astype(bool)
    ref = O.lineofsight_batch(free, seg, threads=4)
    assert np.array_equal(got, ref)
    # symmetry of the canonicalised Bresenham (search.py:47-56)
    rev = seg[:, [2, 3, 0, 1]].copy()
    assert np.array_equal(p.los(rev, layout=layout).cpu().numpy().astype(bool), got)


def test_tile_grid_layout():
    """trrt_tile_grid (include/thetarrt.h K4b): entry [o][K][c] holds, in byte j bit i, pixel (8c+i, 8K-8+j) for
    orientation 0 and pixel (8K-8+j, 8c+i) for orientation 1; everything outside the image is blocked."""
    from theta_rrt_b200 import OccupancyGrid
    for n, seed in ((100, 1), (300, 2), (257, 3), (8, 4), (1, 5)):
        free = np.stack([util.synthetic_map(n, 0.3, 1, seed), util.synthetic_map(n, 0.5, 2, seed + 10)])
        tp = (n + 7) // 8
        got = OccupancyGrid(free).tiles.cpu().numpy().view(np.uint8).reshape(2, 2, tp + 1, tp, 16)
        pad = np.zeros((2, 8 * tp + 16, 8 * tp + 16), bool)  # image at offset (8, 8)
        pad[:, 8:8 + n, 8:8 + n] = free
        K, c, j, i = np.meshgrid(np.arange(tp + 1), np.arange(tp), np.arange(16), np.arange(8), indexing="ij")
        for m in range(2):
            o0 = pad[m][8 * K + j, 8 + 8 * c + i]  # [y + 8, x + 8] with y = 8K-8+j, x = 8c+i
            o1 = pad[m][8 + 8 * c + i, 8 * K + j]  # x = 8K-8+j, y = 8c+i
            for o, want in ((0, o0), (1, o1)):
                assert np.array_equal(got[m, o], np.packbits(want, axis=-1, bitorder="little")[..., 0]), (n, m, o)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 1000, 70001])
def test_los_tiled_refill_mix(O, n):
    """Per-lane refill: a few very long clear rays among many short blocked ones, batch sizes around the warp size."""
    free = util.synthetic_map(1024, 0.02, 2, 11)
    rng = np.random.default_rng(n)
    a = rng.integers(0, 1024, size=(n, 2))
    ln = np.where(rng.random(n) < 0.1, 900, 6)
    d = rng.integers(-1, 2, size=(n, 2)) * ln[:, None] + rng.integers(-3, 4, size=(n, 2))
    seg = np.concatenate([a, a + d], 1).astype(np.int32)
    p = planner_for(free)
    got = p.los(seg).cpu().numpy().astype(bool)
    assert np.array_equal(got, O.lineofsight_batch(free, seg, threads=4))
    assert np.array_equal(got, p.los(seg, layout="rows").cpu().numpy().astype(bool))


def test_los_long_rays_large_map(O):
    """Side 16384: driving-axis lengths up to 16383 (divisors up to 32766 in the block walk's FMA floors), rays that
    cross the whole map on a sparse map, both layouts and the oracle on a subset."""
    n = 16384
    free = util.synthetic_map(n, 0.0005, 16, 21)
    rng = np.random.default_rng(5)
    seg = rng.integers(0, n, size=(60000, 4)).astype(np.int32)
    seg[:20000, 2:] = np.clip(seg[:20000, :2] + rng.integers(-3000, 3001, size=(20000, 2)), 0, n - 1)
    seg[20000:20200] = [[0, 0, n - 1, n - 1], [n - 1, 0, 0, n - 1], [0, 5, n - 1, 6], [7, n - 1, 8, 0]] * 50
    p = planner_for(free)
    got = p.los(seg).cpu().numpy().astype(bool)
    assert np.array_equal(got, p.los(seg, layout="rows").cpu().numpy().astype(bool))
    sub = np.r_[0:2000, 20000:20200, 40000:42000]
    assert np.array_equal(got[sub], O.lineofsight_batch(free, seg[sub], threads=4))
    assert got.any() and not got.all()


def test_los_empty_and_multimap(O):
    free = np.stack([util.synthetic_map(96, 0.2, 3, s) for s in (5, 6, 7)])
    from theta_rrt_b200 import OccupancyGrid, Planner
    p = Planner(OccupancyGrid(free))
    assert p.los(np.zeros((0, 4), np.int32)).numel() == 0
    rng = np.random.default_rng(0)
    seg = rng.integers(0, 96, size=(5000, 4)).astype(np.int32)
    mid = rng.integers(0, 3, size=5000).astype(np.int32)
    for layout in ("tiles", "rows"):
        assert p.los(np.zeros((0, 4), np.int32), layout=layout).numel() == 0
        got = p.los(seg, map_id=mid, layout=layout).cpu().numpy().astype(bool)
        for m in range(3):
            sel = mid == m
            assert np.array_equal(got[sel], O.lineofsight_batch(free[m], seg[sel]))


# ------------------------------------------------------------------ nearest
@pytest.mark.parametrize("n,nq", [(1, 5), (2, 1), (37, 64), (5001, 300), (100003, 700), (1 << 18, 33)])
def test_nearest_vs_oracle(O, n, nq):
    rng = np.random.default_rng(n)
    x = rng.uniform(0, 511, n)
    y = rng.uniform(0, 511, n)
    # exact duplicates and integer nodes to exercise the lowest-index tie-break
    if n > 10:
        x[n // 2] = x[3]; y[n // 2] = y[3]
        x[5] = 100.0; y[5] = 200.0; x[n - 1] = 100.0; y[n - 1] = 200.0
    q = rng.integers(0, 512, size=(nq, 2)).astype(np.int32)
    if n > 10:
        q[0] = (100, 200)
    p = planner_for(np.ones((8, 8), bool))
    idx, d2 = p.nearest(x, y, q, want_d2=True)
    idx = idx.cpu().numpy()
    ref = O.nearest_batch(x, y, q, threads=4)
    assert np.array_equal(idx, ref)
    dx = q[:, 0] - x[idx]; dy = q[:, 1] - y[idx]
    assert bits_equal(d2.cpu().numpy(), dx * dx + dy * dy)
    if n > 10:
        assert idx[0] == 5


def test_nearest_empty_tree():
    p = planner_for(np.ones((8, 8), bool))
    idx = p.nearest(np.zeros(0), np.zeros(0), np.array([[1, 2], [3, 4]], np.int32)).cpu().numpy()
    assert list(idx) == [-1, -1]


# ------------------------------------------------------------------ Theta*
def test_theta_known_answers(maps, O):
    for k in util.theta_kat():
        p = planner_for(maps[k["map"]])
        r = p.theta([[*k["start"], *k["goal"]]], thetastar=k["thetastar"], path_cap=maps[k["map"]].size,
                    log_los=True, lanes=8).host()
        o = O.astar(maps[k["map"]], k["start"], k["goal"], thetastar=k["thetastar"])
        tag = (k["map"], k["start"], k["goal"], k["thetastar"])
        assert int(r["status"][0]) == o["status"], tag
        if k["path"] is False:
            assert int(r["status"][0]) != 0, tag
            continue
        n = int(r["path_len"][0])
        assert [tuple(v) for v in r["path"][0, :n].tolist()] == [tuple(v) for v in k["path"]], tag
        assert int(r["expanded"][0]) == k["expanded"], tag
        assert r["cost"][0] == o["cost"], tag                      # bitwise vs oracle
        assert abs(r["cost"][0] - k["cost"]) <= 1e-9 * k["cost"], tag  # reference, 1e-9 relative
        nl = int(r["n_los"][0])
        assert nl == k["n_los"], tag
        los_ref = np.unpackbits(np.frombuffer(bytes.fromhex(k["los_hex"]), np.uint8))[:nl].astype(bool)
        assert np.array_equal(r["los_log"][0, :nl].astype(bool), los_ref), tag
        assert int(r["pushes"][0]) == o["pushes"], tag


@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_theta_batch_vs_oracle(O, lanes):
    free = np.stack([util.synthetic_map(64, 0.15, 4, 7 + m) for m in range(4)])
    rng = np.random.default_rng(lanes)
    nq = 300
    mid = rng.integers(0, 4, nq).astype(np.int32)
    sg = rng.integers(-1, 65, size=(nq, 4)).astype(np.int32)
    from theta_rrt_b200 import OccupancyGrid, Planner
    p = Planner(OccupancyGrid(free))
    for th in (True, False):
        r = p.theta(sg, thetastar=th, map_id=mid, path_cap=64 * 64, lanes=lanes, n_slots=37).host()
        for q in range(nq):
            o = O.astar(free[mid[q]], sg[q, :2], sg[q, 2:], thetastar=th, log_los=False)
            assert int(r["status"][q]) == o["status"], (q, th)
            if o["status"] == 0:
                n = int(r["path_len"][q])
                assert [tuple(v) for v in r["path"][q, :n].tolist()] == o["path"], (q, th)
                assert r["cost"][q] == o["cost"] and int(r["expanded"][q]) == o["expanded"], (q, th)
            assert int(r["n_los"][q]) == o["n_los"] and int(r["pushes"][q]) == o["pushes"], (q, th)


# ------------------------------------------------------------------ steer / drive / arc single steps
def test_steer_drive_bitwise_vs_oracle(O, maps):
    rng = np.random.default_rng(11)
    n = 20000
    inp = np.stack([rng.uniform(0, 100, n), rng.uniform(0, 100, n), rng.uniform(-180, 180, n),
                    rng.integers(0, 100, n).astype(float), rng.integers(0, 100, n).astype(float),
                    rng.uniform(-180, 180, n)], axis=1)
    inp[:50, 2] = 0.0; inp[:50, 4] = inp[:50, 1] = 40.0  # straight ahead: singular solve
    inp[50:60, 3:5] = inp[50:60, 0:2] = 7.0               # target == origin
    p = planner_for(maps["map1"])
    out, straight = p.steer(inp)
    out = out.cpu().numpy(); straight = straight.cpu().numpy()
    dr_in = []
    for i in range(n):
        o = O.steer(inp[i, :2], inp[i, 2], inp[i, 3:5], inp[i, 5])
        ref = np.array([o["x"], o["y"], o["theta"], o["steer"], o["icc"][0], o["icc"][1], o["rad"], o["dist"]])
        assert bool(straight[i]) == o["straight"], i
        assert np.array_equal(out[i].view(np.int64), ref.view(np.int64)), (i, out[i], ref)
        if not o["straight"]:
            dr_in.append([inp[i, 0], inp[i, 1], inp[i, 2], o["steer"], o["icc"][0], o["icc"][1], o["rad"], o["dist"] / 3])
    dr_in = np.array(dr_in[:5000])
    dout = p.drive(dr_in).cpu().numpy()
    for i in range(len(dr_in)):
        ref = O.drive(dr_in[i, :2], dr_in[i, 2], (dr_in[i, 3], (dr_in[i, 4], dr_in[i, 5]), dr_in[i, 6], dr_in[i, 7]))
        assert np.array_equal(dout[i].view(np.int64), ref.view(np.int64)), i


@pytest.mark.parametrize("lanes", [1, 4, 8, 32])
def test_arc_blocked_vs_oracle(O, maps, lanes):
    free = maps["map1"]
    rng = np.random.default_rng(5)
    rows = []
    for i in range(3000):
        ox, oy = rng.uniform(0, 100, 2)
        o = O.steer((ox, oy), rng.uniform(-180, 180), rng.integers(0, 100, 2), rng.uniform(-180, 180))
        rows.append([ox, oy, o["x"], o["y"], o["steer"], o["icc"][0], o["icc"][1], o["rad"], float(o["straight"])])
    # large radii and centres far outside the image
    for i in range(300):
        r = float(rng.choice([150.3, 1000.7, 41014.2]))
        ang = rng.uniform(0, 2 * np.pi)
        cx, cy = 50 + (r + rng.uniform(-40, 40)) * np.cos(ang), 50 + (r + rng.uniform(-40, 40)) * np.sin(ang)
        rows.append([rng.uniform(0, 100), rng.uniform(0, 100), rng.uniform(0, 100), rng.uniform(0, 100),
                     float(rng.choice([-65, 65, 10.5])), cx, cy, r, 0.0])
    rows = np.array(rows)
    p = planner_for(free)
    got = p.arc_blocked(rows, lanes=lanes).cpu().numpy().astype(bool)
    for i, v in enumerate(rows):
        u = (v[4], None if v[8] else (v[5], v[6]), None if v[8] else v[7], 1.0)
        px = O.getarc(free.shape, v[0:2], v[2:4], u)
        ref = any((not (0 <= x < free.shape[0] and 0 <= y < free.shape[1])) or (not free[y, x]) for x, y in px)
        assert got[i] == ref, (i, v)


# ------------------------------------------------------------------ fused RRT
def run_rrt_pair(O, free, starts, goals, sxy, sth, K, lanes, schedule=0, **params):
    from oracle.c_oracle import Params as OP
    p = planner_for(free, **{k: v for k, v in params.items()})
    res = p.rrt(starts, goals, sxy, sth, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
    op = OP(**{k.lower(): v for k, v in params.items()})
    for q in range(len(starts)):
        o = O.rrt(free, ((starts[q, 0], starts[q, 1]), starts[q, 2]), ((goals[q, 0], goals[q, 1]), goals[q, 2]),
                  sxy[q], sth[q], op, K=K)
        n = o["n_nodes"]
        tag = (q, lanes, schedule)
        assert int(res["status"][q]) == o["status"], tag
        assert int(res["n_nodes"][q]) == n and int(res["sol"][q]) == o["sol"] and int(res["iters"][q]) == o["iters"], tag
        assert np.array_equal(res["it_code"][q], o["it_code"]), tag
        assert np.array_equal(res["it_near"][q], o["it_near"]), tag
        assert np.array_equal(res["it_new"][q], o["it_new"]), tag
        assert np.array_equal(res["parent"][q, :n], o["parent"]), tag
        assert bits_equal(res["node_x"][q, :n], o["x"]) and bits_equal(res["node_y"][q, :n], o["y"]), tag
        assert bits_equal(res["node_theta"][q, :n], o["theta"]), tag
        assert np.array_equal(res["u"][q, :n].view(np.int64), o["u"].view(np.int64)), tag
        nl = int(res["n_los"][q])
        assert nl == o["n_los"] and np.array_equal(res["los_log"][q, :nl].astype(bool), o["los"]), tag
    # SURVEY H3: no nearest decision where the reference's argmin over sqrt() could have kept a lower index than argmin(d2)
    assert (res["counters"][:, 8] == 0).all(), (lanes, schedule)
    return res


@pytest.mark.parametrize("schedule", [0, 1])
@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
def test_rrt_cfg1_golden_and_oracle(O, maps, lanes, schedule):
    """BASELINE cfg 1: map1, ((5,5),0) -> ((90,50),90), seed-0 stream, K=300."""
    run = util.rrt_runs()[0]
    free = maps["map1"]
    K = int(run["K"][0])
    res = run_rrt_pair(O, free, run["start"][None], run["goal"][None], run["sxy"][None], run["sth"][None], K, lanes,
                       schedule=schedule, tol_xy=float(run["tol_xy"][0]))
    n = int(res["n_nodes"][0])
    assert n == len(run["parent"]) and np.array_equal(res["parent"][0, :n], run["parent"])
    assert int(res["sol"][0]) == int(run["sol"][0]) and int(res["iters"][0]) == int(run["iterations"][0])
    near = res["it_near"][0]
    assert np.array_equal(near[run["nearest_it"] - 1], run["nearest_idx"])
    assert np.array_equal(res["los_log"][0, :int(res["n_los"][0])].astype(bool), run["los"])
    for a, b in ((res["node_x"][0, :n], run["x"]), (res["node_y"][0, :n], run["y"]), (res["node_theta"][0, :n], run["theta"])):
        assert np.allclose(a, b, rtol=1e-9, atol=1e-9)


def test_rrt_all_goldens(O, maps):
    """Every committed run of the unmodified reference: CUDA == oracle bitwise, and CUDA == reference on all
    discrete outputs up to the first iteration the oracle's margin audit marks as decided by rounding noise
    (runs without such an iteration must match to the end); coordinates within the documented drift."""
    from oracle.c_oracle import Params as OP
    for i, run in enumerate(util.rrt_runs()):
        free = maps[str(run["map"])]
        K = int(run["K"][0])
        tol = float(run["tol_xy"][0])
        res = run_rrt_pair(O, free, run["start"][None], run["goal"][None], run["sxy"][None], run["sth"][None], K, 8,
                           tol_xy=tol)
        o = O.rrt(free, ((run["start"][0], run["start"][1]), run["start"][2]), ((run["goal"][0], run["goal"][1]), run["goal"][2]),
                  run["sxy"], run["sth"], OP(tol_xy=tol), K=K, audit_eps=util.AUDIT_EPS)
        fa = -1 if i < 2 else o["first_ambiguous"]  # cfg 1 is reproduced to the end (see tests/test_oracle_golden.py)
        n = int(res["n_nodes"][0])
        gpu = dict(n_nodes=n, sol=int(res["sol"][0]), parent=res["parent"][0, :n], it_near=res["it_near"][0],
                   it_new=res["it_new"][0], it_code=res["it_code"][0], los=res["los_log"][0, :int(res["n_los"][0])],
                   x=res["node_x"][0, :n], y=res["node_y"][0, :n], theta=res["node_theta"][0, :n])
        util.compare_rrt_with_reference(gpu, run, fa)


@pytest.mark.parametrize("schedule", [0, 1])
@pytest.mark.parametrize("lanes,nq,K", [(32, 24, 1201), (16, 40, 1001), (8, 96, 801), (4, 64, 801), (1, 64, 401)])
def test_rrt_batch_bitwise_vs_oracle(O, maps, lanes, nq, K, schedule):
    """cfg-3 style batch (random free start/goal, per-query seeded streams, tol_xy=0) -- bitwise vs oracle."""
    from theta_rrt_b200 import samples
    free = maps["map1"]
    starts, goals = util.random_queries(free, nq, 1234)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, q, free.shape)
    res = run_rrt_pair(O, free, starts, goals, sxy, sth, K, lanes, schedule=schedule, tol_xy=0.0)
    # counters are defined on the sequential loop, so both schedules must report the same numbers
    other = run_rrt_pair(O, free, starts[:8], goals[:8], sxy[:8], sth[:8], K, lanes, schedule=1 - schedule, tol_xy=0.0)
    assert np.array_equal(res["counters"][:8, [0, 1, 2, 5, 6]], other["counters"][:, [0, 1, 2, 5, 6]])
    assert (res["counters"][:, 0] > 0).all()


@pytest.mark.parametrize("lanes,schedule", [(32, 0), (16, 0), (16, 1), (4, 0)])
def test_rrt_full_size_one_query_k5001(O, maps, lanes, schedule):
    """BASELINE cfg 3 size for a few queries: K=5001, bitwise vs oracle at full depth."""
    from theta_rrt_b200 import samples
    free = maps["map1"]
    nq, K = 8, 5001
    starts, goals = util.random_queries(free, nq, 1234)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, q, free.shape)
    run_rrt_pair(O, free, starts, goals, sxy, sth, K, lanes, schedule=schedule, tol_xy=0.0)


def test_rrt_full_size_64_distinct_queries_k5001(O, maps):
    """SURVEY 8(d) cfg 3: a >= 32-query subset at full depth.  64 DISTINCT cfg-3 queries (the bench workload's queries
    1000..1063: same generator, same seeds), K = 5001, every tree bit for bit against the oracle (all host threads)."""
    import os
    import bench
    free = maps["map1"]
    nq, K, first = 64, 5001, 1000
    starts, goals, sxy, sth = bench.make_rrt_workload(free, nq, K, first_query=first)
    from oracle.c_oracle import Params as OP
    o = O.rrt_batch(free, starts, goals, sxy, sth, K, OP(tol_xy=0.0), threads=os.cpu_count() or 1, want_nodes=True)
    # the 64 queries ride in a batch large enough to fill the GPU's persistent CTAs (pooled scans, idle warps helping)
    s2, g2, x2, t2 = (np.concatenate([a] * 48) for a in (starts, goals, sxy, sth))
    res = planner_for(free, tol_xy=0.0).rrt(s2, g2, x2, t2, K=K, want_u=False).host()
    assert int(o["iters"].sum()) > 200000 and (o["status"] == 4).sum() > 3  # full-length runs and early ends both present
    for rep in (0, 17, 47):
        sl = slice(rep * nq, (rep + 1) * nq)
        for k in ("n_nodes", "status", "iters", "sol"):
            assert np.array_equal(res[k][sl], o[k]), (k, rep)
        for q in range(nq):
            n = int(o["n_nodes"][q])
            assert np.array_equal(res["parent"][sl][q, :n], o["parent"][q, :n]), (q, rep)
            for j, k in enumerate(("node_x", "node_y", "node_theta")):
                assert bits_equal(res[k][sl][q, :n], o["nodes"][q, :n, j]), (k, q, rep)


@pytest.mark.parametrize("lanes,schedule", [(32, 0), (8, 0), (8, 1), (4, 0)])
def test_rrt_goal_found_and_map2(O, maps, lanes, schedule):
    run = util.rrt_runs()[2]
    run_rrt_pair(O, maps["map2"], run["start"][None], run["goal"][None], run["sxy"][None], run["sth"][None],
                 int(run["K"][0]), lanes, schedule=schedule, tol_xy=float(run["tol_xy"][0]))


def test_rrt_large_radius_arcs_blank_map(O, maps):
    """blank.png (300x300, no obstacles): long gentle arcs with radii far beyond the image exercise the deferred
    (cooperative) raster of the speculative schedule and the out-of-image border logic."""
    from theta_rrt_b200 import samples
    free = maps["blank"].copy()
    free[140:160, 40:260] = False  # one wall so that some arcs are blocked
    nq, K = 12, 601
    starts, goals = util.random_queries(free, nq, 77)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 500 + q, free.shape)
    for lanes, schedule in ((32, 0), (8, 0), (4, 1), (2, 0)):
        run_rrt_pair(O, free, starts, goals, sxy, sth, K, lanes, schedule=schedule, tol_xy=0.0)


def test_findnearest_vs_oracle(O, maps):
    from theta_rrt_b200 import samples
    free = maps["map1"]
    nq, K = 16, 301
    starts, goals = util.random_queries(free, nq, 99)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 100 + q, free.shape)
    p = planner_for(free, tol_xy=0.0)
    res = p.rrt(starts, goals, sxy, sth, K=K, logs=True)
    best, dist = p.findnearest(res, goals)
    h = res.host(); best = best.cpu().numpy(); dist = dist.cpu().numpy()
    for q in range(nq):
        n = int(h["n_nodes"][q])
        sel = h["it_new"][q] >= 0
        b, d = O.findnearest(h["node_x"][q, :n], h["node_y"][q, :n], h["node_theta"][q, :n], h["it_near"][q][sel],
                             h["it_new"][q][sel], ((goals[q, 0], goals[q, 1]), goals[q, 2]))
        assert best[q] == b, q
        if b >= 0:
            assert abs(dist[q] - d) <= 1e-12 * max(1.0, abs(d)), q


def test_cfg5_mixed_maps_rrt_and_theta(O):
    """BASELINE cfg 5 in small: RRT and Theta* queries over several random synthetic 256x256 maps (4x4-block
    Bernoulli obstacles, p = 0.15), each query bound to its map through map_id -- bitwise vs the oracle."""
    from theta_rrt_b200 import OccupancyGrid, Params, Planner, samples
    from oracle.c_oracle import Params as OP
    n_maps, side = 3, 256
    free = np.stack([util.synthetic_map(side, 0.15, 4, 7 + m) for m in range(n_maps)])
    p = Planner(OccupancyGrid(free), Params(tol_xy=0.0))
    rng = np.random.default_rng(55)
    nq, K = 18, 401
    mid = rng.integers(0, n_maps, nq).astype(np.int32)
    starts = np.empty((nq, 3)); goals = np.empty((nq, 3))
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        s, g = util.random_queries(free[mid[q]], 1, 1000 + q)
        starts[q], goals[q] = s[0], g[0]
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 2000 + q, (side, side))
    for lanes, schedule in ((32, 0), (8, 1)):
        res = p.rrt(starts, goals, sxy, sth, K=K, logs=True, map_id=mid, lanes=lanes, schedule=schedule).host()
        for q in range(nq):
            o = O.rrt(free[mid[q]], ((starts[q, 0], starts[q, 1]), starts[q, 2]), ((goals[q, 0], goals[q, 1]), goals[q, 2]),
                      sxy[q], sth[q], OP(tol_xy=0.0), K=K)
            n = o["n_nodes"]
            assert int(res["n_nodes"][q]) == n and int(res["status"][q]) == o["status"], (q, lanes)
            assert np.array_equal(res["parent"][q, :n], o["parent"]) and np.array_equal(res["it_near"][q], o["it_near"]), (q, lanes)
            assert bits_equal(res["node_x"][q, :n], o["x"]) and bits_equal(res["node_theta"][q, :n], o["theta"]), (q, lanes)
    # Theta* on the same maps (unreachable goals allowed -> status)
    nt = 60
    tm = rng.integers(0, n_maps, nt).astype(np.int32)
    sg = np.empty((nt, 4), np.int32)
    for q in range(nt):
        cells = np.argwhere(free[tm[q]])
        a, b = cells[rng.integers(len(cells), size=2)]
        sg[q] = (a[1], a[0], b[1], b[0])
    r = p.theta(sg, map_id=tm, path_cap=4096).host()
    for q in range(nt):
        o = O.astar(free[tm[q]], sg[q, :2], sg[q, 2:], log_los=False)
        assert int(r["status"][q]) == o["status"], q
        if o["status"] == 0:
            n = int(r["path_len"][q])
            assert [tuple(v) for v in r["path"][q, :n].tolist()] == o["path"] and r["cost"][q] == o["cost"], q
            assert int(r["expanded"][q]) == o["expanded"] and int(r["n_los"][q]) == o["n_los"], q


def test_rrt_edge_cases(O, maps):
    """Degenerate sizes and starts the reference accepts: K = 1 (no iteration), K = 2, an empty batch, a start inside
    an obstacle (the reference never tests the start), start == goal (found at the first accepted node or never)."""
    from theta_rrt_b200 import samples
    from oracle.c_oracle import Params as OP
    free = maps["map1"]
    blocked = np.argwhere(~free)[0]
    starts = np.array([[5.0, 5.0, 0.0], [float(blocked[1]), float(blocked[0]), 90.0], [50.0, 20.0, -180.0]])
    goals = np.array([[90.0, 50.0, 90.0], [10.0, 10.0, 0.0], [50.0, 20.0, 180.0]])
    for K in (1, 2, 3, 40):
        nq = len(starts)
        sxy = np.empty((nq, max(K - 1, 0), 2), np.int32); sth = np.empty((nq, max(K - 1, 0)))
        for q in range(nq):
            sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 9 + q, free.shape)
        for lanes, schedule in ((32, 0), (4, 0), (8, 1), (2, 0)):
            p = planner_for(free)
            res = p.rrt(starts, goals, sxy, sth, K=K, logs=True, lanes=lanes, schedule=schedule).host()
            for q in range(nq):
                o = O.rrt(free, ((starts[q, 0], starts[q, 1]), starts[q, 2]), ((goals[q, 0], goals[q, 1]), goals[q, 2]),
                          sxy[q], sth[q], OP(), K=K)
                n = o["n_nodes"]
                tag = (K, q, lanes, schedule)
                assert int(res["n_nodes"][q]) == n and int(res["sol"][q]) == o["sol"] and int(res["status"][q]) == o["status"], tag
                assert int(res["iters"][q]) == o["iters"], tag
                assert np.array_equal(res["parent"][q, :n], o["parent"]), tag
                assert bits_equal(res["node_x"][q, :n], o["x"]) and bits_equal(res["node_theta"][q, :n], o["theta"]), tag
    p = planner_for(free)
    empty = p.rrt(np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 9, 2), np.int32), np.zeros((0, 9)), K=10)
    assert empty.n_nodes.numel() == 0
    assert p.theta(np.zeros((0, 4), np.int32)).path_len.numel() == 0


def test_rrt_host_pipeline_equals_resident(maps):
    """Planner.rrt_host (chunked, side streams, pinned buffers) returns exactly what the resident call returns."""
    import torch
    from theta_rrt_b200 import samples
    free = maps["map1"]
    nq, K = 37, 301
    starts, goals = util.random_queries(free, nq, 4321)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 70 + q, free.shape)
    p = planner_for(free, tol_xy=0.0)
    ref = p.rrt(starts, goals, sxy, sth, K=K).host()
    ins = [torch.from_numpy(a).pin_memory() for a in (starts, goals, sxy, sth)]
    for chunks in (1, 5):
        out = {"node_x": torch.zeros((nq, K), dtype=torch.float64).pin_memory(), "parent": torch.zeros((nq, K), dtype=torch.int32).pin_memory(),
               "n_nodes": torch.zeros(nq, dtype=torch.int32).pin_memory(), "u": torch.zeros((nq, K, 5), dtype=torch.float64).pin_memory()}
        for _ in range(2):  # second call reuses the cached device buffers
            p.rrt_host(*ins, out=out, K=K, chunks=chunks)
            torch.cuda.synchronize()
        for t in out.values():
            t.zero_()
        for _ in range(3):  # streamed batches: nothing waits until host_sync()
            p.rrt_host(*ins, out=out, K=K, chunks=chunks, wait=False)
        p.host_sync()
        torch.cuda.synchronize()
        assert np.array_equal(out["n_nodes"].numpy(), ref["n_nodes"])
        for q in range(nq):
            n = int(ref["n_nodes"][q])
            assert np.array_equal(out["parent"].numpy()[q, :n], ref["parent"][q, :n])
            assert bits_equal(out["node_x"].numpy()[q, :n], ref["node_x"][q, :n])
            assert np.array_equal(out["u"].numpy()[q, 1:n].view(np.int64), ref["u"][q, 1:n].view(np.int64))


def test_rrt_host_valid_rows_only(maps):
    """rrt_host(valid_rows_only=True): the rows that exist arrive packed, bit-identical to the resident result, at
    row_start[q] of the flat host arrays; nothing else is touched."""
    import torch
    from theta_rrt_b200 import samples
    free = maps["map1"]
    nq, K = 41, 401
    starts, goals = util.random_queries(free, nq, 987)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 170 + q, free.shape)
    p = planner_for(free, tol_xy=0.0)
    ref = p.rrt(starts, goals, sxy, sth, K=K).host()
    ins = [torch.from_numpy(a).pin_memory() for a in (starts, goals, sxy, sth)]
    SENT = -12345.5
    for chunks in (1, 6):
        out = {"node_x": torch.full((nq, K), SENT, dtype=torch.float64).pin_memory(),
               "node_y": torch.full((nq, K), SENT, dtype=torch.float64).pin_memory(),
               "node_theta": torch.full((nq, K), SENT, dtype=torch.float64).pin_memory(),
               "parent": torch.full((nq, K), -777, dtype=torch.int32).pin_memory(),
               "u": torch.full((nq, K, 5), SENT, dtype=torch.float64).pin_memory(),
               "n_nodes": torch.zeros(nq, dtype=torch.int32).pin_memory(), "status": torch.zeros(nq, dtype=torch.int32).pin_memory(),
               "row_start": torch.full((nq,), -1, dtype=torch.int64).pin_memory()}
        for _ in range(3):  # three streamed batches: both device result sets of every piece are used
            p.rrt_host(*ins, out=out, K=K, chunks=chunks, wait=False, valid_rows_only=True)
        p.host_sync()
        torch.cuda.synchronize()
        assert np.array_equal(out["n_nodes"].numpy(), ref["n_nodes"]) and np.array_equal(out["status"].numpy(), ref["status"])
        rs = out["row_start"].numpy()
        touched = np.zeros(nq * K, bool)
        flat = {k: out[k].numpy().reshape(nq * K, -1) for k in ("node_x", "node_y", "node_theta", "parent", "u")}
        for q in range(nq):
            n = int(ref["n_nodes"][q])
            c = next(c for c in range(chunks) if nq * c // chunks <= q < nq * (c + 1) // chunks)
            lo = nq * c // chunks
            hi = nq * (c + 1) // chunks
            # inside the block of its piece (queries land in completion order), which is filled without gaps
            assert lo * K <= rs[q] and rs[q] + n <= lo * K + int(ref["n_nodes"][lo:hi].sum()), q
            rows = slice(int(rs[q]), int(rs[q]) + n)
            assert not touched[rows].any(), q  # no two trees overlap
            touched[rows] = True
            for k in ("node_x", "node_y", "node_theta"):
                assert bits_equal(flat[k][rows, 0], ref[k][q, :n]), (k, q)
            assert np.array_equal(flat["parent"][rows, 0], ref["parent"][q, :n])
            assert np.array_equal(flat["u"][rows][1:].view(np.int64), ref["u"][q, 1:n].view(np.int64))
        assert touched.sum() == int(ref["n_nodes"].sum()) < nq * K
        for k in ("node_x", "node_y", "node_theta", "u"):
            assert (flat[k][~touched] == SENT).all(), k
        assert (flat["parent"][~touched] == -777).all()
    # `u` is opt-in: without it neither the copy nor the kernel's u rows exist
    out2 = {k: v for k, v in out.items() if k != "u"}
    for t in out2.values():
        t.zero_()
    p.rrt_host(*ins, out=out2, K=K, chunks=3, valid_rows_only=True)
    torch.cuda.synchronize()
    rs = out2["row_start"].numpy()
    for q in range(nq):
        n = int(ref["n_nodes"][q])
        assert np.array_equal(out2["parent"].numpy().reshape(-1)[rs[q]:rs[q] + n], ref["parent"][q, :n])
    # resident packed result of Planner.rrt
    r = p.rrt(starts, goals, sxy, sth, K=K, pack=True).host()
    assert int(r["pack_total"][0]) == int(ref["n_nodes"].sum())
    for q in range(nq):
        n, r0 = int(ref["n_nodes"][q]), int(r["row_start"][q])
        assert bits_equal(r["pack_x"][r0:r0 + n], ref["node_x"][q, :n]) and np.array_equal(r["pack_parent"][r0:r0 + n], ref["parent"][q, :n])
        assert np.array_equal(r["pack_u"][r0 + 1:r0 + n].view(np.int64), ref["u"][q, 1:n].view(np.int64))
    with pytest.raises(ValueError):
        bad = dict(out); bad["node_x"] = torch.zeros((nq, K), dtype=torch.float64)  # not pinned
        p.rrt_host(*ins, out=bad, K=K, chunks=2, valid_rows_only=True)


# ------------------------------------------------------------------ BASELINE full sizes: properties + exact subsets
def test_cfg4_full_size_nearest_and_raycast(O):
    """BASELINE cfg 4 at full size: 8192 x 8192 grid, 2^20-node tree, 4096 nearest queries, 2^20 rays.
    Nearest: exact against numpy's first-minimum argmin of the same unfused fp64 expression for 128 of the queries,
    and for ALL queries the reported d2 equals the recomputed one and no sampled node is nearer.
    Rays: exact against the oracle on a 10^4 subset, and symmetric (search.py:47-56 canonicalises) on all 2^20."""
    import bench
    rng = np.random.default_rng(3)
    n_nodes, nq = 1 << 20, 4096
    x, y = rng.uniform(0, 8191, n_nodes), rng.uniform(0, 8191, n_nodes)
    x[777] = x[123456]; y[777] = y[123456]  # an exact duplicate: the lower index must win
    qxy = rng.integers(0, 8192, size=(nq, 2)).astype(np.int32)
    qxy[0] = (int(x[123456]), int(y[123456]))
    big = bench.synthetic_map(8192, 0.1, 8, 42)
    p = planner_for(big)
    idx, d2 = p.nearest(x, y, qxy, want_d2=True)
    idx, d2 = idx.cpu().numpy(), d2.cpu().numpy()
    for q in range(128):
        dx, dy = qxy[q, 0] - x, qxy[q, 1] - y
        assert idx[q] == int(np.argmin(dx * dx + dy * dy)), q
    dx, dy = qxy[:, 0] - x[idx], qxy[:, 1] - y[idx]
    assert bits_equal(d2, dx * dx + dy * dy)
    probe = rng.integers(0, n_nodes, 4096)
    dd = (qxy[:, 0:1] - x[probe][None, :]) ** 2 + (qxy[:, 1:2] - y[probe][None, :]) ** 2
    assert (dd.min(axis=1) >= d2).all()
    seg = bench.make_segments(big, 1 << 20, 7)
    got = p.los(seg).cpu().numpy().astype(bool)
    sub = rng.integers(0, len(seg), 10000)
    assert np.array_equal(got[sub], O.lineofsight_batch(big, seg[sub], threads=4))
    assert np.array_equal(p.los(seg[:, [2, 3, 0, 1]].copy()).cpu().numpy().astype(bool), got)
    assert np.array_equal(p.los(seg, layout="rows").cpu().numpy().astype(bool), got)  # both grid layouts agree on all 2^20
    # a ray is clear iff both halves are clear when split at a pixel of the SAME raster: endpoints free is necessary
    free_end = big[seg[:, 1], seg[:, 0]] & big[seg[:, 3], seg[:, 2]]
    assert not (got & ~free_end).any()


def test_cfg3_full_depth_batch_properties(O, maps):
    """BASELINE cfg 3 depth (K = 5001) on a 512-query batch: the result is a well-formed forest, independent of the
    lane count and of repetition (persistent groups pull queries in a different order every run), and the first and
    last query of the batch equal the oracle bit for bit."""
    from theta_rrt_b200 import samples
    from oracle.c_oracle import Params as OP
    free = maps["map1"]
    nq, K = 512, 5001
    starts, goals = util.random_queries(free, nq, 1234)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, q, free.shape)
    p = planner_for(free, tol_xy=0.0)
    a = p.rrt(starts, goals, sxy, sth, K=K, lanes=32).host()
    b = p.rrt(starts, goals, sxy, sth, K=K, lanes=32).host()
    c = p.rrt(starts, goals, sxy, sth, K=K, lanes=16).host()
    for other in (b, c):
        assert np.array_equal(a["n_nodes"], other["n_nodes"]) and np.array_equal(a["status"], other["status"])
        assert np.array_equal(a["iters"], other["iters"])
    for q in range(nq):
        n = int(a["n_nodes"][q])
        assert 1 <= n <= K and a["parent"][q, 0] == -1
        par = a["parent"][q, 1:n]
        assert (par >= 0).all() and (par < n).all()
        for other in (b, c):
            assert np.array_equal(a["parent"][q, :n], other["parent"][q, :n]), q
            assert bits_equal(a["node_x"][q, :n], other["node_x"][q, :n]) and bits_equal(a["node_theta"][q, :n], other["node_theta"][q, :n]), q
    for q in (0, nq - 1):
        o = O.rrt(free, ((starts[q, 0], starts[q, 1]), starts[q, 2]), ((goals[q, 0], goals[q, 1]), goals[q, 2]), sxy[q], sth[q],
                  OP(tol_xy=0.0), K=K)
        n = o["n_nodes"]
        assert int(a["n_nodes"][q]) == n and np.array_equal(a["parent"][q, :n], o["parent"]) and bits_equal(a["node_x"][q, :n], o["x"])


@pytest.mark.parametrize("ps", [
    dict(bikelength=3, LEFTCONSTRAINT=-40, RIGHTCONSTRAINT=40, frontclearance=1.5, maxdrivedist=12, weightxy=0.3, tol_ang=20),
    dict(FORWARDONLY=False, bikelength=7, LEFTCONSTRAINT=-30, RIGHTCONSTRAINT=55, maxdrivedist=45, weightxy=0.9),
    dict(tol_xy=25.0, tol_ang=90.0),  # generous goal test: most queries end with a solution
], ids=["short-bike", "reverse-allowed", "easy-goal"])
def test_rrt_other_parameters_bitwise_vs_oracle(O, maps, ps):
    """builtins.* parameters away from the defaults (main.py:15-32), both schedules, bitwise vs the oracle."""
    from theta_rrt_b200 import samples
    free = maps["map1"]
    nq, K = 24, 601
    starts, goals = util.random_queries(free, nq, 2024)
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 300 + q, free.shape)
    params = dict(tol_xy=0.0)
    params.update(ps)
    for lanes, schedule in ((32, 0), (8, 0), (16, 1), (2, 0)):
        res = run_rrt_pair(O, free, starts, goals, sxy, sth, K, lanes, schedule=schedule, **params)
    if "tol_xy" in ps:
        assert (res["status"] == 0).sum() > 0 and (res["sol"] >= 0).sum() == (res["status"] == 0).sum()
