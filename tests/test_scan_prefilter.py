"""The packed-fp32 prefilter of the fused RRT kernel's pooled nearest scan (`nearest_staged`, trrt_rrt.cuh).

CPU: a numpy model of the kernel's f32x2 arithmetic checks the error bound |F - D| <= SCAN_REL * F + SCAN_ABS * M^2 that the
candidate blocks rest on, on random and adversarial pairs, and a model of the whole procedure (tiles, block minima,
candidate list, blocks rescanned at admission when the list is full, fp64 recheck) returns numpy's first-minimum argmin of
the fp64 d2.
GPU: workloads that stress the filter, bit for bit against the C oracle."""
import os
import re

import numpy as np
import pytest

from tests import util
from tests.util import O, bits_equal  # noqa: F401  (O is a fixture)

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "theta_rrt_b200", "csrc", "trrt_rrt.cuh")


def kernel_constants():
    s = open(SRC).read()
    blk = int(re.search(r"SCAN_BLOCK = (\d+)", s).group(1))
    lst = int(re.search(r"SCAN_LIST = (\d+)", s).group(1))
    rel = float.fromhex(re.search(r"SCAN_REL = (0x1p-\d+)f", s).group(1))
    ab = float.fromhex(re.search(r"SCAN_ABS = (0x1p-\d+)f", s).group(1))
    mx = float.fromhex(re.search(r"SCAN_FP32_MAX = (0x1p\d+)f", s).group(1))
    return blk, lst, rel, ab, mx


BLOCK, LIST, REL, ABS, FP32_MAX = kernel_constants()
TILE = 64  # nodes per staged tile (2 * TILE_PAIRS)
f32 = np.float32


def up32(v):
    """Smallest fp32 >= v (v float64)."""
    r = v.astype(f32)
    return np.where(r.astype(np.float64) < v, np.nextafter(r, f32(np.inf)), r)


def down32(v):
    r = v.astype(f32)
    return np.where(r.astype(np.float64) > v, np.nextafter(r, f32(-np.inf)), r)


def fp64_d2(nx, ny, qx, qy):
    """The kernel's D = rn(rn(dx*dx) + rn(dy*dy)), dx = rn(qx - x)."""
    dx = qx - nx
    dy = qy - ny
    return dx * dx + dy * dy


def fp32_d2(fx, fy, sx, sy):
    """F of the f32x2 sequence: dx = rn(sx - fx), dy = rn(sy - fy), F = rn(fma(dy, dy, rn(dx*dx))).  The fma is computed
    as the float64 sum of the exact dy*dy (48 bits) and rn(dx*dx), rounded to fp32: that can differ from the fused result by
    double rounding, but only to an adjacent fp32 value, so the three candidates (r - ulp, r, r + ulp) are returned and each
    must satisfy the bound.  The unfused variant rn(rn(dy*dy) + rn(dx*dx)) is returned too."""
    dx = (sx - fx).astype(f32)
    dy = (sy - fy).astype(f32)
    p = (dx * dx).astype(f32)
    r = (dy.astype(np.float64) ** 2 + p.astype(np.float64)).astype(f32)
    unf = ((dy * dy).astype(f32) + p).astype(f32)
    return np.stack([np.nextafter(r, f32(-np.inf)), r, np.nextafter(r, f32(np.inf)), unf])


def convert(nx, ny, ox, oy):
    return (nx - ox).astype(f32), (ny - oy).astype(f32)


def check_bound(nx, ny, qx, qy, ox, oy):
    """Every (sample, node) pair given row-wise: nodes nx/ny [S, N], samples qx/qy [S, 1].  M is taken over the row (a row
    stands for one tile: M over a larger set only makes the bound looser)."""
    fx, fy = convert(nx, ny, ox, oy)
    M = np.maximum(np.abs(fx), np.abs(fy)).max(axis=1, keepdims=True)
    assert (M <= FP32_MAX).all()
    c = up32(up32(M.astype(np.float64) ** 2) * ABS)
    sx, sy = f32(qx - ox), f32(qy - oy)
    assert np.array_equal(sx.astype(np.float64), qx - ox)
    D = fp64_d2(nx, ny, qx, qy)
    worst = 0.0
    for F in fp32_d2(fx, fy, sx, sy):
        F = F.astype(np.float64)
        lb = down32(F * (1 - REL) - c)
        ub = up32(F * (1 + REL) + c)
        assert (D >= lb).all() and (D <= ub).all()
        worst = max(worst, float((np.abs(F - D) / (F * REL + c)).max()))
    return worst


@pytest.mark.parametrize("side", [100, 256, 2048])
def test_bound_random_pairs(side):
    """Millions of random pairs: nodes anywhere on the map and its apron, samples on integer pixels."""
    rng = np.random.default_rng(side)
    o = side // 2
    S, N = 2048, 512
    qx = rng.integers(0, side, (S, 1)).astype(np.float64)
    qy = rng.integers(0, side, (S, 1)).astype(np.float64)
    nx = rng.uniform(-20, side + 20, (S, N))
    ny = rng.uniform(-20, side + 20, (S, N))
    # a third of the nodes close to the sample: small distances are where the relative part of the bound matters
    k = N // 3
    nx[:, :k] = qx + rng.normal(0, 2, (S, k))
    ny[:, :k] = qy + rng.normal(0, 2, (S, k))
    assert check_bound(nx, ny, qx, qy, o, o) < 1.0


@pytest.mark.parametrize("side", [256, 2048])
def test_bound_adversarial_pairs(side):
    rng = np.random.default_rng(7 + side)
    o = side // 2
    S = 4096
    qx = rng.integers(0, side, (S, 1)).astype(np.float64)
    qy = rng.integers(0, side, (S, 1)).astype(np.float64)
    cols = []
    # near-ties a few ulps apart, around distances from 1e-6 to the map size
    d = np.exp(rng.uniform(np.log(1e-6), np.log(side), (S, 1)))
    a = rng.uniform(0, 2 * np.pi, (S, 1))
    bx, by = qx + d * np.cos(a), qy + d * np.sin(a)
    for k in range(-3, 4):
        cols.append((bx + k * np.spacing(bx), by - k * np.spacing(by)))
    # the same point reached along two arcs: duplicates and one-ulp neighbours
    cols.append((bx.copy(), by.copy()))
    cols.append((np.nextafter(bx, np.inf), np.nextafter(by, -np.inf)))
    # exactly on the sample, on integer pixels, at the apron and far outside the map
    cols.append((qx.copy(), qy.copy()))
    cols.append((qx + 1.0, qy - 1.0))
    cols.append((np.full_like(qx, -0.5), np.full_like(qy, side - 0.5)))
    cols.append((np.full_like(qx, -3.0 * side), np.full_like(qy, 4.0 * side)))
    cols.append((np.full_like(qx, o + FP32_MAX), np.full_like(qy, o - FP32_MAX)))
    nx = np.concatenate([c[0] for c in cols], axis=1)
    ny = np.concatenate([c[1] for c in cols], axis=1)
    assert check_bound(nx, ny, qx, qy, o, o) < 1.0


def prefilter_argmin(nx, ny, qx, qy, ox, oy, stats=None):
    """The kernel's procedure for one sample over nodes [0, n) (an aligned slice): tiles of 64 nodes converted to fp32,
    block minima, the candidate list of LIST entries (a block admitted to a full list is rescanned in fp64 at once), the
    fp64 rescan of the live entries in slot order, the odd last node in fp64; every fp64 node is folded by (d2, index).
    Returns the index of the first minimum of the fp64 d2."""
    n = len(nx)
    pairs = n // 2
    D = fp64_d2(nx, ny, qx, qy)
    sx, sy = qx - ox, qy - oy
    all64 = not (abs(sx) <= 2.0 ** 24 and abs(sy) <= 2.0 ** 24)
    wide = False
    U = np.float32(np.inf)
    cl = [np.float32(np.inf)] * LIST
    cb = [0] * LIST
    bd, bi = np.inf, 1 << 31

    def scan(j0, j1):
        nonlocal bd, bi
        for j in range(j0, j1):
            if D[j] < bd or (D[j] == bd and j < bi):
                bd, bi = D[j], j

    def settle(b):
        scan(b * BLOCK, min((b + 1) * BLOCK, 2 * pairs))

    for t0 in range(0, 2 * pairs, TILE):
        t1 = min(t0 + TILE, 2 * pairs)
        fx, fy = convert(nx[t0:t1], ny[t0:t1], ox, oy)
        with np.errstate(invalid="ignore"):
            M = np.float32(np.max(np.maximum(np.abs(fx), np.abs(fy))))
        if not (M <= FP32_MAX):
            wide = True
        if wide:
            continue
        c = up32(up32(np.array([float(M) ** 2])) * ABS)[0]
        F = fp32_d2(fx, fy, f32(sx), f32(sy))[1]
        for b0 in range(t0, t1, BLOCK):
            m = np.float32(F[b0 - t0:min(b0 + BLOCK, t1) - t0].min())
            lb = down32(np.array([float(m) * (1 - REL) - float(c)]))[0]
            ub = up32(np.array([float(m) * (1 + REL) + float(c)]))[0]
            U = min(U, ub)
            if stats is not None:
                stats["blocks"] += 1
            if lb <= U:
                for s in range(LIST):
                    if not (cl[s] <= U):
                        cl[s], cb[s] = lb, b0 // BLOCK
                        break
                else:
                    if not all64:
                        settle(b0 // BLOCK)
                        if stats is not None:
                            stats["settled"] += 1
    if all64 or wide:
        scan(0, 2 * pairs)
        if stats is not None:
            stats["fallback"] += 1
    elif pairs > 0:
        for s in range(LIST):
            if cl[s] <= U:
                settle(cb[s])
                if stats is not None:
                    stats["rechecked"] += 1
    scan(2 * pairs, n)
    return bi


def first_argmin(nx, ny, qx, qy):
    return int(np.argmin(fp64_d2(nx, ny, qx, qy)))


def test_procedure_random_trees():
    rng = np.random.default_rng(3)
    stats = dict(blocks=0, rechecked=0, settled=0, fallback=0)
    for side in (100, 256, 2048):
        o = side // 2
        for trial in range(60):
            n = int(rng.integers(1, 700))
            nx = rng.uniform(0, side, n)
            ny = rng.uniform(0, side, n)
            qx, qy = float(rng.integers(0, side)), float(rng.integers(0, side))
            assert prefilter_argmin(nx, ny, qx, qy, o, o, stats) == first_argmin(nx, ny, qx, qy)
    assert stats["rechecked"] > 0


def test_procedure_ties_duplicates_and_overflow():
    """Exact duplicates in different blocks (the first must win), nodes a few ulps apart, a ring of equidistant nodes that
    fills the candidate list (blocks rescanned at admission), far-away nodes (fp64 tiles) and samples off the fp32 range
    (whole slice in fp64)."""
    rng = np.random.default_rng(11)
    stats = dict(blocks=0, rechecked=0, settled=0, fallback=0)
    o = 128
    for trial in range(200):
        n = int(rng.integers(2, 600))
        qx, qy = float(rng.integers(0, 256)), float(rng.integers(0, 256))
        nx = rng.uniform(0, 256, n)
        ny = rng.uniform(0, 256, n)
        kind = trial % 5
        if kind == 0:  # the same nearest point several times, in different blocks
            idx = rng.choice(n, size=min(n, 4), replace=False)
            nx[idx], ny[idx] = qx + 0.3, qy - 0.7
        elif kind == 1:  # a few ulps apart
            idx = rng.choice(n, size=min(n, 6), replace=False)
            nx[idx] = qx + 0.25 + np.arange(len(idx)) * np.spacing(qx + 0.25) * rng.choice([-1, 1], len(idx))
            ny[idx] = qy
        elif kind == 2:  # ring: every block holds a node at the same distance -> the list overflows
            a = rng.uniform(0, 2 * np.pi, n)
            nx, ny = qx + 5 * np.cos(a), qy + 5 * np.sin(a)
            nx[::7], ny[::7] = qx + 5.0, qy
        elif kind == 3:  # a tile beyond the fp32 range
            nx[rng.integers(n)] = 3.0 * FP32_MAX
        else:  # sample beyond the exact fp32 range (the kernel's samples are any int32)
            qx = 2.0 ** 25 + 1
        assert prefilter_argmin(nx, ny, qx, qy, o, o, stats) == first_argmin(nx, ny, qx, qy), (trial, kind)
    assert stats["fallback"] > 0 and stats["settled"] > 0 and stats["rechecked"] > 0


# ------------------------------------------------------------------ GPU, bit for bit against the C oracle
def streams(free, nq, K, seed):
    from theta_rrt_b200 import samples
    starts, goals = util.random_queries(free, nq, seed)
    sxy, sth = samples.make_streams(goals, K - 1, np.arange(nq), free.shape)
    return starts, goals, sxy, sth


def run_vs_oracle(O, free, starts, goals, sxy, sth, K, reps=1, check=None):
    """Runs the batch `reps` times over (enough queries to give the pooled scan several trees per CTA), compares the
    queries listed in `check` (default: all) with the oracle, and every repetition with the first."""
    from oracle.c_oracle import Params as OP
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    nq = len(starts)
    s2, g2, x2, t2 = (np.concatenate([a] * reps) for a in (starts, goals, sxy, sth))
    res = Planner(OccupancyGrid(free), Params(tol_xy=0.0)).rrt(s2, g2, x2, t2, K=K, logs=True, counters=True, lanes=32,
                                                              schedule=0).host()
    assert (res["counters"][:, 8] == 0).all()  # tie audit
    for q in (range(nq) if check is None else check):
        o = O.rrt(free, ((starts[q, 0], starts[q, 1]), starts[q, 2]), ((goals[q, 0], goals[q, 1]), goals[q, 2]),
                  sxy[q], sth[q], OP(tol_xy=0.0), K=K)
        n = o["n_nodes"]
        assert int(res["status"][q]) == o["status"] and int(res["n_nodes"][q]) == n and int(res["iters"][q]) == o["iters"], q
        assert np.array_equal(res["it_near"][q], o["it_near"]), q
        assert np.array_equal(res["it_code"][q], o["it_code"]) and np.array_equal(res["it_new"][q], o["it_new"]), q
        assert np.array_equal(res["parent"][q, :n], o["parent"]), q
        assert bits_equal(res["node_x"][q, :n], o["x"]) and bits_equal(res["node_y"][q, :n], o["y"]), q
        assert bits_equal(res["node_theta"][q, :n], o["theta"]), q
    for r in range(1, reps):
        for k in ("n_nodes", "status", "iters", "it_near"):
            assert np.array_equal(res[k][r * nq:(r + 1) * nq], res[k][:nq]), (k, r)
        for q in range(nq):  # rows beyond n_nodes are not written
            n = int(res["n_nodes"][q])
            assert np.array_equal(res["parent"][r * nq + q, :n], res["parent"][q, :n]), (q, r)


@pytest.mark.gpu
def test_gpu_large_map(O):
    """2048-pixel synthetic map: the largest |coordinate| of a tile and with it the bound's absolute term grow with the map."""
    free = util.synthetic_map(2048, 0.15, 16, 5)
    K = 2001
    starts, goals, sxy, sth = streams(free, 48, K, 21)
    run_vs_oracle(O, free, starts, goals, sxy, sth, K, reps=4)


@pytest.mark.gpu
def test_gpu_small_open_map_long_k(O):
    """An open 64-pixel map and K = 5001: the trees fill with near-coincident nodes, many blocks tie within the bound."""
    free = np.ones((64, 64), bool)
    K = 5001
    starts, goals, sxy, sth = streams(free, 24, K, 4)
    run_vs_oracle(O, free, starts, goals, sxy, sth, K, reps=8)


@pytest.mark.gpu
def test_gpu_cfg3_subset(O, maps):
    """The headline shape: map1, K = 5001, a batch of 32 distinct bench queries repeated to fill the GPU."""
    import bench
    free = maps["map1"]
    K = 5001
    starts, goals, sxy, sth = bench.make_rrt_workload(free, 32, K, first_query=2000)
    run_vs_oracle(O, free, starts, goals, sxy, sth, K, reps=32)
