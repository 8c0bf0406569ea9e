"""Seeded normal streams of reference parity drawn on the device: numpy's legacy RandomState(seed).standard_normal(n)
bit for bit (trrt_rng.cuh, Planner.legacy_normals / rand_conf, seed_stream="device").

CPU: a pure-Python model of the legacy generator, the sequential C restatement (oracle/legacy_normals.c) and the
double-double log of trrt_libm.h against numpy, glibc and decimal.  GPU: the device path against numpy on the same box.
"""
import ctypes as C
import math
from decimal import Decimal, getcontext

import numpy as np
import pytest

from oracle import legacy_normals as L

TL_LOG_EPS = 2.0 ** -66
TL_LOG_MARGIN = 2.0 ** -5
EDGE_SEEDS = [0, 1, 2, 7, 1234, 2 ** 31 - 1, 2 ** 31, 2 ** 31 + 5, 2 ** 32 - 2, 2 ** 32 - 1]


# ------------------------------------------------------------------------------------------- Python model
def init_genrand(s):
    mt = [0] * 624
    mt[0] = s & 0xffffffff
    for i in range(1, 624):
        mt[i] = (1812433253 * (mt[i - 1] ^ (mt[i - 1] >> 30)) + i) & 0xffffffff
    return mt


class MT:
    def __init__(self, seed):
        self.mt = init_genrand(seed)
        self.i = 624

    def twist(self):
        mt = self.mt
        for k in range(624):
            y = (mt[k] & 0x80000000) | (mt[(k + 1) % 624] & 0x7fffffff)
            mt[k] = mt[(k + 397) % 624] ^ (y >> 1) ^ (0x9908b0df if y & 1 else 0)
        self.i = 0

    def u32(self):
        if self.i >= 624:
            self.twist()
        y = self.mt[self.i]
        self.i += 1
        y ^= y >> 11
        y ^= (y << 7) & 0x9d2c5680
        y ^= (y << 15) & 0xefc60000
        y ^= y >> 18
        return y

    def dbl(self):
        a = self.u32() >> 5
        b = self.u32() >> 6
        return (a * 67108864.0 + b) / 9007199254740992.0


def gauss(m, n):
    out = []
    while len(out) < n:
        while True:
            x1 = 2.0 * m.dbl() - 1.0
            x2 = 2.0 * m.dbl() - 1.0
            r2 = x1 * x1 + x2 * x2
            if r2 < 1.0 and r2 != 0.0:
                break
        f = math.sqrt(-2.0 * math.log(r2) / r2)
        out.append(f * x2)
        out.append(f * x1)
    return out[:n]


def numpy_normals(seed, n):
    return np.random.RandomState(seed).standard_normal(n)


def bits(a):
    return np.asarray(a, np.float64).view(np.int64)


def polar_r2(n, seed=0):
    """r2 values of the polar method (accepted candidates) from the Python model's generator."""
    m, out = MT(seed), []
    while len(out) < n:
        x1, x2 = 2.0 * m.dbl() - 1.0, 2.0 * m.dbl() - 1.0
        r2 = x1 * x1 + x2 * x2
        if r2 < 1.0 and r2 != 0.0:
            out.append(r2)
    return np.array(out)


@pytest.mark.parametrize("seed", [0, 1, 7, 1234, 2 ** 31 + 5, 2 ** 32 - 1])
def test_python_model_matches_numpy(seed):
    assert init_genrand(seed) == [int(v) for v in np.random.RandomState(seed).get_state()[1]]
    n = 1501  # odd, and past the first twist block
    assert np.array_equal(bits(gauss(MT(seed), n)), bits(numpy_normals(seed, n)))


# ------------------------------------------------------------------------------------------- C oracle
def test_oracle_init_genrand_matches_numpy():
    for seed in EDGE_SEEDS:
        assert np.array_equal(L.init_genrand(seed), np.random.RandomState(seed).get_state()[1])


def test_oracle_matches_numpy_bitwise_and_decided_logs_match_libm():
    """300 seeds, 2.3e7 normals (1.15e7 polar r2 values): lengths 0, 1, odd ones and ones around twist-block ends."""
    special = [0, 1, 2, 3, 243, 244, 245, 246, 247, 489, 490, 491, 623, 624, 625, 1247, 1248, 1249, 15000, 14999]
    seeds = EDGE_SEEDS + list(range(100, 390))
    lengths = [special[i] if i < len(special) else 77_001 + 2 * i for i in range(len(seeds))]
    stats = np.zeros(3, np.int64)
    total = 0
    for seed, n in zip(seeds, lengths):
        got = L.standard_normal(seed, n, stats)
        assert np.array_equal(bits(got), bits(numpy_normals(seed, n))), (seed, n)
        total += n
    assert len(seeds) >= 256 and total >= 10 ** 7
    logs, undecided, decided_differ = (int(v) for v in stats)
    assert logs >= 10 ** 7
    assert decided_differ == 0
    assert 0.02 < undecided / logs < 0.12  # about 6 % of the polar r2 values lie near a rounding midpoint


# ------------------------------------------------------------------------------------------- tl_log_dd
def exact_ln(x):
    return Decimal(float(x)).ln()


def test_tl_log_dd_bound_against_decimal():
    getcontext().prec = 60
    rng = np.random.default_rng(11)
    k = np.arange(1, 1075)
    xs = np.concatenate([
        rng.random(4000),                                                # random in (0, 1)
        polar_r2(2000, seed=5),                                          # what the generator asks
        1.0 - np.arange(1, 201) * 2.0 ** -53,                            # next to 1
        1.0 - rng.random(300) * 1e-6, 1.0 - rng.random(300) * 1e-12,
        2.0 ** -104 * np.arange(1, 50), 2.0 ** -k[k <= 110],             # tiny polar r2 (x1, x2 multiples of 2^-52)
        2.0 ** -k,                                                       # powers of two, subnormals included
        np.array([5e-324, 1e-320, 2.2250738585072014e-308, 2.2250738585072009e-308]),
        0.7071067811865476 + np.arange(-20, 21) * 2.0 ** -53,            # the reduction's switch point
        0.5 + np.arange(-5, 6) * 2.0 ** -54, 0.25 * (1 + rng.random(100)),
    ])
    xs = xs[(xs > 0) & (xs < 1)]
    hi, lo, decided = L.log_dd(xs)
    worst = Decimal(0)
    for x, h, l, d in zip(xs, hi, lo, decided):
        e = exact_ln(x)
        err = abs((Decimal(float(h)) + Decimal(float(l)) - e) / e)
        worst = max(worst, err)
        if d:  # decided: hi is the correctly rounded log
            assert float(e) == h, x
    assert worst <= Decimal(TL_LOG_EPS), f"relative error 2^{math.log2(float(worst)):.2f} above the stated 2^-66"


def test_glibc_log_error_below_margin():
    """The decided test assumes glibc's log is within 0.5 + 2^-5 ulp; on the polar r2 values it is (largest seen:
    about 0.51 ulp on glibc 2.39, x86-64)."""
    getcontext().prec = 60
    r2 = polar_r2(20000, seed=17)
    worst = 0.0
    for x in r2:
        g = math.log(x)
        worst = max(worst, float(abs(Decimal(g) - exact_ln(x)) / Decimal(math.ulp(g))))
    assert worst < 0.5 + TL_LOG_MARGIN, f"glibc log error {worst:.4f} ulp reaches the margin"


# ------------------------------------------------------------------------------------------- GPU
def planner_for(free=None):
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    if free is None:
        free = np.ones((64, 64), bool)
    return Planner(OccupancyGrid(free, device="cuda:0"), Params())


def abi_draw(p, seeds, ranges, total, fix_cap):
    """trrt_legacy_normals_draw + host log + fixup through the C ABI with caller-given ranges.
    Returns (normals, undecided count)."""
    import torch
    from theta_rrt_b200 import _lib
    dev = p.device
    out = torch.full((max(total, 1),), np.nan, dtype=torch.float64, device=dev)
    s = torch.from_numpy(np.asarray(seeds, np.uint32).view(np.int32)).to(dev)
    r = torch.from_numpy(np.ascontiguousarray(ranges, np.int64)).to(dev)
    fpos = torch.empty(max(fix_cap, 1), dtype=torch.int64, device=dev)
    fr2 = torch.empty(max(fix_cap, 1), dtype=torch.float64, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    work = torch.empty(p.lib.trrt_legacy_normals_workspace_bytes(len(seeds)), dtype=torch.uint8, device=dev)
    a = _lib.CLegacyNormalsArgs(n_seeds=len(seeds), d_seeds=s.data_ptr(), d_range=r.data_ptr(), d_out=out.data_ptr(),
                                d_fix_pos=fpos.data_ptr(), d_fix_r2=fr2.data_ptr(), fix_cap=fix_cap, d_fix_count=cnt.data_ptr(),
                                d_work=work.data_ptr(), work_bytes=work.numel())
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(p.lib.trrt_legacy_normals_draw(C.byref(a), st))
    n_fix = int(cnt.cpu()[0])
    m = min(n_fix, fix_cap)
    if m:
        h = fr2[:m].cpu().numpy()
        lg = np.empty_like(h)
        _lib.check(p.lib.trrt_libm_log_batch(h.ctypes.data, lg.ctypes.data, m))
        # libm's log, the one numpy's legacy_gauss calls (np.log is numpy's own SIMD loop, which rounds differently)
        assert np.array_equal(bits(lg), bits([math.log(v) for v in h]))
        d_log = torch.from_numpy(lg).to(dev)
        _lib.check(p.lib.trrt_legacy_normals_fixup(C.byref(a), d_log.data_ptr(), m, st))
    return out.cpu().numpy(), n_fix


@pytest.mark.gpu
def test_device_cfg3_streams_bitwise():
    """4 096 seeds x 15 000 normals (the cfg-3 rand_conf streams, 5 000 samples each)."""
    p = planner_for()
    n, L_ = 4096, 15000
    seeds = np.arange(n, dtype=np.int64) * 7919 + 3
    ranges = np.stack([np.arange(n) * L_, np.arange(n) * L_ + L_], 1)
    _, n_fix = abi_draw(p, seeds, ranges, n * L_, 1)  # count only: the host-log path is exercised
    assert n_fix > 0
    out, rng = p.legacy_normals(seeds, np.full(n, L_))
    assert np.array_equal(rng.cpu().numpy(), ranges)
    h = out.cpu().numpy()
    for i, seed in enumerate(seeds):
        assert np.array_equal(bits(h[i * L_:(i + 1) * L_]), bits(numpy_normals(int(seed), L_))), seed


@pytest.mark.gpu
def test_device_edge_seeds_odd_lengths_any_order_and_retry():
    p = planner_for()
    seeds = EDGE_SEEDS * 2
    lengths = [0, 1, 2, 3, 245, 246, 491, 624, 1249, 15001, 7, 0, 999, 2, 246, 5000, 1, 313, 3, 10001]
    # ranges in a shuffled order with gaps between them: only [begin, end) of each seed is written
    order = np.random.default_rng(4).permutation(len(seeds))
    ranges = np.zeros((len(seeds), 2), np.int64)
    pos = 0
    for i in order:
        ranges[i] = (pos, pos + lengths[i])
        pos += lengths[i] + 3
    out, n_fix = abi_draw(p, seeds, ranges, pos, 1 << 16)
    assert n_fix > 0
    for i, seed in enumerate(seeds):
        assert np.array_equal(bits(out[ranges[i, 0]:ranges[i, 1]]), bits(numpy_normals(seed, lengths[i]))), (seed, lengths[i])
    gaps = np.ones(pos, bool)
    for b, e in ranges:
        gaps[b:e] = False
    assert np.isnan(out[:pos][gaps]).all()
    # a fixup list of 2 entries overflows: the planner draws once more with the reported count
    out2, rng2 = p.legacy_normals(seeds, lengths, fix_cap=2)
    h2, r2 = out2.cpu().numpy(), rng2.cpu().numpy()
    for i, seed in enumerate(seeds):
        assert np.array_equal(bits(h2[r2[i, 0]:r2[i, 1]]), bits(numpy_normals(seed, lengths[i])))
    with pytest.raises(ValueError, match="Seed must be between"):
        p.legacy_normals([2 ** 32], [4])
    with pytest.raises(ValueError, match="Seed must be between"):
        p.legacy_normals([-1], [4])
    with pytest.raises(ValueError):
        np.random.RandomState(2 ** 32)  # the error numpy raises for the same seed


@pytest.mark.gpu
@pytest.mark.parametrize("xy", ["int32", "int16"])
def test_rand_conf_matches_make_stream(maps, xy):
    import torch
    from theta_rrt_b200 import samples
    free = maps["map2"]
    p = planner_for(free)
    rng = np.random.default_rng(8)
    nq, K = 64, 301
    goals = np.stack([rng.uniform(0, 300, nq), rng.uniform(0, 300, nq), rng.uniform(-900, 900, nq)], 1)
    seeds = rng.integers(0, 2 ** 32, nq)
    sxy, sth = p.rand_conf(goals, seeds, K, xy_dtype=getattr(torch, xy))
    assert sxy.dtype == getattr(torch, xy) and sxy.shape == (nq, K - 1, 2) and sth.shape == (nq, K - 1)
    hx, ht = sxy.cpu().numpy(), sth.cpu().numpy()
    for q in range(nq):
        ex, et = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, int(seeds[q]), free.shape)
        assert np.array_equal(hx[q].astype(np.int32), ex) and np.array_equal(bits(ht[q]), bits(et)), q


@pytest.mark.gpu
def test_missions_device_seed_stream_equals_host(maps):
    from tests.test_missions import map2_queries
    free = maps["map2"]
    sg = map2_queries(free, 256, 2024)
    seeds = np.arange(256) + 9000
    p = planner_for(free)
    hh = p.missions(start_goal=sg, seeds=seeds, K=300).host()
    hd = p.missions(start_goal=sg, seeds=seeds, K=300, seed_stream="device").host()
    assert (hh["n_seg"] > 0).sum() > 200
    fields = [k for k, v in hh.items() if isinstance(v, np.ndarray)]
    assert {"begin", "solution", "nearest", "mindist", "n_nodes", "iters", "seg_status", "status", "path", "path_len"} <= set(fields)
    for k in fields:  # every MissionResult field, bit for bit (NaN payloads included); path rows up to path_len
        if k in ("path", "path_seg"):
            continue
        assert hh[k].dtype == hd[k].dtype and np.array_equal(hh[k].view(np.uint8), hd[k].view(np.uint8)), k
    assert np.array_equal(hh["path_len"], hd["path_len"])
    for m, n in enumerate(np.minimum(hh["path_len"], hh["path"].shape[1])):
        assert np.array_equal(hh["path"][m, :n].view(np.uint8), hd["path"][m, :n].view(np.uint8)), m
        assert np.array_equal(hh["path_seg"][m, :n], hd["path_seg"][m, :n]), m
    with pytest.raises(ValueError):
        p.missions(start_goal=sg[:2], seeds=seeds[:2], K=300, seed_stream="gpu")


@pytest.mark.gpu
def test_rrt_batch_device_seed_stream_equals_host(maps):
    from tests import util
    from theta_rrt_b200 import main as M
    from theta_rrt_b200 import rrt as R
    free = maps["map2"]
    M.set_map(free)
    starts, goals = util.random_queries(free, 48, 21)
    seeds = np.arange(48) * 13 + 2 ** 31
    hh = R.rrt_batch(starts, goals, seeds=seeds, K=300, logs=True).host()
    hd = R.rrt_batch(starts, goals, seeds=seeds, K=300, logs=True, seed_stream="device").host()
    for k in ("n_nodes", "sol", "status", "iters"):
        assert np.array_equal(hh[k], hd[k]), k
    for q in range(48):  # the rows that exist: n_nodes tree rows, iters log entries
        n, it = int(hh["n_nodes"][q]), int(hh["iters"][q])
        for k in ("parent", "node_x", "node_y", "node_theta", "u"):
            assert np.array_equal(hh[k][q, :n].view(np.uint8), hd[k][q, :n].view(np.uint8)), (k, q)
        for k in ("it_near", "it_new", "it_code"):
            assert np.array_equal(hh[k][q, :it], hd[k][q, :it]), (k, q)


@pytest.mark.gpu
def test_plan_batch_device_seed_stream(maps):
    from theta_rrt_b200 import main as M
    free = maps["map2"]
    host = M.plan_batch(free, [(280, 0), (280, 0)], [(8, 280), (280, 0)], seeds=[0, 1])
    dev = M.plan_batch(free, [(280, 0), (280, 0)], [(8, 280), (280, 0)], seeds=[0, 1], seed_stream="device")
    assert repr(host) == repr(dev)
