"""Seed races for RRT batches (trrt_rrt_race_batch, Planner.rrt(race=...), Planner.rrt_race, rrt.rrt_race).

A member of a race group runs no iteration it once a member of its group has found the goal with iters <= it.  The
winner of a group is the lowest query index among the members with the fewest iterations to the goal: the argmin of
full oracle runs of every member, whatever the lanes and schedule.  A member that is cut is PAUSED and holds what the
oracle plans with K = iters + 1; every other member, and every group without a winner, equals the plain call.  The CPU
tests check the host-side rejections and the key helpers (the ABI mirror of the header is checked in test_abi.py)."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from tests import util
from tests.util import O, bits_equal, planner_for  # noqa: F401  (O is a fixture)

OK_FOUND, OK_NOT_FOUND, PAUSED, NOT_RUN = 0, 1, 8, 255
COUNTERS_KEPT = [0, 1, 2, 3, 4, 5, 6, 8]  # every counter but 7 (hash probes of a rebuilt index)
RESUME_CASES = [(32, 0), (16, 0), (8, 0), (1, 0), (8, 1), (32, 1)]


def expected_winners(status, iters, groups, n_groups):
    """(winner, iters) per group from full runs of every member: the lowest query index among the members that found
    the goal in the fewest iterations; -1 where no member found it."""
    winner = np.full(n_groups, -1, np.int64)
    best = np.full(n_groups, -1, np.int64)
    for q in range(len(status)):
        g = int(groups[q])
        if status[q] != OK_FOUND or not 0 <= g < n_groups:
            continue
        if best[g] < 0 or iters[q] < best[g]:  # q ascends: the first member at the minimum is kept
            best[g], winner[g] = iters[q], q
    return winner, best


# ------------------------------------------------------------------ CPU
def test_host_rejections():
    """Rejected before any device work (these calls need no device)."""
    from theta_rrt_b200 import _lib
    lib = _lib.load()
    fake = 4096  # never dereferenced: the call returns before it touches a pointer
    race = _lib.CRrtRace(d_group=fake, n_groups=4, d_key=fake)
    assert lib.trrt_rrt_race_batch(None, C.byref(race), None) == 1
    assert lib.trrt_rrt_batch(None, None) == 1
    a = _lib.CRrtArgs(n_maps=1, H=100, W=100, n_queries=8, K=11, d_row_start=fake)
    assert lib.trrt_rrt_race_batch(C.byref(a), C.byref(race), None) == 1  # packed rows plan whole runs
    a = _lib.CRrtArgs(n_maps=1, H=100, W=100, n_queries=8, K=11)
    for bad in (_lib.CRrtRace(d_group=fake, n_groups=0, d_key=fake), _lib.CRrtRace(d_group=fake, n_groups=-3, d_key=fake),
                _lib.CRrtRace(d_group=None, n_groups=4, d_key=fake), _lib.CRrtRace(d_group=fake, n_groups=4, d_key=None)):
        assert lib.trrt_rrt_race_batch(C.byref(a), C.byref(bad), None) == 1
    a = _lib.CRrtArgs(n_maps=1, H=100, W=100, n_queries=1 << 32, K=11)
    assert lib.trrt_rrt_race_batch(C.byref(a), C.byref(race), None) == 1  # the key holds a 32-bit query index


def test_key_round_trip():
    import torch
    from theta_rrt_b200.planner import race_decode, race_key
    rng = np.random.default_rng(3)
    iters = rng.integers(1, 2 ** 31 - 1, 200)
    q = rng.integers(0, 2 ** 32 - 1, 200)
    keys = np.array([race_key(i, j) for i, j in zip(iters, q)], np.uint64)
    keys = np.concatenate([keys, [np.uint64(2 ** 64 - 1)]])
    w, it = race_decode(torch.from_numpy(keys.view(np.int64)))
    assert np.array_equal(w.numpy().view(np.uint32)[:-1], q.astype(np.uint32))
    assert np.array_equal(it.numpy()[:-1], iters) and w[-1] == -1 and it[-1] == -1
    # the packing orders by iterations first, then by query index
    assert race_key(5, 9) < race_key(6, 0) and race_key(5, 2) < race_key(5, 3)


def test_expected_winners_table():
    status = np.array([1, 0, 0, 4, 0, 0, 6, 0, 1, 0])
    iters = np.array([50, 30, 12, 9, 12, 40, 3, 7, 99, 7])
    groups = np.array([0, 0, 0, 0, 1, 1, 2, 3, 3, 3])
    w, b = expected_winners(status, iters, groups, 5)
    assert w.tolist() == [2, 4, -1, 7, -1] and b.tolist() == [12, 12, -1, 7, -1]
    w, b = expected_winners(status, iters, np.array([0, 0, 0, 0, 9, -1, 2, 3, 3, 3]), 4)  # ids outside [0, 4) race nobody
    assert w.tolist() == [2, -1, -1, 7]


# ------------------------------------------------------------------ GPU
def race_inputs(free, n_prob, S, K, seed):
    """n_prob problems x S seeds: member q = p * S + s plans problem p with the stream of seed seeds[p, s]."""
    from theta_rrt_b200 import samples
    starts, goals = util.random_queries(free, n_prob, seed)
    seeds = (np.arange(n_prob * S).reshape(n_prob, S) * 7 + seed).astype(np.int64)
    ms, mg = np.repeat(starts, S, axis=0), np.repeat(goals, S, axis=0)
    sxy, sth = samples.make_streams(mg, K - 1, seeds.reshape(-1), free.shape)
    return dict(problems=(starts, goals), seeds=seeds, inp=(ms, mg, sxy, sth), groups=np.repeat(np.arange(n_prob), S),
                K=K, free=free)


class OracleRuns:
    """Oracle runs of the members of one workload, by (query, K), computed once."""

    def __init__(self, O, w, params):
        self.O, self.w, self.op = O, w, O.Params(**params)
        ms, mg, sxy, sth = w["inp"]
        full = O.rrt_batch(w["free"], ms, mg, sxy, sth, w["K"], self.op, threads=os.cpu_count() or 1, want_nodes=False)
        self.status, self.iters = full["status"], full["iters"]
        self.cache = {}

    def run(self, qk):
        q, k = qk
        ms, mg, sxy, sth = self.w["inp"]
        return self.O.rrt(self.w["free"], ((ms[q, 0], ms[q, 1]), ms[q, 2]), ((mg[q, 0], mg[q, 1]), mg[q, 2]), sxy[q], sth[q],
                          self.op, K=k)

    def get(self, keys):
        todo = sorted(set(keys) - set(self.cache))
        with ThreadPoolExecutor(os.cpu_count() or 1) as ex:  # the oracle runs outside the GIL
            for qk, r in zip(todo, ex.map(self.run, todo)):
                self.cache[qk] = r
        return [self.cache[qk] for qk in keys]


def check_members(h, orc, groups, winner, best, K, members=None, tag=""):
    """Every member (or those listed): FOUND at its oracle solve iteration, cut members PAUSED within
    [best, K-1], the others as in their full runs; and each equal, bit for bit, to the oracle at K = iters + 1 (cut)
    or at K (otherwise)."""
    members = range(len(h["status"])) if members is None else members
    keys = []
    for q in members:
        st, it = int(h["status"][q]), int(h["iters"][q])
        g = int(groups[q])
        if st == PAUSED:
            assert winner[g] >= 0 and best[g] <= it <= K - 1, (q, it, tag)
            keys.append((q, it + 1))
        else:
            assert st == orc.status[q] and it == orc.iters[q], (q, st, it, tag)
            keys.append((q, K))
    for q, (_, k), o in zip(members, keys, orc.get(keys)):
        t = (q, k, tag)
        want = o["status"]
        if want == OK_NOT_FOUND and o["iters"] == k - 1 and k < K:
            want = PAUSED
        assert int(h["status"][q]) == want and int(h["iters"][q]) == o["iters"], t
        n = o["n_nodes"]
        assert int(h["n_nodes"][q]) == n and int(h["sol"][q]) == o["sol"], t
        for key in ("it_code", "it_near", "it_new"):
            assert np.array_equal(h[key][q, :k - 1], o[key][:k - 1]), (key, t)
        assert (h["it_code"][q, k - 1:] == NOT_RUN).all() and (h["it_near"][q, k - 1:] == -1).all(), t
        assert np.array_equal(h["parent"][q, :n], o["parent"]), t
        for key, ok in (("node_x", "x"), ("node_y", "y"), ("node_theta", "theta")):
            assert bits_equal(h[key][q, :n], o[ok]), (key, t)
        assert np.array_equal(h["u"][q, :n].view(np.int64), o["u"].view(np.int64)), t
        nl = int(h["n_los"][q])
        assert nl == o["n_los"] and np.array_equal(h["los_log"][q, :nl].astype(bool), o["los"]), t


def assert_same_run(a, b, tag, counters=COUNTERS_KEPT):
    for k in ("n_nodes", "sol", "status", "iters", "n_los", "it_near", "it_new", "it_code", "los_log"):
        assert np.array_equal(a[k], b[k]), (k, tag)
    for q in range(len(a["n_nodes"])):
        n = int(a["n_nodes"][q])
        assert np.array_equal(a["parent"][q, :n], b["parent"][q, :n]), ("parent", q, tag)
        for k in ("node_x", "node_y", "node_theta", "u"):
            assert bits_equal(a[k][q, :n], b[k][q, :n]), (k, q, tag)
    assert np.array_equal(a["counters"][:, counters], b["counters"][:, counters]), tag


@pytest.fixture(scope="module")
def race_workloads(O, maps):
    """16 problems x 64 seeds at K = 1201: map2 with the default parameters and map1 with the default tolerance."""
    K = 1201
    out = {}
    for which, seed in (("map2", 11), ("map1", 12)):
        w = race_inputs(maps[which], 16, 64, K, seed)
        orc = OracleRuns(O, w, {})
        win, best = expected_winners(orc.status, orc.iters, w["groups"], 16)
        assert (win >= 0).sum() >= 8, which  # most problems have a winner
        out[which] = (w, orc, win, best)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", RESUME_CASES)
@pytest.mark.parametrize("which", ["map2", "map1"])
def test_race_winner_and_members_equal_oracle(race_workloads, which, lanes, schedule):
    w, orc, win, best = race_workloads[which]
    p = planner_for(w["free"])
    res = p.rrt(*w["inp"], K=w["K"], logs=True, counters=True, lanes=lanes, schedule=schedule, race=w["groups"])
    h = res.host()
    assert np.array_equal(h["race_winner"], win) and np.array_equal(h["race_iters"], best), (which, lanes, schedule)
    key = h["race_key"].view(np.uint64)
    assert np.array_equal(key[win >= 0], (best[win >= 0].astype(np.uint64) << np.uint64(32)) | win[win >= 0].astype(np.uint64))
    assert (key[win < 0] == np.uint64(2 ** 64 - 1)).all()
    assert (h["status"] == PAUSED).any()
    check_members(h, orc, w["groups"], win, best, w["K"], tag=(which, lanes, schedule))


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", RESUME_CASES)
def test_no_winner_no_change(O, maps, lanes, schedule):
    """Singleton groups, ids outside [0, n_groups), and groups on map1 with tol_xy = 0 (nothing is found): the outputs of
    the plain call bit for bit, counters included."""
    import torch
    K = 601
    w2 = race_inputs(maps["map2"], 6, 8, K, 21)
    p2 = planner_for(maps["map2"])
    plain = p2.rrt(*w2["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
    assert (plain["status"] == OK_FOUND).sum() >= 4
    nq = len(plain["status"])
    single = p2.rrt(*w2["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, race=np.arange(nq)).host()
    assert_same_run(single, plain, ("singleton", lanes, schedule), counters=list(range(9)))
    found = plain["status"] == OK_FOUND
    assert np.array_equal(single["race_winner"][found], np.nonzero(found)[0]) and (single["race_winner"][~found] == -1).all()
    ids = torch.tensor(np.where(np.arange(nq) % 2 == 0, -5, 7 + np.arange(nq)), dtype=torch.int32, device="cuda")
    out = p2.rrt(*w2["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, race=ids, race_groups=3).host()
    assert_same_run(out, plain, ("out of range", lanes, schedule), counters=list(range(9)))
    assert (out["race_winner"] == -1).all() and (out["race_key"] == -1).all()
    w1 = race_inputs(maps["map1"], 4, 12, K, 22)
    p1 = planner_for(maps["map1"], tol_xy=0.0)
    plain = p1.rrt(*w1["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
    assert not (plain["status"] == OK_FOUND).any()
    raced = p1.rrt(*w1["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, race=w1["groups"]).host()
    assert_same_run(raced, plain, ("tol 0", lanes, schedule), counters=list(range(9)))
    assert (raced["race_winner"] == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", RESUME_CASES)
def test_race_then_resume(race_workloads, lanes, schedule):
    """Race to the winners, then continue every member without the race: one plain call.  A stop_at pause followed by a
    raced resume: the winners of one raced call."""
    w, orc, win, best = race_workloads["map2"]
    p = planner_for(w["free"])
    K = w["K"]
    plain = p.rrt(*w["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
    res = p.rrt(*w["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, race=w["groups"])
    key = res.race_key.clone()
    p.rrt_resume(res, lanes=lanes, schedule=schedule, race=False)
    h = res.host()
    assert_same_run(h, plain, ("resume without race", lanes, schedule))
    assert np.array_equal(h["race_key"], key.cpu().numpy())  # a plain resume leaves the keys
    res = p.rrt(*w["inp"], K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, race=w["groups"], stop_at=5)
    for stop in (40, None):
        p.rrt_resume(res, stop_at=stop, lanes=lanes, schedule=schedule)
    h = res.host()
    assert np.array_equal(h["race_winner"], win) and np.array_equal(h["race_iters"], best)
    members = range(0, len(h["status"]), 5)
    check_members(h, orc, w["groups"], win, best, K, members=members, tag=("stop, raced resume", lanes, schedule))


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", [(32, 0), (8, 1)])
def test_group_larger_than_one_wave(O, maps, lanes, schedule):
    """One group of 8 192 seeds (more warps than are resident at once): the oracle's winner, and the invariants."""
    free = maps["map2"]
    K = 161
    w = race_inputs(free, 1, 8192, K, 31)
    orc = OracleRuns(O, w, {})
    win, best = expected_winners(orc.status, orc.iters, w["groups"], 1)
    assert win[0] >= 0
    p = planner_for(free)
    h = p.rrt(*w["inp"], K=K, logs=True, lanes=lanes, schedule=schedule, race=w["groups"]).host()
    assert int(h["race_winner"][0]) == win[0] and int(h["race_iters"][0]) == best[0]
    st, it = h["status"], h["iters"]
    paused = st == PAUSED
    assert paused.any() and (it[paused] >= best[0]).all() and (it[paused] <= K - 1).all()
    assert np.array_equal(st[~paused], orc.status[~paused]) and np.array_equal(it[~paused], orc.iters[~paused])
    rng = np.random.default_rng(lanes)
    members = sorted(set(rng.choice(8192, 96, replace=False).tolist()) | {int(win[0])})
    check_members(h, orc, w["groups"], win, best, K, members=members, tag=("wave", lanes, schedule))


@pytest.mark.gpu
def test_planner_rrt_race_streams(race_workloads):
    """Planner.rrt_race with device-drawn and host-drawn streams: the winners, seeds and iters of the explicit call."""
    w, orc, win, best = race_workloads["map2"]
    p = planner_for(w["free"])
    starts, goals = w["problems"]
    for stream in ("device", "host"):
        r = p.rrt_race(starts[:4], goals[:4], w["seeds"][:4], K=w["K"], seed_stream=stream).host()
        assert np.array_equal(r["winner"], np.where(win[:4] >= 0, win[:4], -1)), stream
        assert np.array_equal(r["iters"], best[:4]), stream
        want_seed = np.where(win[:4] >= 0, w["seeds"].reshape(-1)[np.maximum(win[:4], 0)], -1)
        assert np.array_equal(r["winner_seed"], want_seed), stream


def u_equal(a, b):
    """Two cameFrom u tuples (steer, icc array or None, rad or None, dist), bit for bit."""
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        if (x is None) != (y is None):
            return False
        if x is not None and not bits_equal(np.atleast_1d(x), np.atleast_1d(y)):
            return False
    return True


@pytest.mark.gpu
def test_drop_in_rrt_race(O, maps):
    """rrt.rrt_race returns the oracle's winning seed and what rrt.rrt returns under np.random.seed(that seed)."""
    import builtins
    from theta_rrt_b200 import _context, samples
    from theta_rrt_b200 import main as M
    from theta_rrt_b200 import rrt as R
    had = hasattr(builtins, "imarray")
    old = getattr(builtins, "imarray", None)
    free = maps["map2"]
    M.set_map(free)
    try:
        K = int(_context.current_planner().params.K)
        starts, goals = util.random_queries(free, 3, 41)
        for i in range(3):
            start = ((float(starts[i, 0]), float(starts[i, 1])), float(starts[i, 2]))
            goal = ((float(goals[i, 0]), float(goals[i, 1])), float(goals[i, 2]))
            seeds = np.arange(40) * 13 + i
            seed, out = R.rrt_race(start, goal, seeds)
            st = np.array([[start[0][0], start[0][1], R.standardangle(start[1])]] * len(seeds))
            gl = np.array([[goal[0][0], goal[0][1], R.standardangle(goal[1])]] * len(seeds))
            sxy = np.empty((len(seeds), K - 1, 2), np.int32); sth = np.empty((len(seeds), K - 1))
            for q, s in enumerate(seeds):
                sxy[q], sth[q] = samples.make_stream(((gl[q, 0], gl[q, 1]), gl[q, 2]), K - 1, int(s), free.shape)
            full = O.rrt_batch(free, st, gl, sxy, sth, K, O.Params(), threads=os.cpu_count() or 1, want_nodes=False)
            wq, _ = expected_winners(full["status"], full["iters"], np.zeros(len(seeds), np.int64), 1)
            if wq[0] < 0:
                assert (seed, out) == (None, None)
                continue
            assert seed == int(seeds[wq[0]])
            np.random.seed(seed)
            sol, G, cameFrom = R.rrt(start, goal)
            assert out[0] == sol and list(out[1].keys()) == list(G.keys()) and out[1] == G
            assert list(out[2].keys()) == list(cameFrom.keys())
            for k, v in cameFrom.items():
                o = out[2][k]
                if v is None:
                    assert o is None
                    continue
                assert o[0] == v[0] and u_equal(o[1], v[1]), k
    finally:
        if had:
            builtins.imarray = old
        else:
            del builtins.imarray


@pytest.mark.gpu
def test_python_errors(maps):
    import torch
    free = maps["map1"]
    K = 51
    w = race_inputs(free, 2, 3, K, 1)
    p = planner_for(free)
    with pytest.raises(ValueError):
        p.rrt(*w["inp"], K=K, race=w["groups"], pack=True)
    with pytest.raises(ValueError):
        p.rrt(*w["inp"], K=K, race=torch.zeros(6, dtype=torch.int32, device="cuda"))  # no race_groups
    with pytest.raises(ValueError):
        p.rrt(*w["inp"], K=K, race=[0, 0, 0, -1, 1, 1])
    with pytest.raises(ValueError):
        p.rrt(*w["inp"], K=K, race=[0, 0, 1])
    with pytest.raises(ValueError):
        p.rrt_host(*w["inp"], out={"status": torch.empty(6, dtype=torch.int32)}, K=K, race=w["groups"])
    with pytest.raises(ValueError):
        p.rrt_race(w["problems"][0], w["problems"][1], w["seeds"].reshape(-1), K=K)  # seeds must be [P, S]
