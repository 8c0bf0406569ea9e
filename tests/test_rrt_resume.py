"""Pause and resume of RRT batches (trrt_rrt_args d_stop_at / resume, Planner.rrt(stop_at=...), Planner.rrt_resume).

A pause is a window boundary the caller chooses, so every sequence of pauses and resumes, under any lanes and schedule,
must return what one uninterrupted call returns, bit for bit; a query paused at stop_at[q] = k must hold what the
oracle plans with K = k + 1.  The CPU test checks the PAUSED status of the header; the ABI mirror is checked in
test_abi.py."""
import os
import re

import numpy as np
import pytest

from tests import util
from tests.util import O, bits_equal, planner_for  # noqa: F401  (O is a fixture)

PAUSED, OK_FOUND, OK_NOT_FOUND, NOT_RUN = 8, 0, 1, 255
# counter 7 (hash probes) counts probes in the index a resume rebuilds: the one counter that depends on the pauses
COUNTERS_KEPT = [0, 1, 2, 3, 4, 5, 6, 8]


# ------------------------------------------------------------------ CPU
def test_paused_status_in_header_and_names():
    from theta_rrt_b200 import planner
    src = open(os.path.join(util.ROOT, "include", "thetarrt.h")).read()
    assert re.search(r"\bTRRT_PAUSED\s*=\s*8\b", src)
    assert planner.PAUSED == PAUSED and planner.STATUS_NAMES[PAUSED] == "PAUSED"


def test_result_buffers_and_launch_state():
    """host() returns the outputs, not the launch state that rrt_resume plans with; fits() decides which buffers rrt_host
    may reuse."""
    import dataclasses
    from theta_rrt_b200.planner import RrtResult
    res = RrtResult.empty(3, 5, "cpu", want_u=True, logs=True, counters=False)
    assert res.u.shape == (3, 5, 5) and res.it_near.shape == (3, 4) and res.counters is None
    res.launch = object()
    assert set(res.host()) == {f.name for f in dataclasses.fields(RrtResult)} - {"launch"}
    assert res.fits(3, 5, True, True, False)
    for args in ((4, 5, True, True, False), (3, 6, True, True, False), (3, 5, False, True, False),
                 (3, 5, True, False, False), (3, 5, True, True, True)):
        assert not res.fits(*args), args


# ------------------------------------------------------------------ GPU
def streams(free, nq, K, query_seed, stream_seed):
    from theta_rrt_b200 import samples
    starts, goals = util.random_queries(free, nq, query_seed)
    sxy, sth = samples.make_streams(goals, K - 1, np.arange(nq) + stream_seed, free.shape)
    return starts, goals, sxy, sth


def assert_same_run(a, b, tag, counters=True):
    """Every output of two host results: valid tree rows, the full logs, the counters except hash probes."""
    for k in ("n_nodes", "sol", "status", "iters", "n_los", "it_near", "it_new", "it_code", "los_log"):
        assert np.array_equal(a[k], b[k]), (k, tag)
    for q in range(len(a["n_nodes"])):
        n = int(a["n_nodes"][q])
        assert np.array_equal(a["parent"][q, :n], b["parent"][q, :n]), ("parent", q, tag)
        for k in ("node_x", "node_y", "node_theta", "u"):
            assert bits_equal(a[k][q, :n], b[k][q, :n]), (k, q, tag)
    if counters:
        assert np.array_equal(a["counters"][:, COUNTERS_KEPT], b["counters"][:, COUNTERS_KEPT]), tag
    assert (a["counters"][:, 8] == 0).all() and (b["counters"][:, 8] == 0).all(), tag


def run_in_steps(p, inp, K, stops, lanes, schedule, resume_lanes=None, resume_schedule=None):
    """rrt with stop_at = stops[0], then one resume per later entry and a last one without a stop.  After every call
    the queries that have not ended sit exactly at their stop with status PAUSED."""
    rl = lanes if resume_lanes is None else resume_lanes
    rs = schedule if resume_schedule is None else resume_schedule
    res = p.rrt(*inp, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, stop_at=stops[0])
    reached = np.zeros(len(inp[0]), np.int64)
    for i, st in enumerate(list(stops[1:]) + [None]):
        h = res.host()
        want = np.maximum(reached, np.broadcast_to(np.asarray(stops[i], np.int64), reached.shape))
        paused = h["status"] == PAUSED
        assert np.array_equal(h["iters"][paused], want[paused]) and (want[paused] < K - 1).all(), (i, lanes, schedule)
        assert (h["iters"][~paused] <= want[~paused]).all()
        reached = np.where(paused, want, reached)
        p.rrt_resume(res, stop_at=st, lanes=rl, schedule=rs)
    return res.host()


RESUME_CASES = [(32, 0), (16, 0), (8, 0), (1, 0), (8, 1), (32, 1)]


@pytest.fixture(scope="module")
def resume_workloads(maps):
    """map1 with tol_xy = 0 (96 queries, every one runs long) and map2 with the default tolerance (goals found, and the
    reference raising, part-way through a run).  The map1 queries have no node within the tie audit's 4-ulp window of a
    nearest decision, so counter 8 is 0 whatever the schedule."""
    K = 1201
    return {"map1": (maps["map1"], dict(tol_xy=0.0), streams(maps["map1"], 96, K, 1234, 0), K),
            "map2": (maps["map2"], {}, streams(maps["map2"], 64, K, 99, 3000), K)}


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", RESUME_CASES)
@pytest.mark.parametrize("which", ["map1", "map2"])
def test_resume_equals_one_call(resume_workloads, which, lanes, schedule):
    free, params, inp, K = resume_workloads[which]
    p = planner_for(free, **params)
    one = p.rrt(*inp, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
    if which == "map2":  # runs that end mid-way are part of the workload
        assert np.isin(one["status"], (OK_FOUND, 4)).any()
    uniform = run_in_steps(p, inp, K, [0, 1, 31, 32, 33, 500, K - 1], lanes, schedule)
    assert_same_run(uniform, one, ("uniform", which, lanes, schedule))
    rng = np.random.default_rng(lanes * 10 + schedule)
    nq = len(inp[0])
    for trial in range(2):
        m = int(rng.integers(3, 7))
        stops = np.sort(rng.integers(0, K, size=(m, nq)), axis=0)  # per-query stops, repeats included
        stepped = run_in_steps(p, inp, K, list(stops), lanes, schedule)
        assert_same_run(stepped, one, ("random", trial, which, lanes, schedule))
    if (lanes, schedule) == (32, 0):  # paused under one schedule, resumed under the other
        mixed = run_in_steps(p, inp, K, [17, 300, 301, 900], 32, 0, resume_lanes=8, resume_schedule=1)
        assert_same_run(mixed, one, ("mixed", which), counters=False)
        # counters defined on the sequential loop (the rasters of the two schedules count pixels differently)
        assert np.array_equal(mixed["counters"][:, [0, 1, 2, 5, 6, 8]], one["counters"][:, [0, 1, 2, 5, 6, 8]])


@pytest.mark.gpu
def test_full_size_pauses_equal_one_call_and_oracle(O, maps):
    """64 cfg-3 queries (the bench workload's 1000..1063) at K = 5001, paused at 1000, 2500 and 4999 and then resumed:
    equal to the one-shot run and, tree by tree, to the oracle."""
    import bench
    from oracle.c_oracle import Params as OP
    free = maps["map1"]
    nq, K = 64, 5001
    inp = bench.make_rrt_workload(free, nq, K, first_query=1000)
    p = planner_for(free, tol_xy=0.0)
    one = p.rrt(*inp, K=K, logs=True, counters=True).host()
    res = run_in_steps(p, inp, K, [1000, 2500, 4999], 32, 0)
    assert_same_run(res, one, "cfg3")
    starts, goals, sxy, sth = inp
    for q in range(nq):
        o = O.rrt(free, ((starts[q, 0], starts[q, 1]), starts[q, 2]), ((goals[q, 0], goals[q, 1]), goals[q, 2]),
                  sxy[q], sth[q], OP(tol_xy=0.0), K=K)
        n = o["n_nodes"]
        assert int(res["status"][q]) == o["status"], q
        assert int(res["n_nodes"][q]) == n and int(res["sol"][q]) == o["sol"] and int(res["iters"][q]) == o["iters"], q
        for k in ("it_code", "it_near", "it_new"):
            assert np.array_equal(res[k][q], o[k]), (k, q)
        assert np.array_equal(res["parent"][q, :n], o["parent"]), q
        assert bits_equal(res["node_x"][q, :n], o["x"]) and bits_equal(res["node_y"][q, :n], o["y"]), q
        assert bits_equal(res["node_theta"][q, :n], o["theta"]), q
        assert np.array_equal(res["u"][q, :n].view(np.int64), o["u"].view(np.int64)), q
        nl = int(res["n_los"][q])
        assert nl == o["n_los"] and np.array_equal(res["los_log"][q, :nl].astype(bool), o["los"]), q


@pytest.mark.gpu
@pytest.mark.parametrize("which,params,lanes,schedule", [("map1", dict(tol_xy=0.0), 32, 0), ("map2", {}, 8, 1),
                                                          ("map2", {}, 4, 0)])
def test_per_query_budgets_equal_oracle_with_smaller_K(O, maps, which, params, lanes, schedule):
    """stop_at[q] = k_q: query q holds what the oracle plans with K = k_q + 1; PAUSED where that run ran all k_q
    iterations (OK_NOT_FOUND when k_q = K-1)."""
    from oracle.c_oracle import Params as OP
    free = maps[which]
    nq, K = 48, 801
    starts, goals, sxy, sth = streams(free, nq, K, 2024, 40)
    rng = np.random.default_rng(5)
    kq = rng.integers(0, K, nq)
    kq[:4] = (0, 1, K - 1, K - 2)
    p = planner_for(free, **params)
    res = p.rrt(starts, goals, sxy, sth, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, stop_at=kq).host()
    op = OP(**params)
    for q in range(nq):
        k = int(kq[q])
        o = O.rrt(free, ((starts[q, 0], starts[q, 1]), starts[q, 2]), ((goals[q, 0], goals[q, 1]), goals[q, 2]),
                  sxy[q], sth[q], op, K=k + 1)
        n = o["n_nodes"]
        tag = (q, k)
        want = o["status"]
        if want == OK_NOT_FOUND and o["iters"] == k and k < K - 1:
            want = PAUSED
        assert int(res["status"][q]) == want, tag
        assert int(res["n_nodes"][q]) == n and int(res["sol"][q]) == o["sol"] and int(res["iters"][q]) == o["iters"], tag
        for key in ("it_code", "it_near", "it_new"):
            assert np.array_equal(res[key][q, :k], o[key][:k]), (key, tag)
        assert (res["it_code"][q, k:] == NOT_RUN).all() and (res["it_near"][q, k:] == -1).all(), tag
        assert np.array_equal(res["parent"][q, :n], o["parent"]), tag
        for key, ok in (("node_x", "x"), ("node_y", "y"), ("node_theta", "theta")):
            assert bits_equal(res[key][q, :n], o[ok]), (key, tag)
        assert np.array_equal(res["u"][q, :n].view(np.int64), o["u"].view(np.int64)), tag
        nl = int(res["n_los"][q])
        assert nl == o["n_los"] and np.array_equal(res["los_log"][q, :nl].astype(bool), o["los"]), tag
    assert (res["counters"][:, 8] == 0).all()
    if which == "map2":
        assert (res["status"] == PAUSED).any() and np.isin(res["status"], (OK_FOUND, 4)).any()


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", [(32, 0), (4, 0), (8, 1)])
def test_stop_zero_and_stop_last(maps, lanes, schedule):
    free = maps["map1"]
    K = 301
    inp = streams(free, 24, K, 8, 60)
    p = planner_for(free, tol_xy=0.0)
    z = p.rrt(*inp, K=K, logs=True, lanes=lanes, schedule=schedule, stop_at=0).host()
    assert (z["status"] == PAUSED).all() and (z["iters"] == 0).all() and (z["n_nodes"] == 1).all() and (z["sol"] == -1).all()
    assert (z["it_code"] == NOT_RUN).all() and (z["it_near"] == -1).all() and (z["it_new"] == -1).all() and (z["n_los"] == 0).all()
    assert bits_equal(z["node_x"][:, 0], inp[0][:, 0]) and (z["parent"][:, 0] == -1).all()
    one = p.rrt(*inp, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
    last = p.rrt(*inp, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, stop_at=np.full(24, K - 1)).host()
    assert_same_run(last, one, "stop K-1")
    assert np.array_equal(last["counters"], one["counters"])  # same schedule, no resume: every counter


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", [(32, 0), (2, 0), (8, 1)])
def test_k1(maps, lanes, schedule):
    free = maps["map1"]
    p = planner_for(free)
    starts, goals = util.random_queries(free, 5, 3)
    res = p.rrt(starts, goals, np.zeros((5, 0, 2), np.int32), np.zeros((5, 0)), K=1, logs=True, lanes=lanes,
                schedule=schedule, stop_at=0)
    h = res.host()
    assert (h["status"] == OK_NOT_FOUND).all() and (h["iters"] == 0).all() and (h["n_nodes"] == 1).all()
    p.rrt_resume(res, lanes=lanes, schedule=schedule)
    h2 = res.host()
    for k in ("status", "iters", "n_nodes", "sol"):
        assert np.array_equal(h[k], h2[k]), k
    with pytest.raises(ValueError):
        p.rrt(starts, goals, np.zeros((5, 0, 2), np.int32), np.zeros((5, 0)), K=1, stop_at=1)


SENTINEL = {"node_x": 1.25, "node_y": -7.5, "node_theta": 3.0, "parent": -77, "u": 9.5, "n_nodes": 5, "sol": 2,
            "n_los": 3, "it_near": 11, "it_new": 12, "it_code": 7, "los_log": 6, "counters": 123}


def fill_sentinels(res, rows):
    """Every output row of the queries `rows` set to a sentinel (status and iters are left to the caller)."""
    for k, v in SENTINEL.items():
        getattr(res, k)[rows] = v


@pytest.mark.gpu
@pytest.mark.parametrize("lanes,schedule", [(32, 0), (8, 0), (8, 1)])
def test_resume_writes_nothing_it_must_not(maps, lanes, schedule):
    """A resume leaves every byte of a query it does not continue: queries that are not paused (ended, or never
    paused), and paused ones whose stop is <= iters; with no query to continue, no output byte changes."""
    import torch
    free = maps["map2"]
    K = 601
    nq = 40
    inp = streams(free, nq, K, 12, 500)
    p = planner_for(free)
    # no paused query at all: the whole result is sentinels with statuses 0, 1, 4
    res = p.rrt(*inp, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule)
    fill_sentinels(res, slice(None))
    res.status[:] = torch.tensor([0, 1, 4, 6], dtype=torch.int32, device=res.status.device).repeat(nq // 4)
    res.iters[:] = 100
    before = {k: v.clone() for k, v in vars(res).items() if isinstance(v, torch.Tensor)}
    p.rrt_resume(res, lanes=lanes, schedule=schedule)
    p.rrt_resume(res, stop_at=K - 1, lanes=lanes, schedule=schedule)
    for k, v in before.items():
        assert torch.equal(getattr(res, k).view(torch.uint8), v.view(torch.uint8)), k
    # paused at 200: ended queries are never rewritten; paused ones with stop <= iters neither; the rest continue
    res = p.rrt(*inp, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule, stop_at=200)
    h = res.host()
    ended = np.nonzero(h["status"] != PAUSED)[0]
    paused = np.nonzero(h["status"] == PAUSED)[0]
    assert len(ended) and len(paused) > 2
    frozen = paused[:2]  # resumed with a stop at (or below) where they are
    rows = torch.as_tensor(np.concatenate([ended, frozen]), device=res.status.device)
    fill_sentinels(res, rows)
    before = {k: getattr(res, k)[rows].clone() for k in list(SENTINEL) + ["status", "iters"]}
    stop = np.full(nq, K - 1)
    stop[frozen] = (200, 150)
    p.rrt_resume(res, stop_at=stop, lanes=lanes, schedule=schedule)
    for k, v in before.items():
        assert torch.equal(getattr(res, k)[rows], v), k
    one = p.rrt(*inp, K=K, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
    h = res.host()
    go = np.setdiff1d(paused, frozen)
    assert (h["status"][go] != PAUSED).all()
    sub = lambda d: {k: (v[go] if isinstance(v, np.ndarray) and v.ndim and v.shape[0] == nq else v) for k, v in d.items()}  # noqa: E731
    assert_same_run(sub(h), sub(one), ("continued", lanes, schedule))


@pytest.mark.gpu
def test_multimap_map_id(maps):
    """Queries bound to different maps of one grid through map_id pause and resume like one call."""
    from theta_rrt_b200 import OccupancyGrid, Params, Planner, samples
    n_maps, side = 3, 256
    free = np.stack([util.synthetic_map(side, 0.15, 4, 7 + m) for m in range(n_maps)])
    p = Planner(OccupancyGrid(free), Params(tol_xy=0.0))
    rng = np.random.default_rng(55)
    nq, K = 30, 701
    mid = rng.integers(0, n_maps, nq).astype(np.int32)
    starts = np.empty((nq, 3)); goals = np.empty((nq, 3))
    sxy = np.empty((nq, K - 1, 2), np.int32); sth = np.empty((nq, K - 1))
    for q in range(nq):
        s, g = util.random_queries(free[mid[q]], 1, 1000 + q)
        starts[q], goals[q] = s[0], g[0]
        sxy[q], sth[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), K - 1, 2000 + q, (side, side))
    for lanes, schedule in ((32, 0), (8, 1)):
        one = p.rrt(starts, goals, sxy, sth, K=K, map_id=mid, logs=True, counters=True, lanes=lanes, schedule=schedule).host()
        res = p.rrt(starts, goals, sxy, sth, K=K, map_id=mid, logs=True, counters=True, lanes=lanes, schedule=schedule,
                    stop_at=rng.integers(0, K, nq))
        p.rrt_resume(res, stop_at=350, lanes=lanes, schedule=schedule)
        p.rrt_resume(res, lanes=lanes, schedule=schedule)
        assert_same_run(res.host(), one, ("map_id", lanes, schedule))


@pytest.mark.gpu
def test_rrt_batch_device_stream_resumes(maps):
    """rrt.rrt_batch(stop_at=...) with device-drawn samples: the result keeps those samples, and resuming it gives the
    uninterrupted run."""
    import builtins
    from theta_rrt_b200 import _context
    from theta_rrt_b200 import main as M
    from theta_rrt_b200 import rrt as R
    had = hasattr(builtins, "imarray")
    old = getattr(builtins, "imarray", None)
    free = maps["map2"]
    M.set_map(free)
    try:
        starts, goals = util.random_queries(free, 32, 31)
        seeds = np.arange(32) * 7 + 5
        one = R.rrt_batch(starts, goals, seeds=seeds, K=401, logs=True, seed_stream="device").host()
        res = R.rrt_batch(starts, goals, seeds=seeds, K=401, logs=True, seed_stream="device", stop_at=123)
        assert (res.status.cpu().numpy() != OK_NOT_FOUND).all()
        _context.current_planner().rrt_resume(res)
    finally:
        if had:
            builtins.imarray = old
        else:
            del builtins.imarray
    h = res.host()
    for k in ("n_nodes", "sol", "status", "iters", "it_near", "it_new", "it_code", "los_log", "n_los"):
        assert np.array_equal(h[k], one[k]), k


@pytest.mark.gpu
def test_python_value_errors(maps):
    free = maps["map1"]
    K = 51
    inp = streams(free, 6, K, 1, 1)
    p = planner_for(free)
    for bad in (-1, K, [0, 1, 2], [0, 1, 2, 3, 4, K], np.full(7, 3), [0.5] * 6):
        with pytest.raises(ValueError):
            p.rrt(*inp, K=K, stop_at=bad)
    with pytest.raises(ValueError):
        p.rrt(*inp, K=K, stop_at=3, pack=True)
    packed = p.rrt(*inp, K=K, pack=True)
    with pytest.raises(ValueError):
        p.rrt_resume(packed)
    res = p.rrt(*inp, K=K, stop_at=10)
    with pytest.raises(ValueError):
        p.rrt_resume(res, stop_at=K)
    with pytest.raises(ValueError):
        p.rrt_resume(res, stop_at=[K - 1] * 5)
    with pytest.raises(ValueError):
        planner_for(free).rrt_resume(res)  # another planner's grid
