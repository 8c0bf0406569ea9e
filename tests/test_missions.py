"""Batched main.py missions (Planner.missions, trrt_mission_batch, main.plan_batch) against main.chain and the oracle.

The oracle side is tests/mission_oracle.py:mission_chain: main.chain over the oracle's rrt / findnearest / anglebetween,
so every segment record and path row of the device must be bit-identical to it.
"""
import builtins

import numpy as np
import pytest

from tests import util
from tests.mission_oracle import mission_chain
from tests.test_main_chain import check_segments, golden


def seed_normals(seed, K, n_seg):
    return np.random.RandomState(seed).standard_normal(3 * (K - 1) * n_seg)


def bits_equal(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    return np.array_equal(np.where(np.isnan(a), 0.0, a).view(np.int64), np.where(np.isnan(b), 0.0, b).view(np.int64))


def node_row(n):
    return [np.nan] * 3 if n is None else [n[0][0], n[0][1], n[1]]


def compare_with_oracle(h, m, o):
    """Mission m of a host MissionResult against an oracle mission_chain result: bitwise."""
    assert int(h["status"][m]) == o["status"] and int(h["stop_seg"][m]) == o["stop_seg"], m
    for s, rec in enumerate(o["segments"]):
        for key in ("begin", "end", "solution", "nearest"):
            assert bits_equal(h[key][m, s], node_row(rec[key])), (m, s, key)
        assert bits_equal(h["mindist"][m, s], np.nan if rec["mindist"] is None else rec["mindist"]), (m, s)
        got = tuple(int(h[k][m, s]) for k in ("n_nodes", "n_edges", "iters", "seg_status"))
        assert got == (rec["n_nodes"], rec["n_edges"], rec["iters"], rec["status"]), (m, s)
    for s in range(len(o["segments"]), h["seg_status"].shape[1]):
        assert int(h["seg_status"][m, s]) == 255
    n = len(o["path"])
    assert int(h["path_len"][m]) == n, m
    assert bits_equal(h["path"][m, :n], o["path"]), m
    assert np.array_equal(h["path_seg"][m, :n], o["path_seg"]), m


def waypoints_of(h, m):
    return [tuple(map(int, w)) for w in h["waypoints"][m, :int(h["n_waypoints"][m])]]


# ---------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("case", golden(), ids=lambda c: c["map"])
def test_oracle_mission_chain_reproduces_main_kat(maps, case):
    wp = [tuple(w) for w in case["waypoints"]]
    o = mission_chain(maps[case["map"]], wp, seed_normals(case["seed"], case["K"], len(wp) - 1), case["K"])
    assert o["status"] == 0 and o["stop_seg"] == -1
    check_segments(o["segments"], case)
    assert o["path_seg"].tolist() == sorted(o["path_seg"].tolist())


def test_mission_schedule_ragged():
    from theta_rrt_b200.planner import mission_schedule
    order, n_active = mission_schedule([2, 0, 5, 2, 1, 0, 5])
    assert order.tolist() == [2, 6, 0, 3, 4, 1, 5]
    assert n_active.tolist() == [5, 4, 2, 2, 2]
    order, n_active = mission_schedule([0, 0, 0])
    assert order.tolist() == [0, 1, 2] and n_active.tolist() == []
    order, n_active = mission_schedule([])
    assert order.tolist() == [] and n_active.tolist() == []
    with pytest.raises(ValueError):
        mission_schedule([1, -1])


def test_mission_workspace_bytes_formula():
    from theta_rrt_b200 import _lib
    lib = _lib.load()
    for n, K in ((1, 2), (7, 300), (4096, 300), (16384, 1001)):
        assert lib.trrt_mission_workspace_bytes(n, K) == 19 * 256 + n * (104 + 68 * K + 24 * (K - 1)) + \
            lib.trrt_rrt_workspace_bytes(n, K)
    assert lib.trrt_mission_workspace_bytes(0, 300) == 256


def test_mission_records_conversion():
    from theta_rrt_b200.main import mission_records
    nan = np.nan
    h = {"status": np.array([0, 1, 4, 7]), "n_seg": np.array([2, 0, 1, 1]), "path_len": np.array([3, 0, 0, 0]),
         "path": np.zeros((4, 2, 8)), "path_seg": np.zeros((4, 2), np.int32),
         "begin": np.array([[[0, 0, 10.0], [4, 4, 20.0]]] * 4), "end": np.array([[[4, 4, 20.0], [8, 8, 20.0]]] * 4),
         "solution": np.array([[[nan] * 3, [8, 8, 21.0]]] * 4), "nearest": np.array([[[4, 4, 19.0], [nan] * 3]] * 4),
         "mindist": np.array([[0.5, nan]] * 4), "n_nodes": np.array([[3, 4]] * 4), "n_edges": np.array([[2, 3]] * 4)}
    h["path"][0, 0, :3] = (0, 0, 10.0)
    h["path"][0, 1, :3] = (4, 4, 19.0)
    h["path_seg"][0] = [0, 0]
    recs = mission_records(h, 0)
    assert len(recs) == 2
    assert recs[0]["solution"] is None and recs[0]["nearest"] == ((4.0, 4.0), 19.0) and recs[0]["mindist"] == 0.5
    assert recs[1]["solution"] == ((8.0, 8.0), 21.0) and recs[1]["mindist"] is None
    assert recs[0]["path"] == [((0.0, 0.0), 10.0), ((4.0, 4.0), 19.0)] and recs[1]["path"] == []  # truncated at path_cap 2
    assert mission_records(h, 1) is False
    assert isinstance(mission_records(h, 2), TypeError) and isinstance(mission_records(h, 3), TypeError)


# ---------------------------------------------------------------------------------------------------- GPU
def planner_for(free, **kw):
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    return Planner(OccupancyGrid(free, device="cuda:0"), Params(**kw))


def oracle_batch(free, h, seeds, K, maps_by_id=None, params=None):
    out = []
    for m, seed in enumerate(seeds):
        if int(h["n_seg"][m]) == 0:
            out.append(None)
            continue
        wp = waypoints_of(h, m)
        f = free if maps_by_id is None else maps_by_id[int(h["map_id"][m])]
        out.append(mission_chain(f, wp, seed_normals(int(seed), K, len(wp) - 1), K, params))
    return out


def check_batch(h, oracle, route_status=None):
    for m, o in enumerate(oracle):
        if o is None:  # no segment: the route's status is copied
            assert int(h["n_seg"][m]) == 0 and int(h["path_len"][m]) == 0
            if route_status is not None:
                assert int(h["status"][m]) == int(route_status[m])
            assert (h["seg_status"][m] == 255).all()
            continue
        compare_with_oracle(h, m, o)


def map2_queries(free, n, seed):
    starts, goals = util.random_queries(free, n, seed)
    sg = np.concatenate([starts[:, :2], goals[:, :2]], axis=1).astype(np.int32)
    blocked = np.argwhere(~free)[0]
    sg[0] = [sg[0, 0], sg[0, 1], blocked[1], blocked[0]]  # goal on an obstacle
    sg[1] = [-3, 5, sg[1, 2], sg[1, 3]]                     # start outside the map
    sg[2, 2:] = sg[2, :2]                                   # start == goal: search.astar returns False
    return sg


@pytest.mark.gpu
@pytest.mark.parametrize("case", golden(), ids=lambda c: c["map"])
def test_missions_reproduce_main_kat(maps, case):
    from theta_rrt_b200 import main as M
    from theta_rrt_b200.main import mission_records
    free = maps[case["map"]]
    wp = [tuple(w) for w in case["waypoints"]]
    h = planner_for(free).missions(waypoints=[wp], seeds=[case["seed"]], K=case["K"]).host()
    recs = mission_records(h, 0)
    check_segments(recs, case)
    compare_with_oracle(h, 0, mission_chain(free, wp, seed_normals(case["seed"], case["K"], len(wp) - 1), case["K"]))
    M.set_map(free)
    old_k = builtins.K
    builtins.K = case["K"]
    try:
        np.random.seed(case["seed"])
        segs = M.chain(wp)
    finally:
        builtins.K = old_k
    for r, s in zip(recs, segs):
        ref = np.array([node_row(n) for n in M.path_nodes(s)])
        assert np.allclose(np.array([node_row(n) for n in r["path"]]), ref, rtol=0, atol=1e-9)


@pytest.fixture(scope="module")
def map2_batch(maps):
    free = maps["map2"]
    sg = map2_queries(free, 256, 2024)
    seeds = np.arange(256) + 9000
    res = planner_for(free).missions(start_goal=sg, seeds=seeds, K=300)
    h = res.host()
    return free, sg, seeds, h


@pytest.mark.gpu
def test_missions_map2_theta_bitwise(map2_batch):
    from oracle import c_oracle as O
    free, sg, seeds, h = map2_batch
    route_status = h["route"]["status"]
    assert route_status[0] == 3 and route_status[1] == 2 and h["n_seg"][2] == 0 and h["status"][2] == 1
    for m in (3, 4, 5):  # the device's routes are the oracle's A* / Theta* routes
        assert waypoints_of(h, m) == O.astar(free, tuple(sg[m, :2]), tuple(sg[m, 2:]), log_los=False)["path"]
    check_batch(h, oracle_batch(free, h, seeds, 300), route_status)
    assert (h["n_seg"] > 0).sum() > 200
    # stops where the reference raises: in rrt.rrt (rrt.py:170-171) and on a childless tree (main.py:79-81)
    assert (h["status"] == 4).sum() >= 1 and (h["status"] == 7).sum() >= 1


@pytest.mark.gpu
def test_missions_map1_astar_small_k(maps):
    free = maps["map1"]
    from oracle import c_oracle as O
    sg = map2_queries(free, 32, 77)
    seeds = np.arange(32) + 100
    h = planner_for(free, THETASTAR=False).missions(start_goal=sg, seeds=seeds, K=100).host()
    assert h["n_seg"].max() > 50
    check_batch(h, oracle_batch(free, h, seeds, 100, params=O.Params(thetastar=0)), h["route"]["status"])


@pytest.mark.gpu
def test_missions_cfg5_map_ids():
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    maps5 = np.stack([util.synthetic_map(256, 0.15, 4, 7 + m) for m in range(64)])
    rng = np.random.default_rng(5)
    mid = rng.integers(0, 64, 512).astype(np.int32)
    cells = [np.argwhere(f) for f in maps5]
    sg = np.array([[*cells[m][rng.integers(len(cells[m]))][::-1], *cells[m][rng.integers(len(cells[m]))][::-1]]
                   for m in mid], np.int32)
    seeds = np.arange(512) + 31
    h = Planner(OccupancyGrid(maps5, device="cuda:0"), Params()).missions(start_goal=sg, seeds=seeds, K=300,
                                                                          map_id=mid).host()
    h["map_id"] = mid
    check_batch(h, oracle_batch(None, h, seeds, 300, maps_by_id=maps5), h["route"]["status"])


@pytest.mark.gpu
def test_missions_childless_tree_stop(maps, monkeypatch):
    """K = 3: a segment may leave its tree without a child entry; main.chain raises TypeError there (main.py:79-81)."""
    from theta_rrt_b200 import main as M
    from theta_rrt_b200 import rrt as R
    free = maps["map2"]
    wp = [tuple(w) for w in M.REFERENCE_WAYPOINTS]
    seeds = np.arange(16)
    h = planner_for(free).missions(waypoints=[wp] * 16, seeds=seeds, K=3).host()
    stops = 0
    M.set_map(free)
    monkeypatch.setattr(builtins, "K", 3)
    for m, seed in enumerate(seeds):
        o = mission_chain(free, wp, seed_normals(int(seed), 3, len(wp) - 1), 3)
        compare_with_oracle(h, m, o)
        if o["status"] != 7:
            continue
        stops += 1
        calls = []
        real = R.rrt
        monkeypatch.setattr(R, "rrt", lambda *a, **k: (calls.append(1), real(*a, **k))[1])
        np.random.seed(int(seed))
        with pytest.raises(TypeError):
            M.chain(wp)
        monkeypatch.setattr(R, "rrt", real)
        assert len(calls) == int(h["stop_seg"][m]) + 1
    assert stops >= 1


@pytest.mark.gpu
def test_missions_batch_invariance(map2_batch):
    free, sg, seeds, h = map2_batch
    perm = np.random.default_rng(3).permutation(len(sg))[:97]
    h2 = planner_for(free).missions(start_goal=sg[perm], seeds=seeds[perm], K=300).host()
    S2 = h2["seg_status"].shape[1]
    for i, m in enumerate(perm):
        for k in ("status", "stop_seg", "n_seg", "path_len"):
            assert h2[k][i] == h[k][m], (k, m)
        for k in ("begin", "end", "solution", "nearest", "mindist", "n_nodes", "n_edges", "iters", "seg_status"):
            assert bits_equal(h2[k][i], h[k][m][:S2]), (k, m)
            assert (h[k][m][S2:] == 255).all() if k == "seg_status" else True
        n = int(h["path_len"][m])
        assert bits_equal(h2["path"][i, :n], h["path"][m, :n]) and np.array_equal(h2["path_seg"][i, :n], h["path_seg"][m, :n])


@pytest.mark.gpu
def test_missions_path_cap_and_caller_normals(map2_batch):
    import torch
    free, sg, seeds, h = map2_batch
    p = planner_for(free)
    sub = np.nonzero(h["path_len"] > 8)[0][:16]
    hc = p.missions(start_goal=sg[sub], seeds=seeds[sub], K=300, path_cap=5).host()
    assert np.array_equal(hc["path_len"], h["path_len"][sub])
    assert bits_equal(hc["path"], h["path"][sub, :5])
    with pytest.raises(ValueError):
        p.missions(start_goal=sg[sub], normals=torch.zeros((len(sub), 10), dtype=torch.float64, device="cuda:0"), K=300)
    n_seg = h["n_seg"][sub]
    z = torch.randn(len(sub), int(3 * 299 * n_seg.max()), dtype=torch.float64, device="cuda:0")
    hr = p.missions(start_goal=sg[sub], normals=z, K=300).host()
    assert np.array_equal(hr["n_seg"], n_seg) and (hr["status"] == 0).sum() + np.isin(hr["status"], (4, 7)).sum() == len(sub)
    # the same stream through the flat form with ranges gives the same missions
    L = z.shape[1]
    rng = np.stack([np.arange(len(sub)) * L, np.arange(len(sub)) * L + L], axis=1)
    hf = p.missions(start_goal=sg[sub], normals=z.reshape(-1), normal_range=rng, K=300).host()
    assert np.array_equal(hf["path_len"], hr["path_len"]) and np.array_equal(hf["status"], hr["status"])
    for i, n in enumerate(np.minimum(hr["path_len"], hr["path"].shape[1])):
        assert bits_equal(hf["path"][i, :n], hr["path"][i, :n])


@pytest.mark.gpu
def test_plan_batch_png(maps, tmp_path):
    from PIL import Image
    from theta_rrt_b200 import main as M
    p = tmp_path / "map2.png"
    Image.fromarray((maps["map2"].astype(np.uint8) * 255)).convert("RGB").save(p)
    out = M.plan_batch(str(p), [(280, 0), (280, 0)], [(8, 280), (280, 0)], seeds=[0, 1])
    assert [r["end"][0] for r in out[0]] == [tuple(map(float, w)) for w in M.REFERENCE_WAYPOINTS[1:]]
    assert out[1] is False  # start == goal: the start is closed before the goal test, search.astar returns False
    np.random.seed(0)
    segs = M.plan(str(p), start=(280, 0), goal=(8, 280))
    assert [len(s["graph"]) for s in segs] == [r["n_nodes"] for r in out[0]]
    assert [len(M.path_nodes(s)) for s in segs] == [len(r["path"]) for r in out[0]]
