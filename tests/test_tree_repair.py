"""Tree repair after a map edit (trrt_repair_tree, Planner.repair_tree): nodes whose path to the start crosses a newly
blocked edge are pruned, the survivors compacted, cut solutions reopened, and rrt_resume continues the trees on the
edited map as the oracle's loop continued from the repaired tree does (tests/rrt_continue.py)."""
import ctypes as C

import numpy as np
import pytest

from tests import util
from tests.rrt_continue import rrt_continue
from tests.test_map_edits import _assert_tree_valid, _batch, apply_edit, edit_maps, oracle_edge_ok, random_rects
from tests.util import O, bits_equal, planner_for  # noqa: F401  (O is a fixture)
from theta_rrt_b200 import _lib

gpu = pytest.mark.gpu
PAUSED = 8
TREE = ("node_x", "node_y", "node_theta", "u")


# ----------------------------------------------------------------------------- host model of a repair
def host_keep(parent, edge_ok, n):
    """The keep rule: node 0 kept; node i >= 1 kept when following parent from i reaches node 0 within n - 1 steps and
    edge_ok holds for every node the walk leaves before node 0 (all nodes walked at once)."""
    if n == 0:
        return np.zeros(0, bool)
    parent, eok = np.asarray(parent[:n], np.int64), np.asarray(edge_ok[:n], bool)
    pos, ok = np.arange(n), np.ones(n, bool)
    for _ in range(n - 1):
        moving = ok & (pos != 0)
        if not moving.any():
            break
        par = parent[pos]
        ok &= ~moving | (eok[pos] & (par >= 0) & (par < n))
        pos = np.where(moving & ok, par, pos)
    return ok & (pos == 0)


def host_repair(h, edge_ok):
    """The repair of host result h (res.host()) with edge_ok [q, K]: rows compacted in order, parents remapped, the root
    planted again, sol / status / n_nodes updated.  Returns (repaired dict, new_index, n_pruned)."""
    nq, K = h["parent"].shape
    out = {k: h[k].copy() for k in ("parent", "n_nodes", "sol", "status", "iters") + TREE}
    new_index = np.full((nq, K), -1, np.int32)
    n_pruned = np.zeros(nq, np.int32)
    for q in range(nq):
        n = min(max(int(h["n_nodes"][q]), 0), K)
        idx = np.nonzero(host_keep(h["parent"][q], edge_ok[q], n))[0]
        m = len(idx)
        new_index[q, idx] = np.arange(m)
        for k in TREE:
            out[k][q, :m] = h[k][q, idx]
        par = h["parent"][q, idx]
        out["parent"][q, :m] = np.where(idx == 0, -1, new_index[q, np.clip(par, 0, K - 1)])
        if m:
            out["u"][q, 0] = np.nan
        s = int(h["sol"][q])
        ns = int(new_index[q, s]) if 0 <= s < n else -1
        if ns < 0 and h["status"][q] == 0:
            out["status"][q] = PAUSED if h["iters"][q] < K - 1 else 1
        out["sol"][q], out["n_nodes"][q], n_pruned[q] = ns, m, n - m
    return out, new_index, n_pruned


def tree_of(h, q):
    n = int(h["n_nodes"][q])
    return dict(x=h["node_x"][q, :n], y=h["node_y"][q, :n], theta=h["node_theta"][q, :n], parent=h["parent"][q, :n],
                u=h["u"][q, :n])


def query_equal(a, b, q):
    """Query q of two host results: n_nodes, sol, status, iters, and the rows [0, n) bit for bit."""
    if any(int(a[k][q]) != int(b[k][q]) for k in ("n_nodes", "sol", "status", "iters")):
        return False
    n = int(a["n_nodes"][q])
    return np.array_equal(a["parent"][q, :n], b["parent"][q, :n]) and all(bits_equal(a[k][q, :n], b[k][q, :n]) for k in TREE)


def oracle_continued(img, h, q, goals, sxy, sth, K):
    """The oracle's loop continued for query q of h from its own state (rrt_continue), as a host-result row."""
    o = rrt_continue(img, ((goals[q, 0], goals[q, 1]), goals[q, 2]), sxy[q], sth[q], tree_of(h, q), int(h["iters"][q]), K)
    return {"n_nodes": o["n_nodes"], "sol": o["sol"], "status": o["status"], "iters": o["iters"], "parent": o["parent"],
            "node_x": o["x"], "node_y": o["y"], "node_theta": o["theta"], "u": o["u"]}


def row_equal(dev, q, o):
    n = int(o["n_nodes"])
    return all(int(dev[k][q]) == int(o[k]) for k in ("n_nodes", "sol", "status", "iters")) and \
        np.array_equal(dev["parent"][q, :n], o["parent"]) and all(bits_equal(dev[k][q, :n], o[k]) for k in TREE)


def oracle_edges(O, img, h, queries):
    K = h["parent"].shape[1]
    eok = np.zeros((h["parent"].shape[0], K), np.uint8)
    for q in queries:
        for i in range(int(h["n_nodes"][q])):
            eok[q, i] = oracle_edge_ok(O, img, h["parent"][q], h["node_x"][q], h["node_y"][q], h["u"][q], i)
    return eok


def check_repair(h_before, h_after, rep, eok, queries):
    """Device repair (h_after, rep = TreeRepair.host()) against the host model over `queries`."""
    model, new_index, n_pruned = host_repair(h_before, eok)
    for q in queries:
        assert query_equal(h_after, model, q), q
        assert np.array_equal(rep["new_index"][q], new_index[q]), q
        assert rep["n_pruned"][q] == n_pruned[q], q
        assert rep["reopened"][q] == int(h_before["status"][q] == 0 and model["status"][q] == PAUSED), q
    return model


# ----------------------------------------------------------------------------- CPU
def test_ctypes_mirror_and_workspace():
    assert [f[0] for f in _lib.CRepairTreeArgs._fields_] == util.struct_members("trrt_repair_tree_args")
    for s in ("trrt_repair_tree", "trrt_repair_tree_workspace_bytes"):
        assert s in _lib.SIGNATURES
    lib = _lib.load()
    assert lib.trrt_repair_tree_workspace_bytes(4096, 5001) == 256 + 12 * 4096 * 5001
    assert lib.trrt_repair_tree_workspace_bytes(0, 7) == 256
    assert lib.trrt_repair_tree_workspace_bytes(3, 0) == 0


def test_abi_rejects_bad_arguments_before_device_work():
    lib = _lib.load()
    f = 256
    full = dict(n_queries=2, K=8, d_node_x=f, d_node_y=f, d_node_th=f, d_parent=f, d_u=f, d_n_nodes=f, d_sol=f,
                d_status=f, d_iters=f, d_edge_ok=f, d_new_index=f, d_work=f, work_bytes=16)
    assert lib.trrt_repair_tree(None, None) == 1
    for bad in (dict(K=0), dict(K=(1 << 30) + 1), dict(n_queries=-1),
                dict(d_race_key=f),                                 # a key without groups
                dict(d_race_key=f, d_race_group=f),                 # n_race_groups = 0
                dict(d_race_group=f, n_race_groups=2),              # groups without a key
                dict(d_race_key=f, n_race_groups=2),                # no group ids for a non-empty batch
                dict(d_u=None), dict(d_edge_ok=None), dict(d_new_index=None), dict(d_iters=None),
                dict(d_work=f + 2)):                                # misaligned workspace
        a = _lib.CRepairTreeArgs(**{**full, **bad})
        assert lib.trrt_repair_tree(C.byref(a), None) == 1, bad
    a = _lib.CRepairTreeArgs(**full)  # short workspace
    assert lib.trrt_repair_tree(C.byref(a), None) == 4
    a = _lib.CRepairTreeArgs(n_queries=0, K=8)  # nothing to do, and no race
    assert lib.trrt_repair_tree(C.byref(a), None) == 0


def test_repair_tree_refusals_without_gpu():
    import torch
    from theta_rrt_b200.planner import Planner, RrtResult, TreeValidity, _RrtLaunch
    from tests.test_map_edits import _cpu_grid
    p = object.__new__(Planner)
    p.grid = _cpu_grid()

    def result(want_u=True, logs=False, grid=None, packed=False):
        r = RrtResult.empty(2, 5, "cpu", want_u=want_u, logs=logs, counters=False)
        r.launch = _RrtLaunch(None, None, None, None, None, None, grid or p.grid, packed=packed, race=None)
        return r
    with pytest.raises(ValueError, match="want_u"):
        p.repair_tree(result(want_u=False))
    with pytest.raises(ValueError, match="logs"):
        p.repair_tree(result(logs=True))
    with pytest.raises(ValueError, match="pack"):
        p.repair_tree(result(packed=True))
    with pytest.raises(ValueError, match="this planner's grid"):
        p.repair_tree(result(grid=_cpu_grid()))
    bad = TreeValidity(edge_ok=torch.ones((2, 4), dtype=torch.uint8), node_ok=torch.ones((2, 4), dtype=torch.uint8),
                       sol_ok=torch.ones(2, dtype=torch.int8))
    with pytest.raises(ValueError, match="K = 5"):
        p.repair_tree(result(), bad)


def test_host_keep_rule():
    # 0 <- 1 <- 2, 3 -> 2 with a failing edge at 2, 4 an orphan, 5 <-> 6 a cycle, 7 a parent out of range
    parent = [4, 0, 1, 2, -1, 6, 5, 9]
    eok = [0, 1, 0, 1, 1, 1, 1, 1]
    assert host_keep(parent, eok, 8).tolist() == [True, True, False, False, False, False, False, False]
    assert host_keep(parent, np.ones(8), 8).tolist() == [True, True, True, True, False, False, False, False]
    assert host_keep([3, 0, 1, 2], np.ones(4), 4).all()  # a cycle through an overwritten root
    assert host_keep([3, 0, 1, 2], np.ones(4), 3).all()  # the walk's n_nodes cut


@pytest.mark.parametrize("run_index", [0, 1, 2, 4])
def test_oracle_continuation_equals_one_run(maps, run_index):
    """orc_rrt with K' = j + 1 then rrt_continue from j equals one orc_rrt, for j where the goal is not yet found: the
    continuation restates the oracle's loop faithfully."""
    from oracle import c_oracle
    run = util.rrt_runs()[run_index]
    free = maps[str(run["map"])]
    P = c_oracle.Params(tol_xy=float(run["tol_xy"][0]))
    start = ((run["start"][0], run["start"][1]), run["start"][2])
    goal = ((run["goal"][0], run["goal"][1]), run["goal"][2])
    sxy, sth = run["sxy"], run["sth"]
    K = int(run["K"][0])
    full = c_oracle.rrt(free, start, goal, sxy, sth, P, K=K)
    last = full["iters"] - 1 if full["status"] == 0 else K - 1  # the iteration that found the goal, or K-1
    caps = [(K, j) for j in sorted({0, 1, last // 3, last // 2, last})]
    if full["status"] == 0:  # capacity K2 = the solving iteration: j = K2 - 1 continues nothing
        caps.append((full["iters"], full["iters"] - 1))
    for cap, j in caps:
        ref = full if cap == K else c_oracle.rrt(free, start, goal, sxy, sth, P, K=cap)
        head = c_oracle.rrt(free, start, goal, sxy, sth, P, K=j + 1)
        assert head["status"] == 1 and head["iters"] == j
        o = rrt_continue(free, goal, sxy, sth, head, j, cap, P)
        tag = (run_index, cap, j)
        for k in ("status", "n_nodes", "sol", "iters"):
            assert o[k] == ref[k], (tag, k)
        assert np.array_equal(o["parent"], ref["parent"]), tag
        for k in ("x", "y", "theta", "u"):
            assert bits_equal(o[k], ref[k]), (tag, k)
        for k in ("it_near", "it_new", "it_code"):
            assert np.array_equal(np.concatenate([head[k][:j], o[k][j:]]), ref[k]), (tag, k)
        assert np.array_equal(np.concatenate([head["los"], o["los"]]), ref["los"]), tag


# ----------------------------------------------------------------------------- GPU
def _all_bits(res):
    import torch
    out = {}
    for k in ("node_x", "node_y", "node_theta", "u", "parent", "n_nodes", "sol", "status", "iters"):
        t = getattr(res, k)
        out[k] = (t.view(torch.int64) if t.dtype == torch.float64 else t).cpu().numpy().copy()
    return out


@gpu
@pytest.mark.parametrize("which,lanes", [("map1", 0), ("map1", 32), ("map2", 1), ("map2", 32)])
def test_identity_on_unedited_map(maps, which, lanes):
    free = maps[which]
    p = planner_for(free)
    nq, K = 128, 1001
    res = p.rrt(*_batch(free, nq, K, 5), K=K, stop_at=np.where(np.arange(nq) % 3 == 0, 250, K - 1))
    st = res.status.cpu().numpy()
    assert (st == 0).any() and (st == PAUSED).any()
    before = _all_bits(res)
    rep = p.repair_tree(res, lanes=lanes).host()
    after = _all_bits(res)
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    n = before["n_nodes"]
    assert not rep["n_pruned"].any() and not rep["reopened"].any()
    assert np.array_equal(rep["new_index"], np.where(np.arange(K)[None] < n[:, None], np.arange(K)[None], -1))


def _edited_batch(p, free, nq, K, seed, stop_every=4, n_rects=30):
    ins = _batch(free, nq, K, seed)
    res = p.rrt(*ins, K=K, stop_at=np.where(np.arange(nq) % stop_every == 0, K // 3, K - 1))
    rng = np.random.default_rng(seed)
    rects, fl, _ = random_rects(rng, free.shape[0], n_rects, 1)
    fl[:] = False
    img = apply_edit(free[None], rects, fl, np.zeros(n_rects, int))[0]
    p.edit_map(rects, fl)
    return ins, res, img


@gpu
@pytest.mark.parametrize("lanes,schedule", [(0, 0), (0, 1), (1, 0), (1, 1), (32, 0), (32, 1)])
def test_repair_then_resume_vs_oracle(O, maps, lanes, schedule):
    free = maps["map1"]
    p = planner_for(free)
    nq, K = 96, 1001
    (starts, goals, sxy, sth), res, img = _edited_batch(p, free, nq, K, 21 + lanes)
    h0 = res.host()
    eok = oracle_edges(O, img, h0, range(nq))
    rep = p.repair_tree(res, lanes=lanes).host()
    assert np.array_equal(rep["validity"]["edge_ok"], eok)
    h1 = res.host()
    model = check_repair(h0, h1, rep, eok, range(nq))
    assert rep["n_pruned"].sum() > 0 and rep["reopened"].sum() > 0
    _assert_tree_valid(p, res, lanes)
    p.rrt_resume(res, lanes=lanes, schedule=schedule)
    h2 = res.host()
    again = 0
    for q in range(nq):
        if model["status"][q] == PAUSED:
            assert row_equal(h2, q, oracle_continued(img, model, q, goals, sxy, sth, K)), q
            again += bool(rep["reopened"][q] and h2["status"][q] == 0)
        else:
            assert query_equal(h2, model, q), q
    assert again > 0  # reopened queries that reach the goal again on the edited map
    _assert_tree_valid(p, res, lanes)


@gpu
def test_second_repair_is_identity(maps):
    free = maps["map2"]
    p = planner_for(free)
    _, res, _ = _edited_batch(p, free, 64, 801, 7, n_rects=60)
    first = p.repair_tree(res)
    assert first.n_pruned.sum().item() > 0
    before = _all_bits(res)
    rep = p.repair_tree(res).host()
    after = _all_bits(res)
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    assert not rep["n_pruned"].any() and not rep["reopened"].any()


ROWS = ("parent", "n_nodes", "sol", "status", "iters") + TREE


def _rows(arrays, qs):
    """The per-query arrays (a dict, or a result's fields) for queries qs only, on the host (a cfg-3 result holds 0.8 GB
    of u)."""
    import torch
    get = arrays.get if isinstance(arrays, dict) else lambda k: getattr(arrays, k)
    idx = torch.as_tensor(qs, dtype=torch.long, device=get("node_x").device)
    return {k: get(k)[idx].cpu().numpy() for k in ROWS}


@gpu
def test_full_size_cfg3(O, maps):
    free = maps["map1"]
    p = planner_for(free)
    nq, K = 4096, 5001
    starts, goals = util.random_queries(free, nq, 1234)
    sxy_d, sth_d = p.rand_conf(goals, np.arange(nq), K=K)
    res = p.rrt(starts, goals, sxy_d, sth_d, K=K)
    snap = {k: getattr(res, k).clone() for k in ROWS}  # on the device: the state before the repair
    status0 = res.status.cpu().numpy()
    img = apply_edit(free[None], [(40, 40, 60, 60)], [False], [0])[0]
    p.edit_map([[40, 40, 60, 60]], False)
    rep = p.repair_tree(res)
    r = {k: v for k, v in rep.host().items() if k != "validity"}
    r_eok = rep.validity.edge_ok
    reopened = np.nonzero(r["reopened"])[0]
    assert len(reopened) > 0 and (status0[reopened] == 0).all()
    check = np.unique(np.concatenate([reopened[:32], np.arange(0, nq, nq // 32)]))
    _assert_tree_valid(p, res)
    h1 = _rows(res, check)
    p.rrt_resume(res)
    _assert_tree_valid(p, res)
    h2 = _rows(res, check)
    h0 = _rows(snap, check)
    eok = oracle_edges(O, img, h0, range(len(check)))
    assert np.array_equal(r_eok[check].cpu().numpy(), eok)
    sub = {"new_index": r["new_index"][check], "n_pruned": r["n_pruned"][check], "reopened": r["reopened"][check]}
    model = check_repair(h0, h1, sub, eok, range(len(check)))
    sxy, sth = sxy_d[check].cpu().numpy(), sth_d[check].cpu().numpy()
    for j in range(len(check)):
        if model["status"][j] == PAUSED:
            assert row_equal(h2, j, oracle_continued(img, model, j, goals[check], sxy, sth, K)), check[j]
        else:
            assert query_equal(h2, model, j), check[j]


@gpu
def test_multimap_other_map_untouched(maps):
    from theta_rrt_b200 import OccupancyGrid, Params, Planner, samples
    stack = edit_maps(maps)["stack3"][:2]
    pm = Planner(OccupancyGrid(stack), Params())
    nq = 80
    mid = np.arange(nq) % 2
    st, go = np.empty((nq, 3)), np.empty((nq, 3))
    for q in range(nq):
        s, g = util.random_queries(stack[mid[q]], 1, 300 + q)
        st[q], go[q] = s[0], g[0]
    sxy, sth = samples.make_streams(go, 600, np.arange(nq), stack.shape[1:])
    res = pm.rrt(st, go, sxy, sth, K=601, map_id=mid)
    before = _all_bits(res)
    pm.edit_map([[0, 0, 96, 40], [30, 0, 60, 96]], [False, False], map_id=[1, 1])
    rep = pm.repair_tree(res).host()
    after = _all_bits(res)
    on0 = mid == 0
    for k in before:
        assert np.array_equal(before[k][on0], after[k][on0]), k
    assert not rep["n_pruned"][on0].any() and rep["n_pruned"][~on0].sum() > 0


def _race_batch(free, n_prob, S, K, seed):
    from theta_rrt_b200 import samples
    starts, goals = util.random_queries(free, n_prob, seed)
    groups = np.repeat(np.arange(n_prob), S)
    sxy, sth = samples.make_streams(goals[groups], K - 1, np.arange(n_prob * S) + 1000 * seed, free.shape)
    return starts[groups], goals[groups], sxy, sth, groups


def _cutting_rect(O, free, h, q):
    """A small blocked rectangle around a node of query q's solution path that fails an edge of that path."""
    path, c = [], int(h["sol"][q])
    while c > 0:
        path.append(c)
        c = int(h["parent"][q, c])
    for c in path:
        x, y = int(h["node_x"][q, c]), int(h["node_y"][q, c])
        rect = (x - 1, y - 1, x + 2, y + 2)
        img = apply_edit(free[None], [rect], [False], [0])[0]
        if not all(oracle_edge_ok(O, img, h["parent"][q], h["node_x"][q], h["node_y"][q], h["u"][q], i) for i in path):
            return rect, img
    raise AssertionError("no node of the path cuts it")


@gpu
def test_race_keys_and_resume(O, maps):
    free = maps["map1"]
    p = planner_for(free)
    n_prob, S, K = 6, 24, 801
    starts, goals, sxy, sth, groups = _race_batch(free, n_prob, S, K, 3)
    a = p.rrt(starts, goals, sxy, sth, K=K, race=groups)
    b = p.rrt(starts, goals, sxy, sth, K=K, race=groups)
    h = a.host()
    g = int(np.nonzero(h["race_winner"] >= 0)[0][0])
    w = int(h["race_winner"][g])
    rect, img = _cutting_rect(O, free, h, w)
    p.edit_map([rect], False)
    for res in (a, b):
        p.repair_tree(res)
    ha = a.host()
    assert ha["status"][w] != 0  # the winner was cut
    key = np.full(n_prob, -1, np.int64)
    for q in range(len(groups)):
        if ha["status"][q] == 0:
            k = (int(ha["iters"][q]) << 32) | q
            key[groups[q]] = k if key[groups[q]] == -1 else min(key[groups[q]], k)
    assert np.array_equal(ha["race_key"], key)
    assert np.array_equal(b.race_key.cpu().numpy(), key)
    assert ha["race_winner"][g] != w
    p.rrt_resume(a, race=False)
    h2 = a.host()
    for q in range(len(groups)):
        if ha["status"][q] == PAUSED:
            assert row_equal(h2, q, oracle_continued(img, ha, q, goals, sxy, sth, K)), q
        else:
            assert query_equal(h2, ha, q), q
    p.rrt_resume(b, race=True)
    hb = b.host()
    for gi in range(n_prob):
        members = np.nonzero((groups == gi) & (hb["status"] == 0))[0]
        best = min(((int(hb["iters"][q]) << 32) | int(q) for q in members), default=-1)
        assert hb["race_key"][gi] == best, gi


def _hand_built(p, free, K):
    """The parent arrays of test_map_edits.test_hand_built_parent_cycles: a chain in random order, a cycle through an
    overwritten root, a cycle away from the root, over straight edges between random points."""
    import torch
    nq = 4
    res = p.rrt(*_batch(free, nq, K, 31), K=K)
    torch.cuda.synchronize()
    rng = np.random.default_rng(K)
    n = K
    x = rng.uniform(0, 299, (nq, K)); y = rng.uniform(0, 299, (nq, K))
    u = np.full((nq, K, 5), np.nan)
    u[..., 0], u[..., 4] = 0.0, 3.0
    parent = np.empty((nq, K), np.int32)
    for q in range(nq):
        perm = rng.permutation(n)
        parent[q, perm[1:]] = perm[:-1]
        parent[q, perm[0]] = -1
        if q == 1 and n > 3:
            parent[q, perm[0]] = perm[n - 1]
        if q == 2 and n > 5:
            parent[q, perm[n // 2]] = perm[n - 2]
    dev = lambda a, dt: torch.as_tensor(a, dtype=dt, device="cuda:0")
    res.node_x.copy_(dev(x, torch.float64)); res.node_y.copy_(dev(y, torch.float64))
    res.u.copy_(dev(u, torch.float64)); res.parent.copy_(dev(parent, torch.int32))
    res.n_nodes.fill_(n)
    res.sol.copy_(dev([0, n - 1, n // 2, -1], torch.int32))
    res.status.copy_(dev([0, 0, PAUSED, 1], torch.int32))
    res.iters.copy_(dev([K // 2, K - 1, K // 3, K - 1], torch.int32))
    return res


@gpu
@pytest.mark.parametrize("K", [7, 300, 5001])
def test_hand_built_parent_arrays(O, maps, K):
    import torch
    from theta_rrt_b200.planner import TreeValidity
    free = maps["map2"]
    p = planner_for(free)
    for ones in (False, True):
        res = _hand_built(p, free, K)
        h0 = res.host()
        if ones:  # every edge passes: the structure alone decides
            v = TreeValidity(edge_ok=torch.ones((4, K), dtype=torch.uint8, device="cuda:0"),
                             node_ok=torch.ones((4, K), dtype=torch.uint8, device="cuda:0"),
                             sol_ok=torch.ones(4, dtype=torch.int8, device="cuda:0"))
            eok = np.ones((4, K), np.uint8)
        else:
            v = None
            eok = oracle_edges(O, free, h0, range(4))
        rep = p.repair_tree(res, v).host()
        if not ones:
            assert np.array_equal(rep["validity"]["edge_ok"], eok)
        h1 = res.host()
        check_repair(h0, h1, rep, eok, range(4))
        assert (h1["parent"][:, 0] == -1).all() and (h1["n_nodes"] >= 1).all()
        if ones and K > 5:
            assert h1["n_nodes"][1] == K  # the whole cycle reaches node 0


@gpu
def test_edge_cases(maps):
    import torch
    free = maps["map1"]
    p = planner_for(free)
    ins = _batch(free, 8, 101, 9)
    res = p.rrt(*ins, K=101, stop_at=0)  # trees of only the root
    p.edit_map([[0, 0, 100, 100]], False)  # everything blocked
    rep = p.repair_tree(res).host()
    h = res.host()
    assert (h["n_nodes"] == 1).all() and (h["status"] == PAUSED).all() and not rep["n_pruned"].any()
    assert (rep["new_index"][:, 0] == 0).all() and (rep["new_index"][:, 1:] == -1).all()
    p.edit_map([[0, 0, 100, 100]], True)
    empty = p.rrt(np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 100, 2), np.int32), np.zeros((0, 100)), K=101)
    rep = p.repair_tree(empty)
    assert rep.new_index.shape == (0, 101) and rep.n_pruned.shape == (0,)
    one = p.rrt(ins[0], ins[1], np.zeros((8, 0, 2), np.int32), np.zeros((8, 0)), K=1)
    p.edit_map([[0, 0, 100, 100]], False)
    rep = p.repair_tree(one).host()
    h = one.host()
    assert (h["n_nodes"] == 1).all() and (h["status"] == 1).all() and (rep["new_index"] == 0).all()
    torch.cuda.synchronize()
