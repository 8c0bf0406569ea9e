"""Map edits on the device (trrt_grid_edit, OccupancyGrid.edit, Planner.edit_map) and the re-check of planned RRT trees,
Theta* routes and mission paths against the edited map (trrt_validate_tree, trrt_validate_path)."""
import ctypes as C

import numpy as np
import pytest

from tests import util
from tests.util import O, bits_equal, planner_for  # noqa: F401  (O is a fixture)
from theta_rrt_b200 import _lib

gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------- host model of an edit
def apply_edit(img, rects, free, map_ids):
    """imarray[y0:y1, x0:x1] = value per rectangle (clipped), free rectangles first, then the blocked ones."""
    img = img.copy()
    n_maps, H, W = img.shape
    for phase in (True, False):
        for (x0, y0, x1, y1), f, m in zip(rects, free, map_ids):
            if bool(f) == phase and 0 <= m < n_maps:
                img[m, max(y0, 0):max(min(y1, H), 0), max(x0, 0):max(min(x1, W), 0)] = phase
    return img


def random_rects(rng, side, n, n_maps):
    """Rectangles with edges at 0, 1, 7, 8 mod 8 and 31, 32 mod 32, some partly or wholly outside, some empty."""
    def coord():
        k = rng.integers(6)
        if k < 4:
            base = 8 * rng.integers(0, side // 8 + 1) + [0, 1, 7, 8][k]
        elif k == 4:
            base = 32 * rng.integers(0, side // 32 + 1) + [31, 32][rng.integers(2)]
        else:
            base = rng.integers(-20, side + 20)
        return int(base)
    rects = []
    for _ in range(n):
        x0, y0 = coord(), coord()
        kind = rng.integers(8)
        if kind == 0:  # empty
            rects.append((x0, y0, x0 - rng.integers(0, 3), y0 + 5))
        elif kind == 1:  # wholly outside
            rects.append((side + 3, y0, side + 40, y0 + 9))
        elif kind == 2:  # partly outside
            rects.append((x0 - 40, y0 - 40, x0 + 10, y0 + 10))
        else:
            rects.append((x0, y0, x0 + int(rng.integers(1, 70)), y0 + int(rng.integers(1, 70))))
    free = rng.integers(0, 2, n).astype(bool)
    return np.array(rects, np.int64), free, rng.integers(0, n_maps, n)


def fresh(img):
    from theta_rrt_b200 import OccupancyGrid
    return OccupancyGrid(img)


def grids_equal(g, img):
    f = fresh(img)
    return np.array_equal(g.bits.cpu().numpy(), f.bits.cpu().numpy()) and \
        np.array_equal(g.tiles.cpu().numpy(), f.tiles.cpu().numpy())


def trees_equal(a, b):
    """Two host rrt results hold the same trees bit for bit (rows past n_nodes are not written)."""
    if not all(np.array_equal(a[k], b[k]) for k in ("n_nodes", "sol", "status", "iters")):
        return False
    rows = np.arange(a["parent"].shape[1])[None, :] < a["n_nodes"][:, None]
    return np.array_equal(a["parent"][rows], b["parent"][rows]) and \
        all(bits_equal(a[k][rows], b[k][rows]) for k in ("node_x", "node_y", "node_theta", "u"))


def edit_maps(maps):
    stack = np.stack([util.synthetic_map(96, 0.2, 4, 40 + m) for m in range(3)])
    return {"map1": maps["map1"][None], "map2": maps["map2"][None],
            "syn257": util.synthetic_map(257, 0.15, 4, 3)[None], "stack3": stack}


# ----------------------------------------------------------------------------- CPU
def test_ctypes_mirrors_match_header():
    for name, mirror in (("trrt_validate_tree_args", _lib.CValidateTreeArgs),
                         ("trrt_validate_path_args", _lib.CValidatePathArgs)):
        assert [f[0] for f in mirror._fields_] == util.struct_members(name), name
    for s in ("trrt_grid_edit", "trrt_validate_tree", "trrt_validate_tree_workspace_bytes", "trrt_validate_path"):
        assert s in _lib.SIGNATURES
    lib = _lib.load()
    assert lib.trrt_validate_tree_workspace_bytes(4096, 5001) == 256 + 12 * 4096 * 5001


def test_abi_rejects_bad_arguments_before_device_work():
    lib = _lib.load()
    fake = C.c_void_p(256)
    # no bits, negative n, a missing rectangle array, misaligned strip copy, non-square map
    assert lib.trrt_grid_edit(None, None, 1, 8, 8, fake, fake, 1, None) == 1
    assert lib.trrt_grid_edit(fake, None, 1, 8, 8, fake, fake, -1, None) == 1
    assert lib.trrt_grid_edit(fake, None, 1, 8, 8, None, fake, 1, None) == 1
    assert lib.trrt_grid_edit(fake, C.c_void_p(264), 1, 8, 8, fake, fake, 1, None) == 1
    assert lib.trrt_grid_edit(fake, None, 1, 8, 9, fake, fake, 1, None) == 2
    a = _lib.CValidateTreeArgs(d_bits=256, n_maps=1, H=8, W=8, n_queries=1, K=4, lanes=3)
    assert lib.trrt_validate_tree(C.byref(a), None) == 1  # lanes
    a.lanes = 0
    assert lib.trrt_validate_tree(C.byref(a), None) == 1  # NULL arrays
    a.K = (1 << 30) + 1  # the chain tables pack a node index and a bit into an int32
    assert lib.trrt_validate_tree(C.byref(a), None) == 1
    p = _lib.CValidatePathArgs(d_bits=256, n_maps=1, H=8, W=8, mode=2, n_paths=1, path_cap=4)
    assert lib.trrt_validate_path(C.byref(p), None) == 1


def _cpu_grid(n_maps=2, side=16):
    from theta_rrt_b200 import OccupancyGrid
    g = object.__new__(OccupancyGrid)
    g.n_maps, g.H, g.W = n_maps, side, side
    return g


@pytest.mark.parametrize("rects,free,map_id", [
    ([[0, 0, 4]], True, None),              # three columns
    ([[0.5, 0, 4, 4]], True, None),          # not integers
    ([[0, 0, 4, 4], [1, 1, 2, 2]], [True, False, True], None),  # flags do not match
    ([[0, 0, 4, 4]], True, 2),               # map id out of range
    ([[0, 0, 4, 4]], True, [-1]),
    ([[0, 0, 2 ** 31, 4]], True, None),      # does not fit int32
])
def test_edit_rejects_malformed_input(rects, free, map_id):
    with pytest.raises(ValueError):
        _cpu_grid().edit(rects, free, map_id)


def test_validate_tree_refusals_without_gpu():
    from theta_rrt_b200.planner import Planner, RrtResult, _RrtLaunch
    p = object.__new__(Planner)
    p.grid = _cpu_grid()
    res = RrtResult.empty(2, 5, "cpu", want_u=False, logs=False, counters=False)
    res.launch = _RrtLaunch(None, None, None, None, None, None, p.grid, packed=False, race=None)
    with pytest.raises(ValueError, match="want_u"):
        p.validate_tree(res)
    res = RrtResult.empty(2, 5, "cpu", want_u=True, logs=False, counters=False)
    res.launch = _RrtLaunch(None, None, None, None, None, None, _cpu_grid(), packed=False, race=None)
    with pytest.raises(ValueError, match="this planner's grid"):
        p.validate_tree(res)
    with pytest.raises(ValueError):
        p.validate_path(res)


def test_host_model_blocked_wins():
    img = np.ones((1, 8, 8), bool)
    out = apply_edit(img, [(0, 0, 4, 4), (2, 2, 6, 6)], [False, True], [0, 0])
    assert not out[0, 3, 3] and out[0, 5, 5] and not out[0, 0, 0]


# ----------------------------------------------------------------------------- GPU: edits
@gpu
@pytest.mark.parametrize("which", ["map1", "map2", "syn257", "stack3"])
def test_edits_equal_rebuild(maps, which):
    from theta_rrt_b200 import OccupancyGrid
    img = edit_maps(maps)[which].copy()
    nm, side = img.shape[0], img.shape[1]
    rng = np.random.default_rng({"map1": 1, "map2": 2, "syn257": 3, "stack3": 4}[which])
    g = OccupancyGrid(img)
    g.tiles  # strip copy built before the edits: patched in place
    late = OccupancyGrid(img)  # strip copy first built after the edits
    for _ in range(4):
        rects, free, mids = random_rects(rng, side, int(rng.integers(1, 60)), nm)
        before = img
        img = apply_edit(img, rects, free, mids)
        g.edit(rects, free, mids if nm > 1 else None)
        late.edit(rects, free, mids if nm > 1 else None)
        assert grids_equal(g, img)
        # the inverse: every changed pixel back to its old value, as 1x1 rectangles
        m, y, x = np.nonzero(before != img)
        if len(m):
            inv = np.stack([x, y, x + 1, y + 1], 1)
            g.edit(inv, before[m, y, x], m)
            assert grids_equal(g, before)
            g.edit(rects, free, mids if nm > 1 else None)
            assert grids_equal(g, img)
    assert grids_equal(late, img)
    g.edit(np.zeros((0, 4), np.int64), True)  # nothing to do
    assert grids_equal(g, img)


@gpu
def test_edit_cuda_tensors_ignore_foreign_map_ids(maps):
    import torch
    from theta_rrt_b200 import OccupancyGrid
    img = edit_maps(maps)["stack3"].copy()
    g = OccupancyGrid(img)
    g.tiles
    rects = torch.tensor([[0, 0, 50, 50], [10, 10, 20, 20], [5, 5, 90, 9]], dtype=torch.int32, device="cuda:0")
    with pytest.raises(ValueError, match="int32"):  # would be narrowed without a check
        g.edit(rects.to(torch.int64), False, torch.tensor([0, 0, 0], dtype=torch.int32, device="cuda:0"))
    with pytest.raises(ValueError, match="int32"):
        g.edit(rects, False, torch.tensor([0, 0, 0], dtype=torch.int64, device="cuda:0"))
    mids = torch.tensor([7, -1, 2], dtype=torch.int32, device="cuda:0")
    g.edit(rects, torch.tensor([False, False, False], device="cuda:0"), mids)
    img[2, 5:9, 5:90] = False
    assert grids_equal(g, img)


@gpu
def test_consumers_see_the_edit(O, maps):
    import torch
    from theta_rrt_b200 import samples
    free = maps["map2"].copy()
    p = planner_for(free, tol_xy=0.0)
    p.grid.tiles
    rng = np.random.default_rng(5)
    rects, fl, _ = random_rects(rng, 300, 40, 1)
    edited = apply_edit(free[None], rects, fl, np.zeros(40, int))[0]
    p.edit_map(rects, fl)
    q = planner_for(edited, tol_xy=0.0)
    seg = rng.integers(0, 300, size=(20000, 4)).astype(np.int32)
    for layout in ("tiles", "rows"):
        assert np.array_equal(p.los(seg, layout=layout).cpu().numpy(), q.los(seg, layout=layout).cpu().numpy())
    assert np.array_equal(p.los(seg).cpu().numpy().astype(bool), O.lineofsight_batch(edited, seg))
    cells = np.argwhere(edited)
    sg = np.concatenate([cells[rng.integers(len(cells), size=(64,))][:, ::-1],
                         cells[rng.integers(len(cells), size=(64,))][:, ::-1]], 1).astype(np.int32)
    a, b = p.theta(sg).host(), q.theta(sg).host()
    for k in ("path", "path_len", "status", "cost", "expanded"):
        assert np.array_equal(a[k], b[k]), k
    nq, K = 48, 601
    starts, goals = util.random_queries(edited, nq, 77)
    sxy, sth = samples.make_streams(goals, K - 1, np.arange(nq) + 5, edited.shape)
    assert trees_equal(p.rrt(starts, goals, sxy, sth, K=K).host(), q.rrt(starts, goals, sxy, sth, K=K).host())
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------- GPU: validity on the planning map
def _assert_tree_valid(p, res, lanes=0):
    v = p.validate_tree(res, lanes=lanes).host()
    h = res.host()
    rows = np.arange(res.K)[None, :] < h["n_nodes"][:, None]
    assert np.array_equal(v["edge_ok"].astype(bool), rows)
    assert np.array_equal(v["node_ok"].astype(bool), rows)
    assert np.array_equal(v["sol_ok"], np.where(h["sol"] >= 0, 1, -1))
    return v


def _batch(free, nq, K, seed):
    from theta_rrt_b200 import samples
    starts, goals = util.random_queries(free, nq, seed)
    sxy, sth = samples.make_streams(goals, K - 1, np.arange(nq) + seed, free.shape)
    return starts, goals, sxy, sth


@gpu
@pytest.mark.parametrize("which,lanes", [("map1", 0), ("map2", 1), ("map2", 32)])
def test_trees_valid_on_planning_map(maps, which, lanes):
    free = maps[which]
    p = planner_for(free)
    res = p.rrt(*_batch(free, 256, 1001, 3), K=1001)
    st = res.status.cpu().numpy()
    assert (st == 0).any() and (st != 0).any()  # found, not found and the error statuses
    _assert_tree_valid(p, res, lanes)


@gpu
def test_paused_raced_and_multimap_trees_valid(maps):
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    free = maps["map2"]
    p = planner_for(free)
    ins = _batch(free, 64, 801, 11)
    res = p.rrt(*ins, K=801, stop_at=np.arange(64) * 12)
    _assert_tree_valid(p, res)
    p.rrt_resume(res)
    _assert_tree_valid(p, res)
    starts, goals, sxy, sth = _batch(free, 8, 801, 12)
    rs = np.repeat(np.arange(8), 16)
    from theta_rrt_b200 import samples
    sxy, sth = samples.make_streams(goals[rs], 800, np.arange(128) + 500, free.shape)
    raced = p.rrt(starts[rs], goals[rs], sxy, sth, K=801, race=rs)
    _assert_tree_valid(p, raced)
    stack = edit_maps(maps)["stack3"]
    pm = Planner(OccupancyGrid(stack), Params())
    mid = np.arange(60) % 3
    st, go = np.empty((60, 3)), np.empty((60, 3))
    for q in range(60):
        s, g = util.random_queries(stack[mid[q]], 1, 900 + q)
        st[q], go[q] = s[0], g[0]
    sxy, sth = samples.make_streams(go, 400, np.arange(60), stack.shape[1:])
    _assert_tree_valid(pm, pm.rrt(st, go, sxy, sth, K=401, map_id=mid))


@gpu
def test_routes_and_missions_valid_on_planning_map(maps):
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    free = maps["map2"]
    rng = np.random.default_rng(8)
    sg = rng.integers(0, 300, size=(128, 4)).astype(np.int32)  # includes blocked and invalid endpoints
    for thetastar in (True, False):
        p = planner_for(free, THETASTAR=thetastar)
        r = p.theta(sg)
        v = p.validate_path(r).host()
        h = r.host()
        assert np.array_equal(v["ok"], (h["status"] == 0).astype(np.uint8))
        rows = np.arange(r.path.shape[1])[None, :] < np.minimum(h["path_len"], r.path.shape[1])[:, None]
        found = h["status"] == 0
        assert found.any() and not found.all()
        assert np.array_equal(v["step_ok"][found].astype(bool), rows[found])
    p = planner_for(free)
    m = p.missions(start_goal=sg[:64], seeds=np.arange(64) + 9000, K=300)
    v = p.validate_path(m).host()
    h = m.host()
    assert np.array_equal(v["ok"], (h["status"] == 0).astype(np.uint8))
    rows = np.arange(m.path.shape[1])[None, :] < np.minimum(h["path_len"], m.path.shape[1])[:, None]
    assert np.array_equal(v["step_ok"][h["status"] == 0].astype(bool), rows[h["status"] == 0])
    stack = edit_maps(maps)["stack3"]
    pm = Planner(OccupancyGrid(stack), Params())
    mid = np.arange(30) % 3
    cells = [np.argwhere(f) for f in stack]
    sgm = np.array([[*cells[k][rng.integers(len(cells[k]))][::-1], *cells[k][rng.integers(len(cells[k]))][::-1]]
                    for k in mid], np.int32)
    mm = pm.missions(start_goal=sgm, seeds=np.arange(30), K=200, map_id=mid)
    assert np.array_equal(pm.validate_path(mm).ok.cpu().numpy(), (mm.status.cpu().numpy() == 0).astype(np.uint8))
    rr = pm.theta(sgm, map_id=mid)
    assert np.array_equal(pm.validate_path(rr).ok.cpu().numpy(), (rr.status.cpu().numpy() == 0).astype(np.uint8))


# ----------------------------------------------------------------------------- GPU: validity after edits vs the oracle
def oracle_edge_ok(O, img, parent, x, y, u, i):
    p = parent[i]
    if p == -1:
        return True
    b, l = (x[p], y[p]), (x[i], y[i])
    if np.isnan(u[i, 1]):
        px = O.bresenham((int(b[0]), int(b[1])), (int(l[0]), int(l[1])))
    else:
        px = O.getarc(img.shape, b, l, (u[i, 0], (u[i, 1], u[i, 2]), u[i, 3], u[i, 4]))
    H, W = img.shape
    return all(0 <= a < H and 0 <= c < W and img[c, a] for a, c in px)


def host_node_ok(parent, edge_ok, n):
    """The walk of main.path_nodes from every node at once: at most n - 1 parent steps, ending at a node without a
    parent; AND of edge_ok over the nodes it leaves."""
    out = np.zeros(len(parent), bool)
    pos, ok, alive = np.arange(n), np.ones(n, bool), np.ones(n, bool)
    parent, edge_ok = np.asarray(parent[:n]), np.asarray(edge_ok[:n], bool)
    for _ in range(n - 1):
        par = parent[pos]
        alive &= par != -1
        if not alive.any():
            break
        ok &= ~alive | edge_ok[pos]
        pos = np.where(alive, par, pos)
    out[:n] = ok
    return out


def check_tree_vs_oracle(O, img, h, v, queries):
    for q in queries:
        n = int(h["n_nodes"][q])
        eok = np.array([oracle_edge_ok(O, img, h["parent"][q], h["node_x"][q], h["node_y"][q], h["u"][q], i)
                        for i in range(n)])
        assert np.array_equal(v["edge_ok"][q, :n].astype(bool), eok), q
        assert not v["edge_ok"][q, n:].any() and not v["node_ok"][q, n:].any()
        nok = host_node_ok(h["parent"][q], eok, n)
        assert np.array_equal(v["node_ok"][q].astype(bool), nok), q
        s = int(h["sol"][q])
        assert v["sol_ok"][q] == (-1 if s < 0 else int(nok[s]))


@gpu
@pytest.mark.parametrize("lanes", [0, 1, 32])
def test_tree_validity_after_edit_vs_oracle(O, maps, lanes):
    free = maps["map1"]
    p = planner_for(free)
    res = p.rrt(*_batch(free, 96, 1001, 21), K=1001)
    rng = np.random.default_rng(lanes)
    rects, fl, _ = random_rects(rng, 100, 30, 1)
    fl[:] = False
    img = apply_edit(free[None], rects, fl, np.zeros(30, int))[0]
    p.edit_map(rects, fl)
    v = p.validate_tree(res, lanes=lanes).host()
    h = res.host()
    assert 0 < v["edge_ok"].sum() < (np.arange(1001)[None] < h["n_nodes"][:, None]).sum()
    check_tree_vs_oracle(O, img, h, v, range(0, 96, 5))


@gpu
@pytest.mark.parametrize("thetastar,lanes", [(True, 0), (True, 1), (True, 32), (False, 8)])
def test_route_validity_after_edit_vs_oracle(O, maps, thetastar, lanes):
    """Routes planned on map1 between free cells, then checked on the map after blocking edits: step 0 is freespace of
    the first waypoint, step t the oracle's lineofsight(wp[t-1], wp[t]) on the edited image."""
    free = maps["map1"]
    p = planner_for(free, THETASTAR=thetastar)
    rng = np.random.default_rng(40 + lanes)
    cells = np.argwhere(free)
    sg = np.concatenate([cells[rng.integers(len(cells), size=128)][:, ::-1],
                         cells[rng.integers(len(cells), size=128)][:, ::-1]], 1).astype(np.int32)
    r = p.theta(sg)  # planned on the unedited map
    rects, fl, _ = random_rects(rng, 100, 30, 1)
    fl[:] = False
    img = apply_edit(free[None], rects, fl, np.zeros(30, int))[0]
    p.edit_map(rects, fl)
    pv = p.validate_path(r, lanes=lanes).host()
    hr = r.host()
    broken = 0
    for q in range(len(sg)):
        n = min(int(hr["path_len"][q]), r.path.shape[1])
        wp = hr["path"][q]
        exp = ([bool(img[wp[0, 1], wp[0, 0]])] if n else []) + \
            [O.lineofsight(img, tuple(wp[t - 1]), tuple(wp[t])) for t in range(1, n)]
        assert np.array_equal(pv["step_ok"][q, :n].astype(bool), np.array(exp, bool)), q
        assert not pv["step_ok"][q, n:].any()
        assert pv["ok"][q] == int(hr["status"][q] == 0 and all(exp))
        broken += hr["status"][q] == 0 and not all(exp)
    assert (hr["status"] == 0).sum() > 64 and broken > 0  # found routes, some of them cut by the edit


@gpu
@pytest.mark.parametrize("K", [7, 300, 5001])
def test_hand_built_parent_cycles(O, maps, K):
    """Parent arrays with a cycle through an overwritten root and a cycle elsewhere (trees the kernel never builds in
    this shape, but the walk's n_nodes cut defines them)."""
    import torch
    free = maps["map2"]
    p = planner_for(free)
    nq = 4
    res = p.rrt(*_batch(free, nq, K, 31), K=K)
    torch.cuda.synchronize()
    rng = np.random.default_rng(K)
    n = K
    x = rng.uniform(0, 299, (nq, K)); y = rng.uniform(0, 299, (nq, K))
    u = np.full((nq, K, 5), np.nan)  # straight edges: the arcs are covered by test_tree_validity_after_edit_vs_oracle
    u[..., 0], u[..., 4] = 0.0, 3.0
    parent = np.empty((nq, K), np.int32)
    for q in range(nq):
        perm = rng.permutation(n)
        parent[q, perm[1:]] = perm[:-1]  # a chain in random order, pointing to higher and lower indices
        parent[q, perm[0]] = -1
        if q == 1 and n > 3:  # cycle through the overwritten root
            parent[q, perm[0]] = perm[n - 1]
        if q == 2 and n > 5:  # a cycle away from the root
            parent[q, perm[n // 2]] = perm[n - 2]
    dev = lambda a, dt: torch.as_tensor(a, dtype=dt, device="cuda:0")
    res.node_x.copy_(dev(x, torch.float64)); res.node_y.copy_(dev(y, torch.float64))
    res.u.copy_(dev(u, torch.float64)); res.parent.copy_(dev(parent, torch.int32))
    res.n_nodes.fill_(n)
    res.sol.copy_(dev([0, n - 1, n // 2, -1], torch.int32))
    v = p.validate_tree(res).host()
    h = res.host()
    assert v["edge_ok"].any() and not v["edge_ok"].all()
    check_tree_vs_oracle(O, free, h, v, range(nq))


@gpu
@pytest.mark.parametrize("lanes", [0, 1, 32])
def test_mission_validity_after_edit_vs_oracle(O, maps, lanes):
    free = maps["map2"]
    p = planner_for(free)
    rng = np.random.default_rng(4)
    cells = np.argwhere(free)
    sg = np.concatenate([cells[rng.integers(len(cells), size=32)][:, ::-1],
                         cells[rng.integers(len(cells), size=32)][:, ::-1]], 1).astype(np.int32)
    m = p.missions(start_goal=sg, seeds=np.arange(32) + 70, K=300)
    rects, fl, _ = random_rects(rng, 300, 60, 1)
    fl[:] = False
    img = apply_edit(free[None], rects, fl, np.zeros(60, int))[0]
    p.edit_map(rects, fl)
    v = p.validate_path(m, lanes=lanes).host()
    h = m.host()
    bad = 0
    for q in range(32):
        n = min(int(h["path_len"][q]), m.path.shape[1])
        rows, seg = h["path"][q], h["path_seg"][q]
        exp = []
        for r in range(n):
            if r == 0 or seg[r] != seg[r - 1]:
                exp.append(True)
                continue
            par = np.array([-1, 0], np.int32)
            exp.append(oracle_edge_ok(O, img, par, rows[[r - 1, r], 0], rows[[r - 1, r], 1],
                                      np.stack([rows[r - 1, 3:], rows[r, 3:]]), 1))
        assert np.array_equal(v["step_ok"][q, :n].astype(bool), np.array(exp, bool)), q
        assert not v["step_ok"][q, n:].any()
        assert v["ok"][q] == int(h["status"][q] == 0 and all(exp))
        bad += not all(exp)
    assert bad > 0


# ----------------------------------------------------------------------------- GPU: ordering
@gpu
def test_edit_map_waits_for_inflight_rrt_host(maps):
    import torch
    free = maps["map2"]
    p = planner_for(free, tol_xy=0.0)
    nq, K = 96, 1501
    ins = _batch(free, nq, K, 61)
    ref = p.rrt(*ins, K=K).host()
    pins = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in ins]
    out = {"parent": torch.zeros((nq, K), dtype=torch.int32).pin_memory(),
           "n_nodes": torch.zeros(nq, dtype=torch.int32).pin_memory()}
    p.rrt_host(*pins, out=out, K=K, chunks=3, wait=False)
    p.edit_map([[0, 0, 300, 300]], False)  # the whole map blocked
    p.host_sync()
    torch.cuda.synchronize()
    assert np.array_equal(out["n_nodes"].numpy(), ref["n_nodes"])
    for q in range(nq):
        n = int(ref["n_nodes"][q])
        assert np.array_equal(out["parent"].numpy()[q, :n], ref["parent"][q, :n])
    assert not p.grid.bits.any().item()


@gpu
def test_pause_edit_revert_resume_equals_one_call(maps):
    free = maps["map2"]
    p = planner_for(free)
    ins = _batch(free, 64, 1201, 71)
    ref = p.rrt(*ins, K=1201).host()
    res = p.rrt(*ins, K=1201, stop_at=400)
    rects = np.array([[100, 100, 200, 200], [0, 0, 40, 300]])
    before = free[None].copy()
    img = apply_edit(before, rects, [False, True], [0, 0])
    p.edit_map(rects, [False, True])
    m, y, x = np.nonzero(before != img)
    p.edit_map(np.stack([x, y, x + 1, y + 1], 1), before[m, y, x])
    p.rrt_resume(res)
    assert trees_equal(res.host(), ref)
