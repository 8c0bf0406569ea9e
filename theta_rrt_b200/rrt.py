"""Drop-in for the reference's `rrt` module (rrt.py) on the GPU path.

`rrt(start, goal, debug=False)` keeps the reference's contract: it returns
`(sol, G, cameFrom)` with `G` an insertion-ordered dict node -> [children],
`cameFrom` a dict node -> (parent, u) (start -> None), nodes of the form
`((x, y), theta)`, and it draws its samples from numpy's global legacy
generator exactly like `rand_conf` does, so a script that seeds `np.random`
and calls `rrt.rrt` sees the same sample stream as with the reference.
The whole expansion loop runs in one fused CUDA kernel (trrt_rrt_batch).
"""
from __future__ import annotations

import builtins

import numpy as np

from . import _context, samples
from .planner import IT_ARC_BLOCKED, IT_NOT_RUN, IT_QRAND_BLOCKED, IT_QRAND_IN_TREE, Planner, RrtResult, _check_seed_stream
from .samples import standardangle as _standardangle_np


def standardangle(angle):
    """rrt.py:9-14."""
    while angle > 180:
        angle = angle - 360
    while angle <= -180:
        angle = angle + 360
    return angle


def linefrompoints(p, q):
    """rrt.py:42-46."""
    a = q[1] - p[1]
    b = p[0] - q[0]
    c = a * p[0] + b * p[1]
    return a, b, c


def angle_to_arclength(radius, angle):
    """rrt.py:48-51."""
    while angle < 0:
        angle = angle + 360
    return (np.pi * 2 * radius) * angle / 360


def arclength_to_angle(radius, arclength):
    """rrt.py:70-71."""
    return arclength * 360 / (np.pi * 2 * radius)


def anglebetween(vec1, vec2):
    """rrt.py:73-77 -- host helper of the driver (main.py:59,66); the kernels carry their own copy."""
    dot = np.dot(vec1[:2], vec2)
    det = vec2[0] * vec1[1] - vec1[0] * vec2[1]
    return standardangle(np.rad2deg(np.arctan2(det, dot)))


def anglediff(angle1, angle2):
    """rrt.py:108-115: wrapped angle2 - angle1 in degrees, through the device's quaternion evaluation."""
    p = _context.current_planner()
    return float(p.anglediff([[float(angle1), float(angle2)]]).cpu()[0])


def bike_clear(node):
    """rrt.py:208-213."""
    p = _context.current_planner()
    return bool(p.clearance([[node[0][0], node[0][1], node[1]]]).cpu()[0, 0])


def front_of_bike_clear(node):
    """rrt.py:215-222."""
    p = _context.current_planner()
    return bool(p.clearance([[node[0][0], node[0][1], node[1]]]).cpu()[0, 1])


def rand_conf(mean):
    """rrt.py:53-68: one sample from numpy's global generator."""
    p = _context.current_planner()
    xy, th = samples.draw_stream_global(((mean[0][0], mean[0][1]), mean[1]), 1, p.grid.shape,
                                        p.params.xystdv, p.params.anglestdv)
    return ((int(xy[0, 0]), int(xy[0, 1])), float(th[0]))


# ---------------------------------------------------------------------------
# result conversion
# ---------------------------------------------------------------------------
def _u_tuple(row):
    steer_, iccx, iccy, rad, dist = (float(v) for v in row)
    if np.isnan(rad):
        return (0, None, None, dist)  # rrt.py:541 (dist is 1, or 1/3 never: the reference raises first)
    return (steer_, np.array([iccx, iccy]), rad, dist)


def result_to_dicts(h, q, start_node):
    """Arrays of query q (host dict from RrtResult.host()) -> (sol, G, cameFrom) like rrt.py:206."""
    n = int(h["n_nodes"][q])
    xs, ys, ths = h["node_x"][q], h["node_y"][q], h["node_theta"][q]
    keys = [start_node] + [((float(xs[i]), float(ys[i])), float(ths[i])) for i in range(1, n)]
    G = {k: [] for k in keys}
    if h.get("it_new") is not None:
        near, new = h["it_near"][q], h["it_new"][q]
        for it in np.nonzero(new >= 0)[0]:
            G[keys[int(near[it])]].append(keys[int(new[it])])
    cameFrom = {}
    par = h["parent"][q]
    for i in range(n):
        if par[i] < 0:
            if i == 0:
                cameFrom[keys[0]] = None
            continue
        cameFrom[keys[i]] = (keys[int(par[i])], _u_tuple(h["u"][q, i]))
    s = int(h["sol"][q])
    return (keys[s] if s >= 0 else None), G, cameFrom


def rrt(start, goal, debug=False):
    """rrt.py:130-206."""
    p = _context.current_planner()
    P = p.params
    K = int(P.K)
    start = (start[0], standardangle(start[1]))
    goal = (goal[0], standardangle(goal[1]))
    n_it = max(K - 1, 0)
    state = np.random.get_state()
    sxy, sth = samples.draw_stream_global(goal, n_it, p.grid.shape, P.xystdv, P.anglestdv)
    res = p.rrt([[start[0][0], start[0][1], start[1]]], [[goal[0][0], goal[0][1], goal[1]]], sxy[None], sth[None],
                K=K, logs=True, want_u=True)
    h = res.host()
    iters = int(h["iters"][0])
    status = int(h["status"][0])
    if iters < n_it or status == 4:
        # the reference stops drawing at its `break` / exception: leave the global generator where it would be
        used = iters + (1 if status == 4 else 0)
        np.random.set_state(state)
        np.random.standard_normal(3 * used)
    if debug:
        codes = h["it_code"][0]
        for it in range(min(iters + (1 if status == 4 else 0), n_it)):
            print(it + 1)
            if codes[it] == IT_QRAND_BLOCKED:
                print('Qrand not in freespace')
            elif codes[it] == IT_QRAND_IN_TREE:
                print("Qrand already in keys")
            elif codes[it] == IT_ARC_BLOCKED:
                print('Path to qnew intersects obstacles')
    if status == 4:
        # rrt.py:170-171 -> drive() -> arclength_to_angle(None, ...) (rrt.py:275,71)
        raise TypeError("unsupported operand type(s) for *: 'float' and 'NoneType'")
    sol, G, cameFrom = result_to_dicts(h, 0, start)
    if sol is not None:
        print('Found goal!')
    print("Nodes in tree: ", len(G.keys()))
    return sol, G, cameFrom


def rrt_batch(starts, goals, seeds=None, sample_xy=None, sample_th=None, K=None, logs=False, lanes=0,
              seed_stream="host", stop_at=None) -> RrtResult:
    """Many independent rrt() calls in one launch.  Either pass per-query `seeds` (the stream of query q equals
    `np.random.seed(seeds[q])` followed by K-1 rand_conf calls, drawn by numpy on the host with seed_stream="host" or
    on the device with seed_stream="device", Planner.rand_conf: the same bits) or explicit sample arrays.
    stop_at: per-query iteration stops (Planner.rrt); Planner.rrt_resume continues the paused queries with the samples
    the result keeps."""
    _check_seed_stream(seed_stream)
    p = _context.current_planner()
    P = p.params
    K = int(K or P.K)
    starts = np.asarray(starts, dtype=np.float64).reshape(-1, 3).copy()
    goals = np.asarray(goals, dtype=np.float64).reshape(-1, 3).copy()
    starts[:, 2] = _standardangle_np(starts[:, 2])
    goals[:, 2] = _standardangle_np(goals[:, 2])
    if sample_xy is None:
        if seeds is None:
            raise ValueError("pass seeds or sample arrays")
        sample_xy, sample_th = p._seeded_samples(goals, seeds, K, seed_stream, P)
    return p.rrt(starts, goals, sample_xy, sample_th, K=K, logs=logs, lanes=lanes, stop_at=stop_at)


def rrt_race(start, goal, seeds, K=None):
    """Seed race for one problem: rrt(start, goal) under np.random.seed(seed) for every seed of `seeds`, planned in one
    launch whose members stop once one of them has reached the goal (Planner.rrt_race, device-drawn streams).  Returns
    (seed, (sol, G, cameFrom)) for the winner -- the seed that reaches the goal in the fewest iterations, the first of
    them in `seeds` on a tie -- where the tuple is what `np.random.seed(seed); rrt(start, goal)` returns; (None, None)
    when no seed reaches the goal.  numpy's global generator is not touched."""
    p = _context.current_planner()
    K = int(K or p.params.K)
    start = (start[0], standardangle(start[1]))
    goal = (goal[0], standardangle(goal[1]))
    seeds = np.asarray(seeds).reshape(1, -1)
    r = p.rrt_race([[start[0][0], start[0][1], start[1]]], [[goal[0][0], goal[0][1], goal[1]]], seeds, K=K, logs=True)
    w = int(r.winner.cpu()[0])
    if w < 0:
        return None, None
    res = r.result
    h = {k: getattr(res, k)[w:w + 1].cpu().numpy() for k in ("n_nodes", "node_x", "node_y", "node_theta", "parent", "u",
                                                               "sol", "it_near", "it_new")}
    return int(seeds[0, w]), result_to_dicts(h, 0, start)


def findnearest(tree, goal):
    """rrt.py:117-128 for a G dict as returned by rrt()."""
    p = _context.current_planner()
    keys = list(tree.keys())
    if not keys:
        return (None, None)
    index = {k: i for i, k in enumerate(keys)}
    ep, ec = [], []
    for parent in keys:
        for child in tree[parent]:
            ep.append(index[parent])
            ec.append(index[child])
    if not ep:
        return (None, None)
    import torch
    n = len(keys)
    E = len(ep)
    K = max(n, E + 1)
    dev = p.device
    def pad(vals, fill, dt):
        a = np.full(K if dt == np.float64 else K - 1, fill, dt)
        a[:len(vals)] = vals
        return torch.from_numpy(a).to(dev)
    fake = RrtResult(K=K, node_x=pad([float(k[0][0]) for k in keys], np.nan, np.float64).reshape(1, K),
                     node_y=pad([float(k[0][1]) for k in keys], np.nan, np.float64).reshape(1, K),
                     node_theta=pad([float(k[1]) for k in keys], np.nan, np.float64).reshape(1, K),
                     parent=torch.zeros((1, K), dtype=torch.int32, device=dev),
                     n_nodes=torch.tensor([n], dtype=torch.int32, device=dev),
                     sol=torch.zeros(1, dtype=torch.int32, device=dev), status=torch.zeros(1, dtype=torch.int32, device=dev),
                     iters=torch.zeros(1, dtype=torch.int32, device=dev),
                     it_near=pad(ep, -1, np.int32).reshape(1, K - 1), it_new=pad(ec, -1, np.int32).reshape(1, K - 1))
    best, dist = p.findnearest(fake, [[goal[0][0], goal[0][1], goal[1]]])
    b = int(best.cpu()[0])
    if b < 0:
        return (None, None)
    return (keys[b], float(dist.cpu()[0]))


def steer(bikeorigin, theta, bikegoal, thetagoal, plot=False):
    """rrt.py:306-541 (plot is accepted and ignored: drawing is out of scope)."""
    p = _context.current_planner()
    out, straight = p.steer([[bikeorigin[0], bikeorigin[1], theta, bikegoal[0], bikegoal[1], thetagoal]])
    o = out.cpu().numpy()[0]
    if int(straight.cpu()[0]):
        if o[0] == bikegoal[0] and o[1] == bikegoal[1]:
            return (bikegoal, theta), (0, None, None, 1)
        return (np.array([o[0], o[1]]), theta), (0, None, None, 1)
    return (np.array([o[0], o[1]]), float(o[2])), (float(o[3]), np.array([o[4], o[5]]), float(o[6]), float(o[7]))


def drive(bikeorigin, u):
    """rrt.py:272-304."""
    if u[1] is None or u[2] is None:
        raise TypeError("unsupported operand type(s) for *: 'float' and 'NoneType'")  # rrt.py:275,71
    p = _context.current_planner()
    out = p.drive([[bikeorigin[0][0], bikeorigin[0][1], bikeorigin[1], u[0], u[1][0], u[1][1], u[2], u[3]]])
    o = out.cpu().numpy()[0]
    return ((float(o[0]), float(o[1])), float(o[2])), u


def edge_blocked(begin, land, u):
    """`False in [search.freespace(px) for px in search.getArc(begin, land, u)]` (rrt.py:173-174)."""
    p = _context.current_planner()
    straight = u[1] is None
    row = [begin[0], begin[1], land[0], land[1], u[0], np.nan if straight else u[1][0], np.nan if straight else u[1][1],
           np.nan if straight else u[2], 1.0 if straight else 0.0]
    return bool(p.arc_blocked([row]).cpu()[0])


# ---------------------------------------------------------------------------
# visual adapters (rrt.py:16-40, 79-106, 224-270): display lists from theta_rrt_b200.draw, painted when matplotlib exists
# ---------------------------------------------------------------------------
def _draw_kw():
    return dict(bikelength=float(getattr(builtins, "bikelength", 5)), forwardonly=bool(getattr(builtins, "FORWARDONLY", True)))


def _paint(display_list):
    from . import draw
    try:
        draw.render(display_list, ax=getattr(builtins, "ax", None), bikelength=_draw_kw()["bikelength"])
    except ImportError:
        pass  # no matplotlib: the display list is still returned
    return display_list


def draw_bicycle(bike_loc, theta, alpha, color='blue'):
    """rrt.py:16-40."""
    return _paint([("bike", (float(bike_loc[0]), float(bike_loc[1])), float(theta), float(alpha), color)])


def draw_path_segment(bike1, bike2, u, colors=None, bikes=True):
    """rrt.py:224-270."""
    from . import draw
    return _paint(draw.segment_primitives(bike1, bike2, u, colors=colors or draw.SEGMENT_COLORS, bikes=bikes, **_draw_kw()))


def drawpath(solution, camefrom):
    """rrt.py:79-98."""
    from . import draw
    return _paint(draw.path_display_list(solution, camefrom, **_draw_kw()))


def drawtree(begin, graph, camefrom):
    """rrt.py:100-106."""
    from . import draw
    return _paint(draw.tree_display_list(graph, camefrom, **_draw_kw()))
