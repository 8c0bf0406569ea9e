"""Drop-in for the reference's `main` module (main.py): parameters in `builtins`, map PNG in,
chained RRT path out.

Importing this module installs the reference's default parameters into `builtins`
(main.py:15-32), exactly like `import main` does there.  `plan()` is the flow of
main.py:35-84 without the matplotlib calls: load the map (main.py:37-42), take the Theta*
waypoints (the reference hard-codes the result of `search.astar((280,0),(8,280))` at
main.py:57; here they are computed on the GPU unless passed in), then run one RRT per
consecutive waypoint pair with headings from `rrt.anglebetween`, restarting from the
`rrt.findnearest` node when a segment does not reach its goal (main.py:58-81).

    python -m theta_rrt_b200.main [map.png] [--start X Y --goal X Y] [--seed S]
"""
from __future__ import annotations

import builtins
import sys

import numpy as np

# ---- PARAMETERS (main.py:15-32) -------------------------------------------------------------
builtins.THETASTAR = True
builtins.bikelength = 5
builtins.FORWARDONLY = True
builtins.LEFTCONSTRAINT = -65
builtins.RIGHTCONSTRAINT = 65
builtins.frontclearance = 2
builtins.K = 300
builtins.showtree = False
builtins.maxdrivedist = 30
builtins.tol_xy = 10
builtins.tol_ang = 45
builtins.weightxy = .6
builtins.xystdv = 0.4
builtins.anglestdv = 100

from . import rrt, search  # noqa: E402  (after the parameters, like the reference's import order)
from .grid import load_png  # noqa: E402

REFERENCE_WAYPOINTS = [(280, 0), (73, 38), (72, 39), (33, 130), (15, 190), (8, 280)]  # main.py:57


def set_map(image):
    """main.py:37-42: `builtins.imarray = np.array(Image.open(p).convert('1'))`; arrays are taken as they are."""
    if isinstance(image, (str, bytes)) or hasattr(image, "__fspath__"):
        image = load_png(image)
    builtins.imarray = np.asarray(image)
    return builtins.imarray


def chain(waypoints, debug=False):
    """main.py:56-84 for a list of (x, y) waypoints.  Returns one record per segment:
    {begin, end, solution, graph, camefrom, nearest, mindist} with the reference's node tuples."""
    path = list(waypoints) + [None]
    nearest = None
    segments = []
    for first, second, third in zip(path, path[1:], path[2:]):
        angle1 = rrt.anglebetween([1, 0], np.subtract(second, first))
        if nearest is not None:          # main.py:60-62: a failed segment moves every later start
            angle1 = nearest[1]
            first = nearest[0]
        if third is None:
            angle2 = angle1
        else:
            angle2 = rrt.anglebetween([1, 0], np.subtract(third, second))
        begin = (first, rrt.standardangle(angle1))
        end = (second, rrt.standardangle(angle2))
        solution, graph, camefrom = rrt.rrt(begin, end, debug=debug)
        rec = {"begin": begin, "end": end, "solution": solution, "graph": graph, "camefrom": camefrom,
               "nearest": None, "mindist": None}
        if solution is None:
            print("Didn't find solution")
            found, mindist = rrt.findnearest(graph, end)
            if found is None:
                # main.py:79-81: the reference indexes the (None, None) result of a childless tree
                raise TypeError("'NoneType' object is not subscriptable")
            nearest = found
            rec["nearest"], rec["mindist"] = found, mindist
        segments.append(rec)
    return segments


def plan(image, start=None, goal=None, waypoints=None, debug=False):
    """Map in, chained path out.  `waypoints` defaults to the Theta* path from `start` to `goal`
    (the computation the reference keeps commented out at main.py:48-52); with neither given, the
    reference's own waypoint list (main.py:57) is used.  plan_batch() plans many missions at once."""
    set_map(image)
    if waypoints is None:
        if start is None or goal is None:
            waypoints = REFERENCE_WAYPOINTS
        else:
            waypoints = search.astar(tuple(start), tuple(goal))
            if waypoints is False:
                return False
    return chain(waypoints, debug=debug)


def path_nodes(segment):
    """Nodes from a segment's begin to its solution (or nearest) node, walking camefrom (rrt.py:79-98 without drawing)."""
    node = segment["solution"] if segment["solution"] is not None else segment["nearest"]
    out = []
    while node is not None:
        out.append(node)
        prev = segment["camefrom"].get(node)
        node = prev[0] if prev else None
    return out[::-1]


def _node(row):
    return None if np.isnan(row[0]) else ((float(row[0]), float(row[1])), float(row[2]))


def mission_records(h, m):
    """Mission m of a host MissionResult (`Planner.missions(...).host()`) as main.plan would return it: False when
    the route search finds no path (search.py:222-227, :307), the exception the reference raises when it raises, else
    one record per segment with the keys of chain(); `n_nodes` / `n_edges` stand for the graph / camefrom dicts,
    and `path` is path_nodes() of the segment (the rows that fit the result's path_cap)."""
    status, n_seg = int(h["status"][m]), int(h["n_seg"][m])
    if status == 4:
        return TypeError("unsupported operand type(s) for *: 'float' and 'NoneType'")  # rrt.py:170-171, :275
    if status == 7:
        return TypeError("'NoneType' object is not subscriptable")  # main.py:79-81
    if status == 5:
        return ValueError("attempt to get argmin of an empty sequence")  # search.py:262
    if status in (1, 2, 3):
        return False
    if status != 0:
        return RuntimeError(f"mission status {status} (capacity of the call exceeded)")
    n_rows = min(int(h["path_len"][m]), h["path"].shape[1])
    rows, row_seg = h["path"][m, :n_rows], h["path_seg"][m, :n_rows]
    out = []
    for s in range(n_seg):
        mind = float(h["mindist"][m, s])
        out.append({"begin": _node(h["begin"][m, s]), "end": _node(h["end"][m, s]),
                    "solution": _node(h["solution"][m, s]), "nearest": _node(h["nearest"][m, s]),
                    "mindist": None if np.isnan(mind) else mind, "n_nodes": int(h["n_nodes"][m, s]),
                    "n_edges": int(h["n_edges"][m, s]), "path": [_node(r) for r in rows[row_seg == s]]})
    return out


def plan_batch(image, starts, goals, seeds, K=None, seed_stream="host"):
    """plan() for many (start, goal, seed) missions on one map: Theta* (A* with THETASTAR=False) waypoints and the
    segment chain of every mission in one batched device call (Planner.missions).  Mission m draws its samples like
    plan() after np.random.seed(seeds[m]), with numpy on the host (seed_stream="host") or on the device
    (seed_stream="device", the same bits).  Returns one mission_records() entry per mission."""
    set_map(image)
    from . import _context
    p = _context.current_planner()
    sg = np.concatenate([np.asarray(starts, np.int32).reshape(-1, 2), np.asarray(goals, np.int32).reshape(-1, 2)], axis=1)
    h = p.missions(start_goal=sg, seeds=seeds, K=K if K is not None else int(p.params.K), seed_stream=seed_stream).host()
    return [mission_records(h, m) for m in range(len(sg))]


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="theta-rrt main.py flow on the GPU path (no plotting)")
    ap.add_argument("map", nargs="?", default="map2.png")
    ap.add_argument("--start", type=int, nargs=2)
    ap.add_argument("--goal", type=int, nargs=2)
    ap.add_argument("--seed", type=int, default=None, help="np.random.seed before planning")
    args = ap.parse_args(argv)
    if args.seed is not None:
        np.random.seed(args.seed)
    segs = plan(args.map, start=args.start, goal=args.goal, debug=True)
    if segs is False:
        return 1
    for i, s in enumerate(segs):
        nodes = path_nodes(s)
        tag = "reached" if s["solution"] is not None else "nearest"
        print(f"segment {i}: {s['begin']} -> {s['end']}  {tag}, {len(s['graph'])} tree nodes, {len(nodes)} path nodes")
    return 0


if __name__ == "__main__":
    sys.exit(main())
