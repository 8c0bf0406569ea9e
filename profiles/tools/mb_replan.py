"""Map edits and re-validation of planned results: what an edit and a re-check cost next to a rebuild and a re-plan.

  (a) edits of 1, 64 and 4 096 random rectangles (sides 1-64 px, half free, half blocked) on the cfg-4 8192^2 grid with
      its strip copy built (Planner.edit_map: rows + strip patch), against rebuilding the grid from the host image
      (OccupancyGrid + tiles);
  (b) validate_tree on a cfg-3 result (4 096 queries x K = 5 001 on map1, u kept) after a blocking edit, next to the rrt
      call that planned it, in the same run;
  (c) validate_path on 8 192 map2 Theta* routes, and on cfg-5-style missions (512 missions over 64 random 256^2 maps,
      K = 300).
CUDA events around each call after warm-up; median of --reps timed calls.  The GPU's name, power limit and max SM clock
are read in the same run.  Writes mb_replan.json to the output directory.

    python profiles/tools/mb_replan.py --out DIR [--reps 10]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import util  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    name, power, clk = out[0].split(", ")
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def timed(fn, reps, warm=2):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}


def random_rects(rng, side, n):
    xy = rng.integers(0, side, (n, 2))
    wh = rng.integers(1, 65, (n, 2))
    return np.concatenate([xy, xy + wh], 1), rng.integers(0, 2, n).astype(bool)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for mb_replan.json")
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    import torch
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    if not torch.cuda.is_available():
        sys.exit("mb_replan.py measures on the GPU: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info()}
    rng = np.random.default_rng(9)

    # (a) edits against a rebuild, cfg-4 grid
    big = util.synthetic_map(8192, 0.1, 8, 42)
    p4 = Planner(OccupancyGrid(big), Params())
    p4.grid.tiles
    a = {}
    for n in (1, 64, 4096):
        rects, free = random_rects(rng, 8192, n)
        d_rects = torch.from_numpy(rects.astype(np.int32)).cuda()
        d_free = torch.from_numpy(free).cuda()
        a[f"edit_{n}"] = timed(lambda: p4.edit_map(d_rects, d_free), args.reps)
    a["rebuild"] = timed(lambda: OccupancyGrid(big).tiles, max(3, args.reps // 3), warm=1)
    res["a_edit_cfg4"] = a

    # (b) validate_tree on a cfg-3 result
    z = np.load(os.path.join(ROOT, "tests", "golden", "maps.npz"))
    m1 = z["map1"].astype(bool)
    p3 = Planner(OccupancyGrid(m1), Params())
    nq, K = 4096, 5001
    starts, goals = util.random_queries(m1, nq, 1234)
    sxy, sth = p3.rand_conf(goals, np.arange(nq), K=K)
    torch.cuda.synchronize()
    t_rrt = timed(lambda: p3.rrt(starts, goals, sxy, sth, K=K), 3, warm=1)
    r = p3.rrt(starts, goals, sxy, sth, K=K)
    p3.edit_map([[40, 40, 60, 60]], False)
    t_val = timed(lambda: p3.validate_tree(r), args.reps)
    v = p3.validate_tree(r)
    edges = int(r.n_nodes.sum().item())
    res["b_validate_tree_cfg3"] = {"rrt": t_rrt, "validate_tree": t_val, "edges": edges,
                                   "edges_per_sec": edges / (t_val["median_ms"] / 1e3),
                                   "edges_ok": int(v.edge_ok.sum().item()), "sol_ok": int((v.sol_ok == 1).sum().item()),
                                   "sol_found": int((r.sol >= 0).sum().item())}
    # (c) validate_path: map2 Theta* routes, cfg-5-style missions
    m2 = z["map2"].astype(bool)
    p2 = Planner(OccupancyGrid(m2), Params())
    cells = np.argwhere(m2)
    rq = np.random.default_rng(5)
    A, B = cells[rq.integers(len(cells), size=8192)], cells[rq.integers(len(cells), size=8192)]
    sg = torch.from_numpy(np.stack([A[:, 1], A[:, 0], B[:, 1], B[:, 0]], 1).astype(np.int32)).cuda()
    routes = p2.theta(sg, path_cap=64)
    p2.edit_map([[140, 140, 160, 160]], False)
    tr = timed(lambda: p2.validate_path(routes), args.reps)
    rows = int(torch.clamp(routes.path_len, max=64).sum().item())
    res["c_validate_routes_map2"] = {"validate_path": tr, "routes": 8192, "rows": rows,
                                     "ok": int(p2.validate_path(routes).ok.sum().item()),
                                     "found": int((routes.status == 0).sum().item())}
    maps5 = np.stack([util.synthetic_map(256, 0.15, 4, 7 + m) for m in range(64)])
    p5 = Planner(OccupancyGrid(maps5), Params())
    mid = rng.integers(0, 64, 512).astype(np.int32)
    c5 = [np.argwhere(f) for f in maps5]
    sg5 = np.array([[*c5[m][rng.integers(len(c5[m]))][::-1], *c5[m][rng.integers(len(c5[m]))][::-1]] for m in mid], np.int32)
    ms = p5.missions(start_goal=sg5, seeds=np.arange(512), K=300, map_id=mid, seed_stream="device")
    p5.edit_map(rng.integers(0, 200, (64, 2)).repeat(2, 1) + [0, 0, 24, 24], False, map_id=rng.integers(0, 64, 64))
    tm = timed(lambda: p5.validate_path(ms), args.reps)
    mrows = int(torch.clamp(ms.path_len, max=ms.path.shape[1]).sum().item())
    res["c_validate_missions_cfg5"] = {"validate_path": tm, "missions": 512, "rows": mrows, "path_cap": ms.path.shape[1],
                                       "ok": int(p5.validate_path(ms).ok.sum().item()),
                                       "status0": int((ms.status == 0).sum().item())}
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out, "mb_replan.json"), "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
