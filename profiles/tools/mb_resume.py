"""Pause and resume on the headline workload: cfg 3 (4 096 queries x K = 5 001 on map1, tol_xy = 0, bench.py's seeded
streams, device-resident inputs) planned three ways with the default kernel (speculative window, one warp per query):
  one       one Planner.rrt call
  5x1000    Planner.rrt(stop_at=1000), then rrt_resume up to 2000, 3000, 4000 and the end (5 calls)
  50x100    the same in steps of 100 iterations (50 calls)
Reported: ms per full step of each (CUDA events around the whole sequence, after one untimed warm-up step of each
way), the cost of one extra resume call ((ms of the split step - ms of one call) / (calls - 1): the index rebuild plus
a launch and its tail), and whether the three ways return identical trees, logs-free outputs and statuses.

    python profiles/tools/mb_resume.py [--reps 3] [--json OUT]
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

import bench  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    name, power, clk = out[0].split(", ")
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--queries", type=int, default=bench.NQ_PER_GPU)
    ap.add_argument("--json", help="also write the result line to this file")
    args = ap.parse_args()
    import torch
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    if not torch.cuda.is_available():
        sys.exit("mb_resume.py measures on the GPU: no CUDA device")
    K = bench.K_RRT
    z = np.load(os.path.join(ROOT, "tests", "golden", "maps.npz"))
    free = z["map1"].astype(bool)
    inp = bench.make_rrt_workload(free, args.queries, K)
    dev = torch.device("cuda:0")
    d_in = [torch.from_numpy(a).to(dev) for a in inp]
    p = Planner(OccupancyGrid(free, device=dev), Params(tol_xy=0.0, K=K))
    ways = {"one": [K - 1], "5x1000": list(range(1000, K, 1000)), "50x100": list(range(100, K, 100))}

    def step(stops):
        if len(stops) == 1:
            return p.rrt(*d_in, K=K)
        res = p.rrt(*d_in, K=K, stop_at=stops[0])
        for s in stops[1:]:
            p.rrt_resume(res, stop_at=s)
        return res

    out = {"workload": f"cfg3: {args.queries} queries on map1 (100x100), K={K}, tol_xy=0", "gpu": gpu_info(), "ways": {}}
    results = {}
    for name, stops in ways.items():
        step(stops)  # warm-up
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = step(stops)
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        results[name] = res.host()
        out["ways"][name] = {"calls": len(stops), "ms": ms, "ms_min": min(ms), "ms_median": float(np.median(ms))}
    base = out["ways"]["one"]["ms_median"]
    for name in ("5x1000", "50x100"):
        w = out["ways"][name]
        w["ms_per_extra_call"] = (w["ms_median"] - base) / (w["calls"] - 1)
    a = results["one"]
    identical = {}
    for name in ("5x1000", "50x100"):
        b = results[name]
        same = all(np.array_equal(a[k], b[k]) for k in ("n_nodes", "sol", "status", "iters"))
        for q in range(len(a["n_nodes"])):
            n = int(a["n_nodes"][q])
            same = same and np.array_equal(a["parent"][q, :n], b["parent"][q, :n]) and all(
                np.array_equal(a[k][q, :n].view(np.uint8), b[k][q, :n].view(np.uint8)) for k in ("node_x", "node_y", "node_theta", "u"))
            if not same:
                break
        identical[name] = bool(same)
    out["identical_to_one_call"] = identical
    out["statuses"] = {int(s): int(c) for s, c in zip(*np.unique(a["status"], return_counts=True))}
    line = json.dumps(out)
    print(line, flush=True)
    if args.json:
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
