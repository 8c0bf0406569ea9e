"""Tree repair after a map edit: what repair_tree costs, and what it buys against planning the cut queries again.

  (a) repair_tree alone (validity given) and validate_tree + repair_tree on a cfg-3 result (4 096 queries x K = 5 001 on
      map1, u kept, device-drawn seeded streams) after the 20x20 blocking edit of profiles/r9 ([40, 40, 60, 60));
  (b) for the queries whose solution that edit cut, two ways back on the edited map: repair_tree + rrt_resume of the
      whole result (only the reopened queries grow), and a fresh rrt of just those queries with their seeded streams;
      each with its time and the number of those queries that reach the goal;
  (c) with --parent DIR (a built checkout of the parent commit): bench.py run alternately from DIR and from this tree,
      --pairs times, each run dumping its outputs, which must be identical.
Every timed call restores the planned result from a device copy first (untimed), so each one repairs the same trees.
CUDA events around each call after warm-up; median of --reps timed calls.  The GPU's name, power limit and SM clock are
read in the same run.  Writes mb_repair.json (and bench_alternated.json with --parent) to the output directory.

    python profiles/tools/mb_repair.py --out DIR [--reps 10] [--parent DIR --pairs 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import util  # noqa: E402

ARRAYS = ("node_x", "node_y", "node_theta", "parent", "u", "n_nodes", "sol", "status", "iters")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    name, power, clk, max_clk = out[0].split(", ")
    return {"name": name, "power_limit": power, "sm_clock": clk, "max_sm_clock": max_clk}


def timed(fn, reps, setup, warm=2):
    """fn timed with CUDA events, setup (untimed) before each call."""
    import torch
    for _ in range(warm):
        setup()
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        setup()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}


def bench_alternated(parent, pairs, out):
    """bench.py from the parent checkout and from this tree, alternated; outputs dumped to temporary directories and
    compared array by array."""
    args = ["--gpus", "1", "--steps", "5", "--warmup", "3", "--skip-secondary", "--skip-cpu", "--skip-python-ref"]
    runs, same = {}, []
    for i in range(1, pairs + 1):
        dumps = {}
        for tag, tree in (("parent", parent), ("change", ROOT)):
            d = tempfile.mkdtemp(prefix=f"dump_{tag}_")
            r = subprocess.run([sys.executable, "bench.py", *args, "--dump-outputs", d], cwd=tree, capture_output=True,
                               text=True, timeout=1800)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
            runs[f"{tag}_{i}"] = json.loads(line)
            runs[f"{tag}_{i}"]["gpu"] = gpu_info()
            dumps[tag] = d
        names = sorted(f for f in os.listdir(dumps["parent"]) if f.endswith(".npy"))
        assert names == sorted(f for f in os.listdir(dumps["change"]) if f.endswith(".npy"))
        same.append({"pair": i, "arrays": len(names),
                     "identical": all(np.array_equal(np.load(os.path.join(dumps["parent"], f)).view(np.uint8),
                                                     np.load(os.path.join(dumps["change"], f)).view(np.uint8))
                                      for f in names)})
    res = {"runs": runs, "dumps": same}
    with open(os.path.join(out, "bench_alternated.json"), "w") as f:
        f.write(json.dumps(res) + "\n")
    summary = {}
    for tag in ("parent", "change"):
        v = [runs[f"{tag}_{i}"]["ms_per_step"] for i in range(1, pairs + 1)]
        summary[tag] = {"resident_ms": v, "median": float(np.median(v)), "min": min(v), "max": max(v)}
    summary["dumps_identical"] = all(s["identical"] for s in same)
    return summary


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for mb_repair.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--parent", help="a built checkout of the parent commit: also run bench.py alternately (c)")
    ap.add_argument("--pairs", type=int, default=3)
    args = ap.parse_args()
    import torch
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    if not torch.cuda.is_available():
        sys.exit("mb_repair.py measures on the GPU: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info()}

    z = np.load(os.path.join(ROOT, "tests", "golden", "maps.npz"))
    m1 = z["map1"].astype(bool)
    p = Planner(OccupancyGrid(m1), Params())
    nq, K = 4096, 5001
    starts, goals = util.random_queries(m1, nq, 1234)
    sxy, sth = p.rand_conf(goals, np.arange(nq), K=K)
    r = p.rrt(starts, goals, sxy, sth, K=K)
    snap = {k: getattr(r, k).clone() for k in ARRAYS}
    p.edit_map([[40, 40, 60, 60]], False)

    def restore():
        for k in ARRAYS:
            getattr(r, k).copy_(snap[k])

    restore()
    v = p.validate_tree(r)
    t_rep = timed(lambda: p.repair_tree(r, v), args.reps, restore)
    t_both = timed(lambda: p.repair_tree(r), args.reps, restore)
    restore()
    rep = p.repair_tree(r, v)
    rows = int(snap["n_nodes"].sum().item())
    kept = int(r.n_nodes.sum().item())
    moved_bytes = 2 * kept * (3 * 8 + 4 + 5 * 8) + nq * K * 4  # rows read and written, new_index written
    res["a_repair_cfg3"] = {"repair_tree": t_rep, "validate_tree+repair_tree": t_both, "rows": rows, "rows_kept": kept,
                            "rows_pruned": int(rep.n_pruned.sum().item()), "found_before": int((snap["status"] == 0).sum().item()),
                            "reopened": int(rep.reopened.sum().item()), "bytes_moved_estimate": moved_bytes}

    # (b) the cut queries: repair + resume of the whole result, against a fresh plan of just those queries
    cut = torch.nonzero(rep.reopened).flatten()
    n_cut = int(cut.numel())
    t_resume = timed(lambda: (p.repair_tree(r, v), p.rrt_resume(r)), args.reps, restore)
    restore()
    p.repair_tree(r, v)
    p.rrt_resume(r)
    found_resume = int((r.status[cut] == 0).sum().item())
    c_starts, c_goals = starts[cut.cpu().numpy()], goals[cut.cpu().numpy()]
    c_sxy, c_sth = sxy[cut].contiguous(), sth[cut].contiguous()
    t_fresh = timed(lambda: p.rrt(c_starts, c_goals, c_sxy, c_sth, K=K), args.reps, lambda: None)
    fresh = p.rrt(c_starts, c_goals, c_sxy, c_sth, K=K)
    res["b_cut_queries"] = {"cut": n_cut,
                            "repair_tree+rrt_resume": dict(t_resume, found=found_resume),
                            "fresh_rrt": dict(t_fresh, found=int((fresh.status == 0).sum().item()))}
    res["gpu_after"] = gpu_info()
    if args.parent:
        res["c_bench_alternated"] = bench_alternated(os.path.abspath(args.parent), args.pairs, args.out)
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out, "mb_repair.json"), "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
