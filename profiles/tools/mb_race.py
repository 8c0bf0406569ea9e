"""Seed races: time to solution of one planning problem raced over S seeds in one call (Planner.rrt_race).

For each map (map1 with the default tolerance, map2; 32 random problems each, K = 5 001) and each seed count S:
  race      rand_conf streams of the S seeds drawn on the device, then one raced trrt_rrt_race_batch call
  no race   the same S members planned by one plain call (every member runs to its end); winner taken afterwards
  oracle    the C oracle on one host core: seeds tried in order (numpy stream, then a full run) until one reaches the goal,
            capped at ORACLE_SEEDS seeds and ORACLE_S seconds per problem
Per problem, CUDA events around the call and its synchronisation (the streams are drawn before the event pair; their
draw is reported apart).  Reported per (map, S): median and p90 ms, the winner's iterations (median), the fraction of
problems solved.  Every problem is warmed up once per S before it is timed.

    python profiles/tools/mb_race.py [--problems 32] [--seeds 1,148,1024,4144,16384] [--json OUT]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import util  # noqa: E402

ORACLE_SEEDS, ORACLE_S = 4096, 3.0


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    name, power, clk = out[0].split(", ")
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def stats(ms):
    ms = np.asarray(ms, np.float64)
    return {"median_ms": float(np.median(ms)), "p90_ms": float(np.percentile(ms, 90)), "min_ms": float(ms.min())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--problems", type=int, default=32)
    ap.add_argument("--seeds", default="1,148,1024,4144,16384")
    ap.add_argument("--K", type=int, default=5001)
    ap.add_argument("--skip-oracle", action="store_true")
    ap.add_argument("--json", help="also write the result line to this file")
    args = ap.parse_args()
    import torch
    from oracle import c_oracle as O
    from theta_rrt_b200 import OccupancyGrid, Params, Planner, samples
    if not torch.cuda.is_available():
        sys.exit("mb_race.py measures on the GPU: no CUDA device")
    K, NP = args.K, args.problems
    S_list = [int(s) for s in args.seeds.split(",")]
    z = np.load(os.path.join(ROOT, "tests", "golden", "maps.npz"))
    dev = torch.device("cuda:0")
    out = {"workload": f"{NP} random problems per map, K={K}, device-drawn rand_conf streams, default params",
           "gpu": gpu_info(), "maps": {}}

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        e1.synchronize()
        return r, e0.elapsed_time(e1)

    for which in ("map1", "map2"):
        free = z[which].astype(bool)
        p = Planner(OccupancyGrid(free, device=dev), Params(K=K))
        starts, goals = util.random_queries(free, NP, 777 if which == "map1" else 778)
        per_map = {}
        for S in S_list:
            race_ms, plain_ms, draw_ms, win_it, solved, agree = [], [], [], [], 0, 0
            for i in range(NP):
                seeds = np.arange(S, dtype=np.int64) + 100_000 * i
                st, gl = np.repeat(starts[i:i + 1], S, 0), np.repeat(goals[i:i + 1], S, 0)
                (sxy, sth), d_ms = timed(lambda: p.rand_conf(gl, seeds, K))
                draw_ms.append(d_ms)
                groups = torch.zeros(S, dtype=torch.int32, device=dev)
                d_st, d_gl = torch.from_numpy(st).to(dev), torch.from_numpy(gl).to(dev)
                run_race = lambda: p.rrt(d_st, d_gl, sxy, sth, K=K, race=groups, race_groups=1)  # noqa: E731
                run_plain = lambda: p.rrt(d_st, d_gl, sxy, sth, K=K)  # noqa: E731
                run_race(); run_plain()  # warm-up of this shape
                res, ms = timed(run_race)
                race_ms.append(ms)
                w = int(res.race_winner.cpu()[0])
                if w >= 0:
                    solved += 1
                    win_it.append(int(res.race_iters.cpu()[0]))
                del res
                res, ms = timed(run_plain)
                plain_ms.append(ms)
                h_st, h_it = res.status.cpu().numpy(), res.iters.cpu().numpy()
                f = np.nonzero(h_st == 0)[0]
                pw = int(f[np.argmin(h_it[f])]) if len(f) else -1  # argmin keeps the lowest index on ties
                agree += int(pw == w)
                del res, sxy, sth
            per_map[str(S)] = {"race": stats(race_ms), "no_race": stats(plain_ms), "draw": stats(draw_ms),
                               "winner_iters_median": float(np.median(win_it)) if win_it else None,
                               "solved_fraction": solved / NP, "winner_equals_no_race_argmin": agree / NP}
            print(which, S, json.dumps(per_map[str(S)]), flush=True)
        if not args.skip_oracle:
            # the CPU way: one host core tries the seeds in order until one reaches the goal
            P = O.Params()
            ms, tried, solved = [], [], 0
            for i in range(NP):
                g = ((goals[i, 0], goals[i, 1]), goals[i, 2])
                s0 = ((starts[i, 0], starts[i, 1]), starts[i, 2])
                t0 = time.perf_counter()
                n = 0
                while n < ORACLE_SEEDS and time.perf_counter() - t0 < ORACLE_S:
                    sxy, sth = samples.make_stream(g, K - 1, 100_000 * i + n, free.shape)
                    o = O.rrt(free, s0, g, sxy, sth, P, K=K, log_los=False)
                    n += 1
                    if o["status"] == 0:
                        solved += 1
                        break
                ms.append((time.perf_counter() - t0) * 1e3)
                tried.append(n)
            per_map["oracle_in_order"] = {**stats(ms), "seeds_tried_median": float(np.median(tried)),
                                          "solved_fraction": solved / NP, "cap": f"{ORACLE_SEEDS} seeds or {ORACLE_S} s"}
            print(which, "oracle", json.dumps(per_map["oracle_in_order"]), flush=True)
        out["maps"][which] = per_map
        del p
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line, flush=True)
    if args.json:
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
