"""Batched main.py missions (Planner.missions / trrt_mission_batch) against the serial main.chain flow.

Workloads (K = 300, main.py's default; Theta* waypoints; seeded rand_conf streams, reference parity):
  map2   4 096 missions on map2 (300 x 300), random free start / goal cells (bench.random_queries, seed 31)
  cfg5  16 384 missions over the 64 cfg-5 maps (256 x 256, bench.synthetic_map(256, 0.15, 4, 7 + m)), per-mission map ids
Reported per workload: missions/s end to end (route, the one host read, host-side seeded normals, chain); CUDA-event
times of Theta* alone and of the chain alone (device normals, so no host generation in the window); the kernel split
of the chain (mission stage / commit kernels vs the fused RRT kernel) from one torch.profiler run; the host time to
generate the seeded normals; the stage count and n_active per stage.  On map2 also: the drop-in main.chain per
mission (32 missions) and mission_chain over the C oracle (tests/mission_oracle.py) on one host core (64 missions).  The first 16 missions of
each workload are checked bitwise against the oracle.

    python profiles/tools/mb_missions.py [--out profiles/r3] [--reps 3] [--seed-stream host|device]

--seed-stream device draws the seeded normals of the end-to-end runs on the GPU (Planner.missions(seed_stream="device"),
the same bits); host_seeded_normals_s is still numpy's time for them.
"""
from __future__ import annotations

import argparse
import builtins
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from tests.mission_oracle import mission_chain  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power = out[0].split(", ")
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def seeded_normals(n_seg, seeds, K):
    need = 3 * (K - 1) * np.asarray(n_seg)
    t = time.perf_counter()
    flat = np.empty(int(need.sum()))
    o = 0
    for m, s in enumerate(seeds):
        flat[o:o + need[m]] = np.random.RandomState(int(s)).standard_normal(int(need[m]))
        o += need[m]
    return time.perf_counter() - t, flat


def bits_equal(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    return np.array_equal(np.where(np.isnan(a), 0, a).view(np.int64), np.where(np.isnan(b), 0, b).view(np.int64))


def check_oracle(h, free_of, seeds, K, n):
    bad = 0
    for m in range(n):
        if int(h["n_seg"][m]) == 0:
            continue
        wp = [tuple(map(int, w)) for w in h["waypoints"][m, :int(h["n_waypoints"][m])]]
        z = np.random.RandomState(int(seeds[m])).standard_normal(3 * (K - 1) * (len(wp) - 1))
        o = mission_chain(free_of(m), wp, z, K)
        ok = int(h["status"][m]) == o["status"] and int(h["path_len"][m]) == len(o["path"])
        ok = ok and bits_equal(h["path"][m, :len(o["path"])], o["path"])
        for s, r in enumerate(o["segments"]):
            ok = ok and int(h["n_nodes"][m, s]) == r["n_nodes"] and int(h["iters"][m, s]) == r["iters"]
        bad += not ok
    return bad


def run(torch, planner, sg, seeds, K, map_id, reps, tag, seed_stream="host"):
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    res = planner.missions(start_goal=sg, seeds=seeds, K=K, map_id=map_id, seed_stream=seed_stream)  # warm-up (and the checked result)
    torch.cuda.synchronize()
    h = res.host()
    n_seg = h["n_seg"]
    order, n_active = res.schedule
    gen_s, _ = seeded_normals(n_seg, seeds, K)
    # end to end: route, host read, seeded normals, chain
    e2e = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        planner.missions(start_goal=sg, seeds=seeds, K=K, map_id=map_id, seed_stream=seed_stream)
        torch.cuda.synchronize()
        e2e.append(time.perf_counter() - t)
    # Theta* alone
    th = []
    for _ in range(reps):
        a, b = ev(), ev()
        a.record()
        planner.theta(sg, map_id=map_id)
        b.record()
        torch.cuda.synchronize()
        th.append(a.elapsed_time(b) / 1e3)
    # chain alone: the same waypoints, device normals (one row per mission, the length the longest needs)
    wps = [h["waypoints"][m, :int(h["n_waypoints"][m])] if n_seg[m] else h["waypoints"][m, :1] for m in range(len(sg))]
    L = max(int(3 * (K - 1) * n_seg.max()), 1)
    z = torch.randn(len(sg), L, dtype=torch.float64, device=planner.device)
    planner.missions(waypoints=wps, normals=z, K=K, map_id=map_id)
    ch = []
    for _ in range(reps):
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        planner.missions(waypoints=wps, normals=z, K=K, map_id=map_id)
        b.record()
        torch.cuda.synchronize()
        ch.append(a.elapsed_time(b) / 1e3)
    # kernel split of the chain (separate, profiled run)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        planner.missions(waypoints=wps, normals=z, K=K, map_id=map_id)
        torch.cuda.synchronize()
    split = {}
    for e in prof.key_averages():
        name = e.key
        for k in ("mission_stage_kernel", "mission_commit_kernel", "mission_init_kernel", "rrt_kernel_spec"):
            if k in name:
                split[k] = split.get(k, 0.0) + e.device_time_total / 1e3  # ms
    n = len(sg)
    return h, {
        "missions": n, "K": K, "segments_total": int(n_seg.sum()), "stages": int(len(n_active)),
        "n_active": [int(v) for v in n_active], "status_counts": {str(k): int(v) for k, v in zip(*np.unique(h["status"], return_counts=True))},
        "e2e_s": e2e, "missions_per_s_e2e": n / float(np.median(e2e)),
        "theta_s": th, "chain_s_device_normals": ch, "missions_per_s_chain": n / float(np.median(ch)),
        "host_seeded_normals_s": gen_s, "kernel_ms_profiled": split, "tag": tag, "seed_stream": seed_stream,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed-stream", choices=("host", "device"), default="host",
                    help="where the seeded normals of the end-to-end runs are drawn")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mb_missions needs a CUDA device")
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    from theta_rrt_b200 import main as M
    out = {"gpu": gpu_info(), "workloads": {}}
    K = 300
    maps = bench.load_maps()
    free2 = maps["map2"]
    starts, goals = bench.random_queries(free2, 4096, 31)
    sg2 = np.concatenate([starts[:, :2], goals[:, :2]], axis=1).astype(np.int32)
    seeds2 = np.arange(4096) + 1_000_000
    p2 = Planner(OccupancyGrid(free2, device="cuda:0"), Params())
    h2, r2 = run(torch, p2, sg2, seeds2, K, None, args.reps, "map2", args.seed_stream)
    r2["oracle_mismatches_first16"] = check_oracle(h2, lambda m: free2, seeds2, K, 16)
    # serial references on the same missions
    M.set_map(free2)
    builtins.K = K
    import contextlib
    import io
    t = time.perf_counter()
    n_serial = 0
    for m in range(32):
        if int(h2["n_seg"][m]) == 0:
            continue
        wp = [tuple(map(int, w)) for w in h2["waypoints"][m, :int(h2["n_waypoints"][m])]]
        np.random.seed(int(seeds2[m]))
        with contextlib.redirect_stdout(io.StringIO()):
            try:
                M.chain(wp)
            except TypeError:
                pass
        n_serial += 1
    r2["serial_dropin_chain_s_per_mission"] = (time.perf_counter() - t) / max(n_serial, 1)
    r2["serial_dropin_missions"] = n_serial
    t = time.perf_counter()
    n_or = 0
    for m in range(64):
        if int(h2["n_seg"][m]) == 0:
            continue
        wp = [tuple(map(int, w)) for w in h2["waypoints"][m, :int(h2["n_waypoints"][m])]]
        mission_chain(free2, wp, np.random.RandomState(int(seeds2[m])).standard_normal(3 * (K - 1) * (len(wp) - 1)), K)
        n_or += 1
    r2["oracle_one_core_s_per_mission"] = (time.perf_counter() - t) / max(n_or, 1)
    r2["oracle_missions"] = n_or
    out["workloads"]["map2_4096"] = r2
    print(json.dumps({"map2": {k: r2[k] for k in ("missions_per_s_e2e", "missions_per_s_chain", "oracle_mismatches_first16")}}), flush=True)
    # cfg-5 maps
    maps5 = np.stack([bench.synthetic_map(256, 0.15, 4, 7 + m) for m in range(64)])
    rng = np.random.default_rng(55)
    mid = rng.integers(0, 64, 16384).astype(np.int32)
    cells = [np.argwhere(f) for f in maps5]
    u = rng.random((2, 16384))
    a = np.stack([cells[m][int(u[0, i] * len(cells[m]))] for i, m in enumerate(mid)])
    b = np.stack([cells[m][int(u[1, i] * len(cells[m]))] for i, m in enumerate(mid)])
    sg5 = np.stack([a[:, 1], a[:, 0], b[:, 1], b[:, 0]], 1).astype(np.int32)
    seeds5 = np.arange(16384) + 2_000_000
    p5 = Planner(OccupancyGrid(maps5, device="cuda:0"), Params())
    h5, r5 = run(torch, p5, sg5, seeds5, K, mid, args.reps, "cfg5", args.seed_stream)
    r5["oracle_mismatches_first16"] = check_oracle(h5, lambda m: maps5[mid[m]], seeds5, K, 16)
    out["workloads"]["cfg5_16384"] = r5
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "missions.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
