"""Seeded sample streams (reference parity): numpy's RandomState on the host against the device generator
(Planner.legacy_normals / Planner.rand_conf, trrt_rng.cuh).

Workloads:
  cfg3     4 096 rand_conf streams of 5 000 samples (15 000 normals each), seeds 0..4095, goals on map1
  map2     the normals of mb_missions.py's map2 missions (4 096, Theta* routes, 3 * 299 normals per segment)
  cfg5     the normals of mb_missions.py's cfg-5 missions (16 384 over 64 maps)
Reported per workload: host numpy time (one RandomState per seed, as the host paths do), device time end to end
(host clock around the call and a device synchronise), and the device path split into its parts in a separate
instrumented run: draw kernel (CUDA events), the count read, the r2 copy + host libm log, the log copy + fixup kernel
(CUDA events), and on cfg3 the rand_conf kernel.  Also the undecided fraction (pairs that took the host's log) and a
bitwise comparison of the device output with numpy's.  Medians of --reps runs after a warm-up.

    python profiles/tools/mb_seeded_streams.py [--out DIR] [--reps 5]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import bench  # noqa: E402
from mb_missions import gpu_info  # noqa: E402


def host_normals(seeds, counts):
    t = time.perf_counter()
    flat = np.empty(int(np.sum(counts)))
    o = 0
    for s, n in zip(seeds, counts):
        flat[o:o + n] = np.random.RandomState(int(s)).standard_normal(int(n))
        o += n
    return time.perf_counter() - t, flat


def split_run(torch, p, seeds, counts):
    """The steps of Planner.legacy_normals, each timed."""
    from theta_rrt_b200 import _lib
    from theta_rrt_b200.planner import legacy_seeds
    dev = p.device
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    seeds = legacy_seeds(seeds)
    n = len(seeds)
    rng = np.zeros((n, 2), np.int64)
    rng[:, 1] = np.cumsum(counts)
    rng[1:, 0] = rng[:-1, 1]
    total = int(rng[-1, 1])
    out = torch.empty(total, dtype=torch.float64, device=dev)
    s_d = torch.from_numpy(seeds.view(np.int32)).to(dev)
    r_d = torch.from_numpy(rng).to(dev)
    cap = total // 16 + 1024
    fpos = torch.empty(cap, dtype=torch.int64, device=dev)
    fr2 = torch.empty(cap, dtype=torch.float64, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    work = torch.empty(256, dtype=torch.uint8, device=dev)
    a = _lib.CLegacyNormalsArgs(n_seeds=n, d_seeds=s_d.data_ptr(), d_range=r_d.data_ptr(), d_out=out.data_ptr(),
                                d_fix_pos=fpos.data_ptr(), d_fix_r2=fr2.data_ptr(), fix_cap=cap, d_fix_count=cnt.data_ptr(),
                                d_work=work.data_ptr(), work_bytes=256)
    st = torch.cuda.current_stream(dev).cuda_stream
    h_r2 = torch.empty(cap, dtype=torch.float64).pin_memory()
    h_log = torch.empty(cap, dtype=torch.float64).pin_memory()
    torch.cuda.synchronize()
    e0, e1, e2, e3 = ev(), ev(), ev(), ev()
    e0.record()
    _lib.check(p.lib.trrt_legacy_normals_draw(C.byref(a), st))
    e1.record()
    t0 = time.perf_counter()
    n_fix = int(cnt.cpu()[0])
    t1 = time.perf_counter()
    assert n_fix <= cap
    h_r2[:n_fix].copy_(fr2[:n_fix], non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    t2 = time.perf_counter()
    _lib.check(p.lib.trrt_libm_log_batch(h_r2.data_ptr(), h_log.data_ptr(), n_fix))
    t3 = time.perf_counter()
    e2.record()
    d_log = h_log[:n_fix].to(dev, non_blocking=True)
    _lib.check(p.lib.trrt_legacy_normals_fixup(C.byref(a), d_log.data_ptr(), n_fix, st))
    e3.record()
    torch.cuda.synchronize()
    return out, {"draw_kernel_ms": e0.elapsed_time(e1), "count_read_ms": (t1 - t0) * 1e3, "r2_copy_ms": (t2 - t1) * 1e3,
                 "host_log_ms": (t3 - t2) * 1e3, "log_copy_and_fixup_ms": e2.elapsed_time(e3), "undecided_pairs": n_fix,
                 "undecided_fraction_of_pairs": n_fix / max(1, int(sum((int(c) + 1) // 2 for c in counts)))}


def normals_workload(torch, p, seeds, counts, reps):
    host_s, flat = host_normals(seeds, counts)
    p.legacy_normals(seeds, counts)  # warm-up
    torch.cuda.synchronize()
    dev_s = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out, _ = p.legacy_normals(seeds, counts)
        torch.cuda.synchronize()
        dev_s.append(time.perf_counter() - t)
    same = bool(np.array_equal(out.cpu().numpy().view(np.int64), flat.view(np.int64)))
    _, split = split_run(torch, p, seeds, counts)
    return {"seeds": len(seeds), "normals": int(np.sum(counts)), "host_numpy_s": host_s, "device_s": dev_s,
            "device_s_median": float(np.median(dev_s)), "speedup": host_s / float(np.median(dev_s)),
            "bitwise_equal_numpy": same, "split": split}


def mission_counts(torch, p, sg, K, map_id=None):
    r = p.theta(sg, map_id=map_id)
    n_wp, st = r.path_len.cpu().numpy(), r.status.cpu().numpy()
    n_seg = np.where((st == 0) & (n_wp <= r.path.shape[1]), np.maximum(n_wp - 1, 0), 0)
    return 3 * (K - 1) * n_seg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mb_seeded_streams needs a CUDA device")
    from theta_rrt_b200 import OccupancyGrid, Params, Planner, samples
    out = {"gpu": gpu_info(), "host_threads_for_log": os.cpu_count(), "workloads": {}}
    K = 300
    maps = bench.load_maps()
    # cfg3: rand_conf streams
    free1 = maps["map1"]
    p1 = Planner(OccupancyGrid(free1, device="cuda:0"), Params())
    nq, S = 4096, 5000
    starts, goals = bench.random_queries(free1, nq, 3)
    seeds = np.arange(nq)
    t = time.perf_counter()
    hx = np.empty((nq, S, 2), np.int32)
    ht = np.empty((nq, S))
    for q in range(nq):
        hx[q], ht[q] = samples.make_stream(((goals[q, 0], goals[q, 1]), goals[q, 2]), S, int(seeds[q]), free1.shape)
    host_s = time.perf_counter() - t
    p1.rand_conf(goals, seeds, S + 1)
    torch.cuda.synchronize()
    dev_s = []
    for _ in range(args.reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        sxy, sth = p1.rand_conf(goals, seeds, S + 1)
        torch.cuda.synchronize()
        dev_s.append(time.perf_counter() - t)
    same = bool(np.array_equal(sxy.cpu().numpy(), hx) and np.array_equal(sth.cpu().numpy().view(np.int64), ht.view(np.int64)))
    nz, split = split_run(torch, p1, seeds, np.full(nq, 3 * S))
    g = torch.from_numpy(goals).to("cuda:0")
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    p1.lib.trrt_rand_conf_batch(free1.shape[0], free1.shape[1], 0.4, 100.0, nq, S, g.data_ptr(), nz.data_ptr(), sxy.data_ptr(), 0,
                                sth.data_ptr(), torch.cuda.current_stream().cuda_stream)
    b.record()
    torch.cuda.synchronize()
    split["rand_conf_kernel_ms"] = a.elapsed_time(b)
    out["workloads"]["cfg3_rand_conf_4096x5000"] = {"host_numpy_make_stream_s": host_s, "device_s": dev_s,
                                                    "device_s_median": float(np.median(dev_s)),
                                                    "speedup": host_s / float(np.median(dev_s)), "bitwise_equal_numpy": same,
                                                    "split": split}
    print(json.dumps({"cfg3": out["workloads"]["cfg3_rand_conf_4096x5000"]}), flush=True)
    # map2 missions (mb_missions.py's queries and seeds)
    free2 = maps["map2"]
    st2, gl2 = bench.random_queries(free2, 4096, 31)
    sg2 = np.concatenate([st2[:, :2], gl2[:, :2]], axis=1).astype(np.int32)
    p2 = Planner(OccupancyGrid(free2, device="cuda:0"), Params())
    c2 = mission_counts(torch, p2, sg2, K)
    out["workloads"]["map2_missions_normals"] = normals_workload(torch, p2, np.arange(4096) + 1_000_000, c2, args.reps)
    print(json.dumps({"map2": out["workloads"]["map2_missions_normals"]}), flush=True)
    # cfg-5 missions
    maps5 = np.stack([bench.synthetic_map(256, 0.15, 4, 7 + m) for m in range(64)])
    rng = np.random.default_rng(55)
    mid = rng.integers(0, 64, 16384).astype(np.int32)
    cells = [np.argwhere(f) for f in maps5]
    u = rng.random((2, 16384))
    pa = np.stack([cells[m][int(u[0, i] * len(cells[m]))] for i, m in enumerate(mid)])
    pb = np.stack([cells[m][int(u[1, i] * len(cells[m]))] for i, m in enumerate(mid)])
    sg5 = np.stack([pa[:, 1], pa[:, 0], pb[:, 1], pb[:, 0]], 1).astype(np.int32)
    p5 = Planner(OccupancyGrid(maps5, device="cuda:0"), Params())
    c5 = mission_counts(torch, p5, sg5, K, map_id=mid)
    out["workloads"]["cfg5_missions_normals"] = normals_workload(torch, p5, np.arange(16384) + 2_000_000, c5, args.reps)
    print(json.dumps({"cfg5": out["workloads"]["cfg5_missions_normals"]}), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "seeded_streams.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
