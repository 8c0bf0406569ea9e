#!/usr/bin/env python
"""bench.py -- theta-rrt planning inner loop on B200: RRT expansions/s (+ LOS checks/s, Theta* expansions/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[2], SURVEY.md 8d cfg 3): batched RRT, 4096 independent
queries per GPU on map1 (100x100), K=5001 (5000 expansions each), tol_xy=0 so every query runs all
iterations, start/goal uniform over free cells (default_rng(1234)), per-query sample stream equal to
np.random.seed(q) + 5000 x rand_conf(goal_q).  One "step" = one fused-kernel pass over the batch.

The single JSON line carries
  value      RRT expansions/s with all inputs resident in HBM (CUDA events on the launch stream)
  e2e        the same metric through the public host-buffer API (pinned H2D of the sample streams,
             kernel, D2H of the trees) inside the timed region
  roofline   the fused rrt kernel against the roof that physically bounds it (the fp64 pipe; peaks
             measured by profiles/tools/mb_peaks.cu -> profiles/peaks.json, per-launch instruction /
             byte counts from the committed ncu captures -> profiles/kernel_counts.json), with the
             SURVEY 8(d) algorithmic-byte figure kept as `algorithmic_equiv`
  parity     the first queries of the timed launch compared with the CPU oracle (trees bit for bit)
  secondary  cfg 4 (LOS checks/s over an 8192^2 grid, nearest-node scan over a 2^20-node tree), Theta* on
             map2 and cfg 5 (65536 mixed RRT / Theta* queries over 64 random maps); under --gpus N the
             rays and the mixed queries are sharded over the ranks, each with its own roofline
  cpu_baseline  the C oracle (a port of the reference) and the unmodified Python reference (oracle/_ref)
             on the host cores, bounded samples

--impl reference times the reference's algorithm on the host CPU: the C port on all host threads (the
line's value) and the unmodified Python sources, one process and one per core, when oracle/_ref is
present.  Multi-GPU (torchrun, one rank per GPU): queries are sharded by rank, no data-path collective;
a gather of the per-query summaries over NCCL closes each step ("scaling": "weak").

--dump-outputs DIR writes what the last timed step of the headline workload returned (rank 0's queries) as float64
.npy files in DIR (dump_outputs).  The inputs are seeded, so two builds run with the same arguments can be compared
file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NQ_PER_GPU = 4096
K_RRT = 5001
MAP_SEED = 1234
K_PYREF = 601  # the Python reference is timed on the first 600 iterations of a query per process (about 10 s)
DUMP_TREES = 96  # --dump-outputs: trees of 96 queries are at most 96 x K_RRT rows x 112 B = 54 MB
WORKLOAD = ("cfg3: batched RRT, %d independent queries per GPU on map1.png (100x100), K=%d "
            "(5000 expansions each), tol_xy=0, seeded rand_conf streams")


# --------------------------------------------------------------------------- workload
def load_maps():
    z = np.load(os.path.join(ROOT, "tests", "golden", "maps.npz"))
    return {k: z[k].astype(bool) for k in z.files}


def random_queries(free, nq, seed, offset=0):
    rng = np.random.default_rng(seed)
    cells = np.argwhere(free)
    n_all = offset + nq
    a = cells[rng.integers(len(cells), size=n_all)]
    b = cells[rng.integers(len(cells), size=n_all)]
    hs, hg = rng.uniform(-180, 180, n_all), rng.uniform(-180, 180, n_all)
    starts = np.stack([a[:, 1], a[:, 0], hs], axis=1).astype(np.float64)[offset:]
    goals = np.stack([b[:, 1], b[:, 0], hg], axis=1).astype(np.float64)[offset:]
    return starts, goals


def make_rrt_workload(free, nq, K, first_query=0):
    from theta_rrt_b200 import samples
    starts, goals = random_queries(free, nq, MAP_SEED, offset=first_query)
    sxy = np.empty((nq, K - 1, 2), np.int32)
    sth = np.empty((nq, K - 1), np.float64)
    for q in range(nq):
        g = ((goals[q, 0], goals[q, 1]), goals[q, 2])
        sxy[q], sth[q] = samples.make_stream(g, K - 1, first_query + q, free.shape)
    return starts, goals, sxy, sth


def synthetic_map(n, p, block, seed):
    rng = np.random.default_rng(seed)
    nb = (n + block - 1) // block
    coarse = rng.random((nb, nb)) >= p
    return np.kron(coarse, np.ones((block, block), bool))[:n, :n]


def make_segments(free, n, seed, maxlen=512):
    """cfg 4 raycast input: n segments from a random free cell, length uniform [1, maxlen] px, uniform direction."""
    rng = np.random.default_rng(seed)
    side = free.shape[0]
    cells = np.argwhere(free)
    c = cells[rng.integers(len(cells), size=n)]
    length = rng.uniform(1, maxlen, n)
    ang = rng.uniform(0, 2 * np.pi, n)
    x0, y0 = c[:, 1], c[:, 0]
    x1 = np.clip((x0 + length * np.cos(ang)).astype(np.int64), 0, side - 1)
    y1 = np.clip((y0 + length * np.sin(ang)).astype(np.int64), 0, side - 1)
    return np.stack([x0, y0, x1, y1], axis=1).astype(np.int32)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            if t0 is not None and (ts < t0 - 0.1 or ts > t1 + 0.3):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(np.max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _load_json(name):
    p = os.path.join(ROOT, "profiles", name)
    try:
        return json.load(open(p))
    except Exception:
        return {}


def pipe_peaks():
    """Peaks of the pipes and on-chip memories, measured on this pool's B200 by profiles/tools/mb_peaks.cu."""
    return _load_json("peaks.json")


def kernel_counts(kernel):
    """Per-launch instruction / byte counts of a kernel on ITS bench workload, from the committed ncu capture
    (profiles/kernel_counts.json; the workload is deterministic, so counts of one launch hold for every launch)."""
    return _load_json("kernel_counts.json").get(kernel, {})


def physical_roofline(kernel, ms, bound, alg=None, note=""):
    """roofline object for a kernel that is not HBM-bound: achieved rate on the pipe / memory that bounds it (ncu counts per
    launch / live CUDA-event time) over the peak measured by mb_peaks; the L2 / shared-memory / DRAM rates ride along."""
    pk, kc = pipe_peaks(), kernel_counts(kernel)
    sec = ms / 1e3
    r = {"kernel": kernel, "bound": bound, "achieved": None, "peak": None, "unit": None, "frac": None,
         "traffic": kc.get("dram_bytes"), "peak_source": "profiles/peaks.json (mb_peaks.cu on this pool's B200)",
         "counts_source": kc.get("source")}
    if bound == "fp64" and kc.get("fp64_warp_inst") and pk.get("fp64_dadd_lane_inst_per_s"):
        # a warp instruction occupies the pipe for all 32 lanes whatever its predicate mask: lane slots = warp instructions x 32
        r.update(achieved=kc["fp64_warp_inst"] * 32 / sec / 1e12, peak=pk["fp64_dadd_lane_inst_per_s"] / 1e12, unit="T fp64 lane-slots/s",
                 fp64_thread_inst_per_launch=kc.get("fp64_thread_inst"), fp64_warp_inst_per_launch=kc["fp64_warp_inst"])
    elif bound == "issue" and kc.get("warp_inst") and pk.get("issue_warp_inst_per_s_nominal"):
        r.update(achieved=kc["warp_inst"] / sec / 1e9, peak=pk["issue_warp_inst_per_s_nominal"] / 1e9, unit="G warp-inst/s")
    if r["achieved"] is not None:
        r["frac"] = r["achieved"] / r["peak"]
    if kc.get("l2_bytes") and pk.get("l2_read_GBps"):
        r["l2"] = {"achieved_GBps": kc["l2_bytes"] / sec / 1e9, "peak_GBps": pk["l2_read_GBps"],
                   "frac": kc["l2_bytes"] / sec / 1e9 / pk["l2_read_GBps"], "metric": "lts__t_bytes.sum"}
    if kc.get("smem_wavefronts") and pk.get("smem_read_GBps"):
        gbs = kc["smem_wavefronts"] * 128 / sec / 1e9
        r["smem"] = {"achieved_GBps": gbs, "peak_GBps": pk["smem_read_GBps"], "frac": gbs / pk["smem_read_GBps"],
                     "metric": "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum x 128 B"}
    if kc.get("dram_bytes"):
        hbm, _ = measured_peaks()
        r["dram"] = {"achieved_GBps": kc["dram_bytes"] / sec / 1e9, "peak_GBps": hbm, "frac": kc["dram_bytes"] / sec / 1e9 / hbm}
    if alg is not None:
        r["algorithmic_equiv"] = alg
    if note:
        r["note"] = note
    return r


# --------------------------------------------------------------------------- reference arm (CPU)
def python_reference(free, starts, goals, sxy, sth, cores):
    """The UNMODIFIED Python reference (rrt.rrt, rrt.py:130) on this box's host cores: one process, and one process per
    core (BASELINE.md section 3), on the first K_PYREF-1 iterations of the step's first queries.  None when the files are
    absent (oracle/_ref is a git-ignored verbatim copy made by oracle/make_ref.py at build time)."""
    from oracle import py_reference_bench as R
    if R.reference_dir() is None:
        return {"unavailable": "oracle/_ref (copy of the Python reference) not present on this box"}
    try:
        import scipy  # noqa: F401  (rrt.py:4)
    except Exception as e:  # pragma: no cover
        return {"unavailable": f"scipy missing on this box: {e}"}
    n = min(cores, len(starts))
    one = max((R.time_reference(free, starts, goals, sxy, sth, K_PYREF, procs=1) for _ in range(2)), key=lambda r: r[0])  # best of two
    allc = R.time_reference(free, starts, goals, sxy, sth, K_PYREF, procs=n)
    return {"kind": "reference", "unit": "expansions/s", "single_core_value": one[0], "all_cores_value": allc[0], "cores": n,
            "sample": f"first {K_PYREF - 1} iterations of one query per process (queries 0..{n - 1} of the step; single core: query 0), "
                      f"tol_xy=0, injected rand_conf stream; {allc[1]} iterations in {allc[2]:.1f} s wall with {n} processes",
            "source": R.reference_dir()}


def run_reference_arm(args, rank, world):
    """The reference's algorithm on the host CPU: C oracle port, all host threads, bounded sample per step; next to it the
    unmodified Python reference, single process and one process per core."""
    if rank != 0:
        return
    from oracle import c_oracle as O
    free = load_maps()["map1"]
    cores = os.cpu_count() or 1
    nq = max(4 * cores, 32)  # ~0.2 s of one core per query, four queries per thread: a step is about a second of wall
    starts, goals, sxy, sth = make_rrt_workload(free, nq, K_RRT)
    P = O.Params(tol_xy=0.0)
    O.lib()
    for _ in range(max(args.warmup, 1)):
        O.rrt_batch(free, starts[:cores], goals[:cores], sxy[:cores], sth[:cores], K_RRT, P, threads=cores, want_nodes=False)
    t0 = time.perf_counter()
    done = 0
    for _ in range(args.steps):
        r = O.rrt_batch(free, starts, goals, sxy, sth, K_RRT, P, threads=cores, want_nodes=True)
        done += int(r["iters"].sum())  # executed loop iterations (queries the reference would abort stop early)
    dt = time.perf_counter() - t0
    value = done / dt
    sample = f"{nq} of the {NQ_PER_GPU} queries per step, K={K_RRT}, {cores} threads"
    line = {"impl": "reference", "metric": "rrt_expansions_per_sec", "value": value, "unit": "expansions/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD % (NQ_PER_GPU, K_RRT), "queries_per_gpu": NQ_PER_GPU, "K": K_RRT,
                       "sample_queries_per_step": nq, "host_threads": cores},
            "cpu_baseline": {"value": value, "unit": "expansions/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "expansions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "python_reference": python_reference(free, starts, goals, sxy, sth, cores),
            "note": "value = the reference's algorithm as its C restatement (oracle/, kind 'port') on all host threads: the "
                    "fastest CPU form of the path, hence the conservative denominator; python_reference = the unmodified "
                    "Python sources (kind 'reference') timed in the same run"}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm
def time_steps(torch, fn, steps, warmup, dist_on):
    """W warm-up calls, then `steps` timed calls with per-step CUDA events on the current stream."""
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
        torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0 = time.time()
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t1 = time.time()
    if dist_on:
        dist.barrier()
        torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in ev]
    return ms, t0, t1


def max_over_ranks(torch, dist_on, dev, v):
    t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
    if dist_on:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(torch, dist_on, dev, vals):
    t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device=dev)
    if dist_on:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return [float(x) for x in t.tolist()]


def check_parity(free, starts, goals, sxy, sth, K, res, n):
    """The first n queries of the timed launch against the CPU oracle: tree size, parents, status, iteration count and the
    node coordinates bit for bit.  Raises on the first difference (a fast kernel with other results is not done)."""
    from oracle import c_oracle as O
    cores = os.cpu_count() or 1
    r = O.rrt_batch(free, starts[:n], goals[:n], sxy[:n], sth[:n], K, O.Params(tol_xy=0.0), threads=cores, want_nodes=True)
    g = {k: getattr(res, k)[:n].cpu().numpy() for k in ("n_nodes", "status", "iters", "sol", "parent", "node_x", "node_y", "node_theta")}
    for k in ("n_nodes", "status", "iters", "sol"):
        if not np.array_equal(g[k], r[k]):
            raise SystemExit(f"PARITY FAILURE: {k} differs from the oracle on the first {n} queries")
    rows = 0
    for q in range(n):
        m = int(r["n_nodes"][q])
        rows += m
        if not np.array_equal(g["parent"][q, :m], r["parent"][q, :m]):
            raise SystemExit(f"PARITY FAILURE: parents of query {q} differ from the oracle")
        for j, k in enumerate(("node_x", "node_y", "node_theta")):
            if not np.array_equal(g[k][q, :m].view(np.int64), np.ascontiguousarray(r["nodes"][q, :m, j]).view(np.int64)):
                raise SystemExit(f"PARITY FAILURE: {k} of query {q} differs bitwise from the oracle")
    return {"checked_queries": n, "tree_rows_compared_bitwise": rows, "against": "oracle/trrt_oracle.c (C restatement, pinned to the reference)",
            "fields": "n_nodes, status, iters, sol, parent, node_x/y/theta (bit patterns)", "result": "identical"}


def dump_outputs(out_dir, res, first_query):
    """What one Planner.rrt call returned, as float64 .npy files in out_dir:
      n_nodes, sol, status, iters         [q]      every query of the call
      queries                             [s]      ids of DUMP_TREES queries drawn with default_rng(0), ascending
      node_x, node_y, node_theta, parent  [rows]   tree rows 0 .. n_nodes-1 of those queries, concatenated in the
      u, u_nan                            [rows,5] order of `queries` (rows past n_nodes are never written)
    u holds 0 where the kernel returns NaN (the root row, icc and rad of a straight edge) and u_nan is 1 there, so that
    equal outputs compare equal without NaN-aware comparisons.  The per-query arrays take 32 B a query; a B200 cannot
    hold the outputs of enough queries to take them past 16 MB."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = {k: getattr(res, k).cpu().numpy().astype(np.float64) for k in ("n_nodes", "sol", "status", "iters")}
    nq = len(out["n_nodes"])
    pick = np.sort(np.random.default_rng(0).choice(nq, size=min(DUMP_TREES, nq), replace=False))
    idx = torch.from_numpy(pick).to(res.node_x.device)
    n = out["n_nodes"][pick].astype(np.int64)
    for k in ("node_x", "node_y", "node_theta", "parent", "u"):
        a = getattr(res, k)[idx].cpu().numpy()
        out[k] = np.concatenate([a[j, :n[j]] for j in range(len(pick))]).astype(np.float64)
    out["u_nan"] = np.isnan(out["u"]).astype(np.float64)
    out["u"][out["u_nan"] == 1] = 0.0
    out["queries"] = (first_query + pick).astype(np.float64)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    mb = sum(v.nbytes for v in out.values()) / 2**20
    print(f"bench: {len(out)} output arrays ({mb:.1f} MiB) written to {out_dir}", file=sys.stderr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--queries", type=int, default=NQ_PER_GPU, help="queries per GPU (default: the cfg-3 size)")
    ap.add_argument("--lanes", type=int, default=0, help="lanes per query of the fused kernel (0 = auto)")
    ap.add_argument("--schedule", type=int, default=0, help="0 = speculative window (default), 1 = cooperative")
    ap.add_argument("--dense-d2h", action="store_true", help="e2e: copy the full [q][K] tree arrays instead of the packed rows")
    ap.add_argument("--chunks", type=int, default=4, help="pieces of the e2e host-buffer pipeline (Planner.rrt_host)")
    ap.add_argument("--skip-secondary", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-python-ref", action="store_true", help="do not time the Python reference (about 30 s of CPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from theta_rrt_b200 import OccupancyGrid, Params, Planner, shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist_on = world > 1
    # one process per GPU: stay on the GPU's NUMA node before any pinned buffer exists (not at N = 1, where the CPU
    # baseline legs of this process use every host core)
    numa = shard.bind_host_to_device(local_rank) if (dist_on and not os.environ.get("TRRT_NO_NUMA_BIND")) else None
    if dist_on:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    maps = load_maps()
    free = maps["map1"]
    nq = args.queries
    K = K_RRT
    total_q = nq * world
    lo, hi = shard.shard_range(total_q, rank, world)  # contiguous block of query ids of this rank
    starts, goals, sxy, sth = make_rrt_workload(free, hi - lo, K, first_query=lo)
    planner = Planner(OccupancyGrid(free, device=dev), Params(tol_xy=0.0, K=K))

    # ---- device-resident inputs (value) and pinned host inputs (e2e; sample coordinates as int16 pairs)
    h_in = [torch.from_numpy(a).pin_memory() for a in (starts, goals, sxy, sth)]
    d_in = [t.to(dev) for t in h_in]
    h_in16 = [h_in[0], h_in[1], torch.from_numpy(sxy.astype(np.int16)).pin_memory(), h_in[3]]
    torch.cuda.synchronize()

    # one untimed instrumented run: counters for the algorithmic-byte accounting
    r0 = planner.rrt(*d_in, K=K, counters=True, lanes=args.lanes, schedule=args.schedule)
    torch.cuda.synchronize()
    counters = r0.counters.sum(dim=0).cpu().numpy().astype(np.int64)
    n_nodes_total = int(r0.n_nodes.sum().item())
    iters_total = int(r0.iters.sum().item())
    # tol_xy=0 disables the goal test, but a query still ends early when the reference itself would raise
    # (quirk Q7: rrt.py:170-171 calls drive() on a straight-line steer -> TypeError); such queries are
    # reported with status 4 and only their executed iterations count as work
    status_bad = int((r0.status > 1).sum().item())
    del r0

    launches = {"n": 0}
    keep = {}

    def step_resident():
        keep["res"] = planner.rrt(*d_in, K=K, lanes=args.lanes, schedule=args.schedule)
        launches["n"] += 1
        if dist_on:  # optional gather of the per-query summaries (SURVEY.md 8e)
            rec = torch.stack([keep["res"].n_nodes, keep["res"].sol, keep["res"].status], dim=1)
            keep["gathered"] = shard.gather_records(rec, total_q)

    clocks = ClockSampler(local_rank)
    clocks.start()
    ms, t0, t1 = time_steps(torch, step_resident, args.steps, args.warmup, dist_on)
    clk = clocks.stop(t0, t1)
    launches_timed = args.steps
    total_ms = float(sum(ms))
    total_ms_max = max_over_ranks(torch, dist_on, dev, total_ms)
    it_all = sum_over_ranks(torch, dist_on, dev, [iters_total, n_nodes_total, status_bad])
    expansions_per_step_all = int(it_all[0])  # loop iterations actually executed (rrt.py:141)
    value = expansions_per_step_all * args.steps / (total_ms_max / 1e3)

    # ---- parity of the timed launch (rank 0): the first queries against the CPU oracle
    parity = None
    if rank == 0 and not args.skip_cpu:
        parity = check_parity(free, starts, goals, sxy, sth, K, keep["res"], min(64, hi - lo))
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, keep["res"], lo)

    # ---- roofline of the fused kernel (this rank's launch)
    alg_bytes = 16 * int(counters[0]) + 16 * iters_total + (28 + 40) * n_nodes_total
    ms_kernel = total_ms / args.steps
    peak, peak_src = measured_peaks()
    alg_gbs = alg_bytes / (ms_kernel / 1e3) / 1e9
    roofline = physical_roofline(
        "rrt_kernel", ms_kernel, "fp64",
        alg={"achieved": alg_gbs, "peak": peak, "unit": "GB/s", "frac": alg_gbs / peak, "peak_source": peak_src,
             "algorithmic_bytes_per_launch": alg_bytes, "pairs_scanned_per_launch": int(counters[0]),
             "definition": "SURVEY 8(d): 16 B per scanned (query,node) pair of the sequential loop + 16 B per sample + 68 B per "
                           "inserted node, over the measured HBM copy peak; NOT a physical HBM figure (trees are L1/L2/shared-memory "
                           "resident), kept for comparison with round 1"},
        note="bound by the fp64 pipe: the nearest scan issues 6 fp64-pipe instructions per (sample, node) pair and the steer / libm "
             "chain is fp64 too; achieved = fp64-pipe warp instructions per launch x 32 (ncu, smsp__inst_executed_pipe_fp64) / "
             "CUDA-event time of this run, peak = DADD rate measured by mb_peaks.cu")
    if nq != NQ_PER_GPU or args.lanes or args.schedule:
        roofline["counts_note"] = "ncu counts were taken on the default cfg-3 launch; this run uses other options"

    # ---- e2e through the host-buffer API: pinned H2D of the inputs, kernel, D2H of the trees
    nql = hi - lo
    shapes = {"node_x": ((nql, K), torch.float64), "node_y": ((nql, K), torch.float64), "node_theta": ((nql, K), torch.float64),
              "parent": ((nql, K), torch.int32), "u": ((nql, K, 5), torch.float64), "n_nodes": ((nql,), torch.int32),
              "sol": ((nql,), torch.int32), "status": ((nql,), torch.int32), "iters": ((nql,), torch.int32),
              "row_start": ((nql,), torch.int64)}
    h_all = {k: torch.empty(sh, dtype=dt).pin_memory() for k, (sh, dt) in shapes.items()}
    vro = not args.dense_d2h
    small = ("n_nodes", "sol", "status", "iters") + (("row_start",) if vro else ())

    def e2e_run(with_u):
        """`steps` streamed batches through Planner.rrt_host; returns (ms per step, H2D bytes, D2H bytes)."""
        out = {k: v for k, v in h_all.items() if (k != "u" or with_u) and (k != "row_start" or vro)}
        h2d = sum(t.numel() * t.element_size() for t in h_in16)
        row = 28 + (40 if with_u else 0)
        d2h = (n_nodes_total * row if vro else nql * K * row) + sum(out[k].numel() * out[k].element_size() for k in small)

        def step():
            planner.rrt_host(*h_in16, out=out, K=K, chunks=args.chunks, wait=False, lanes=args.lanes, schedule=args.schedule, valid_rows_only=vro)
        for _ in range(2):
            step()
        planner.host_sync(); torch.cuda.synchronize()
        if dist_on:
            dist.barrier()
            torch.cuda.synchronize()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        for _ in range(args.steps):
            step()
        planner.host_sync()
        eb.record()
        torch.cuda.synchronize()
        if dist_on:
            dist.barrier()
            torch.cuda.synchronize()
        msx = max_over_ranks(torch, dist_on, dev, ea.elapsed_time(eb)) / args.steps
        # the host really received this step's trees: sizes, and the last row of every tree against the resident result
        assert int(out["n_nodes"].sum()) == n_nodes_total
        last_dev = (keep["res"].n_nodes.long() - 1).clamp(min=0)
        rows = torch.arange(nql, device=dev)
        if vro:
            last_host = out["row_start"] + last_dev.cpu()
            assert torch.equal(out["node_x"].view(-1)[last_host], keep["res"].node_x[rows, last_dev].cpu())
            assert torch.equal(out["parent"].view(-1)[last_host], keep["res"].parent[rows, last_dev].cpu())
        else:
            assert torch.equal(out["node_x"][rows.cpu(), last_dev.cpu()], keep["res"].node_x[rows, last_dev].cpu())
        # the same call with every step completed before the next starts
        def serial():
            planner.rrt_host(*h_in16, out=out, K=K, chunks=args.chunks, wait=True, lanes=args.lanes, schedule=args.schedule, valid_rows_only=vro)
            torch.cuda.synchronize()
        mss, _, _ = time_steps(torch, serial, min(args.steps, 3), 1, dist_on)
        return msx, int(h2d), int(d2h), float(sum(mss)) / len(mss)

    ms_e2e, h2d, d2h, serial_ms = e2e_run(with_u=False)
    ms_e2e_u, h2d_u, d2h_u, serial_ms_u = e2e_run(with_u=True)
    e2e_value = expansions_per_step_all / (ms_e2e / 1e3)
    launches_e2e = args.steps * args.chunks  # one fused kernel per piece (it packs its own rows)
    keep.clear()
    del h_all
    torch.cuda.empty_cache()

    line = {"metric": "rrt_expansions_per_sec", "value": value, "unit": "expansions/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD % (nq, K),
                       "queries_per_gpu": nq, "K": K, "lanes_per_query": args.lanes or 32,
                       "schedule": "speculative window" if args.schedule == 0 else "cooperative",
                       "parallelism": "query-sharded x%d, no data-path collective" % world,
                       "l2_policy": "inputs+outputs per step (%.2f GB) exceed the 126 MB L2" %
                                    ((16 * iters_total + 68 * n_nodes_total) / 1e9)},
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "expansions/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e,
                    "api": "Planner.rrt_host(pinned inputs with int16 sample coordinates, pinned outputs node_x/y/theta, parent, "
                           "n_nodes, sol, status, iters%s, chunks=%d, wait=False%s) per step, host_sync() after the last step"
                           % (", row_start" if vro else "", args.chunks, ", valid_rows_only=True" if vro else ""),
                    "serial_ms_per_step": serial_ms, "host_numa_binding": numa,
                    "with_u": {"value": expansions_per_step_all / (ms_e2e_u / 1e3), "ms_per_step": ms_e2e_u, "h2d_bytes_per_step": h2d_u,
                               "d2h_bytes_per_step": d2h_u, "serial_ms_per_step": serial_ms_u,
                               "note": "the same call with `u` (steer, icc, rad, dist of cameFrom, 40 B per node) among the outputs"},
                    "note": "steps are streamed: the transfers of a step overlap the planning of its neighbours; the trees travel as "
                            "the rows that exist (packed by the fused kernel itself); `u` is opt-in for the host transfer; "
                            "serial_ms_per_step is the same call with every step completed before the next starts"},
            "gpu_launches": launches_timed, "gpu_launches_e2e": launches_e2e,
            "roofline": roofline,
            "parity": parity,
            "expansions_per_step": expansions_per_step_all,
            "accepted_nodes_per_sec": (int(it_all[1]) - total_q) * args.steps / (total_ms_max / 1e3),
            "queries_ended_by_reference_TypeError": int(it_all[2])}

    if not args.skip_secondary:
        sec = secondary_benchmarks(torch, dev, maps, peak, peak_src, args, rank, world, dist_on)
        if rank == 0:
            line["secondary"] = sec
    if rank == 0 and world == 1 and not args.skip_cpu:
        line["cpu_baseline"] = cpu_baseline(free, starts, goals, sxy, sth, args)
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line), flush=True)


def make_cfg5(rank, world, nq5=32768, K5=1001):
    """BASELINE cfg 5: 65 536 queries = 32 768 RRT (as cfg 3, K = 1 001) + 32 768 Theta*, each bound to one of 64 random
    256 x 256 maps (4x4-block Bernoulli obstacles, p = 0.15, default_rng(7 + map)); this rank's contiguous shard."""
    from theta_rrt_b200 import samples, shard
    n_maps5, side5 = 64, 256
    maps5 = np.stack([synthetic_map(side5, 0.15, 4, 7 + m) for m in range(n_maps5)])
    r5 = np.random.default_rng(77)
    mid_r = r5.integers(0, n_maps5, nq5).astype(np.int32)
    mid_t = r5.integers(0, n_maps5, nq5).astype(np.int32)
    free_cells = [np.argwhere(m) for m in maps5]
    u = r5.random((4, nq5))  # one free cell per (query, endpoint), drawn for all queries so that shards agree

    def pick(mids, col):
        return np.stack([free_cells[m][int(u[col, i] * len(free_cells[m]))] for i, m in enumerate(mids)])
    a5, b5, ta, tb = pick(mid_r, 0), pick(mid_r, 1), pick(mid_t, 2), pick(mid_t, 3)
    hs, hg = r5.uniform(-180, 180, nq5), r5.uniform(-180, 180, nq5)
    lo, hi = shard.shard_range(nq5, rank, world)
    starts5 = np.stack([a5[:, 1], a5[:, 0], hs], 1).astype(np.float64)[lo:hi]
    goals5 = np.stack([b5[:, 1], b5[:, 0], hg], 1).astype(np.float64)[lo:hi]
    n = hi - lo
    sxy5 = np.empty((n, K5 - 1, 2), np.int32); sth5 = np.empty((n, K5 - 1))
    for q in range(n):
        sxy5[q], sth5[q] = samples.make_stream(((goals5[q, 0], goals5[q, 1]), goals5[q, 2]), K5 - 1, 500000 + lo + q, (side5, side5))
    sg5 = np.stack([ta[:, 1], ta[:, 0], tb[:, 1], tb[:, 0]], 1).astype(np.int32)[lo:hi]
    return dict(maps=maps5, K=K5, nq_total=nq5, lo=lo, hi=hi, starts=starts5, goals=goals5, sxy=sxy5, sth=sth5, sg=sg5,
                mid_r=mid_r[lo:hi], mid_t=mid_t[lo:hi])


def secondary_benchmarks(torch, dev, maps, peak, peak_src, args, rank, world, dist_on):
    """cfg 4 microbenchmarks, Theta* on map2 and cfg 5; each timed with CUDA events after warm-up.  The cfg-4 rays and the
    cfg-5 queries are sharded over the ranks (contiguous shards, maps replicated, no collective; the rates are totals over
    all ranks divided by the slowest rank's time); the single-tree nearest scan and the map2 searches are replicas-only work
    and run on rank 0."""
    from theta_rrt_b200 import OccupancyGrid, Params, Planner, shard
    out = {}
    steps = max(args.steps, 5)
    cores = os.cpu_count() or 1

    def timed(fn, n=steps, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        if dist_on:
            import torch.distributed as dist
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    # ---- cfg 4: 8192^2 grid, 2^20 segments (sharded), 2^20-node tree, 4096 queries
    big = synthetic_map(8192, 0.1, 8, 42)
    pl = Planner(OccupancyGrid(big, device=dev))
    seg_all = make_segments(big, 1 << 20, 7)
    slo, shi = shard.shard_range(len(seg_all), rank, world)
    seg = seg_all[slo:shi]
    d_seg = torch.from_numpy(seg).to(dev)
    d_out = torch.empty(len(seg), dtype=torch.uint8, device=dev)
    ms_rows = timed(lambda: pl.los(d_seg, out=d_out, layout="rows"))
    vis_rows = d_out.cpu().numpy().astype(bool)
    ms = timed(lambda: pl.los(d_seg, out=d_out))
    vis = d_out.cpu().numpy().astype(bool)
    assert np.array_equal(vis, vis_rows), "los: strip and row layouts disagree"
    px = np.maximum(np.abs(seg[:, 2] - seg[:, 0]), np.abs(seg[:, 3] - seg[:, 1])) + 1
    los_bytes = 4.0 * float(px[vis].sum()) + 17.0 * len(seg)
    ms_all = max_over_ranks(torch, dist_on, dev, ms)
    ms_rows_all = max_over_ranks(torch, dist_on, dev, ms_rows)
    nvis, npx = sum_over_ranks(torch, dist_on, dev, [float(vis.sum()), float(px.sum())])
    alg = los_bytes / (ms / 1e3) / 1e9
    out["los_cfg4"] = {"metric": "los_checks_per_sec", "value": len(seg_all) / (ms_all / 1e3), "unit": "checks/s", "ms": ms_all,
                       "segments": len(seg_all), "segments_per_rank": len(seg), "n_gpus": world, "scaling": "strong",
                       "grid": "8192x8192: strip copy (32 MiB, L2 resident) of the bit-packed rows (8 MiB), replicated per rank",
                       "visible_fraction": nvis / len(seg_all),
                       "pixel_tests_per_sec_upper": npx / (ms_all / 1e3),
                       "rows_layout_ms": ms_rows_all, "rows_layout_checks_per_sec": len(seg_all) / (ms_rows_all / 1e3),
                       "roofline": physical_roofline(
                           "los_tiled_kernel", ms, "issue",
                           alg={"achieved": alg, "peak": peak, "unit": "GB/s", "frac": alg / peak, "peak_source": peak_src,
                                "definition": "SURVEY 8(d): one 4-B word per pixel test of the fully walked (visible) rays + 16 B segment "
                                              "in + 1 B out, over the HBM copy peak; not a physical HBM figure"},
                           note="bound by instruction issue (integer / FMA pipes) and the dependent 16-byte strip loads from L2; counts are "
                                "those of the full 2^20-ray launch, so the fractions hold for the one-GPU run")}
    if rank == 0:
        rng = np.random.default_rng(3)
        n_nodes = 1 << 20
        x = torch.from_numpy(rng.uniform(0, 8191, n_nodes)).to(dev)
        y = torch.from_numpy(rng.uniform(0, 8191, n_nodes)).to(dev)
        qxy = torch.from_numpy(rng.integers(0, 8192, size=(4096, 2)).astype(np.int32)).to(dev)
    if rank == 0:
        def timed0(fn, n=steps, warm=3):  # rank-0-only work: no barrier
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        ms = timed0(lambda: pl.nearest(x, y, qxy))
        ach = 16.0 * n_nodes * 4096 / (ms / 1e3) / 1e9
        out["nearest_cfg4"] = {"metric": "nearest_queries_per_sec", "value": 4096 / (ms / 1e3), "unit": "queries/s",
                               "ms": ms, "nodes": n_nodes, "queries": 4096, "n_gpus": 1, "scaling": "replicas only (one tree)",
                               "roofline": physical_roofline(
                                   "nearest_tile_kernel", ms, "fp64",
                                   alg={"achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                                        "definition": "SURVEY 8(d): 16 B per (query, node) over the HBM copy peak; 8 queries share every node "
                                                      "load in registers, so this exceeds 1 and is not a physical figure"},
                                   note="4096 queries x 2^20 nodes: 6 fp64-pipe instructions per pair, the fp64 pipe is the roof")}
        # single-query scans over a tree larger than L2 (2^24 nodes = 256 MiB): the pure HBM-streaming case
        n_big = 1 << 24
        xb = torch.from_numpy(rng.uniform(0, 8191, n_big)).to(dev)
        yb = torch.from_numpy(rng.uniform(0, 8191, n_big)).to(dev)
        q1 = qxy[:1].contiguous()
        ms = timed0(lambda: pl.nearest(xb, yb, q1))
        ach = 16.0 * n_big / (ms / 1e3) / 1e9
        out["nearest_single_query_hbm"] = {"metric": "nearest_scan_GBps", "value": ach, "unit": "GB/s", "ms": ms,
                                           "nodes": n_big, "queries": 1,
                                           "roofline": {"kernel": "nearest_tile_kernel", "bound": "hbm", "achieved": ach,
                                                        "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": 16 * n_big,
                                                        "peak_source": peak_src,
                                                        "note": "one query, 256 MiB SoA tree (> L2): every byte comes from HBM; the "
                                                                "whole call (counter memset + one kernel with the last-CTA fold, "
                                                                "launch gaps included) is timed"}}
        ko = kernel_counts("nearest_tile_kernel_single_query")
        if ko.get("ncu_duration_us"):
            gbs = 16.0 * n_big / (ko["ncu_duration_us"] * 1e-6) / 1e9
            out["nearest_single_query_hbm"]["kernel_only"] = {"us": ko["ncu_duration_us"], "achieved": gbs, "peak": peak, "unit": "GB/s",
                                                              "frac": gbs / peak, "source": ko.get("source"),
                                                              "note": "device time of the kernel alone (ncu launch list of this bench command)"}
        del xb, yb, x, y
        if not args.skip_cpu:
            # CPU port (oracle) on a bounded sample of the same rays, all host threads
            from oracle import c_oracle as O
            O.lib()
            ns = min(1 << 17, len(seg))
            O.lineofsight_batch(big, seg[:4096], threads=cores)
            t = time.perf_counter()
            cpu_vis = O.lineofsight_batch(big, seg[:ns], threads=cores)
            dt = time.perf_counter() - t
            assert np.array_equal(cpu_vis, vis[:ns])  # same booleans as the kernel
            out["los_cfg4"]["cpu_baseline"] = {"value": ns / dt, "unit": "checks/s", "cores": cores, "kind": "port",
                                               "sample": f"first {ns} of the {len(seg_all)} rays on {cores} threads"}
        # ---- Theta* on map2: the reference's single query and a batch of random free-cell queries
        m2 = maps["map2"]
        pt = Planner(OccupancyGrid(m2, device=dev))
        one = torch.tensor([[280, 0, 8, 280]], dtype=torch.int32, device=dev)
        ms1 = timed0(lambda: pt.theta(one, lanes=32), n=3, warm=2)
        r = pt.theta(one, lanes=32).host()
        out["theta_cfg2"] = {"metric": "theta_single_query_ms", "value": ms1, "unit": "ms", "expanded": int(r["expanded"][0]),
                             "los_checks": int(r["n_los"][0]), "cost": float(r["cost"][0]),
                             "expansions_per_sec": int(r["expanded"][0]) / (ms1 / 1e3),
                             "note": "one search is a serial chain of 30 384 pops on one warp; open list = global-memory 32-ary heap "
                                     "(L1 resident), measured faster than the shared-memory heap north_star names (DESIGN.md K3)"}
        cells = np.argwhere(m2)
        rq = np.random.default_rng(5)
        nqt = 8192
        a, b = cells[rq.integers(len(cells), size=nqt)], cells[rq.integers(len(cells), size=nqt)]
        sg = torch.from_numpy(np.stack([a[:, 1], a[:, 0], b[:, 1], b[:, 0]], 1).astype(np.int32)).to(dev)
        msb = timed0(lambda: pt.theta(sg, path_cap=64), n=3, warm=3)
        rb = pt.theta(sg, path_cap=64).host()
        out["theta_batch_map2"] = {"metric": "theta_expansions_per_sec", "value": float(rb["expanded"].sum()) / (msb / 1e3),
                                   "unit": "expansions/s", "ms": msb, "queries": nqt,
                                   "los_checks_per_sec": float(rb["n_los"].sum()) / (msb / 1e3),
                                   "found": int((rb["status"] == 0).sum()),
                                   "roofline": physical_roofline("theta_kernel", msb, "issue",
                                                                 note="latency-bound pointer chasing (heap, cells): issue slots are the "
                                                                      "nearest physical roof; the L1/L2 rates ride along")}
        # The 8 192-query batch is bounded by its longest search (one warp, ~59 k expansions); four times the queries show
        # what the kernel sustains when that tail is amortised.
        nql = 4 * nqt
        a, b = cells[rq.integers(len(cells), size=nql)], cells[rq.integers(len(cells), size=nql)]
        sgl = torch.from_numpy(np.stack([a[:, 1], a[:, 0], b[:, 1], b[:, 0]], 1).astype(np.int32)).to(dev)
        msl = timed0(lambda: pt.theta(sgl, path_cap=64), n=2, warm=2)
        rl = pt.theta(sgl, path_cap=64)
        out["theta_batch_map2"]["longest_search_expansions"] = int(rb["expanded"].max())
        out["theta_batch_map2"]["large_batch"] = {"queries": nql, "ms": msl, "value": float(rl.expanded.sum()) / (msl / 1e3),
                                                  "unit": "expansions/s", "longest_search_expansions": int(rl.expanded.max()),
                                                  "note": "same kernel and map, 4x the queries: the batch above ends with its longest "
                                                          "search running alone on one warp"}
        del sgl, rl
        if not args.skip_cpu:
            from oracle import c_oracle as O
            nsmp = min(nqt, 4 * cores)
            sgh = sg[:nsmp].cpu().numpy()
            t = time.perf_counter()
            rc = O.astar_batch(m2, sgh, thetastar=True, threads=cores)
            dt = time.perf_counter() - t
            assert np.array_equal(rc["expanded"], rb["expanded"][:nsmp])  # same searches as the kernel
            out["theta_batch_map2"]["cpu_baseline"] = {"value": float(rc["expanded"].sum()) / dt, "unit": "expansions/s",
                                                       "cores": cores, "kind": "port",
                                                       "sample": f"first {nsmp} of the {nqt} queries on {cores} threads"}
            t = time.perf_counter()
            O.astar(m2, (280, 0), (8, 280))
            out["theta_cfg2"]["cpu_port_single_core_ms"] = (time.perf_counter() - t) * 1e3
        del pt
    del pl, d_seg, d_out
    torch.cuda.empty_cache()
    # ---- cfg 5: 65 536 mixed queries over 64 random maps, sharded over the ranks
    c5 = make_cfg5(rank, world)
    p5 = Planner(OccupancyGrid(c5["maps"], device=dev), Params(tol_xy=0.0, K=c5["K"]))
    d5 = [torch.from_numpy(v).to(dev) for v in (c5["starts"], c5["goals"], c5["sxy"], c5["sth"])]
    sg5 = torch.from_numpy(c5["sg"]).to(dev)
    dm_r, dm_t = torch.from_numpy(c5["mid_r"]).to(dev), torch.from_numpy(c5["mid_t"]).to(dev)
    res5 = {}

    def step5r():
        res5["rrt"] = p5.rrt(*d5, K=c5["K"], map_id=dm_r, want_u=False)

    def step5t():
        res5["theta"] = p5.theta(sg5, map_id=dm_t, path_cap=64)
    # (three warm-up calls: the result tensors of a call are freed when the next call's replace them, so the caching allocator
    # needs two generations of them before the timed calls stop reaching cudaMalloc)
    ms5r = max_over_ranks(torch, dist_on, dev, timed(step5r, n=3, warm=3))
    ms5t = max_over_ranks(torch, dist_on, dev, timed(step5t, n=3, warm=3))
    it5, ex5, los5, found5 = sum_over_ranks(torch, dist_on, dev, [float(res5["rrt"].iters.sum()), float(res5["theta"].expanded.sum()),
                                                                  float(res5["theta"].n_los.sum()), float((res5["theta"].status == 0).sum())])
    ms5 = ms5r + ms5t
    out["cfg5_mixed"] = {
        "metric": "mixed_queries_per_sec", "value": 2 * c5["nq_total"] / (ms5 / 1e3), "unit": "queries/s", "ms": ms5,
        "n_gpus": world, "scaling": "strong", "queries": 2 * c5["nq_total"], "queries_per_rank": 2 * (c5["hi"] - c5["lo"]),
        "rrt_queries": c5["nq_total"], "K": c5["K"], "theta_queries": c5["nq_total"], "maps": "64 x 256x256",
        "rrt_ms": ms5r, "theta_ms": ms5t,
        "rrt_expansions_per_sec": it5 / (ms5r / 1e3), "theta_expansions_per_sec": ex5 / (ms5t / 1e3),
        "theta_los_checks_per_sec": los5 / (ms5t / 1e3), "theta_found": int(found5),
        "note": "BASELINE cfg 5: 32 768 RRT (K = 1 001) + 32 768 Theta* queries over 64 random maps, contiguous shards of both halves "
                "per rank, maps replicated, no collective; the RRT batch and the Theta* batch back to back, slowest rank's time"}
    if rank == 0 and not args.skip_cpu:
        from oracle import c_oracle as O
        nsmp = min(4 * cores, c5["hi"] - c5["lo"])
        t = time.perf_counter()
        done_r = 0
        for m in np.unique(c5["mid_r"][:nsmp]):  # the oracle takes one map per call
            sel = np.nonzero(c5["mid_r"][:nsmp] == m)[0]
            rr = O.rrt_batch(c5["maps"][m], c5["starts"][sel], c5["goals"][sel], c5["sxy"][sel], c5["sth"][sel], c5["K"], O.Params(tol_xy=0.0),
                             threads=cores, want_nodes=False)
            done_r += int(rr["iters"].sum())
            assert np.array_equal(rr["n_nodes"], res5["rrt"].n_nodes[torch.from_numpy(sel).to(dev)].cpu().numpy())
        dtr = time.perf_counter() - t
        t = time.perf_counter()
        done_t = 0
        for m in np.unique(c5["mid_t"][:nsmp]):
            sel = np.nonzero(c5["mid_t"][:nsmp] == m)[0]
            rt = O.astar_batch(c5["maps"][m], c5["sg"][sel], thetastar=True, threads=cores)
            done_t += int(rt["expanded"].sum())
            assert np.array_equal(rt["expanded"], res5["theta"].expanded[torch.from_numpy(sel).to(dev)].cpu().numpy())
        dtt = time.perf_counter() - t
        out["cfg5_mixed"]["cpu_baseline"] = {"value": 2 * nsmp / (dtr + dtt), "unit": "queries/s", "cores": cores, "kind": "port",
                                             "rrt_expansions_per_sec": done_r / dtr, "theta_expansions_per_sec": done_t / dtt,
                                             "sample": f"first {nsmp} RRT and first {nsmp} Theta* queries of rank 0's shard on {cores} threads "
                                                       "(same results as the kernels, asserted)"}
    return out


def cpu_baseline(free, starts, goals, sxy, sth, args):
    """The C oracle (a port of the reference's algorithm) on the host: one core and all cores, bounded sample; plus the
    unmodified Python reference, one process and one per core."""
    from oracle import c_oracle as O
    cores = os.cpu_count() or 1
    P = O.Params(tol_xy=0.0)
    K = sth.shape[1] + 1
    O.lib()
    n1 = min(8, len(starts))
    t = time.perf_counter()
    r = O.rrt_batch(free, starts[:n1], goals[:n1], sxy[:n1], sth[:n1], K, P, threads=1, want_nodes=False)
    one = int(r["iters"].sum()) / (time.perf_counter() - t)
    nall = min(len(starts), max(4 * cores, 32))
    t = time.perf_counter()
    r = O.rrt_batch(free, starts[:nall], goals[:nall], sxy[:nall], sth[:nall], K, P, threads=cores, want_nodes=False)
    allc = int(r["iters"].sum()) / (time.perf_counter() - t)
    out = {"value": allc, "unit": "expansions/s", "cores": cores, "kind": "port",
           "sample": f"first {nall} of the step's queries on {cores} threads (single thread: first {n1} queries)",
           "single_core_value": one}
    if not args.skip_python_ref:
        out["python_reference"] = python_reference(free, starts, goals, sxy, sth, cores)
    return out


if __name__ == "__main__":
    main()
