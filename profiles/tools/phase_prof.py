"""Where does a window of the fused RRT kernel spend its time, warp by warp?  Needs the experiment build:
    nvcc ... -DTRRT_PHASE_PROF -o profiles/tools/_libthetarrt_prof.so   (python profiles/tools/phase_prof.py build)
    python profiles/tools/phase_prof.py [nq] [K]
clock64 sums per warp: scan (loop top -> barrier arrival), barrier wait, expansion, predicted re-expansion, commit."""
import ctypes, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
SO = os.path.join(ROOT, "profiles", "tools", "_libthetarrt_prof.so")
if len(sys.argv) > 1 and sys.argv[1] == "build":
    from theta_rrt_b200 import build as B
    cmd = [B.nvcc_path(), *B.NVCC_FLAGS, "-DTRRT_PHASE_PROF", *sys.argv[2:], "-o", SO, os.path.join(B.CSRC, "thetarrt.cu")]
    subprocess.check_call(cmd)
    sys.exit(0)
import numpy as np, torch
from theta_rrt_b200 import _lib
_lib.SO_PATH = SO
import bench
from theta_rrt_b200 import OccupancyGrid, Params, Planner
nq = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
K = int(sys.argv[2]) if len(sys.argv) > 2 else 5001
dev = torch.device("cuda:0")
free = bench.load_maps()["map1"]
starts, goals, sxy, sth = bench.make_rrt_workload(free, nq, K)
p = Planner(OccupancyGrid(free, device=dev), Params(tol_xy=0.0, K=K))
d = [torch.from_numpy(a).to(dev) for a in (starts, goals, sxy, sth)]
lib = _lib.load()
lib.trrt_debug_phase_prof.argtypes = [ctypes.c_void_p]
buf = (ctypes.c_uint64 * 24)()
for _ in range(2):
    p.rrt(*d, K=K)
lib.trrt_debug_phase_prof(buf)
nn = (ctypes.c_uint64 * 8)()
if hasattr(lib, "trrt_debug_nn_stats"):
    lib.trrt_debug_nn_stats.argtypes = [ctypes.c_void_p]
    lib.trrt_debug_nn_stats(nn)
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(); r = p.rrt(*d, K=K); b.record(); torch.cuda.synchronize()
lib.trrt_debug_phase_prof(buf)
if hasattr(lib, "trrt_debug_nn_stats"):
    lib.trrt_debug_nn_stats(nn)
    s_ = [int(x) for x in nn]
    if s_[0]:
        print(f"cell-index lookups {s_[0]}: decided by the cells {100 * s_[1] / s_[0]:.1f}%, pages {s_[2] / s_[0]:.2f} nodes {s_[3] / s_[0]:.1f} per lookup; "
              f"per warp-window {s_[5] / s_[4]:.2f} samples left to the full scan in {s_[6] / s_[4]:.2f} passes")
v = [int(x) for x in buf]
W = v[10]
print(f"kernel {a.elapsed_time(b):.2f} ms, windows (warp x window) {W}, iterations {int(r.iters.sum())}")
names = [("sample, publish", 19, None), ("wait at barrier 1", 18, None), ("pooled scan", 0, 1), ("wait at barrier 2", 2, None), ("expansion", 3, 4), ("pass + commit", 7, 8)]
WR = v[20] or W  # warp-rounds (idle warps take part in the pooled scan and the barriers)
print(f"warp-rounds {WR}, of which with a query {W}")
tot = v[0] + v[2] + v[3] + v[7] + v[18] + v[19]
for nm, i, j in names:
    Wn = W if i in (3, 7) else WR
    mean = v[i] / Wn
    line = f"  {nm:28s} mean {mean:9.0f} cycles  {100 * v[i] / tot:5.1f}%"
    if j is not None:
        var = v[j] * 1024 / Wn - mean * mean
        line += f"  std {max(var, 0) ** 0.5:9.0f}"
    print(line)
if v[21]: print(f"  of 'sample, publish': nearest lookup {v[21] / WR:.0f} cycles, of which the walk over the cells {v[22] / WR:.0f}")
if v[14]:  # fp32 prefilter of the pooled scan (per lane: one sample against one slice of a tree)
    print(f"  scan prefilter: lane-slices {v[14]}, fp32 blocks {v[15] / v[14]:.1f} per lane-slice; rechecked in fp64 {v[11] / v[14]:.2f} "
          f"blocks per lane-slice ({100 * v[11] / max(v[15], 1):.2f}% of the blocks), {v[11] / (32 * WR):.2f} per lane-window; "
          f"rescanned at admission (list full) {v[12] / v[14]:.4f} blocks per lane-slice; whole slice in fp64 {100 * v[13] / v[14]:.3f}% of lane-slices")
    print(f"  of 'pooled scan', mean per lane-window: cp.async waits {v[5] / (32 * WR):.0f} cycles, fp64 rescans {v[6] / (32 * WR):.0f} cycles")
post = (v[3] + v[7]) / W
print(f"  after-barrier work per window: mean {post:.0f}, std {max(v[9] * 1024 / W - post * post, 0) ** 0.5:.0f}")
print(f"  iterations committed per window: {v[17] / max(v[16], 1):.2f} of 32")
