"""LOS microbenchmark on the cfg-4 grid (8192^2, 2^20 random rays): python profiles/tools/mb_los.py
Rows layout (one thread per ray / G lanes per ray) against the tiled layout with per-lane refill."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import bench
from theta_rrt_b200 import OccupancyGrid, Planner
dev = torch.device("cuda:0")
big = bench.synthetic_map(8192, 0.1, 8, 42)
pl = Planner(OccupancyGrid(big, device=dev))
seg = bench.make_segments(big, 1 << 20, 7)
d_seg = torch.from_numpy(seg).to(dev)
out = torch.empty(len(seg), dtype=torch.uint8, device=dev)
ref = None


def run(label, **kw):
    global ref
    for _ in range(3): pl.los(d_seg, out=out, **kw)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20): pl.los(d_seg, out=out, **kw)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 20
    res = out.cpu().numpy()
    if ref is None: ref = res.copy()
    print(f"{label}: {ms*1e3:8.1f} us  {len(seg)/ms/1e6:8.2f} G checks/s  same as first: {bool((res == ref).all())}", flush=True)


run("rows  (one thread per ray)", layout="rows")
run("tiles default", layout="tiles")
# sorted by length (what a caller could do for the rows kernel): upper bound on what refill can recover
px = np.maximum(np.abs(seg[:, 2] - seg[:, 0]), np.abs(seg[:, 3] - seg[:, 1]))
d_seg = torch.from_numpy(np.ascontiguousarray(seg[np.argsort(px)])).to(dev); ref = None
run("rows  lanes 1, rays sorted by length", layout="rows")
run("tiles default, rays sorted by length", layout="tiles")
