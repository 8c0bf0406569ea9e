"""Host logic of bench.py (no GPU): workload generators are deterministic and shard-consistent, the roofline arithmetic
reads the committed peaks / counts, and the reference arm prints a line with the contract's keys."""
import json
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_generators_are_deterministic(maps):
    free = maps["map1"]
    a = bench.make_rrt_workload(free, 6, 101, first_query=10)
    b = bench.make_rrt_workload(free, 16, 101, first_query=0)
    for x, y in zip(a, b):
        assert np.array_equal(x, y[10:16])  # a shard is a slice of the whole: same starts, goals and per-query stream seeds
    s1, s2 = bench.make_segments(free, 100, 7, maxlen=40), bench.make_segments(free, 100, 7, maxlen=40)
    assert np.array_equal(s1, s2) and s1.dtype == np.int32 and s1.min() >= 0 and s1.max() < 100
    m = bench.synthetic_map(64, 0.15, 4, 9)
    assert m.shape == (64, 64) and np.array_equal(m, bench.synthetic_map(64, 0.15, 4, 9)) and 0.5 < m.mean() < 1.0


def test_cfg5_shards_partition_the_workload():
    whole = bench.make_cfg5(0, 1, nq5=24, K5=21)
    parts = [bench.make_cfg5(r, 3, nq5=24, K5=21) for r in range(3)]
    assert [p["lo"] for p in parts] == [0, 8, 16] and parts[-1]["hi"] == 24
    for k in ("starts", "goals", "sxy", "sth", "sg", "mid_r", "mid_t"):
        assert np.array_equal(np.concatenate([p[k] for p in parts]), whole[k]), k
    assert whole["maps"].shape == (64, 256, 256)
    # start / goal cells are free cells of the query's own map
    for q in range(24):
        mp = whole["maps"][whole["mid_r"][q]]
        assert mp[int(whole["starts"][q, 1]), int(whole["starts"][q, 0])] and mp[int(whole["goals"][q, 1]), int(whole["goals"][q, 0])]


def test_physical_roofline_uses_committed_peaks_and_counts():
    pk, kc = bench.pipe_peaks(), bench.kernel_counts("rrt_kernel")
    assert pk.get("fp64_dadd_lane_inst_per_s", 0) > 1e13 and kc.get("fp64_warp_inst", 0) > 1e9
    r = bench.physical_roofline("rrt_kernel", 40.0, "fp64", alg={"x": 1})
    assert r["bound"] == "fp64" and r["unit"].startswith("T fp64")
    assert abs(r["achieved"] - kc["fp64_warp_inst"] * 32 / 0.040 / 1e12) < 1e-9 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert 0 < r["frac"] < 1 and 0 < r["l2"]["frac"] < 1 and 0 < r["smem"]["frac"] < 1 and r["algorithmic_equiv"] == {"x": 1}
    i = bench.physical_roofline("los_tiled_kernel", 0.07, "issue")
    assert i["unit"] == "G warp-inst/s" and 0 < i["frac"] < 1
    assert bench.physical_roofline("no_such_kernel", 1.0, "fp64")["frac"] is None  # nothing invented when counts are missing


def test_reference_arm_line_without_python_reference(monkeypatch, capsys):
    """--impl reference on a tiny step (the Python reference leg is stubbed out: it is timed for real on the GPU box)."""
    monkeypatch.setattr(bench, "python_reference", lambda *a, **k: {"unavailable": "stubbed in this test"})
    monkeypatch.setattr(bench, "K_RRT", 201)
    monkeypatch.setattr(bench.os, "cpu_count", lambda: 2)
    args = type("A", (), {"steps": 1, "warmup": 1, "gpus": 1})()
    bench.run_reference_arm(args, rank=0, world=1)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
              "data", "config", "cpu_baseline", "e2e", "python_reference"):
        assert k in line, k
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    bench.run_reference_arm(args, rank=1, world=2)  # other ranks print nothing
    assert capsys.readouterr().out == ""


def test_dump_outputs_writes_valid_tree_rows_of_a_fixed_sample(tmp_path):
    import torch
    from theta_rrt_b200.planner import RrtResult
    nq, K = 300, 9
    rng = np.random.default_rng(1)
    n = rng.integers(1, K + 1, nq)
    f = lambda *s: torch.from_numpy(rng.normal(size=s))  # noqa: E731
    i = lambda *s: torch.from_numpy(rng.integers(-1, K, size=s).astype(np.int32))  # noqa: E731
    res = RrtResult(K=K, node_x=f(nq, K), node_y=f(nq, K), node_theta=f(nq, K), parent=i(nq, K),
                    n_nodes=torch.from_numpy(n.astype(np.int32)), sol=i(nq), status=i(nq), iters=i(nq), u=f(nq, K, 5))
    res.u[:, 0] = float("nan")  # root rows
    res.u[::3, 1:, 1:4] = float("nan")  # straight edges
    bench.dump_outputs(str(tmp_path / "a"), res, 1000)
    bench.dump_outputs(str(tmp_path / "b"), res, 1000)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(k + ".npy" for k in ("n_nodes", "sol", "status", "iters", "queries", "node_x", "node_y", "node_theta",
                                                "parent", "u", "u_nan"))
    d = {p[:-4]: np.load(tmp_path / "a" / p) for p in names}
    assert all(v.dtype == np.float64 and np.array_equal(v, np.load(tmp_path / "b" / (k + ".npy"))) for k, v in d.items())
    assert np.array_equal(d["n_nodes"], n) and np.array_equal(d["status"], res.status.numpy())
    q = d["queries"].astype(np.int64) - 1000
    assert len(q) == bench.DUMP_TREES and np.all(np.diff(q) > 0)
    rows = np.concatenate([np.stack([np.full(n[j], j), np.arange(n[j])], 1) for j in q])
    assert len(d["node_x"]) == len(rows) == n[q].sum() and d["u"].shape == d["u_nan"].shape == (len(rows), 5)
    for k in ("node_x", "node_y", "node_theta", "parent"):
        assert np.array_equal(d[k], getattr(res, k).numpy()[rows[:, 0], rows[:, 1]]), k
    u = res.u.numpy()[rows[:, 0], rows[:, 1]]
    assert d["u_nan"].sum() > 0 and np.array_equal(d["u_nan"] == 1, np.isnan(u))
    assert np.array_equal(d["u"], np.where(np.isnan(u), 0.0, u))


def test_bench_rejects_zero_steps_and_dump_of_the_reference_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True)
        assert p.returncode == 2 and "error" in p.stderr, extra
