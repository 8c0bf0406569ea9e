"""Shared helpers for the parity tests."""
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def O():
    """The C oracle, built and loaded (a module imports this fixture by name)."""
    from oracle import c_oracle
    c_oracle.lib()
    return c_oracle


def planner_for(free=None, device=None, **params):
    """A Planner over `free` (default: an open 64 x 64 map) on `device` (default: OccupancyGrid's, cuda:0) with
    Params(**params)."""
    from theta_rrt_b200 import OccupancyGrid, Params, Planner
    if free is None:
        free = np.ones((64, 64), bool)
    grid = OccupancyGrid(free) if device is None else OccupancyGrid(free, device=device)
    return Planner(grid, Params(**params))


def bits_equal(a, b):
    """float64 arrays equal bit for bit (NaN payloads included)."""
    a = np.ascontiguousarray(a, np.float64)
    b = np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def bits_equal_nan(a, b):
    """float64 arrays equal bit for bit, where any NaN equals any NaN."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    return np.array_equal(np.where(np.isnan(a), 0.0, a).view(np.int64), np.where(np.isnan(b), 0.0, b).view(np.int64))


def struct_members(name):
    """Member names of `typedef struct name {...} name;` in include/thetarrt.h, in declaration order."""
    src = open(os.path.join(ROOT, "include", "thetarrt.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, flags=re.S).group(1)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            head, *rest = decl.split(",")
            names.append(re.findall(r"\w+", head)[-1])
            names += [r.strip().lstrip("*").strip() for r in rest]
    return names


def synthetic_map(n, p, block, seed):
    """Square Bernoulli-obstacle map (True = free), obstacles in block x block tiles (SURVEY.md 8d cfg 4/5)."""
    rng = np.random.default_rng(seed)
    nb = (n + block - 1) // block
    coarse = rng.random((nb, nb)) >= p
    return np.kron(coarse, np.ones((block, block), bool))[:n, :n]


def rrt_runs():
    z = np.load(os.path.join(GOLDEN, "rrt_kat.npz"))
    n = int(z["n_runs"][0])
    runs = []
    for i in range(n):
        p = f"r{i}_"
        runs.append({k[len(p):]: z[k] for k in z.files if k.startswith(p)})
    return runs


def theta_kat():
    return json.load(open(os.path.join(GOLDEN, "theta_kat.json")))


def random_queries(free, nq, seed):
    """starts/goals drawn uniformly from free cells, headings uniform (-180, 180] (SURVEY.md 8d cfg 3)."""
    rng = np.random.default_rng(seed)
    cells = np.argwhere(free)  # (y, x)
    a = cells[rng.integers(len(cells), size=nq)]
    b = cells[rng.integers(len(cells), size=nq)]
    starts = np.stack([a[:, 1], a[:, 0], rng.uniform(-180, 180, nq)], axis=1).astype(np.float64)
    goals = np.stack([b[:, 1], b[:, 0], rng.uniform(-180, 180, nq)], axis=1).astype(np.float64)
    return starts, goals


AUDIT_EPS = 1e-6


def compare_rrt_with_reference(res, run, first_ambiguous, coord_atol=1e-5):
    """Compare one RRT result (dict with n_nodes, parent, it_near, it_new, it_code, los, x, y, theta, sol)
    with a golden run of the unmodified reference.

    Discrete outputs must be identical for every iteration before `first_ambiguous` (the first
    iteration whose outcome the oracle's margin audit marks as decided by rounding noise; -1 = none,
    compare everything).  Returns the number of iterations compared.
    """
    K = int(run["K"][0])
    n_it = int(run["iterations"][0])
    limit = n_it if first_ambiguous < 0 else min(first_ambiguous, n_it)
    ref_near = np.full(K - 1, -1, np.int64)
    ref_near[run["nearest_it"] - 1] = run["nearest_idx"]
    assert np.array_equal(np.asarray(res["it_near"])[:limit], ref_near[:limit]), "nearest-node indices"
    # LOS booleans of the compared iterations, in call order
    n_los_ref = int(np.sum(run["los_it"] <= limit))
    assert np.array_equal(np.asarray(res["los"])[:n_los_ref].astype(bool), run["los"][:n_los_ref]), "LOS booleans"
    # nodes created before `limit`: index = insertion order, so they form a prefix
    it_code = np.asarray(res["it_code"])
    n_pref = 1 + int(np.sum(it_code[:limit] == 0))
    assert n_pref <= len(run["parent"])
    if limit == n_it:
        assert int(res["n_nodes"]) == len(run["parent"]), "tree size"
        assert int(res["sol"]) == int(run["sol"][0]), "solution node"
        assert np.array_equal(np.asarray(res["parent"])[:n_pref], run["parent"][:n_pref]), "parent array"
    else:
        # parents of prefix nodes may still be overwritten by later (uncompared) iterations (rrt.py:187-188):
        # compare the creating edge instead
        created = np.nonzero(it_code[:limit] == 0)[0]
        new_idx = np.asarray(res["it_new"])[created]
        assert np.array_equal(new_idx, np.arange(1, n_pref)), "insertion order"
    for a, b in ((res["x"], run["x"]), (res["y"], run["y"]), (res["theta"], run["theta"])):
        assert np.allclose(np.asarray(a)[:n_pref], b[:n_pref], rtol=0, atol=coord_atol), "node coordinates"
    return limit
