"""main.py missions on the C parity oracle: the CPU side of the tests of Planner.missions / trrt_mission_batch.

TEST INFRASTRUCTURE ONLY -- used by tests/test_missions.py and profiles/tools/mb_missions.py.  `mission_chain` is
main.chain (main.py:56-84) over the oracle's rrt / findnearest / anglebetween (oracle/c_oracle.py), with headings from
the oracle's anglebetween (the same trrt_libm atan2 the device uses), so device results can be compared bit for bit.
"""
import numpy as np

from oracle.c_oracle import Params, anglebetween, findnearest, rrt


def mission_chain(free, waypoints, normals, K, params=None, xystdv=0.4, anglestdv=100):
    """main.chain (main.py:56-84) over the oracle's rrt / findnearest / anglebetween for one mission.

    Segment s runs from waypoint s to s+1; once a segment has failed, every later one starts at the most recent
    findnearest node with its heading.  `normals` is the mission's stream of standard normals in draw order: segment s
    turns the next 3*(K-1) of them into rand_conf samples around its end (samples.stream_from_normals), and the stream
    then advances by 3 * iterations run, where the reference stops drawing.  Returns dict(segments, path, path_seg,
    status, stop_seg); `path` rows are (x, y, theta, u[5]) of main.path_nodes, segment after segment.  status 4 (the
    reference raises in rrt.rrt) and 7 (findnearest of a childless tree, main.py:79-81) stop the chain at stop_seg."""
    from theta_rrt_b200 import samples
    from theta_rrt_b200.rrt import standardangle
    P = params or Params()
    wp = [tuple(int(v) for v in w) for w in waypoints]
    normals = np.asarray(normals, np.float64)
    path = wp + [None]
    nearest = None
    off = 0
    segs, rows, row_seg = [], [], []
    status, stop_seg = 0, -1
    for s, (first, second, third) in enumerate(zip(path, path[1:], path[2:])):
        angle1 = anglebetween((1, 0), (second[0] - first[0], second[1] - first[1]))
        if nearest is not None:
            angle1, first = nearest[1], nearest[0]
        angle2 = angle1 if third is None else anglebetween((1, 0), (third[0] - second[0], third[1] - second[1]))
        begin = ((float(first[0]), float(first[1])), standardangle(angle1))
        end = ((float(second[0]), float(second[1])), standardangle(angle2))
        sxy, sth = samples.stream_from_normals(normals[off:off + 3 * (K - 1)], end, free.shape, xystdv, anglestdv)
        o = rrt(free, begin, end, sxy, sth, P, K=K)
        node = lambda i: ((float(o["x"][i]), float(o["y"][i])), float(o["theta"][i]))  # noqa: E731
        sel = o["it_new"] >= 0
        rec = dict(begin=begin, end=end, solution=None, nearest=None, mindist=None, n_nodes=o["n_nodes"],
                   n_edges=int(sel.sum()), iters=o["iters"], status=o["status"])
        segs.append(rec)
        if o["status"] not in (0, 1):
            status, stop_seg = o["status"], s
            break
        if o["sol"] >= 0:
            term = o["sol"]
            rec["solution"] = node(term)
        else:
            b, d = findnearest(o["x"], o["y"], o["theta"], o["it_near"][sel], o["it_new"][sel], end, P)
            if b < 0:
                status, stop_seg = 7, s
                break
            term = b
            nearest = node(b)
            rec["nearest"], rec["mindist"] = nearest, d
        chain = []
        c = term
        while c >= 0 and len(chain) < o["n_nodes"]:
            chain.append(c)
            c = int(o["parent"][c])
        for c in reversed(chain):
            rows.append(np.concatenate([[o["x"][c], o["y"][c], o["theta"][c]], o["u"][c]]))
            row_seg.append(s)
        off += 3 * o["iters"]
    return dict(segments=segs, path=np.array(rows, np.float64).reshape(-1, 8), path_seg=np.array(row_seg, np.int32),
                status=status, stop_seg=stop_seg)
