"""Batched planner front-end over libthetarrt.so.

Every method accepts either host data (numpy / sequences, copied to the GPU
through pinned memory) or torch CUDA tensors (used in place) and returns torch
tensors resident on the device; `.host()` on a result copies it back.  The
calls only enqueue work on torch's current stream of the planner's device.
There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import operator
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from .grid import OccupancyGrid
from .params import Params

STATUS_NAMES = {0: "OK_FOUND", 1: "OK_NOT_FOUND", 2: "ERR_ENDPOINT_INVALID", 3: "ERR_ENDPOINT_BLOCKED",
                4: "ERR_REF_RAISES_DRIVE_NONE", 5: "ERR_REF_RAISES_ARGMIN_EMPTY", 6: "ERR_CAPACITY",
                7: "ERR_REF_RAISES_NO_NEAREST"}
SEG_NOT_RUN = 255
IT_NEW_NODE, IT_EXISTING_NODE, IT_QRAND_BLOCKED, IT_QRAND_IN_TREE, IT_STEER_CONSTRAINT, IT_ARC_BLOCKED = range(6)
IT_NOT_RUN = 255
COUNTER_NAMES = ("nodes_scanned", "los_calls", "los_pixels", "arc_candidate_pixels", "arc_angle_tests",
                 "steer_calls", "drive_calls", "hash_probes", "nearest_sqrt_ties")


def _host_dict(obj):
    out = {}
    for k, v in obj.__dict__.items():
        out[k] = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v
    return out


@dataclass
class RrtResult:
    K: int
    node_x: torch.Tensor
    node_y: torch.Tensor
    node_theta: torch.Tensor
    parent: torch.Tensor
    n_nodes: torch.Tensor
    sol: torch.Tensor
    status: torch.Tensor
    iters: torch.Tensor
    u: torch.Tensor | None = None
    it_near: torch.Tensor | None = None
    it_new: torch.Tensor | None = None
    it_code: torch.Tensor | None = None
    los_log: torch.Tensor | None = None
    n_los: torch.Tensor | None = None
    counters: torch.Tensor | None = None
    lanes: int = 0
    # packed copy of the rows that exist (rrt(..., pack=True)): rows row_start[q] ... + n_nodes[q] - 1 of the pack_* arrays
    row_start: torch.Tensor | None = None
    pack_total: torch.Tensor | None = None  # int64 [1]: rows in use
    pack_x: torch.Tensor | None = None
    pack_y: torch.Tensor | None = None
    pack_theta: torch.Tensor | None = None
    pack_parent: torch.Tensor | None = None
    pack_u: torch.Tensor | None = None

    def host(self):
        return _host_dict(self)


@dataclass
class ThetaResult:
    path: torch.Tensor
    path_len: torch.Tensor
    cost: torch.Tensor
    expanded: torch.Tensor
    status: torch.Tensor
    los_log: torch.Tensor | None = None
    n_los: torch.Tensor | None = None
    pushes: torch.Tensor | None = None
    extra: dict = field(default_factory=dict)

    def host(self):
        return _host_dict(self)


@dataclass
class MissionResult:
    """Planner.missions output.  Per segment [B, S] (S = largest segment count): begin, end, solution, nearest
    (float64 [.., 3] = x, y, theta; NaN where the reference has None), mindist (NaN when none), n_nodes, n_edges,
    iters, seg_status (trrt_status of the segment's RRT, SEG_NOT_RUN = 255 where no segment ran).  Per mission:
    status (0 = the chain ran to its end; 4 / 7 = it stopped where the reference raises; otherwise the route search's
    status), stop_seg (-1 when the chain ran to its end), n_seg, waypoints (int32 [B, wp_cap, 2], n_waypoints of them
    valid), path (float64 [B, path_cap, 8] = x, y, theta, u[5] of main.path_nodes, segment after segment), path_seg
    (segment of each row) and path_len (full length, also when it exceeds path_cap; rows past it are not written)."""
    K: int
    begin: torch.Tensor
    end: torch.Tensor
    solution: torch.Tensor
    nearest: torch.Tensor
    mindist: torch.Tensor
    n_nodes: torch.Tensor
    n_edges: torch.Tensor
    iters: torch.Tensor
    seg_status: torch.Tensor
    status: torch.Tensor
    stop_seg: torch.Tensor
    n_seg: torch.Tensor
    waypoints: torch.Tensor
    n_waypoints: torch.Tensor
    path: torch.Tensor
    path_seg: torch.Tensor
    path_len: torch.Tensor
    route: ThetaResult | None = None

    def host(self):
        out = _host_dict(self)
        if self.route is not None:
            out["route"] = self.route.host()
        return out


SEED_STREAMS = ("host", "device")


def legacy_seeds(seeds):
    """Seeds of np.random.RandomState(int) as uint32 [n]; raises numpy's ValueError outside [0, 2**32)."""
    a = np.asarray(seeds).reshape(-1)
    if a.dtype.kind == "O" or a.dtype.kind == "b":
        a = np.array([operator.index(v) for v in a], dtype=object)
        if any(v < 0 or v > 0xffffffff for v in a):
            raise ValueError("Seed must be between 0 and 2**32 - 1")
        return a.astype(np.uint32)
    if a.dtype.kind not in "iu":
        raise TypeError(f"seeds must be integers, got {a.dtype}")
    if a.size and (int(a.min()) < 0 or int(a.max()) > 0xffffffff):
        raise ValueError("Seed must be between 0 and 2**32 - 1")
    return a.astype(np.uint32)


def mission_schedule(n_seg):
    """Dispatch order of trrt_mission_batch: missions by decreasing segment count (stable), so that the missions
    with a segment s are the first n_active[s] slots.  Returns (order int32 [B], n_active int32 [max(n_seg)])."""
    n_seg = np.asarray(n_seg, dtype=np.int64).reshape(-1)
    if n_seg.size and n_seg.min() < 0:
        raise ValueError("segment counts must be >= 0")
    order = np.argsort(-n_seg, kind="stable").astype(np.int32)
    S = int(n_seg.max()) if n_seg.size else 0
    n_active = (n_seg[None, :] > np.arange(S)[:, None]).sum(axis=1).astype(np.int32)
    return order, n_active


class Planner:
    """Device-resident planner for one OccupancyGrid (one or several same-size maps)."""

    def __init__(self, grid: OccupancyGrid, params: Params | None = None):
        if not torch.cuda.is_available():
            raise _lib.TrrtError("no CUDA device: theta_rrt_b200 has no CPU fallback")
        self.lib = _lib.load()
        self.grid = grid
        self.device = grid.device
        self.params = params or Params()
        self._work = {}

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _dev(self, a, dtype, shape=None):
        """numpy/sequence -> device tensor through pinned memory; CUDA tensors pass through."""
        if isinstance(a, torch.Tensor):
            t = a
            if t.device != self.device:
                t = t.to(self.device, non_blocking=True)
            if t.dtype != dtype:
                t = t.to(dtype)
            t = t.contiguous()
        else:
            npdt = {torch.float64: np.float64, torch.int32: np.int32, torch.uint8: np.uint8, torch.int16: np.int16,
                    torch.int64: np.int64}[dtype]
            h = torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=npdt)))
            t = h.pin_memory().to(self.device, non_blocking=True) if h.numel() else h.to(self.device)
        if shape is not None:
            t = t.reshape(shape)
        return t

    def _scratch(self, key, nbytes):
        """Grow-only scratch buffers (caller-owned workspace of the C ABI), one per kernel family AND stream: calls issued on
        different streams never share a workspace, and a buffer is only ever replaced by the stream that uses it (the caching
        allocator hands a freed block back to the stream it was allocated on, behind the work already queued there)."""
        key = (key, torch.cuda.current_stream(self.device).cuda_stream)
        cur = self._work.get(key)
        if cur is None or cur.numel() < nbytes:
            cur = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=self.device)
            self._work[key] = cur
        return cur

    def _map_ids(self, map_id, n):
        if map_id is None:
            return None
        t = self._dev(map_id, torch.int32, (n,))
        return t

    # ------------------------------------------------------------------ K4
    def los(self, seg, map_id=None, out=None, layout="tiles"):
        """search.lineofsight for segments int32 [n,4] = (x0,y0,x1,y1).  Returns uint8 [n] (1 = visible).
        layout "tiles" (default) tests 8 pixels per step on the strip copy of the grid with per-lane refill (trrt_los_batch_tiled),
        "rows" the packed rows with one thread per ray (trrt_los_batch); the results are identical."""
        if layout not in ("tiles", "rows"):
            raise ValueError("layout must be 'tiles' or 'rows'")
        with torch.cuda.device(self.device):
            seg = self._dev(seg, torch.int32).reshape(-1, 4)
            n = seg.shape[0]
            mid = self._map_ids(map_id, n)
            if out is None:
                out = torch.empty(n, dtype=torch.uint8, device=self.device)
            g = self.grid
            if layout == "tiles":
                _lib.check(self.lib.trrt_los_batch_tiled(g.tiles.data_ptr(), g.n_maps, g.H, g.W,
                                                         mid.data_ptr() if mid is not None else None, seg.data_ptr(),
                                                         n, out.data_ptr(), self._stream()), "trrt_los_batch_tiled")
            else:
                _lib.check(self.lib.trrt_los_batch(g.bits.data_ptr(), g.n_maps, g.H, g.W,
                                                   mid.data_ptr() if mid is not None else None, seg.data_ptr(), n,
                                                   out.data_ptr(), self._stream()), "trrt_los_batch")
        return out

    # ------------------------------------------------------------------ K1
    def nearest(self, x, y, qxy, want_d2=False):
        """Nearest tree node (rrt.py:156-158) for integer query points int32 [q,2] over SoA x, y float64 [n]."""
        with torch.cuda.device(self.device):
            x = self._dev(x, torch.float64).reshape(-1)
            y = self._dev(y, torch.float64).reshape(-1)
            qxy = self._dev(qxy, torch.int32).reshape(-1, 2)
            n, nq = x.shape[0], qxy.shape[0]
            idx = torch.empty(nq, dtype=torch.int32, device=self.device)
            d2 = torch.empty(nq, dtype=torch.float64, device=self.device) if want_d2 else None
            wb = self.lib.trrt_nearest_workspace_bytes(n, nq)
            work = self._scratch("nearest", wb)
            _lib.check(self.lib.trrt_nearest_batch(x.data_ptr(), y.data_ptr(), n, qxy.data_ptr(), nq, idx.data_ptr(),
                                                   d2.data_ptr() if want_d2 else None, work.data_ptr(), work.numel(),
                                                   self._stream()), "trrt_nearest_batch")
        return (idx, d2) if want_d2 else idx

    # ------------------------------------------------------------------ K2
    def rrt(self, starts, goals, sample_xy, sample_th, K=None, params=None, map_id=None, logs=False, want_u=True,
            counters=False, lanes=0, schedule=0, work_key="rrt", reuse=None, pack=False, packed=None):
        """rrt.rrt for a batch.  starts/goals float64 [q,3] (x, y, theta_deg); sample_xy int32 [q,K-1,2];
        sample_th float64 [q,K-1].  K = builtins.K (node capacity; K-1 iterations).
        pack=True: the kernel also leaves a packed copy of the tree rows that exist (pack_x, pack_y, pack_theta,
        pack_parent, pack_u; query q owns rows row_start[q] ... + n_nodes[q] - 1, pack_total rows in all); `packed` may
        pass a dict of such arrays to use; its pack_total must then hold the first row to use (0 for arrays of this call's own)."""
        P = params or self.params
        with torch.cuda.device(self.device):
            starts = self._dev(starts, torch.float64).reshape(-1, 3)
            goals = self._dev(goals, torch.float64).reshape(-1, 3)
            nq = starts.shape[0]
            sample_th = self._dev(sample_th, torch.float64)
            if K is None:
                K = (sample_th.numel() // nq if nq else 0) + 1
            K = int(K)
            if sample_th.numel() != nq * (K - 1):
                raise ValueError(f"sample stream has {sample_th.numel()} values, expected {nq} x (K-1 = {K - 1})")
            sample_th = sample_th.reshape(nq, K - 1)
            # int16 sample coordinates are taken as they are (half the host-to-device bytes of the stream's xy part)
            xy16 = isinstance(sample_xy, torch.Tensor) and sample_xy.dtype == torch.int16
            sample_xy = self._dev(sample_xy, torch.int16 if xy16 else torch.int32).reshape(nq, K - 1, 2)
            mid = self._map_ids(map_id, nq)
            dev = self.device
            f64 = dict(dtype=torch.float64, device=dev)
            i32 = dict(dtype=torch.int32, device=dev)
            if reuse is not None and reuse.K == K and reuse.node_x.shape[0] == nq and (reuse.u is not None) == bool(want_u) \
                    and (reuse.it_near is not None) == bool(logs) and (reuse.counters is not None) == bool(counters):
                res = reuse  # caller-provided result buffers of the right shape (rrt_host keeps one set per stream)
                if counters:
                    res.counters.zero_()
            else:
                res = RrtResult(K=K, node_x=torch.empty((nq, K), **f64), node_y=torch.empty((nq, K), **f64),
                                node_theta=torch.empty((nq, K), **f64), parent=torch.empty((nq, K), **i32),
                                n_nodes=torch.empty(nq, **i32), sol=torch.empty(nq, **i32), status=torch.empty(nq, **i32),
                                iters=torch.empty(nq, **i32))
                if want_u:
                    res.u = torch.empty((nq, K, 5), **f64)
                if logs:
                    res.it_near = torch.empty((nq, K - 1), **i32)
                    res.it_new = torch.empty((nq, K - 1), **i32)
                    res.it_code = torch.empty((nq, K - 1), dtype=torch.uint8, device=dev)
                    res.los_log = torch.zeros((nq, 2 * (K - 1)), dtype=torch.uint8, device=dev)
                    res.n_los = torch.empty(nq, **i32)
                if counters:
                    res.counters = torch.zeros((nq, 9), dtype=torch.int64, device=dev)
            if pack:
                if packed is None:
                    packed = {"pack_x": torch.empty(nq * K, **f64), "pack_y": torch.empty(nq * K, **f64),
                              "pack_theta": torch.empty(nq * K, **f64), "pack_parent": torch.empty(nq * K, **i32),
                              "row_start": torch.empty(nq, dtype=torch.int64, device=dev),
                              "pack_total": torch.empty(1, dtype=torch.int64, device=dev)}
                    if want_u:
                        packed["pack_u"] = torch.empty((nq * K, 5), **f64)
                    packed["pack_total"].zero_()
                for k, v in packed.items():  # a reused set: the caller has set pack_total to the first row to use
                    setattr(res, k, v)
            wb = self.lib.trrt_rrt_workspace_bytes(nq, K)
            work = self._scratch(work_key, wb)  # concurrent launches (rrt_host) must not share a workspace
            g = self.grid
            ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
            a = _lib.CRrtArgs(d_bits=g.bits.data_ptr(), n_maps=g.n_maps, H=g.H, W=g.W, d_map_id=ptr(mid),
                              params=P.to_c(), n_queries=nq, K=K, lanes_per_query=int(lanes), schedule=int(schedule),
                              sample_xy_i16=int(xy16),
                              d_start=starts.data_ptr(), d_goal=goals.data_ptr(), d_sample_xy=sample_xy.data_ptr(),
                              d_sample_th=sample_th.data_ptr(), d_node_x=res.node_x.data_ptr(),
                              d_node_y=res.node_y.data_ptr(), d_node_th=res.node_theta.data_ptr(),
                              d_parent=res.parent.data_ptr(), d_u=ptr(res.u), d_n_nodes=res.n_nodes.data_ptr(),
                              d_sol=res.sol.data_ptr(), d_status=res.status.data_ptr(), d_iters=res.iters.data_ptr(),
                              d_it_near=ptr(res.it_near), d_it_new=ptr(res.it_new), d_it_code=ptr(res.it_code),
                              d_los_log=ptr(res.los_log), d_n_los=ptr(res.n_los), d_counters=ptr(res.counters),
                              d_work=work.data_ptr(), work_bytes=work.numel(),
                              d_pack_rows=ptr(res.pack_total) if pack else None, d_row_start=ptr(res.row_start) if pack else None,
                              d_pack_x=ptr(res.pack_x) if pack else None, d_pack_y=ptr(res.pack_y) if pack else None,
                              d_pack_th=ptr(res.pack_theta) if pack else None,
                              d_pack_parent=ptr(res.pack_parent) if pack else None,
                              d_pack_u=ptr(res.pack_u) if (pack and want_u) else None)
            _lib.check(self.lib.trrt_rrt_batch(C.byref(a), self._stream()), "trrt_rrt_batch")
            res.lanes = int(lanes)
            # keep inputs alive until the stream has consumed them
            res._keep = (starts, goals, sample_xy, sample_th, mid)
        return res

    _TREE = ("node_x", "node_y", "node_theta", "parent", "u")
    _PACKED = {"node_x": "pack_x", "node_y": "pack_y", "node_theta": "pack_theta", "parent": "pack_parent", "u": "pack_u"}

    def rrt_host(self, starts, goals, sample_xy, sample_th, out, K=None, chunks=4, wait=True, valid_rows_only=False, **kw):
        """rrt.rrt for a batch whose inputs and outputs live in (pinned) HOST memory: the queries are cut into
        `chunks` contiguous pieces, each on its own stream (host->device copy, fused kernel, device->host copy), so
        that the PCIe transfers of one piece overlap the planning of the others.  `out` maps RrtResult field names
        (node_x, node_y, node_theta, parent, u, n_nodes, sol, status, iters, ...) to host tensors with a leading
        query dimension; they are filled in place, and only the fields that are present travel (leave `u` out and the
        kernel does not even produce it).  The call returns after enqueuing.  With wait=True the planner's
        current stream waits for every piece (synchronise it before reading `out`).  With wait=False nothing waits:
        successive calls queue piece c of the next batch behind piece c of this one on the same stream, so the
        transfers of one batch also overlap the planning of the next (double-buffered streaming of batches); call
        host_sync() before reading the outputs or reusing the host buffers.

        valid_rows_only=True: a tree holds n_nodes[q] <= K nodes (about half of K on cfg 3) and only those rows are
        brought back.  The fused kernel itself packs them (one row reservation per finished query, trrt_rrt_args
        d_pack_*), and every piece is fetched with one linear copy per array; in the host arrays (contiguous pinned
        tensors of the usual [q, K(, 5)] shape, viewed as flat row arrays) the rows of query q are rows
        out["row_start"][q] ... + n_nodes[q] - 1, anything else is not touched.  `out` must contain n_nodes and
        row_start (int64 [q]).  The size of a piece's copy is known once its row count has reached the host, so the
        copies of a batch are issued one call later (or in host_sync()), on copy streams of their own, while the next
        batch is already being planned; the packed rows are double-buffered per piece."""
        ins = [t if isinstance(t, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(t))
               for t in (starts, goals, sample_xy, sample_th)]
        nq = ins[0].shape[0]
        chunks = max(1, min(int(chunks), nq))
        defer = bool(valid_rows_only)
        want_u = "u" in out
        if defer:
            if "n_nodes" not in out or "row_start" not in out:
                raise ValueError("valid_rows_only needs 'n_nodes' and 'row_start' among the outputs")
            for k in self._TREE:
                if k in out and not (out[k].is_pinned() and out[k].is_contiguous()):
                    raise ValueError(f"valid_rows_only needs a contiguous pinned host tensor for '{k}'")
        with torch.cuda.device(self.device):
            main = torch.cuda.current_stream(self.device)
            if not hasattr(self, "_streams") or len(self._streams) < chunks:
                self.host_sync()  # nothing may be in flight on streams that are about to be replaced
                self._streams = [torch.cuda.Stream(self.device) for _ in range(chunks)]
                self._copy_streams = [torch.cuda.Stream(self.device) for _ in range(chunks)]
            if not hasattr(self, "_host_cache"):
                self._host_cache = {}
            Kc = int(K) if K is not None else ins[3].numel() // nq + 1
            pk = None
            if defer:
                # packed rows of the whole batch: two sets used alternately (one is fetched while the other is filled).  Piece c
                # owns rows [lo*K, hi*K) of every array and its own row counter, which starts at lo*K, so the kernel's
                # row_start values are positions in the batch-wide arrays -- and in the flat host arrays.  No small kernel
                # runs between the pieces' persistent kernels (it would wait for an SM until one of them retires): the
                # counters are initialised and read back by copies.
                pkey = ("packed", nq, Kc, chunks, want_u)
                pc = self._host_cache.get(pkey)
                if pc is None:
                    def new_set():
                        d = {"pack_x": torch.empty(nq * Kc, dtype=torch.float64, device=self.device),
                             "pack_y": torch.empty(nq * Kc, dtype=torch.float64, device=self.device),
                             "pack_theta": torch.empty(nq * Kc, dtype=torch.float64, device=self.device),
                             "pack_parent": torch.empty(nq * Kc, dtype=torch.int32, device=self.device),
                             "row_start": torch.empty(nq, dtype=torch.int64, device=self.device),
                             "pack_total": torch.empty(chunks, dtype=torch.int64, device=self.device),
                             "total_host": torch.zeros(chunks, dtype=torch.int64).pin_memory(), "free": [None] * chunks}
                        if want_u:
                            d["pack_u"] = torch.empty((nq * Kc, 5), dtype=torch.float64, device=self.device)
                        return d
                    first = torch.tensor([nq * c // chunks * Kc for c in range(chunks)], dtype=torch.int64).pin_memory()
                    pc = {"sets": [new_set(), new_set()], "turn": 0, "first": first}
                    self._host_cache[pkey] = pc
                pk = pc["sets"][pc["turn"]]
                pc["turn"] = 1 - pc["turn"]
            start = torch.cuda.Event()
            start.record(main)
            keep, deferred = [], []
            for c in range(chunks):
                lo, hi = nq * c // chunks, nq * (c + 1) // chunks
                st = self._streams[c]
                st.wait_event(start)
                with torch.cuda.stream(st):
                    # device buffers of a piece are allocated once and reused by later calls of the same shape
                    key = (c, chunks, want_u, tuple((tuple(t[lo:hi].shape), t.dtype) for t in ins))
                    cached = self._host_cache.get(key)
                    if cached is None:
                        cached = {"din": [torch.empty(t[lo:hi].shape, dtype=t.dtype, device=self.device) for t in ins], "res": None}
                        self._host_cache[key] = cached
                    din = cached["din"]
                    for d, t in zip(din, ins):
                        d.copy_(t[lo:hi], non_blocking=True)
                    packed = None
                    if defer:
                        if pk["free"][c] is not None:
                            st.wait_event(pk["free"][c])  # the copies that still read this set's rows of the piece
                            pk["free"][c] = None
                        packed = {k: pk[k] for k in ("pack_x", "pack_y", "pack_theta", "pack_parent", "pack_u") if k in pk}
                        packed["row_start"] = pk["row_start"][lo:hi]
                        packed["pack_total"] = pk["pack_total"][c:c + 1]
                        packed["pack_total"].copy_(pc["first"][c:c + 1], non_blocking=True)
                    res = self.rrt(*din, K=K, work_key=("rrt", c), reuse=cached["res"], want_u=want_u, pack=defer, packed=packed, **kw)
                    cached["res"] = res
                    for name, t in out.items():
                        if defer and name in self._TREE:
                            continue
                        t[lo:hi].copy_(getattr(res, name), non_blocking=True)
                    if defer:
                        pk["total_host"][c:c + 1].copy_(res.pack_total, non_blocking=True)
                    keep.append((din, res))
                done = torch.cuda.Event()
                done.record(st)
                if defer:
                    deferred.append((c, lo, hi, res.K, pk, done, out))
                elif wait:
                    main.wait_event(done)
                else:
                    self._pending = [e for e in getattr(self, "_pending", []) if not e.query()] + [done]
            self._inflight = keep  # tensors stay referenced until the next call
            if defer:
                # the previous batch first (its row counts are on the host by now), this one only if the caller waits
                previous, self._deferred = getattr(self, "_deferred", []), deferred
                self._issue_tree_copies(previous)
                if wait:
                    self._issue_tree_copies(self._deferred)
                    self._deferred = []
                    self.host_sync()
        return out

    def _issue_tree_copies(self, items):
        """Second half of rrt_host(valid_rows_only=True) for the pieces in `items`: wait until the piece's row count is on
        the host, then fetch its packed rows with one linear copy per array on the piece's copy stream."""
        for c, lo, hi, K, pk, done, out in items:
            done.synchronize()
            rows = min(max(int(pk["total_host"][c]) - lo * K, 0), (hi - lo) * K)
            cs = self._copy_streams[c]
            cs.wait_event(done)
            with torch.cuda.stream(cs):
                for name, pname in self._PACKED.items():
                    if name not in out or pname not in pk:
                        continue
                    m = 5 if name == "u" else 1
                    sl = slice(lo * K * m, (lo * K + rows) * m)
                    out[name].view(-1)[sl].copy_(pk[pname].view(-1)[sl], non_blocking=True)
            copied = torch.cuda.Event()
            copied.record(cs)
            pk["free"][c] = copied
            self._pending = [e for e in getattr(self, "_pending", []) if not e.query()] + [copied]

    def host_sync(self):
        """Make the planner's current stream wait for every piece enqueued by rrt_host(..., wait=False)."""
        with torch.cuda.device(self.device):
            if getattr(self, "_deferred", None):
                self._issue_tree_copies(self._deferred)
                self._deferred = []
            main = torch.cuda.current_stream(self.device)
            for e in getattr(self, "_pending", []):
                main.wait_event(e)
            self._pending = []

    def findnearest(self, res: RrtResult, goals, params=None):
        """rrt.findnearest (rrt.py:117-128) for every query of an RrtResult produced with logs=True."""
        if res.it_near is None:
            raise ValueError("findnearest needs the edge log: run rrt(..., logs=True)")
        P = params or self.params
        with torch.cuda.device(self.device):
            goals = self._dev(goals, torch.float64).reshape(-1, 3)
            nq = goals.shape[0]
            best = torch.empty(nq, dtype=torch.int32, device=self.device)
            dist = torch.empty(nq, dtype=torch.float64, device=self.device)
            cp = P.to_c()
            _lib.check(self.lib.trrt_findnearest_batch(C.byref(cp), nq, res.K, res.node_x.data_ptr(),
                                                       res.node_y.data_ptr(), res.node_theta.data_ptr(),
                                                       res.n_nodes.data_ptr(), res.it_near.data_ptr(),
                                                       res.it_new.data_ptr(), goals.data_ptr(), best.data_ptr(),
                                                       dist.data_ptr(), self._stream()), "trrt_findnearest_batch")
        return best, dist

    # ------------------------------------------------------------------ single steps
    def steer(self, inputs, params=None):
        """rrt.steer for rows (ox, oy, theta, gx, gy, thetagoal).  Returns (out float64 [n,8], straight uint8 [n])."""
        P = params or self.params
        with torch.cuda.device(self.device):
            inp = self._dev(inputs, torch.float64).reshape(-1, 6)
            n = inp.shape[0]
            out = torch.empty((n, 8), dtype=torch.float64, device=self.device)
            straight = torch.empty(n, dtype=torch.uint8, device=self.device)
            cp = P.to_c()
            _lib.check(self.lib.trrt_steer_batch(C.byref(cp), n, inp.data_ptr(), out.data_ptr(), straight.data_ptr(),
                                                 self._stream()), "trrt_steer_batch")
        return out, straight

    def drive(self, inputs, params=None):
        """rrt.drive for rows (ox, oy, theta, u.steer, iccx, iccy, rad, dist).  Returns float64 [n,3]."""
        P = params or self.params
        with torch.cuda.device(self.device):
            inp = self._dev(inputs, torch.float64).reshape(-1, 8)
            n = inp.shape[0]
            out = torch.empty((n, 3), dtype=torch.float64, device=self.device)
            cp = P.to_c()
            _lib.check(self.lib.trrt_drive_batch(C.byref(cp), n, inp.data_ptr(), out.data_ptr(), self._stream()),
                       "trrt_drive_batch")
        return out

    def arc_blocked(self, inputs, map_id=None, lanes=0):
        """rrt.py:173-174 for rows (bx, by, lx, ly, u.steer, iccx, iccy, rad, straight).  Returns uint8 [n]."""
        with torch.cuda.device(self.device):
            inp = self._dev(inputs, torch.float64).reshape(-1, 9)
            n = inp.shape[0]
            mid = self._map_ids(map_id, n)
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
            g = self.grid
            _lib.check(self.lib.trrt_arc_batch(g.bits.data_ptr(), g.n_maps, g.H, g.W,
                                               mid.data_ptr() if mid is not None else None, n, inp.data_ptr(),
                                               out.data_ptr(), int(lanes), self._stream()), "trrt_arc_batch")
        return out

    def arc_pixels(self, inputs, cap=None):
        """Pixel lists of search.getArc (mode 0), search.bresenham (mode 1) and search.getCircle (mode 2) in the reference's
        list order, for rows (bx, by, lx, ly, u.steer, iccx, iccy, rad, mode).  Returns a list of int32 arrays [len, 2]."""
        with torch.cuda.device(self.device):
            inp = self._dev(inputs, torch.float64).reshape(-1, 9)
            n = inp.shape[0]
            g = self.grid
            if cap is None:
                cap = 16 * (g.H + g.W) + 64
            while True:
                pix = torch.empty((n, cap, 2), dtype=torch.int32, device=self.device)
                cnt = torch.empty(n, dtype=torch.int32, device=self.device)
                _lib.check(self.lib.trrt_arc_pixels_batch(g.H, g.W, n, inp.data_ptr(), int(cap), pix.data_ptr(), cnt.data_ptr(),
                                                          self._stream()), "trrt_arc_pixels_batch")
                c = cnt.cpu().numpy()
                if n == 0 or int(c.max()) <= cap:
                    break
                cap = int(c.max())  # a list was longer than the buffer: once more with room for the longest
            h = pix.cpu().numpy()
        return [h[i, :int(c[i])].copy() for i in range(n)]

    def clearance(self, nodes, map_id=None, params=None):
        """rrt.bike_clear / rrt.front_of_bike_clear (rrt.py:208-222) for rows (x, y, theta).  Returns uint8 [n, 2]."""
        P = params or self.params
        with torch.cuda.device(self.device):
            inp = self._dev(nodes, torch.float64).reshape(-1, 3)
            n = inp.shape[0]
            mid = self._map_ids(map_id, n)
            out = torch.empty((n, 2), dtype=torch.uint8, device=self.device)
            g = self.grid
            cp = P.to_c()
            _lib.check(self.lib.trrt_clearance_batch(g.bits.data_ptr(), g.n_maps, g.H, g.W, mid.data_ptr() if mid is not None else None,
                                                     C.byref(cp), n, inp.data_ptr(), out.data_ptr(), self._stream()),
                       "trrt_clearance_batch")
        return out

    def anglediff(self, pairs):
        """rrt.anglediff (rrt.py:108-115) for rows (a1, a2) in degrees.  Returns float64 [n]."""
        with torch.cuda.device(self.device):
            inp = self._dev(pairs, torch.float64).reshape(-1, 2)
            n = inp.shape[0]
            out = torch.empty(n, dtype=torch.float64, device=self.device)
            _lib.check(self.lib.trrt_anglediff_batch(n, inp.data_ptr(), out.data_ptr(), self._stream()), "trrt_anglediff_batch")
        return out

    # ------------------------------------------------------------------ K3
    def theta(self, start_goal, thetastar=None, map_id=None, path_cap=None, log_los=False, lanes=0, n_slots=0,
              heap_cap=0, longest_first=True, mem_budget=None):
        """search.astar for queries int32 [q,4] = (sx, sy, gx, gy).  longest_first: dispatch the queries to the
        persistent slots by decreasing start-goal distance (a batch ends with its longest search; results stay
        indexed by query).  mem_budget: bytes the search workspace may take (default: half of the free device memory); the
        number of concurrent searches is cut down to fit."""
        if thetastar is None:
            thetastar = self.params.THETASTAR
        with torch.cuda.device(self.device):
            sg = self._dev(start_goal, torch.int32).reshape(-1, 4)
            nq = sg.shape[0]
            mid = self._map_ids(map_id, nq)
            g = self.grid
            if path_cap is None:
                path_cap = 4 * (g.H + g.W)
            dev = self.device
            i32 = dict(dtype=torch.int32, device=dev)
            res = ThetaResult(path=torch.full((nq, path_cap, 2), -1, **i32), path_len=torch.empty(nq, **i32),
                              cost=torch.empty(nq, dtype=torch.float64, device=dev), expanded=torch.empty(nq, **i32),
                              status=torch.empty(nq, **i32), n_los=torch.empty(nq, **i32),
                              pushes=torch.empty(nq, **i32))
            los_cap = 0
            if log_los:
                los_cap = g.H * g.W
                res.los_log = torch.zeros((nq, los_cap), dtype=torch.uint8, device=dev)
            ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
            a = _lib.CThetaArgs(d_bits=g.bits.data_ptr(), n_maps=g.n_maps, H=g.H, W=g.W, d_map_id=ptr(mid),
                                thetastar=int(bool(thetastar)), lanes_per_query=int(lanes), n_queries=nq,
                                d_start_goal=sg.data_ptr(), d_path=res.path.data_ptr(), path_cap=int(path_cap),
                                d_path_len=res.path_len.data_ptr(), d_cost=res.cost.data_ptr(),
                                d_expanded=res.expanded.data_ptr(), d_status=res.status.data_ptr(),
                                d_los_log=ptr(res.los_log), los_cap=int(los_cap), d_n_los=res.n_los.data_ptr(),
                                d_pushes=res.pushes.data_ptr(), n_slots=int(n_slots), heap_cap=int(heap_cap),
                                d_work=None, work_bytes=0, d_order=None)
            order = None
            if longest_first and nq > 1:
                d = (sg[:, 2] - sg[:, 0]).to(torch.float32) ** 2 + (sg[:, 3] - sg[:, 1]).to(torch.float32) ** 2
                order = torch.argsort(d, descending=True).to(torch.int32)
                a.d_order = order.data_ptr()
            wb = self.lib.trrt_theta_workspace_bytes(C.byref(a))  # fills n_slots / heap_cap
            if wb == 0:
                raise _lib.TrrtError("trrt_theta_batch: map too large for the search workspace (2*H*W heap entries must fit an int32)")
            if mem_budget is None:  # half of what is free now plus what the cached workspace already holds
                have = self._work.get(("theta", torch.cuda.current_stream(self.device).cuda_stream))
                mem_budget = (torch.cuda.mem_get_info(self.device)[0] + (have.numel() if have is not None else 0)) // 2
            if wb > mem_budget:  # fewer concurrent searches: a slot costs (H*W + heap_cap) * 16 bytes
                per_slot = (g.H * g.W + int(a.heap_cap)) * 16
                a.n_slots = max(1, int((mem_budget - 256) // per_slot))
                wb = self.lib.trrt_theta_workspace_bytes(C.byref(a))
                if wb > mem_budget:
                    raise _lib.TrrtError(f"trrt_theta_batch: one search slot needs {per_slot} bytes, budget {mem_budget}")
            work = self._scratch("theta", wb)
            a.d_work = work.data_ptr()
            a.work_bytes = work.numel()
            _lib.check(self.lib.trrt_theta_batch(C.byref(a), self._stream()), "trrt_theta_batch")
            res.extra = dict(n_slots=int(a.n_slots), heap_cap=int(a.heap_cap), workspace_bytes=int(wb))
            res._keep = (sg, mid, order)
        return res

    # ------------------------------------------------------------------ seeded streams
    def legacy_normals(self, seeds, counts, fix_cap=None):
        """np.random.RandomState(seeds[i]).standard_normal(counts[i]) for every i, bit for bit, drawn on the device
        (trrt_legacy_normals_draw).  Returns (normals float64 [sum(counts)], ranges int64 [n, 2]): seed i's stream is
        normals[ranges[i, 0]:ranges[i, 1]], both on the device.  Integer seeds in [0, 2**32) only (init_genrand
        seeding).  The logs the device cannot settle (about 6 % of the pairs) come from this process's libm, the one
        numpy calls: their count is the one host read, then the r2 values travel to pinned memory and the logs back.
        fix_cap: room of the list of such pairs (default a sixteenth of the normals); an overflow draws once more with
        the reported count."""
        seeds = legacy_seeds(seeds)
        counts = np.asarray(counts, dtype=np.int64).reshape(-1)
        n = len(seeds)
        if len(counts) != n:
            raise ValueError(f"{len(counts)} counts for {n} seeds")
        if n and counts.min() < 0:
            raise ValueError("counts must be >= 0")
        rng = np.zeros((n, 2), np.int64)
        rng[:, 1] = np.cumsum(counts)
        rng[1:, 0] = rng[:-1, 1]
        total = int(rng[-1, 1]) if n else 0
        dev = self.device
        with torch.cuda.device(dev):
            out = torch.empty(total, dtype=torch.float64, device=dev)
            rng_d = self._dev(rng, torch.int64) if n else torch.zeros((0, 2), dtype=torch.int64, device=dev)
            if total == 0:
                return out, rng_d
            seeds_d = self._dev(seeds.view(np.int32), torch.int32)
            cap = int(fix_cap) if fix_cap is not None else total // 16 + 1024
            count = torch.zeros(1, dtype=torch.int64, device=dev)
            work = self._scratch("legacy_normals", self.lib.trrt_legacy_normals_workspace_bytes(n))
            for _ in range(2):  # a second draw only when the fixup list overflowed
                fix_pos = torch.empty(max(cap, 1), dtype=torch.int64, device=dev)
                fix_r2 = torch.empty(max(cap, 1), dtype=torch.float64, device=dev)
                a = _lib.CLegacyNormalsArgs(n_seeds=n, d_seeds=seeds_d.data_ptr(), d_range=rng_d.data_ptr(), d_out=out.data_ptr(),
                                            d_fix_pos=fix_pos.data_ptr(), d_fix_r2=fix_r2.data_ptr(), fix_cap=cap,
                                            d_fix_count=count.data_ptr(), d_work=work.data_ptr(), work_bytes=work.numel())
                _lib.check(self.lib.trrt_legacy_normals_draw(C.byref(a), self._stream()), "trrt_legacy_normals_draw")
                n_fix = int(count.cpu()[0])  # the one host read
                if n_fix <= cap:
                    break
                cap = n_fix  # the list overflowed: once more with room for every entry
            if n_fix:
                h_r2, h_log = self._pinned("legacy_normals", n_fix)
                h_r2.copy_(fix_r2[:n_fix], non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
                _lib.check(self.lib.trrt_libm_log_batch(h_r2.data_ptr(), h_log.data_ptr(), n_fix), "trrt_libm_log_batch")
                d_log = h_log.to(dev, non_blocking=True)
                _lib.check(self.lib.trrt_legacy_normals_fixup(C.byref(a), d_log.data_ptr(), n_fix, self._stream()),
                           "trrt_legacy_normals_fixup")
        return out, rng_d

    def _pinned(self, key, n):
        """Two grow-only pinned float64 host buffers of at least n values per key and stream.  A call that reuses them has
        synchronised the stream first, so the copies of the previous call that read them have completed."""
        key = (key, torch.cuda.current_stream(self.device).cuda_stream)
        cur = getattr(self, "_pin", {}).get(key)
        if cur is None or cur[0].numel() < n:
            cur = tuple(torch.empty(max(int(n), 1024), dtype=torch.float64).pin_memory() for _ in range(2))
            self.__dict__.setdefault("_pin", {})[key] = cur
        return cur[0][:n], cur[1][:n]

    def rand_conf(self, goals, seeds, K=None, xy_dtype=torch.int32, params=None):
        """The K-1 rand_conf samples (rrt.py:53-68) of query q after np.random.seed(seeds[q]), around goals[q] float64
        [q, 3] = (x, y, theta_deg), i.e. samples.make_stream(goal, K-1, seeds[q], ...) per query, drawn on the device
        (legacy_normals, then trrt_rand_conf_batch).  Returns (sample_xy xy_dtype [q, K-1, 2], sample_th float64
        [q, K-1]) on the device, the sample layout of rrt(); xy_dtype is torch.int32 or torch.int16."""
        P = params or self.params
        K = int(K if K is not None else P.K)
        if K < 1:
            raise ValueError("K must be >= 1")
        if xy_dtype not in (torch.int32, torch.int16):
            raise ValueError("xy_dtype must be torch.int32 or torch.int16")
        with torch.cuda.device(self.device):
            goals = self._dev(goals, torch.float64).reshape(-1, 3)
            nq, S = goals.shape[0], K - 1
            seeds = legacy_seeds(seeds)
            if len(seeds) != nq:
                raise ValueError(f"{len(seeds)} seeds for {nq} queries")
            nz, _ = self.legacy_normals(seeds, np.full(nq, 3 * S, np.int64))
            sxy = torch.empty((nq, S, 2), dtype=xy_dtype, device=self.device)
            sth = torch.empty((nq, S), dtype=torch.float64, device=self.device)
            g = self.grid
            _lib.check(self.lib.trrt_rand_conf_batch(g.H, g.W, float(P.xystdv), float(P.anglestdv), nq, S, goals.data_ptr(),
                                                     nz.data_ptr(), sxy.data_ptr(), int(xy_dtype == torch.int16),
                                                     sth.data_ptr(), self._stream()), "trrt_rand_conf_batch")
        return sxy, sth

    # ------------------------------------------------------------------ main.py missions
    def missions(self, start_goal=None, waypoints=None, seeds=None, normals=None, normal_range=None, map_id=None, K=None,
                 thetastar=None, path_cap=None, params=None, seed_stream="host") -> MissionResult:
        """main.plan for a batch of missions (main.py:56-84): a route, then one RRT per consecutive waypoint pair with
        the headings of main.chain, restarting from the rrt.findnearest node once a segment has failed.  The segment
        chain runs on the device (trrt_mission_batch): per stage, one kernel builds every mission's start, goal and
        samples, the fused RRT kernel runs, and one kernel commits the segment records and path rows.

        Routes: `waypoints` (one (n_i, 2) integer sequence per mission), or Theta* / A* (`thetastar`, default
        Params.THETASTAR) over `start_goal` int32 [B, 4] = (sx, sy, gx, gy).  The route lengths are read back once to
        build the schedule; nothing else waits for the device.
        Samples: `seeds` gives mission m the normals of np.random.RandomState(seeds[m]) in draw order, i.e. the stream
        main.chain consumes after np.random.seed(seeds[m]) (reference parity), drawn by numpy on the host
        (seed_stream="host") or on the device (seed_stream="device", legacy_normals: the same bits).  Or `normals`: a float64 stream (e.g. a
        device torch.randn tensor) with `normal_range` int64 [B, 2] = [begin, end) per mission, or a [B, L] tensor with one
        row per mission; mission m needs 3 * (K-1) * n_seg[m] values.
        map_id: [B] map of each mission.  path_cap: path rows kept per mission (default n_seg_max * K, which never
        truncates)."""
        P = params or self.params
        K = int(K if K is not None else P.K)
        if K < 2:
            raise ValueError("K must be >= 2")
        if (seeds is None) == (normals is None):
            raise ValueError("pass exactly one of seeds and normals")
        if seed_stream not in SEED_STREAMS:
            raise ValueError(f"seed_stream must be one of {SEED_STREAMS}")
        g = self.grid
        with torch.cuda.device(self.device):
            route = None
            if waypoints is None:
                if start_goal is None:
                    raise ValueError("pass start_goal or waypoints")
                route = self.theta(start_goal, thetastar=thetastar if thetastar is not None else P.THETASTAR, map_id=map_id)
                wp, n_wp, route_status = route.path, route.path_len, route.status
                hr = torch.stack([n_wp, route_status]).cpu().numpy()  # the one host read: segment counts for the schedule
                n_wp_h, rs_h = hr[0].astype(np.int64), hr[1]
                B = len(n_wp_h)
                ok = (rs_h == 0) & (n_wp_h <= wp.shape[1])
                n_seg = np.where(ok, np.maximum(n_wp_h - 1, 0), 0)
            else:
                wl = [np.asarray(w, dtype=np.int64).reshape(-1, 2) for w in waypoints]
                B = len(wl)
                n_wp_h = np.array([len(w) for w in wl], np.int64)
                wp_h = np.zeros((B, max(int(n_wp_h.max()) if B else 1, 1), 2), np.int32)
                for m, w in enumerate(wl):
                    wp_h[m, :len(w)] = w
                wp = self._dev(wp_h, torch.int32)
                n_wp = self._dev(n_wp_h, torch.int32)
                route_status = None
                n_seg = np.maximum(n_wp_h - 1, 0)
            order, n_active = mission_schedule(n_seg)
            S = len(n_active)
            need = 3 * (K - 1) * n_seg
            if seeds is not None:
                seeds = np.asarray(seeds).reshape(-1)
                if len(seeds) != B:
                    raise ValueError(f"{len(seeds)} seeds for {B} missions")
                if seed_stream == "device":
                    nz, rng_d = self.legacy_normals(seeds, need)
                    if nz.numel() == 0:
                        nz = torch.zeros(1, dtype=torch.float64, device=self.device)
                else:
                    rng = np.zeros((B, 2), np.int64)
                    rng[:, 1] = np.cumsum(need)
                    rng[1:, 0] = rng[:-1, 1]
                    flat = np.empty(int(need.sum()), np.float64)
                    for m in range(B):
                        if need[m]:
                            flat[rng[m, 0]:rng[m, 1]] = np.random.RandomState(int(seeds[m])).standard_normal(int(need[m]))
                    nz = self._dev(flat, torch.float64) if flat.size else torch.zeros(1, dtype=torch.float64, device=self.device)
            else:
                nz = self._dev(normals, torch.float64)
                if normal_range is None:
                    if nz.dim() != 2 or nz.shape[0] != B:
                        raise ValueError("normals without normal_range must be a [missions, L] array")
                    L = nz.shape[1]
                    rng = np.stack([np.arange(B) * L, np.arange(B) * L + L], axis=1).astype(np.int64)
                else:
                    rng = (normal_range.cpu().numpy() if isinstance(normal_range, torch.Tensor) else np.asarray(normal_range))
                    rng = rng.astype(np.int64).reshape(B, 2)
                nz = nz.reshape(-1)
                if B and (rng.min() < 0 or rng[:, 1].max() > nz.numel() or (rng[:, 1] < rng[:, 0]).any()):
                    raise ValueError("normal_range outside the normals")
                short = np.nonzero(rng[:, 1] - rng[:, 0] < need)[0]
                if len(short):
                    m = int(short[0])
                    raise ValueError(f"mission {m} has {int(rng[m, 1] - rng[m, 0])} normals, its {int(n_seg[m])} segments "
                                     f"need {int(need[m])} (3 * (K-1) per segment)")
                if nz.numel() == 0:
                    nz = torch.zeros(1, dtype=torch.float64, device=self.device)
            if not (seeds is not None and seed_stream == "device"):
                rng_d = self._dev(rng, torch.int64) if B else None
            order_d = self._dev(order, torch.int32)
            mid = self._map_ids(map_id, B)
            if path_cap is None:
                path_cap = max(S * K, 1)
            dev = self.device
            f64 = dict(dtype=torch.float64, device=dev)
            i32 = dict(dtype=torch.int32, device=dev)
            Sc = max(S, 1)
            res = MissionResult(K=K, begin=torch.empty((B, Sc, 3), **f64), end=torch.empty((B, Sc, 3), **f64),
                                solution=torch.empty((B, Sc, 3), **f64), nearest=torch.empty((B, Sc, 3), **f64),
                                mindist=torch.empty((B, Sc), **f64), n_nodes=torch.empty((B, Sc), **i32),
                                n_edges=torch.empty((B, Sc), **i32), iters=torch.empty((B, Sc), **i32),
                                seg_status=torch.empty((B, Sc), **i32), status=torch.empty(B, **i32),
                                stop_seg=torch.empty(B, **i32), n_seg=torch.empty(B, **i32), waypoints=wp,
                                n_waypoints=n_wp, path=torch.empty((B, int(path_cap), 8), **f64),
                                path_seg=torch.empty((B, int(path_cap)), **i32), path_len=torch.empty(B, **i32), route=route)
            if B == 0:
                return res
            wb = self.lib.trrt_mission_workspace_bytes(B, K)
            work = self._scratch("mission", wb)
            ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
            n_active_h = np.ascontiguousarray(n_active, dtype=np.int32)
            a = _lib.CMissionArgs(d_bits=g.bits.data_ptr(), n_maps=g.n_maps, H=g.H, W=g.W, d_map_id=ptr(mid),
                                  params=P.to_c(), xystdv=float(P.xystdv), anglestdv=float(P.anglestdv), n_missions=B, K=K,
                                  d_waypoints=wp.data_ptr(), wp_cap=int(wp.shape[1]), d_n_waypoints=n_wp.data_ptr(),
                                  d_route_status=ptr(route_status), d_normals=nz.data_ptr(), d_normal_range=rng_d.data_ptr(),
                                  d_order=order_d.data_ptr(), n_stages=S, n_active=n_active_h.ctypes.data if S else None,
                                  seg_cap=Sc, d_seg_begin=res.begin.data_ptr(), d_seg_end=res.end.data_ptr(),
                                  d_seg_solution=res.solution.data_ptr(), d_seg_nearest=res.nearest.data_ptr(),
                                  d_seg_mindist=res.mindist.data_ptr(), d_seg_n_nodes=res.n_nodes.data_ptr(),
                                  d_seg_n_edges=res.n_edges.data_ptr(), d_seg_iters=res.iters.data_ptr(),
                                  d_seg_status=res.seg_status.data_ptr(), d_status=res.status.data_ptr(),
                                  d_stop_seg=res.stop_seg.data_ptr(), d_n_seg=res.n_seg.data_ptr(),
                                  d_path=res.path.data_ptr(), d_path_seg=res.path_seg.data_ptr(), path_cap=int(path_cap),
                                  d_path_len=res.path_len.data_ptr(), d_work=work.data_ptr(), work_bytes=work.numel())
            _lib.check(self.lib.trrt_mission_batch(C.byref(a), self._stream()), "trrt_mission_batch")
            res._keep = (nz, rng_d, order_d, mid)
            res.schedule = (order, n_active)
        return res
