"""ctypes binding of libthetarrt.so (include/thetarrt.h).

There is no CPU fallback: if the library is missing, was not built, or no CUDA
device is present, the calls raise.  The oracle under /oracle is never imported
from here.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libthetarrt.so")

c_i32p = C.POINTER(C.c_int32)
c_u32p = C.POINTER(C.c_uint32)
c_u64p = C.POINTER(C.c_uint64)
c_u8p = C.POINTER(C.c_uint8)
c_dp = C.POINTER(C.c_double)


class TrrtError(RuntimeError):
    pass


class CParams(C.Structure):
    """struct trrt_params (main.py:15-32)."""
    _fields_ = [("thetastar", C.c_int32), ("forwardonly", C.c_int32), ("bikelength", C.c_double),
                ("leftconstraint", C.c_double), ("rightconstraint", C.c_double), ("frontclearance", C.c_double),
                ("maxdrivedist", C.c_double), ("tol_xy", C.c_double), ("tol_ang", C.c_double), ("weightxy", C.c_double)]


class CRrtArgs(C.Structure):
    """struct trrt_rrt_args."""
    _fields_ = [
        ("d_bits", C.c_void_p), ("n_maps", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("d_map_id", C.c_void_p),
        ("params", CParams),
        ("n_queries", C.c_int64), ("K", C.c_int32), ("lanes_per_query", C.c_int32),
        ("schedule", C.c_int32), ("sample_xy_i16", C.c_int32),
        ("d_start", C.c_void_p), ("d_goal", C.c_void_p), ("d_sample_xy", C.c_void_p), ("d_sample_th", C.c_void_p),
        ("d_node_x", C.c_void_p), ("d_node_y", C.c_void_p), ("d_node_th", C.c_void_p), ("d_parent", C.c_void_p),
        ("d_u", C.c_void_p), ("d_n_nodes", C.c_void_p), ("d_sol", C.c_void_p), ("d_status", C.c_void_p),
        ("d_iters", C.c_void_p),
        ("d_it_near", C.c_void_p), ("d_it_new", C.c_void_p), ("d_it_code", C.c_void_p), ("d_los_log", C.c_void_p),
        ("d_n_los", C.c_void_p), ("d_counters", C.c_void_p),
        ("d_work", C.c_void_p), ("work_bytes", C.c_size_t),
        ("d_pack_rows", C.c_void_p), ("d_row_start", C.c_void_p), ("d_pack_x", C.c_void_p), ("d_pack_y", C.c_void_p),
        ("d_pack_th", C.c_void_p), ("d_pack_parent", C.c_void_p), ("d_pack_u", C.c_void_p),
        ("d_stop_at", C.c_void_p), ("resume", C.c_int32),
    ]


class CRrtRace(C.Structure):
    """struct trrt_rrt_race."""
    _fields_ = [("d_group", C.c_void_p), ("n_groups", C.c_int64), ("d_key", C.c_void_p)]


class CThetaArgs(C.Structure):
    """struct trrt_theta_args."""
    _fields_ = [
        ("d_bits", C.c_void_p), ("n_maps", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("d_map_id", C.c_void_p),
        ("thetastar", C.c_int32), ("lanes_per_query", C.c_int32), ("n_queries", C.c_int64),
        ("d_start_goal", C.c_void_p),
        ("d_path", C.c_void_p), ("path_cap", C.c_int32), ("d_path_len", C.c_void_p), ("d_cost", C.c_void_p),
        ("d_expanded", C.c_void_p), ("d_status", C.c_void_p),
        ("d_los_log", C.c_void_p), ("los_cap", C.c_int32), ("d_n_los", C.c_void_p), ("d_pushes", C.c_void_p),
        ("n_slots", C.c_int32), ("heap_cap", C.c_int32), ("d_work", C.c_void_p), ("work_bytes", C.c_size_t),
        ("d_order", C.c_void_p),
    ]


class CMissionArgs(C.Structure):
    """struct trrt_mission_args."""
    _fields_ = [
        ("d_bits", C.c_void_p), ("n_maps", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("d_map_id", C.c_void_p),
        ("params", CParams), ("xystdv", C.c_double), ("anglestdv", C.c_double),
        ("n_missions", C.c_int64), ("K", C.c_int32),
        ("d_waypoints", C.c_void_p), ("wp_cap", C.c_int32), ("d_n_waypoints", C.c_void_p), ("d_route_status", C.c_void_p),
        ("d_normals", C.c_void_p), ("d_normal_range", C.c_void_p),
        ("d_order", C.c_void_p), ("n_stages", C.c_int32), ("n_active", C.c_void_p),
        ("seg_cap", C.c_int32), ("d_seg_begin", C.c_void_p), ("d_seg_end", C.c_void_p), ("d_seg_solution", C.c_void_p),
        ("d_seg_nearest", C.c_void_p), ("d_seg_mindist", C.c_void_p), ("d_seg_n_nodes", C.c_void_p),
        ("d_seg_n_edges", C.c_void_p), ("d_seg_iters", C.c_void_p), ("d_seg_status", C.c_void_p),
        ("d_status", C.c_void_p), ("d_stop_seg", C.c_void_p), ("d_n_seg", C.c_void_p),
        ("d_path", C.c_void_p), ("d_path_seg", C.c_void_p), ("path_cap", C.c_int32), ("d_path_len", C.c_void_p),
        ("d_work", C.c_void_p), ("work_bytes", C.c_size_t),
    ]


class CLegacyNormalsArgs(C.Structure):
    """struct trrt_legacy_normals_args."""
    _fields_ = [
        ("n_seeds", C.c_int64), ("d_seeds", C.c_void_p), ("d_range", C.c_void_p), ("d_out", C.c_void_p),
        ("d_fix_pos", C.c_void_p), ("d_fix_r2", C.c_void_p), ("fix_cap", C.c_int64), ("d_fix_count", C.c_void_p),
        ("d_work", C.c_void_p), ("work_bytes", C.c_size_t),
    ]


class CValidateTreeArgs(C.Structure):
    """struct trrt_validate_tree_args."""
    _fields_ = [
        ("d_bits", C.c_void_p), ("n_maps", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("d_map_id", C.c_void_p),
        ("n_queries", C.c_int64), ("K", C.c_int32), ("lanes", C.c_int32),
        ("d_node_x", C.c_void_p), ("d_node_y", C.c_void_p), ("d_parent", C.c_void_p), ("d_u", C.c_void_p),
        ("d_n_nodes", C.c_void_p), ("d_sol", C.c_void_p),
        ("d_edge_ok", C.c_void_p), ("d_node_ok", C.c_void_p), ("d_sol_ok", C.c_void_p),
        ("d_work", C.c_void_p), ("work_bytes", C.c_size_t),
    ]


class CRepairTreeArgs(C.Structure):
    """struct trrt_repair_tree_args."""
    _fields_ = [
        ("n_queries", C.c_int64), ("K", C.c_int32),
        ("d_node_x", C.c_void_p), ("d_node_y", C.c_void_p), ("d_node_th", C.c_void_p), ("d_parent", C.c_void_p),
        ("d_u", C.c_void_p), ("d_n_nodes", C.c_void_p), ("d_sol", C.c_void_p), ("d_status", C.c_void_p),
        ("d_iters", C.c_void_p), ("d_edge_ok", C.c_void_p), ("d_new_index", C.c_void_p), ("d_n_pruned", C.c_void_p),
        ("d_race_group", C.c_void_p), ("n_race_groups", C.c_int64), ("d_race_key", C.c_void_p),
        ("d_work", C.c_void_p), ("work_bytes", C.c_size_t),
    ]


class CValidatePathArgs(C.Structure):
    """struct trrt_validate_path_args."""
    _fields_ = [
        ("d_bits", C.c_void_p), ("n_maps", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("d_map_id", C.c_void_p),
        ("mode", C.c_int32), ("lanes", C.c_int32), ("n_paths", C.c_int64), ("path_cap", C.c_int32),
        ("d_route", C.c_void_p), ("d_rows", C.c_void_p), ("d_row_seg", C.c_void_p),
        ("d_path_len", C.c_void_p), ("d_status", C.c_void_p), ("d_step_ok", C.c_void_p), ("d_ok", C.c_void_p),
    ]


# every symbol include/thetarrt.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "trrt_version": (C.c_int, []),
    "trrt_error_string": (C.c_char_p, [C.c_int]),
    "trrt_last_cuda_error": (C.c_char_p, []),
    "trrt_default_params": (None, [C.POINTER(CParams)]),
    "trrt_grid_words": (C.c_size_t, [C.c_int, C.c_int]),
    "trrt_pack_grid": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "trrt_los_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                 C.c_void_p, C.c_void_p]),
    "trrt_tile_words": (C.c_size_t, [C.c_int, C.c_int]),
    "trrt_tile_grid": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "trrt_los_batch_tiled": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p]),
    "trrt_grid_edit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                 C.c_void_p]),
    "trrt_validate_tree_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "trrt_validate_tree": (C.c_int, [C.POINTER(CValidateTreeArgs), C.c_void_p]),
    "trrt_validate_path": (C.c_int, [C.POINTER(CValidatePathArgs), C.c_void_p]),
    "trrt_repair_tree_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "trrt_repair_tree": (C.c_int, [C.POINTER(CRepairTreeArgs), C.c_void_p]),
    "trrt_nearest_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "trrt_nearest_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "trrt_rrt_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "trrt_rrt_batch": (C.c_int, [C.POINTER(CRrtArgs), C.c_void_p]),
    "trrt_rrt_race_batch": (C.c_int, [C.POINTER(CRrtArgs), C.POINTER(CRrtRace), C.c_void_p]),
    "trrt_steer_batch": (C.c_int, [C.POINTER(CParams), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "trrt_drive_batch": (C.c_int, [C.POINTER(CParams), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "trrt_arc_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p,
                                 C.c_void_p, C.c_int, C.c_void_p]),
    "trrt_arc_pixels_batch": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "trrt_clearance_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(CParams), C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "trrt_anglediff_batch": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "trrt_findnearest_batch": (C.c_int, [C.POINTER(CParams), C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "trrt_theta_workspace_bytes": (C.c_size_t, [C.POINTER(CThetaArgs)]),
    "trrt_theta_batch": (C.c_int, [C.POINTER(CThetaArgs), C.c_void_p]),
    "trrt_mission_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "trrt_mission_batch": (C.c_int, [C.POINTER(CMissionArgs), C.c_void_p]),
    "trrt_legacy_normals_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "trrt_legacy_normals_draw": (C.c_int, [C.POINTER(CLegacyNormalsArgs), C.c_void_p]),
    "trrt_libm_log_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "trrt_legacy_normals_fixup": (C.c_int, [C.POINTER(CLegacyNormalsArgs), C.c_void_p, C.c_int64, C.c_void_p]),
    "trrt_rand_conf_batch": (C.c_int, [C.c_int, C.c_int, C.c_double, C.c_double, C.c_int64, C.c_int32, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
}

_lib = None


def load():
    """Load libthetarrt.so; raises TrrtError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise TrrtError(f"{SO_PATH} not found: build it with `python -m theta_rrt_b200.build` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = ABI mismatch, let it surface
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(err: int, what: str = ""):
    if err != 0:
        lib = load()
        msg = lib.trrt_error_string(err).decode()
        cuda = lib.trrt_last_cuda_error().decode()
        raise TrrtError(f"{what or 'libthetarrt'}: {msg}" + (f" [{cuda}]" if cuda and err in (5, 6) else ""))
