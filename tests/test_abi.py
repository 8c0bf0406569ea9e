"""The C-ABI library loads and exports every symbol include/thetarrt.h declares (no compute calls)."""
import ctypes as C
import os
import re

from tests import util
from theta_rrt_b200 import _lib


def header_symbols():
    src = open(os.path.join(util.ROOT, "include", "thetarrt.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(trrt_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_expected_entry_points():
    syms = header_symbols()
    for s in ("trrt_los_batch", "trrt_nearest_batch", "trrt_rrt_batch", "trrt_theta_batch", "trrt_pack_grid",
              "trrt_steer_batch", "trrt_drive_batch", "trrt_arc_batch", "trrt_findnearest_batch"):
        assert s in syms


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.SO_PATH), "libthetarrt.so missing: run __graft_entry__.build()"
    lib = C.CDLL(_lib.SO_PATH)
    for s in header_symbols():
        assert hasattr(lib, s), s
    assert set(_lib.SIGNATURES) == set(header_symbols())


def test_trivial_host_calls():
    lib = _lib.load()
    assert lib.trrt_version() == 200
    assert lib.trrt_grid_words(100, 100) == 400 and lib.trrt_grid_words(300, 300) == 3000
    assert lib.trrt_error_string(2).decode().startswith("map must be square")
    p = _lib.CParams()
    lib.trrt_default_params(C.byref(p))
    assert (p.thetastar, p.forwardonly, p.bikelength, p.leftconstraint, p.rightconstraint) == (1, 1, 5, -65, 65)
    assert (p.frontclearance, p.maxdrivedist, p.tol_xy, p.tol_ang, p.weightxy) == (2, 30, 10, 45, .6)
    assert lib.trrt_rrt_workspace_bytes(4096, 5001) == 4096 * 16384 * 4 + 256  # work counter + one index table per query


def test_struct_layouts_match_header():
    # every ctypes mirror has the header's members in the header's order
    for name, mirror in (("trrt_params", _lib.CParams), ("trrt_rrt_args", _lib.CRrtArgs), ("trrt_rrt_race", _lib.CRrtRace),
                         ("trrt_theta_args", _lib.CThetaArgs), ("trrt_mission_args", _lib.CMissionArgs),
                         ("trrt_legacy_normals_args", _lib.CLegacyNormalsArgs)):
        assert [f[0] for f in mirror._fields_] == util.struct_members(name), name
    # members added after d_pack_u keep the offsets of the earlier ones
    assert _lib.CRrtArgs._fields_[-2:] == [("d_stop_at", C.c_void_p), ("resume", C.c_int32)]
    assert "trrt_rrt_race_batch" in _lib.SIGNATURES
    # sizes the CUDA side was compiled with (offsets are exercised by the GPU tests)
    assert C.sizeof(_lib.CParams) == 8 + 8 * 8
    assert C.sizeof(_lib.CRrtArgs) % 8 == 0 and C.sizeof(_lib.CThetaArgs) % 8 == 0
    assert C.sizeof(_lib.CRrtRace) == 24
