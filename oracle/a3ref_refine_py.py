"""ctypes view of oracle/liba3ref_refine.so (corner refinement, kernel K5) — TEST INFRASTRUCTURE ONLY (see a3ref_refine.h)."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from .a3ref_py import Intrinsics, Pose

HERE = Path(__file__).resolve().parent
_lib = None


def build() -> Path:
    subprocess.run(["make", "-s", "-C", str(HERE), "-f", "refine.mk"], check=True)
    return HERE / "liba3ref_refine.so"


def lib():
    global _lib
    if _lib is None:
        so = HERE / "liba3ref_refine.so"
        if not so.exists():
            build()
        L = C.CDLL(str(so))
        fp, u32p, PP = C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(Pose)
        L.a3ref_refine_corners.restype = C.c_int
        L.a3ref_refine_corners.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, u32p, fp]
        L.a3ref_solve_with_undistorted_points_f32.argtypes = [fp, C.c_float, C.c_uint32, C.c_uint32, PP, PP]
        L.a3ref_solve_with_intrinsics_f32.argtypes = [fp, C.c_float, C.POINTER(Intrinsics), PP, PP]
        _lib = L
    return _lib


def refine_corners(grey: np.ndarray, corners):
    """grey uint8 [H, W]; corners: 4 (x, y) integer corners (or 8 values) -> (refined float32 [4, 2], ok)."""
    g = np.ascontiguousarray(grey, np.uint8)
    c = np.ascontiguousarray(np.asarray(corners).reshape(8), np.uint32)
    out = np.zeros(8, np.float32)
    ok = lib().a3ref_refine_corners(g.ctypes.data, g.shape[1], g.shape[0], c.ctypes.data_as(C.POINTER(C.c_uint32)),
                                    out.ctypes.data_as(C.POINTER(C.c_float)))
    return out.reshape(4, 2), bool(ok)


def _fc(corners):
    c = np.ascontiguousarray(np.asarray(corners, np.float32).reshape(8))
    return c, c.ctypes.data_as(C.POINTER(C.c_float))


def solve_with_undistorted_points_f32(corners, size: float, image_size):
    c, pc = _fc(corners)
    a, b = Pose(), Pose()
    lib().a3ref_solve_with_undistorted_points_f32(pc, size, image_size[0], image_size[1], C.byref(a), C.byref(b))
    return a, b


def solve_with_intrinsics_f32(corners, size: float, k: Intrinsics):
    c, pc = _fc(corners)
    a, b = Pose(), Pose()
    lib().a3ref_solve_with_intrinsics_f32(pc, size, C.byref(k), C.byref(a), C.byref(b))
    return a, b
