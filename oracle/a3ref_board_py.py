"""ctypes view of oracle/liba3ref_board.so (board pose, kernel K6) — TEST INFRASTRUCTURE ONLY (see a3ref_board.h)."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from .a3ref_py import Intrinsics, Pose

HERE = Path(__file__).resolve().parent
_lib = None

UNDISTORTED, INTRINSICS = 1, 2


def build() -> Path:
    subprocess.run(["make", "-s", "-C", str(HERE), "-f", "board.mk"], check=True)
    return HERE / "liba3ref_board.so"


def lib():
    global _lib
    if _lib is None:
        so = HERE / "liba3ref_board.so"
        if not so.exists():
            build()
        L = C.CDLL(str(so))
        vp, u32, PP = C.c_void_p, C.c_uint32, C.POINTER(Pose)
        L.a3ref_board_solve.restype = C.c_int
        L.a3ref_board_solve.argtypes = [vp, vp, u32, PP, PP]
        L.a3ref_board_frame.restype = C.c_int
        L.a3ref_board_frame.argtypes = [vp, vp, u32, u32, u32, u32, C.POINTER(Intrinsics), vp, vp, u32, PP, PP, C.POINTER(u32)]
        _lib = L
    return _lib


def solve(uv, xy):
    """Normalised image points uv [n, 2] and board points xy [n, 2] (f32) -> (best Pose, alt Pose, ok)."""
    u = np.ascontiguousarray(np.asarray(uv, np.float32).reshape(-1, 2))
    x = np.ascontiguousarray(np.asarray(xy, np.float32).reshape(-1, 2))
    a, b = Pose(), Pose()
    ok = lib().a3ref_board_solve(u.ctypes.data, x.ctypes.data, u.shape[0], C.byref(a), C.byref(b))
    return a, b, bool(ok)


def solve_frame(board_ids, board_corners, ids, corners, image_size=None, k: Intrinsics | None = None):
    """One frame's markers (ids [n], f32 corners [n, 4, 2] in a3_marker.corners order) against a board (ids [m], corners
    [m, 4, 2]); `k` = intrinsics mode, else undistorted at image_size (w, h) -> (best, alt, n_markers, ok)."""
    bi = np.ascontiguousarray(board_ids, np.uint64)
    bc = np.ascontiguousarray(np.asarray(board_corners, np.float32).reshape(-1, 8))
    mi = np.ascontiguousarray(ids, np.uint64).reshape(-1)
    mc = np.ascontiguousarray(np.asarray(corners, np.float32).reshape(-1, 8))
    a, b, nm = Pose(), Pose(), C.c_uint32()
    w, h = image_size if image_size is not None else (0, 0)
    ok = lib().a3ref_board_frame(bi.ctypes.data, bc.ctypes.data, bi.size, INTRINSICS if k is not None else UNDISTORTED, w, h,
                                 C.byref(k) if k is not None else None, mi.ctypes.data, mc.ctypes.data, mi.size, C.byref(a),
                                 C.byref(b), C.byref(nm))
    return a, b, int(nm.value), bool(ok)
