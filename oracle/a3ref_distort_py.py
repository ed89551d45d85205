"""ctypes view of oracle/liba3ref_distort.so (corner undistortion, kernel K7, and the board pose on undistorted corners)
— TEST INFRASTRUCTURE ONLY (see a3ref_distort.h)."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

from .a3ref_py import Intrinsics, Pose

HERE = Path(__file__).resolve().parent
_lib = None


class Distortion(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("k1", "k2", "p1", "p2", "k3")]


def build() -> Path:
    subprocess.run(["make", "-s", "-C", str(HERE), "-f", "distort.mk"], check=True)
    return HERE / "liba3ref_distort.so"


def lib():
    global _lib
    if _lib is None:
        so = HERE / "liba3ref_distort.so"
        if not so.exists():
            build()
        L = C.CDLL(str(so))
        vp, u32, PP, PK, PD = C.c_void_p, C.c_uint32, C.POINTER(Pose), C.POINTER(Intrinsics), C.POINTER(Distortion)
        L.a3ref_undistort_points.restype = None
        L.a3ref_undistort_points.argtypes = [PK, PD, vp, u32, vp, vp]
        L.a3ref_board_frame_distorted.restype = C.c_int
        L.a3ref_board_frame_distorted.argtypes = [vp, vp, u32, PK, PD, vp, vp, u32, PP, PP, C.POINTER(u32)]
        _lib = L
    return _lib


def distortion(k1=0.0, k2=0.0, p1=0.0, p2=0.0, k3=0.0) -> Distortion:
    return Distortion(k1, k2, p1, p2, k3)


def undistort_points(points, k: Intrinsics, d: Distortion):
    """Pixels [n, 2] (pixel-centre convention) -> (normalised undistorted f32 [n, 2], ok bool [n]); a failed point reads (0, 0)."""
    p = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 2))
    out = np.zeros_like(p)
    ok = np.zeros(p.shape[0], np.uint8)
    lib().a3ref_undistort_points(C.byref(k), C.byref(d), p.ctypes.data, p.shape[0], out.ctypes.data, ok.ctypes.data)
    return out, ok.astype(bool)


def solve_frame(board_ids, board_corners, ids, corners, k: Intrinsics, d: Distortion):
    """One frame's markers (ids [n], f32 corners [n, 4, 2] in a3_marker.corners order, pixels) against a board, in
    intrinsics mode with distortion d -> (best, alt, n_markers, ok), as a3ref_board_py.solve_frame."""
    bi = np.ascontiguousarray(board_ids, np.uint64)
    bc = np.ascontiguousarray(np.asarray(board_corners, np.float32).reshape(-1, 8))
    mi = np.ascontiguousarray(ids, np.uint64).reshape(-1)
    mc = np.ascontiguousarray(np.asarray(corners, np.float32).reshape(-1, 8))
    a, b, nm = Pose(), Pose(), C.c_uint32()
    ok = lib().a3ref_board_frame_distorted(bi.ctypes.data, bc.ctypes.data, bi.size, C.byref(k), C.byref(d), mi.ctypes.data, mc.ctypes.data,
                                           mi.size, C.byref(a), C.byref(b), C.byref(nm))
    return a, b, int(nm.value), bool(ok)
