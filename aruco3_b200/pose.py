"""Host-side mirror of the reference's `pose` module and `CameraIntrinsics` over the C ABI.

  `MarkerPose`                      /root/reference/src/pose.rs:8-50
  `solve_with_intrinsics`           /root/reference/src/pose.rs:52-55
  `solve_with_undistorted_points`   /root/reference/src/pose.rs:59-62
  `solve_with_normalized_points`    /root/reference/src/pose.rs:64-81
  `CameraIntrinsics`                /root/reference/src/pinhole.rs:11-94
  `CameraDistortion`                not in the reference: OpenCV's five lens coefficients (kernel K7)

The solvers run on the device (kernel K4, csrc/k4_pose.cu) and therefore need a `Detector` handle; each accepts one
marker (4 corners, returns `(best, alt)` like the reference) or a batch [n,4,2] (returns two lists).  With
`Detector.set_pose(...)` the same kernel runs inside `detect_batch` right behind the decode kernel.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _ffi
from ._ffi import A3CameraDistortion, A3CameraIntrinsics, A3Pose, check, lib


@dataclass
class MarkerPose:
    """src/pose.rs:8-12; default src/pose.rs:42-50."""
    error: float = float(np.float32(1e31))
    rotation: np.ndarray = field(default_factory=lambda: np.eye(3, dtype=np.float32))
    translation: np.ndarray = field(default_factory=lambda: np.zeros(3, np.float32))

    @staticmethod
    def from_c(p: A3Pose) -> "MarkerPose":
        return MarkerPose(float(p.error), np.array(p.rotation, np.float32).reshape(3, 3), np.array(p.translation, np.float32))

    def to_c(self) -> A3Pose:
        p = A3Pose()
        p.error = self.error
        p.rotation[:] = np.asarray(self.rotation, np.float32).ravel().tolist()
        p.translation[:] = np.asarray(self.translation, np.float32).ravel().tolist()
        return p

    def _apply(self, points, inverse: bool):
        pts = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
        out = np.empty_like(pts)
        c = self.to_c()
        lib().a3_pose_apply_transform(C.byref(c), pts.ctypes.data, pts.shape[0], int(inverse), out.ctypes.data)
        return [tuple(float(v) for v in row) for row in out]

    def apply_transform_to_points(self, points):
        """src/pose.rs:17-20"""
        return self._apply(points, False)

    apply_transform_to_vectors = apply_transform_to_points  # src/pose.rs:24-28

    def apply_inverse_transform_to_points(self, points):
        """src/pose.rs:30-33"""
        return self._apply(points, True)

    apply_inverse_transform_to_vectors = apply_inverse_transform_to_points  # src/pose.rs:35-39


class CameraIntrinsics:
    """src/pinhole.rs:11-18."""

    def __init__(self, image_width: int, image_height: int, focal_x: float, focal_y: float, principal_x: float | None = None,
                 principal_y: float | None = None):
        """`CameraIntrinsics::new` (src/pinhole.rs:26-35): a missing principal point is the image centre."""
        self._c = A3CameraIntrinsics()
        px = C.byref(C.c_float(principal_x)) if principal_x is not None else None
        py = C.byref(C.c_float(principal_y)) if principal_y is not None else None
        lib().a3_camera_intrinsics_new(image_width, image_height, focal_x, focal_y,
                                       C.cast(px, C.POINTER(C.c_float)) if px else None,
                                       C.cast(py, C.POINTER(C.c_float)) if py else None, C.byref(self._c))

    @staticmethod
    def new_from_fov_horizontal(horizontal_fov_radians: float, sensor_width_mm: float, resolution_x: int,
                                resolution_y: int) -> "CameraIntrinsics":
        """src/pinhole.rs:37-60"""
        k = CameraIntrinsics.__new__(CameraIntrinsics)
        k._c = A3CameraIntrinsics()
        lib().a3_camera_intrinsics_from_fov_horizontal(horizontal_fov_radians, sensor_width_mm, resolution_x, resolution_y,
                                                       C.byref(k._c))
        return k

    image_width = property(lambda s: int(s._c.image_width))
    image_height = property(lambda s: int(s._c.image_height))
    focal_x = property(lambda s: float(s._c.focal_x))
    focal_y = property(lambda s: float(s._c.focal_y))
    principal_x = property(lambda s: float(s._c.principal_x))
    principal_y = property(lambda s: float(s._c.principal_y))

    def project(self, x: float, y: float, z: float):
        """src/pinhole.rs:65-71"""
        out = (C.c_float * 3)()
        lib().a3_camera_project(C.byref(self._c), x, y, z, out)
        return tuple(out)

    def project_culled(self, x: float, y: float, z: float):
        """src/pinhole.rs:76-84 -> (u, v) or None when z <= 0"""
        out = (C.c_float * 2)()
        return tuple(out) if lib().a3_camera_project_culled(C.byref(self._c), x, y, z, out) else None

    def unproject(self, x: float, y: float):
        """src/pinhole.rs:88-93"""
        out = (C.c_float * 2)()
        lib().a3_camera_unproject(C.byref(self._c), x, y, out)
        return tuple(out)

    def to_matrix3(self) -> np.ndarray:
        """`From<CameraIntrinsics> for Matrix3<f32>` (src/pinhole.rs:97-105)"""
        return np.array([[self.focal_x, 0, self.principal_x], [0, self.focal_y, self.principal_y], [0, 0, 1]], np.float32)

    def to_matrix3x4(self) -> np.ndarray:
        """`From<CameraIntrinsics> for Matrix3x4<f32>` (src/pinhole.rs:107-115)"""
        return np.concatenate([self.to_matrix3(), np.zeros((3, 1), np.float32)], axis=1)


class CameraDistortion:
    """A lens distortion: OpenCV's five-coefficient Brown-Conrady model in OpenCV's order (the `distCoeffs` of
    `calibrateCamera`), on the normalised coordinates of `CameraIntrinsics`.  Give it to `Detector(distortion=...)` /
    `Detector.set_distortion` and the marker and board poses in intrinsics mode solve from undistorted corners."""

    def __init__(self, k1: float = 0.0, k2: float = 0.0, p1: float = 0.0, p2: float = 0.0, k3: float = 0.0):
        self._c = A3CameraDistortion(k1, k2, p1, p2, k3)

    k1 = property(lambda s: float(s._c.k1))
    k2 = property(lambda s: float(s._c.k2))
    p1 = property(lambda s: float(s._c.p1))
    p2 = property(lambda s: float(s._c.p2))
    k3 = property(lambda s: float(s._c.k3))

    def coefficients(self) -> np.ndarray:
        """(k1, k2, p1, p2, k3) as f32, OpenCV's distCoeffs"""
        return np.array([self._c.k1, self._c.k2, self._c.p1, self._c.p2, self._c.k3], np.float32)

    def __repr__(self):
        return "CameraDistortion(k1={}, k2={}, p1={}, p2={}, k3={})".format(*self.coefficients().tolist())


def _solve(detector, mode, pts, dtype, marker_size_mm, extra):
    a = np.ascontiguousarray(pts, dtype)
    single = a.ndim == 2
    a = a.reshape(-1, 8)
    n = a.shape[0]
    best, alt = (A3Pose * max(n, 1))(), (A3Pose * max(n, 1))()
    L, h = lib(), detector._h
    if mode == _ffi.POSE_INTRINSICS:
        check(L.a3_solve_with_intrinsics(h, a.ctypes.data, n, marker_size_mm, C.byref(extra._c), best, alt))
    elif mode == _ffi.POSE_UNDISTORTED:
        check(L.a3_solve_with_undistorted_points(h, a.ctypes.data, n, marker_size_mm, extra[0], extra[1], best, alt))
    else:
        check(L.a3_solve_with_normalized_points(h, a.ctypes.data, n, marker_size_mm, best, alt))
    b = [MarkerPose.from_c(best[i]) for i in range(n)]
    c = [MarkerPose.from_c(alt[i]) for i in range(n)]
    return (b[0], c[0]) if single else (b, c)


def solve_with_intrinsics(detector, image_points, marker_size_mm: float, camera_intrinsics: CameraIntrinsics):
    """src/pose.rs:52-55; image_points: [(x, y)] * 4 (u32, `Marker.corners`) or [n,4,2]."""
    return _solve(detector, _ffi.POSE_INTRINSICS, image_points, np.uint32, marker_size_mm, camera_intrinsics)


def solve_with_undistorted_points(detector, image_points, marker_size_mm: float, image_size):
    """src/pose.rs:59-62; image_size = (width, height)."""
    return _solve(detector, _ffi.POSE_UNDISTORTED, image_points, np.uint32, marker_size_mm, image_size)


def solve_with_normalized_points(detector, normalized_image_points, marker_size_mm: float):
    """src/pose.rs:64-81; points are f32."""
    return _solve(detector, _ffi.POSE_NORMALIZED, normalized_image_points, np.float32, marker_size_mm, None)
