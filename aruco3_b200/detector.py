"""Host-side mirror of the reference's detection API over the C ABI (include/aruco3_b200.h).

Names and argument meaning follow the reference so tests read like its own:
  `DetectorConfig`  /root/reference/src/aruco.rs:23-43      `Detector`   /root/reference/src/aruco.rs:46-52
  `Detection`       /root/reference/src/aruco.rs:16-21      `Marker`     /root/reference/src/aruco.rs:8-13
  `ARDictionary`    /root/reference/src/dictionaries.rs:22-28, 115-232

This module only marshals numpy buffers through ctypes; every stage runs in libaruco3_b200.so (CUDA kernels
for the pixel and decode stages, C++ for the contour / quad stage).  There is no Python or CPU fallback:
without the library or without a CUDA device `Detector(...)` raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _ffi
from ._ffi import A3Config, A3Decode, A3Dictionary, A3Error, A3Marker, A3Outputs, A3Pose, A3Stats, check, lib


@dataclass
class DetectorConfig:
    """src/aruco.rs:23-30; defaults src/aruco.rs:32-43."""
    threshold_window: int = 7
    contour_simplification_epsilon: float = 0.05
    min_side_length_factor: float = 0.2
    min_corner_separation_factor: float = 0.1
    homography_sample_size: int = 49
    filter_high_bit_errors: bool = True

    def to_c(self) -> A3Config:
        return A3Config(self.threshold_window, self.contour_simplification_epsilon, self.min_side_length_factor,
                        self.min_corner_separation_factor, self.homography_sample_size,
                        1 if self.filter_high_bit_errors else 0)


class ARDictionary:
    """src/dictionaries.rs:22-28. `code_list` is a read-only uint64 view of the table inside the library."""

    def __init__(self, c: A3Dictionary, name: str = ""):
        self._c = c
        self.name = name
        self.num_bits = int(c.num_bits)
        self.tau = int(c.tau)
        self.code_list = np.ctypeslib.as_array(c.codes, (c.n_codes,)) if c.n_codes else np.zeros(0, np.uint64)

    @staticmethod
    def new_from_named_dict(name: str) -> "ARDictionary":
        """src/dictionaries.rs:140-145 — case-insensitive; the reference panics on an unknown name, we raise."""
        c = A3Dictionary()
        check(lib().a3_dictionary_by_name(name.encode(), C.byref(c)))
        return ARDictionary(c, name.upper())

    @staticmethod
    def get_dictionary_names() -> list:
        """src/dictionaries.rs:147-149"""
        L = lib()
        return [L.a3_dictionary_name(i).decode() for i in range(L.a3_dictionary_count())]

    def get_mark_size(self) -> int:
        """src/dictionaries.rs:154-156"""
        return int(lib().a3_dictionary_mark_size(C.byref(self._c)))

    def find_nearest(self, bits: int):
        """src/dictionaries.rs:160-196 -> (index, distance)"""
        idx, dist = C.c_uint64(), C.c_uint8()
        lib().a3_find_nearest(C.byref(self._c), bits, C.byref(idx), C.byref(dist))
        return idx.value, dist.value

    def try_find_nearest(self, bits: int):
        """src/dictionaries.rs:200-207 -> (index, distance) or None"""
        idx, dist = C.c_uint64(), C.c_uint8()
        ok = lib().a3_try_find_nearest(C.byref(self._c), bits, C.byref(idx), C.byref(dist))
        return (idx.value, dist.value) if ok else None

    def make_binary_image(self, marker_id: int):
        """src/dictionaries.rs:212-232 -> (width, bool list), the reference's order"""
        buf = np.zeros(256, np.uint8)
        n = C.c_uint32()
        w = lib().a3_make_binary_image(C.byref(self._c), marker_id, buf.ctypes.data, buf.size, C.byref(n))
        return int(w), [bool(v) for v in buf[:n.value]]


def hamming_distance(a: int, b: int) -> int:
    """src/lib.rs:11-21"""
    return int(lib().a3_hamming_distance(a, b))


@dataclass
class Marker:
    """src/aruco.rs:8-13 (+ the winning rotation, which the reference folds into `corners`)."""
    id: int
    code: int
    corners: list            # [(x, y)] * 4, already rotate_left(rotation)
    hamming_distance: int
    rotation: int = 0
    candidate: int = 0
    poses: tuple | None = None   # (best, alt) MarkerPose when the detector has a pose mode (Detector.set_pose)
    # corners="refined": [(x, y)] * 4 f32 sub-pixel corners in the order of `corners` (pixel-centre convention: grey pixel
    # (x, y) is the point (x, y)); `refined` is False where the refinement fell back to the integer corners
    corners_refined: list | None = None
    refined: bool = False


@dataclass
class Detection:
    """src/aruco.rs:16-21"""
    grey: np.ndarray | None = None          # uint8 [H, W]
    candidates: list = field(default_factory=list)    # [[(x, y)] * 4]
    homographies: list = field(default_factory=list)  # uint8 [hs, hs] per candidate ([1, 1] zeros when the projection failed)
    markers: list = field(default_factory=list)
    # extras for stage-by-stage parity checks (not in the reference struct)
    mask: np.ndarray | None = None
    decodes: list = field(default_factory=list)
    board_pose: object | None = None  # BoardPose of the detector's board (Detector.set_board), else None


_FMT = {("rgb", 3): _ffi.FMT_RGB8, ("rgb", 4): _ffi.FMT_RGBA8, ("bgr", 3): _ffi.FMT_BGR8, ("bgr", 4): _ffi.FMT_BGRA8}


def _frames_view(frames: np.ndarray, order: str = "rgb"):
    """-> (contiguous uint8 array, format, n, h, w, pitch, frame_stride) for [n,H,W,3|4] or [n,H,W]; `order` "bgr" =
    camera byte order B,G,R[,A] (A3_FMT_BGR8 / A3_FMT_BGRA8)."""
    a = np.asarray(frames)
    if a.dtype == np.uint16 and order == "rgb" and (a.ndim == 3 or (a.ndim == 4 and a.shape[3] in (2, 3, 4))):
        # Luma16 [n,H,W], LumaA16 [n,H,W,2], Rgb16 [n,H,W,3], Rgba16 [n,H,W,4]: native-endian u16 subpixels
        fmt = _ffi.FMT_LUMA16 if a.ndim == 3 else {2: _ffi.FMT_LUMAA16, 3: _ffi.FMT_RGB16, 4: _ffi.FMT_RGBA16}[a.shape[3]]
    elif a.dtype != np.uint8:
        raise A3Error(_ffi.A3_ERR_UNSUPPORTED, "only 8- and 16-bit integer images are supported (convert float images with into_luma8 on the host)")
    elif a.ndim == 3:
        fmt = _ffi.FMT_LUMA8
    elif a.ndim == 4 and a.shape[3] == 2 and order == "rgb":
        fmt = _ffi.FMT_LUMAA8
    elif a.ndim == 4 and (order, a.shape[3]) in _FMT:
        fmt = _FMT[(order, a.shape[3])]
    else:
        raise A3Error(_ffi.A3_ERR_INVALID_ARGUMENT, f"bad frame array shape {a.shape}")
    a = np.ascontiguousarray(a)
    n, h, w = a.shape[:3]
    pitch = w * (a.shape[3] if a.ndim == 4 else 1) * a.itemsize  # not a.strides: a size-1 axis of a C-contiguous view may report any stride
    return a, fmt, n, h, w, pitch, pitch * h


class Detector:
    """`Detector { config, dictionary }` (src/aruco.rs:46-49) bound to one CUDA device.

    Thread-compatible like the C handle: one Detector per (host thread, device).
    """

    def __init__(self, config: DetectorConfig | None = None, dictionary: ARDictionary | str = "ARUCO", device: int = 0,
                 host_threads: int | None = None, contours: str = "device", corners: str = "integer", board=None,
                 board_intrinsics=None, distortion=None):
        self.config = config or DetectorConfig()
        self.dictionary = ARDictionary.new_from_named_dict(dictionary) if isinstance(dictionary, str) else dictionary
        self.device = device
        self._h = C.c_void_p()
        cfg = self.config.to_c()
        check(lib().a3_detector_create(C.byref(cfg), C.byref(self.dictionary._c), device, C.byref(self._h)))
        if host_threads:
            check(lib().a3_detector_set_host_threads(self._h, host_threads))
        # where find_contours + the quad filters run: "device" (kernel K3, host redo of flagged frames) or "host"
        check(lib().a3_detector_set_contour_mode(self._h, {"host": _ffi.CONTOURS_HOST, "device": _ffi.CONTOURS_DEVICE}[contours]))
        self.last_stats: dict = {}
        self._pose_mode = _ffi.POSE_OFF
        self._corner_mode = _ffi.CORNERS_INTEGER
        self.set_corner_refinement(corners)
        self._board = None
        if board is not None:
            self.set_board(board, board_intrinsics)
        self.set_distortion(distortion)

    def set_distortion(self, distortion=None):
        """Give the camera intrinsics of the pose and board modes a lens distortion (`pose.CameraDistortion`): `detect` /
        `detect_batch` then undistort every corner the pose kernels read (kernel K7) and the marker and board poses solve from
        the undistorted points.  Only with intrinsics modes (`set_pose` / `set_board` with `camera_intrinsics`); `None` or all
        coefficients zero switches it off."""
        check(lib().a3_detector_set_distortion(self._h, C.byref(distortion._c) if distortion is not None else None))
        self._distortion = distortion

    def set_board(self, board, camera_intrinsics=None):
        """Also solve the pose of a planar `Board` in every frame inside `detect` / `detect_batch` (kernel K6 behind the
        decode kernel and K5) into `Detection.board_pose`, from every accepted marker on the board: its refined corners when
        the detector refines corners, else the integer ones.  Normalisation as `set_pose`: `camera_intrinsics`, or
        undistorted at the frame size when None.  `board=None` switches it off."""
        if board is None:
            check(lib().a3_detector_set_board(self._h, None, _ffi.POSE_OFF, None))
            self._board = None
            return
        mode = _ffi.POSE_INTRINSICS if camera_intrinsics is not None else _ffi.POSE_UNDISTORTED
        c = board.to_c()
        check(lib().a3_detector_set_board(self._h, C.byref(c), mode,
                                          C.byref(camera_intrinsics._c) if camera_intrinsics is not None else None))
        self._board = board

    def set_corner_refinement(self, corners: str = "refined"):
        """`"refined"`: `detect` / `detect_batch` also return each marker's sub-pixel corners (`Marker.corners_refined`,
        kernel K5 behind the decode kernel), and the pose step (set_pose) solves from them.  `"integer"` (the default)
        switches it off: only the reference's integer corners, and nothing more runs."""
        mode = {"integer": _ffi.CORNERS_INTEGER, "refined": _ffi.CORNERS_REFINED}[corners]
        check(lib().a3_detector_set_corner_refinement(self._h, mode))
        self._corner_mode = mode

    def set_pose(self, marker_size_mm: float | None, camera_intrinsics=None):
        """Also solve every marker's pose pair inside `detect` / `detect_batch` (kernel K4 behind the decode kernel):
        `pose::solve_with_intrinsics(&m.corners, size, &k)` when `camera_intrinsics` is given
        (examples/macroquad_detect.rs:150), else `pose::solve_with_undistorted_points(&m.corners, size, (w, h))`
        (examples/webcam_kamera.rs:68).  `marker_size_mm=None` switches it off."""
        if marker_size_mm is None:
            mode = _ffi.POSE_OFF
        else:
            mode = _ffi.POSE_INTRINSICS if camera_intrinsics is not None else _ffi.POSE_UNDISTORTED
        check(lib().a3_detector_set_pose(self._h, mode, marker_size_mm or 0.0,
                                         C.byref(camera_intrinsics._c) if camera_intrinsics is not None else None))
        self._pose_mode = mode

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().a3_detector_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- the reference's entry point -------------------------------------------------------------------
    def detect(self, image: np.ndarray, order: str = "rgb") -> Detection:
        """`Detector::detect(&self, image: DynamicImage) -> Detection` (src/aruco.rs:52-121): one image [H,W,3|4] or [H,W]."""
        return self.detect_batch(np.asarray(image)[None], full=True, order=order)[0]

    def detect_batch(self, frames: np.ndarray, full: bool = False, want_mask: bool = False, cand_capacity: int = 0,
                     marker_capacity: int = 0, order: str = "rgb") -> list:
        """`detect` over n equally sized frames -> [Detection].  `full` also returns grey, candidates, homographies
        and the per-candidate decode records (what `Detection` holds in the reference); without it only markers.
        `order="bgr"`: frames are B,G,R[,A] as cameras deliver them; the result is that of the swizzled image."""
        a, fmt, n, h, w, pitch, fstride = _frames_view(frames, order)
        hs = self.config.homography_sample_size
        cap_m = marker_capacity or max(64 * n, 1024)
        cap_c = cand_capacity or max(128 * n, 2048)
        while True:
            markers = (A3Marker * cap_m)()
            n_markers = C.c_uint32()
            stats = A3Stats()
            outs = A3Outputs()
            offsets = np.zeros(n + 1, np.uint32)
            outs.frame_marker_offsets = offsets.ctypes.data
            keep = []
            poses = None
            if self._pose_mode != _ffi.POSE_OFF:
                poses = (A3Pose * (2 * cap_m))()
                outs.marker_poses = C.cast(poses, C.c_void_p).value
            refined = None
            if self._corner_mode == _ffi.CORNERS_REFINED:
                refined = np.zeros((cap_m, 4, 2), np.float32)
                outs.marker_corners = refined.ctypes.data
            bposes = None
            if self._board is not None:
                bposes = (_ffi.A3BoardPose * n)()
                outs.board_poses = C.cast(bposes, C.c_void_p).value
            if full:
                grey = np.empty((n, h, w), np.uint8)
                cands = np.zeros((cap_c, 8), np.uint32)
                cframe = np.zeros(cap_c, np.uint32)
                patches = np.zeros((cap_c, hs, hs), np.uint8)
                decs = (A3Decode * cap_c)()
                outs.grey = grey.ctypes.data
                outs.candidates = cands.ctypes.data
                outs.candidate_frame = cframe.ctypes.data
                outs.homographies = patches.ctypes.data
                outs.decodes = C.cast(decs, C.c_void_p).value
                outs.cand_capacity = cap_c
                keep = [grey, cands, cframe, patches, decs]
            if want_mask:
                mask = np.empty((n, h, w), np.uint8)
                outs.mask = mask.ctypes.data
            st = lib().a3_detect_batch(self._h, a.ctypes.data, fmt, _ffi.MEM_HOST, n, w, h, pitch, fstride,
                                       C.cast(markers, C.c_void_p), cap_m, C.byref(n_markers), C.byref(outs),
                                       C.byref(stats))
            if st == _ffi.A3_ERR_CAPACITY:  # two-call sizing: counts are valid
                cap_m = max(cap_m, n_markers.value)
                cap_c = max(cap_c, outs.n_candidates)
                continue
            check(st)
            break
        self.last_stats = stats.as_dict()
        dets = [Detection() for _ in range(n)]
        for i in range(n_markers.value):
            m = markers[i]
            dets[m.frame].markers.append(Marker(int(m.id), int(m.code), [(int(m.corners[2 * k]), int(m.corners[2 * k + 1])) for k in range(4)],
                                                int(m.hamming_distance), int(m.rotation), int(m.candidate)))
            if poses is not None:
                from .pose import MarkerPose
                dets[m.frame].markers[-1].poses = (MarkerPose.from_c(poses[2 * i]), MarkerPose.from_c(poses[2 * i + 1]))
            if refined is not None:
                dets[m.frame].markers[-1].corners_refined = [(refined[i, k, 0], refined[i, k, 1]) for k in range(4)]
                dets[m.frame].markers[-1].refined = bool(m.corners_refined)
        if bposes is not None:
            from .board import BoardPose
            for f in range(n):
                dets[f].board_pose = BoardPose.from_c(bposes[f])
        if full:
            for f in range(n):
                dets[f].grey = grey[f]
            for k in range(outs.n_candidates):
                d = dets[int(cframe[k])]
                d.candidates.append([(int(cands[k, 2 * j]), int(cands[k, 2 * j + 1])) for j in range(4)])
                dc = decs[k]
                d.homographies.append(patches[k] if dc.homography_ok else np.zeros((1, 1), np.uint8))  # src/aruco.rs:256
                d.decodes.append(dict(codes=[int(c) for c in dc.codes], id=int(dc.id), has_codes=bool(dc.has_codes),
                                      homography_ok=bool(dc.homography_ok), otsu=int(dc.otsu), rotation=int(dc.rotation),
                                      hamming_distance=int(dc.hamming_distance), accepted=bool(dc.accepted)))
        if want_mask:
            for f in range(n):
                dets[f].mask = mask[f]
        del keep
        return dets

    # ---- stage probes (the same kernels) -----------------------------------------------------------------
    def gray_threshold(self, frames: np.ndarray, want_bits: bool = False, order: str = "rgb"):
        """into_luma8 + adaptive_threshold over [n,H,W,C] host frames -> (grey [n,H,W], mask [n,H,W][, bits [n,H,ceil(W/32)]])."""
        a, fmt, n, h, w, pitch, fstride = _frames_view(frames, order)
        grey = np.empty((n, h, w), np.uint8)
        mask = np.empty((n, h, w), np.uint8)
        bits = np.empty((n, h, (w + 31) // 32), np.uint32) if want_bits else None
        check(lib().a3_gray_threshold_batch(self._h, a.ctypes.data, fmt, _ffi.MEM_HOST, n, w, h, pitch, fstride,
                                            grey.ctypes.data, mask.ctypes.data, bits.ctypes.data if want_bits else None, None))
        return (grey, mask, bits) if want_bits else (grey, mask)

    def quads_from_masks_device(self, masks: np.ndarray, quad_capacity: int = 1024):
        """find_contours + quad filters on the device (kernel K3) for host masks [n,H,W] -> (list of uint32 [m,8] per frame,
        flags uint32 [n], contours uint32 [n], points uint64 [n]); a frame with a non-zero flag must be redone by the host stage."""
        m = np.ascontiguousarray(masks, dtype=np.uint8)
        if m.ndim == 2:
            m = m[None]
        n, h, w = m.shape
        quads = np.zeros((n, quad_capacity, 8), np.uint32)
        counts, flags, contours = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint32)
        points = np.zeros(n, np.uint64)
        check(lib().a3_quads_from_masks_device(self._h, m.ctypes.data, n, w, h, quads.ctypes.data, quad_capacity, counts.ctypes.data,
                                               flags.ctypes.data, contours.ctypes.data, points.ctypes.data))
        return [quads[f, :counts[f]].copy() for f in range(n)], flags, contours, points

    def decode_candidates(self, grey: np.ndarray, quads: np.ndarray, quad_frame: np.ndarray | None = None):
        """extract_homographies + homography_to_code_permutations + match for quads uint32 [m,8] over grey [n,H,W]
        -> (decode dicts, patches uint8 [m,hs,hs])."""
        g = np.ascontiguousarray(grey, dtype=np.uint8)
        if g.ndim == 2:
            g = g[None]
        n, h, w = g.shape
        q = np.ascontiguousarray(quads, dtype=np.uint32).reshape(-1, 8)
        m = q.shape[0]
        hs = self.config.homography_sample_size
        decs = (A3Decode * max(m, 1))()
        patches = np.zeros((m, hs, hs), np.uint8)
        qf = np.ascontiguousarray(quad_frame, dtype=np.uint32) if quad_frame is not None else None
        check(lib().a3_decode_candidates(self._h, g.ctypes.data, n, w, h, q.ctypes.data, qf.ctypes.data if qf is not None else None,
                                         m, C.cast(decs, C.c_void_p), patches.ctypes.data))
        out = [dict(codes=[int(c) for c in decs[k].codes], id=int(decs[k].id), has_codes=bool(decs[k].has_codes),
                    homography_ok=bool(decs[k].homography_ok), otsu=int(decs[k].otsu), rotation=int(decs[k].rotation),
                    hamming_distance=int(decs[k].hamming_distance), accepted=bool(decs[k].accepted)) for k in range(m)]
        return out, patches

    def refine_corners(self, grey: np.ndarray, corners: np.ndarray, corner_frame: np.ndarray | None = None):
        """The corner refinement (kernel K5) for integer corners uint32 [m,4,2] or [m,8] (screen-clockwise, as
        `Marker.corners`) over grey [n,H,W] or [H,W] -> (refined float32 [m,4,2], ok bool [m])."""
        g = np.ascontiguousarray(grey, dtype=np.uint8)
        if g.ndim == 2:
            g = g[None]
        n, h, w = g.shape
        c = np.ascontiguousarray(corners, dtype=np.uint32).reshape(-1, 8)
        m = c.shape[0]
        out = np.zeros((m, 4, 2), np.float32)
        ok = np.zeros(m, np.uint8)
        cf = np.ascontiguousarray(corner_frame, dtype=np.uint32) if corner_frame is not None else None
        check(lib().a3_refine_corners(self._h, g.ctypes.data, n, w, h, c.ctypes.data, cf.ctypes.data if cf is not None else None, m,
                                      out.ctypes.data, ok.ctypes.data))
        return out, ok.astype(bool)

    def undistort_points(self, points, camera_intrinsics, distortion):
        """The undistortion (kernel K7's device function) as a probe: pixels [n, 2] (pixel-centre convention) -> (normalised
        undistorted float32 [n, 2], ok bool [n]); a point that fails (fold of the model, no convergence, non-finite) reads
        (0, 0).  `pose.solve_with_normalized_points` on its result is what the marker pose with distortion computes."""
        p = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 2))
        out = np.zeros_like(p)
        ok = np.zeros(p.shape[0], np.uint8)
        check(lib().a3_undistort_points(self._h, p.ctypes.data, p.shape[0], C.byref(camera_intrinsics._c), C.byref(distortion._c),
                                        out.ctypes.data, ok.ctypes.data))
        return out, ok.astype(bool)

    def solve_board(self, ids, corners, frame=None, n_frames: int | None = None, image_size=None) -> list:
        """The board solve (kernel K6) with this detector's board and mode, as a probe: markers' ids [m], f32 corners
        [m, 4, 2] (image pixels, the order of `Marker.corners`), non-decreasing frame index [m] (None = all frame 0);
        image_size (w, h) for undistorted mode -> [BoardPose] * n_frames."""
        from .board import BoardPose
        i = np.ascontiguousarray(np.asarray(ids, np.uint64).reshape(-1))
        c = np.ascontiguousarray(np.asarray(corners, np.float32).reshape(-1, 8))
        f = np.ascontiguousarray(np.asarray(frame, np.uint32).reshape(-1)) if frame is not None else None
        nf = n_frames if n_frames is not None else (int(f.max()) + 1 if f is not None and f.size else 1)
        out = (_ffi.A3BoardPose * max(nf, 1))()
        w, h = image_size if image_size is not None else (0, 0)
        check(lib().a3_solve_board(self._h, i.ctypes.data, c.ctypes.data, f.ctypes.data if f is not None else None, i.size, nf, w, h,
                                   C.cast(out, C.c_void_p)))
        return [BoardPose.from_c(out[k]) for k in range(nf)]


def quads_from_mask(mask: np.ndarray, config: DetectorConfig | None = None) -> np.ndarray:
    """find_contours + contours_to_candidates + enforce_clockwise_corners + discard_too_near (src/aruco.rs:64-69)
    on one host mask -> uint32 [n,8].  Host stage of the product; needs no device."""
    cfg = (config or DetectorConfig()).to_c()
    m = np.ascontiguousarray(mask, dtype=np.uint8)
    h, w = m.shape
    cap = 1024
    while True:
        quads = np.zeros((cap, 8), np.uint32)
        n = C.c_uint32()
        st = lib().a3_quads_from_mask(C.byref(cfg), m.ctypes.data, w, h, quads.ctypes.data, cap, C.byref(n), None)
        if st == _ffi.A3_ERR_CAPACITY:
            cap = n.value
            continue
        check(st)
        return quads[:n.value].copy()
