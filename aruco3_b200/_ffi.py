"""ctypes binding of libaruco3_b200.so — the same C ABI (include/aruco3_b200.h) a Rust -sys crate would bind."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
# A3_LIB_PATH: load another build of the same library (A/B timing of kernel variants, tools/k1_variants.sh); never a fallback
LIB_PATH = Path(os.environ["A3_LIB_PATH"]).resolve() if os.environ.get("A3_LIB_PATH") else PKG / "libaruco3_b200.so"

A3_OK, A3_ERR_INVALID_ARGUMENT, A3_ERR_UNKNOWN_DICTIONARY, A3_ERR_CUDA, A3_ERR_CAPACITY, A3_ERR_UNSUPPORTED, \
    A3_ERR_OUT_OF_MEMORY = range(7)
FMT_RGB8, FMT_RGBA8, FMT_LUMA8, FMT_BGR8, FMT_BGRA8 = 0, 1, 2, 3, 4
FMT_LUMAA8, FMT_LUMA16, FMT_LUMAA16, FMT_RGB16, FMT_RGBA16 = 5, 6, 7, 8, 9
MEM_HOST, MEM_DEVICE = 0, 1
CONTOURS_HOST, CONTOURS_DEVICE = 0, 1
POSE_OFF, POSE_UNDISTORTED, POSE_INTRINSICS, POSE_NORMALIZED = 0, 1, 2, 3
CORNERS_INTEGER, CORNERS_REFINED = 0, 1


class A3Config(C.Structure):
    _fields_ = [("threshold_window", C.c_uint32), ("contour_simplification_epsilon", C.c_double),
                ("min_side_length_factor", C.c_float), ("min_corner_separation_factor", C.c_float),
                ("homography_sample_size", C.c_uint32), ("filter_high_bit_errors", C.c_uint8)]


class A3Dictionary(C.Structure):
    _fields_ = [("num_bits", C.c_uint8), ("tau", C.c_uint8), ("n_codes", C.c_uint32),
                ("codes", C.POINTER(C.c_uint64))]


class A3Marker(C.Structure):
    _fields_ = [("id", C.c_uint64), ("code", C.c_uint64), ("corners", C.c_uint32 * 8), ("frame", C.c_uint32),
                ("candidate", C.c_uint32), ("hamming_distance", C.c_uint8), ("rotation", C.c_uint8),
                ("corners_refined", C.c_uint8), ("reserved", C.c_uint8 * 5)]


class A3Decode(C.Structure):
    _fields_ = [("codes", C.c_uint64 * 4), ("id", C.c_uint64), ("has_codes", C.c_uint8), ("homography_ok", C.c_uint8),
                ("otsu", C.c_uint8), ("rotation", C.c_uint8), ("hamming_distance", C.c_uint8), ("accepted", C.c_uint8),
                ("reserved", C.c_uint8 * 2)]


class A3Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_frames", "n_contours", "n_contour_points", "n_candidates_before_discard",
                                          "n_candidates", "n_markers")] + \
               [(n, C.c_double) for n in ("ms_h2d", "ms_pixel_kernel", "ms_contour_kernels", "ms_mask_d2h", "ms_host_quads",
                                          "ms_decode_kernel", "ms_host_cpu", "ms_total")] + \
               [(n, C.c_uint32) for n in ("pixel_kernel_launches", "decode_kernel_launches", "host_threads", "contour_kernel_launches",
                                          "host_fallback_frames", "pose_kernel_launches", "one_shot", "one_shot_retry", "input_staged", "output_staged",
                                          "refine_kernel_launches")] + \
               [("ms_refine_kernel", C.c_double), ("board_kernel_launches", C.c_uint32), ("ms_board_kernel", C.c_double),
                ("undistort_kernel_launches", C.c_uint32), ("ms_undistort_kernel", C.c_double)]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


class A3Outputs(C.Structure):
    _fields_ = [("grey", C.c_void_p), ("mask", C.c_void_p), ("candidates", C.c_void_p), ("candidate_frame", C.c_void_p),
                ("homographies", C.c_void_p), ("decodes", C.c_void_p), ("cand_capacity", C.c_uint32),
                ("n_candidates", C.c_uint32), ("frame_marker_offsets", C.c_void_p), ("marker_poses", C.c_void_p),
                ("marker_corners", C.c_void_p), ("board_poses", C.c_void_p)]


class A3Pose(C.Structure):
    _fields_ = [("error", C.c_float), ("rotation", C.c_float * 9), ("translation", C.c_float * 3)]


class A3Board(C.Structure):
    _fields_ = [("n_markers", C.c_uint32), ("ids", C.POINTER(C.c_uint64)), ("corners", C.POINTER(C.c_float))]


class A3BoardPose(C.Structure):
    _fields_ = [("best", A3Pose), ("alt", A3Pose), ("n_markers", C.c_uint32), ("ok", C.c_uint8), ("reserved", C.c_uint8 * 3)]


class A3CameraIntrinsics(C.Structure):
    _fields_ = [("image_width", C.c_uint32), ("image_height", C.c_uint32), ("focal_x", C.c_float), ("focal_y", C.c_float),
                ("principal_x", C.c_float), ("principal_y", C.c_float)]


class A3CameraDistortion(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("k1", "k2", "p1", "p2", "k3")]


class A3K1Tuning(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("strip_cols", "seg_rows", "force_no_tma", "force_generic", "chunk_frames")] + \
               [("reserved", C.c_uint32 * 3)]


class A3Error(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"aruco3_b200 status {status}: {message}")
        self.status = status


_lib = None


def build(force: bool = False) -> Path:
    """Compile the CUDA library in-tree (nvcc, sm_100a)."""
    if force:
        subprocess.run(["make", "-s", "-C", str(PKG / "csrc"), "clean"], check=True)
    subprocess.run(["make", "-s", "-C", str(PKG / "csrc")], check=True)
    return LIB_PATH


def lib():
    """Load the CUDA library. There is no fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if os.environ.get("A3_NO_AUTOBUILD"):
            raise A3Error(A3_ERR_CUDA, f"{LIB_PATH} is missing (run `python -c 'import __graft_entry__ as g; g.build()'`)")
        build()
    L = C.CDLL(str(LIB_PATH))
    vp, u32, u64, sz = C.c_void_p, C.c_uint32, C.c_uint64, C.c_size_t
    L.a3_version.restype = C.c_char_p
    L.a3_last_error.restype = C.c_char_p
    L.a3_status_string.restype = C.c_char_p
    L.a3_status_string.argtypes = [C.c_int32]
    L.a3_device_count.restype = C.c_int32
    L.a3_dictionary_count.restype = C.c_int32
    L.a3_dictionary_name.restype = C.c_char_p
    L.a3_dictionary_name.argtypes = [C.c_int32]
    L.a3_dictionary_by_name.argtypes = [C.c_char_p, C.POINTER(A3Dictionary)]
    L.a3_dictionary_mark_size.restype = C.c_uint8
    L.a3_dictionary_mark_size.argtypes = [C.POINTER(A3Dictionary)]
    L.a3_hamming_distance.restype = C.c_uint8
    L.a3_hamming_distance.argtypes = [u64, u64]
    L.a3_find_nearest.restype = None
    L.a3_find_nearest.argtypes = [C.POINTER(A3Dictionary), u64, C.POINTER(u64), C.POINTER(C.c_uint8)]
    L.a3_try_find_nearest.restype = C.c_int32
    L.a3_try_find_nearest.argtypes = L.a3_find_nearest.argtypes
    L.a3_make_binary_image.restype = C.c_uint8
    L.a3_make_binary_image.argtypes = [C.POINTER(A3Dictionary), u64, vp, u32, C.POINTER(u32)]
    L.a3_config_default.restype = None
    L.a3_config_default.argtypes = [C.POINTER(A3Config)]
    L.a3_detector_create.argtypes = [C.POINTER(A3Config), C.POINTER(A3Dictionary), C.c_int32, C.POINTER(vp)]
    L.a3_detector_destroy.restype = None
    L.a3_detector_destroy.argtypes = [vp]
    L.a3_detector_acquire.argtypes = [C.POINTER(A3Config), C.POINTER(A3Dictionary), C.c_int32, C.POINTER(vp)]
    L.a3_detector_release.restype = None
    L.a3_detector_release.argtypes = [vp]
    L.a3_detector_cache_clear.restype = None
    L.a3_detector_create_count.restype = C.c_uint64
    L.a3_detector_set_host_threads.argtypes = [vp, u32]
    L.a3_detector_set_contour_mode.argtypes = [vp, u32]
    L.a3_detector_set_corner_refinement.argtypes = [vp, u32]
    L.a3_detector_set_k1_tuning.argtypes = [vp, C.POINTER(A3K1Tuning)]
    L.a3_detect_batch.argtypes = [vp, vp, C.c_int, C.c_int, u32, u32, u32, sz, sz, vp, u32, C.POINTER(u32),
                                  C.POINTER(A3Outputs), C.POINTER(A3Stats)]
    L.a3_gray_threshold_batch.argtypes = [vp, vp, C.c_int, C.c_int, u32, u32, u32, sz, sz, vp, vp, vp, vp]
    L.a3_quads_from_mask.argtypes = [C.POINTER(A3Config), vp, u32, u32, vp, u32, C.POINTER(u32), C.POINTER(A3Stats)]
    L.a3_quads_from_masks_device.argtypes = [vp, vp, u32, u32, u32, vp, u32, vp, vp, vp, vp]
    L.a3_decode_candidates.argtypes = [vp, vp, u32, u32, u32, vp, vp, u32, vp, vp]
    L.a3_refine_corners.argtypes = [vp, vp, u32, u32, u32, vp, vp, u32, vp, vp]
    fp, f32, PK, PP = C.POINTER(C.c_float), C.c_float, C.POINTER(A3CameraIntrinsics), C.POINTER(A3Pose)
    L.a3_detector_set_pose.argtypes = [vp, u32, f32, PK]
    L.a3_detector_set_board.argtypes = [vp, C.POINTER(A3Board), u32, PK]
    L.a3_solve_board.argtypes = [vp, vp, vp, vp, u32, u32, u32, u32, vp]
    PD = C.POINTER(A3CameraDistortion)
    L.a3_detector_set_distortion.argtypes = [vp, PD]
    L.a3_undistort_points.argtypes = [vp, vp, u32, PK, PD, vp, vp]
    L.a3_solve_with_intrinsics.argtypes = [vp, vp, u32, f32, PK, vp, vp]
    L.a3_solve_with_undistorted_points.argtypes = [vp, vp, u32, f32, u32, u32, vp, vp]
    L.a3_solve_with_normalized_points.argtypes = [vp, vp, u32, f32, vp, vp]
    L.a3_pose_default.restype = None
    L.a3_pose_default.argtypes = [PP]
    L.a3_pose_apply_transform.restype = None
    L.a3_pose_apply_transform.argtypes = [PP, vp, u32, C.c_int32, vp]
    L.a3_camera_intrinsics_new.restype = None
    L.a3_camera_intrinsics_new.argtypes = [u32, u32, f32, f32, fp, fp, PK]
    L.a3_camera_intrinsics_from_fov_horizontal.restype = None
    L.a3_camera_intrinsics_from_fov_horizontal.argtypes = [f32, f32, u32, u32, PK]
    L.a3_camera_project.restype = None
    L.a3_camera_project.argtypes = [PK, f32, f32, f32, fp]
    L.a3_camera_project_culled.restype = C.c_int32
    L.a3_camera_project_culled.argtypes = [PK, f32, f32, f32, fp]
    L.a3_camera_unproject.restype = None
    L.a3_camera_unproject.argtypes = [PK, f32, f32, fp]
    _lib = L
    return L


def check(status: int):
    if status != A3_OK:
        raise A3Error(status, lib().a3_last_error().decode(errors="replace"))
