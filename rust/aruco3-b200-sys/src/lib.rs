//! Raw bindings, one to one with `include/aruco3_b200.h`. Not compiled in this repository's environment.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

pub type a3_status = i32;
pub const A3_OK: a3_status = 0;
pub const A3_ERR_INVALID_ARGUMENT: a3_status = 1;
pub const A3_ERR_UNKNOWN_DICTIONARY: a3_status = 2;
pub const A3_ERR_CUDA: a3_status = 3;
pub const A3_ERR_CAPACITY: a3_status = 4;
pub const A3_ERR_UNSUPPORTED: a3_status = 5;
pub const A3_ERR_OUT_OF_MEMORY: a3_status = 6;

pub const A3_FMT_RGB8: i32 = 0;
pub const A3_FMT_RGBA8: i32 = 1;
pub const A3_FMT_LUMA8: i32 = 2;
pub const A3_FMT_BGR8: i32 = 3; // camera byte order: what examples/webcam_kamera.rs:38-52 swizzles on the host
pub const A3_FMT_BGRA8: i32 = 4;
pub const A3_FMT_LUMAA8: i32 = 5; // the other integer DynamicImage variants: into_luma8 runs on the device (kernel K0)
pub const A3_FMT_LUMA16: i32 = 6;
pub const A3_FMT_LUMAA16: i32 = 7;
pub const A3_FMT_RGB16: i32 = 8;
pub const A3_FMT_RGBA16: i32 = 9;
pub const A3_MEM_HOST: i32 = 0;
pub const A3_MEM_DEVICE: i32 = 1;

/// `DetectorConfig`, field for field (reference `src/aruco.rs:23-30`).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct a3_config {
    pub threshold_window: u32,
    pub contour_simplification_epsilon: f64,
    pub min_side_length_factor: f32,
    pub min_corner_separation_factor: f32,
    pub homography_sample_size: u32,
    pub filter_high_bit_errors: u8,
}

/// `ARDictionary` (reference `src/dictionaries.rs:22-28`); `codes` points at static storage inside the library.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct a3_dictionary {
    pub num_bits: u8,
    pub tau: u8,
    pub n_codes: u32,
    pub codes: *const u64,
}

/// `Marker` (reference `src/aruco.rs:8-13`) plus frame / candidate / rotation.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct a3_marker {
    pub id: u64,
    pub code: u64,
    pub corners: [u32; 8],
    pub frame: u32,
    pub candidate: u32,
    pub hamming_distance: u8,
    pub rotation: u8,
    /// 1 when K5 refined this marker's corners (`a3_outputs.marker_corners`), 0 when off or fell back
    pub corners_refined: u8,
    pub reserved: [u8; 5],
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct a3_decode {
    pub codes: [u64; 4],
    pub id: u64,
    pub has_codes: u8,
    pub homography_ok: u8,
    pub otsu: u8,
    pub rotation: u8,
    pub hamming_distance: u8,
    pub accepted: u8,
    pub reserved: [u8; 2],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct a3_stats {
    pub n_frames: u64,
    pub n_contours: u64,
    pub n_contour_points: u64,
    pub n_candidates_before_discard: u64,
    pub n_candidates: u64,
    pub n_markers: u64,
    pub ms_h2d: f64,
    pub ms_pixel_kernel: f64,
    pub ms_contour_kernels: f64,
    pub ms_mask_d2h: f64,
    pub ms_host_quads: f64,
    pub ms_decode_kernel: f64,
    pub ms_host_cpu: f64,
    pub ms_total: f64,
    pub pixel_kernel_launches: u32,
    pub decode_kernel_launches: u32,
    pub host_threads: u32,
    pub contour_kernel_launches: u32,
    pub host_fallback_frames: u32,
    pub pose_kernel_launches: u32,
    pub one_shot: u32,
    pub one_shot_retry: u32,
    pub input_staged: u32,
    pub output_staged: u32,
    pub refine_kernel_launches: u32,
    pub ms_refine_kernel: f64,
    /// board pose (K6, `a3_detector_set_board`): launches and the sum of its CUDA-event intervals
    pub board_kernel_launches: u32,
    pub ms_board_kernel: f64,
    /// corner undistortion (K7, `a3_detector_set_distortion`): launches and the sum of its CUDA-event intervals
    pub undistort_kernel_launches: u32,
    pub ms_undistort_kernel: f64,
}

/// MarkerPose, reference `src/pose.rs:8-12`; rotation row-major
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct a3_pose {
    pub error: f32,
    pub rotation: [f32; 9],
    pub translation: [f32; 3],
}

/// CameraIntrinsics, reference `src/pinhole.rs:11-18`
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct a3_camera_intrinsics {
    pub image_width: u32,
    pub image_height: u32,
    pub focal_x: f32,
    pub focal_y: f32,
    pub principal_x: f32,
    pub principal_y: f32,
}

/// Lens distortion of the intrinsics: OpenCV's k1 k2 p1 p2 k3 (not in the reference's pinhole model).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct a3_camera_distortion {
    pub k1: f32,
    pub k2: f32,
    pub p1: f32,
    pub p2: f32,
    pub k3: f32,
}

pub const A3_CORNERS_INTEGER: u32 = 0;
pub const A3_CORNERS_REFINED: u32 = 1;
pub const A3_POSE_OFF: u32 = 0;
pub const A3_POSE_UNDISTORTED: u32 = 1;
pub const A3_POSE_INTRINSICS: u32 = 2;
pub const A3_POSE_NORMALIZED: u32 = 3;

#[repr(C)]
pub struct a3_outputs {
    pub grey: *mut u8,
    pub mask: *mut u8,
    pub candidates: *mut u32,
    pub candidate_frame: *mut u32,
    pub homographies: *mut u8,
    pub decodes: *mut a3_decode,
    pub cand_capacity: u32,
    pub n_candidates: u32,
    pub frame_marker_offsets: *mut u32,
    pub marker_poses: *mut a3_pose,
    /// marker_capacity * 8 f32 (A3_CORNERS_REFINED), may be null
    pub marker_corners: *mut f32,
    /// n board poses (`a3_detector_set_board`), may be null
    pub board_poses: *mut a3_board_pose,
}

/// A rigid planar board: `n_markers` distinct ids and their corners on the board plane (x right, y up), `n_markers * 8`
/// f32 in the order of `a3_marker.corners`
#[repr(C)]
pub struct a3_board {
    pub n_markers: u32,
    pub ids: *const u64,
    pub corners: *const f32,
}

/// The board's pose in one frame (kernel K6): board points `(x, y, 0)` -> camera; error = RMS reprojection distance
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct a3_board_pose {
    pub best: a3_pose,
    pub alt: a3_pose,
    pub n_markers: u32,
    pub ok: u8,
    pub reserved: [u8; 3],
}

#[repr(C)]
pub struct a3_detector {
    _private: [u8; 0],
}

extern "C" {
    pub fn a3_version() -> *const c_char;
    pub fn a3_last_error() -> *const c_char;
    pub fn a3_status_string(s: a3_status) -> *const c_char;
    pub fn a3_device_count() -> i32;

    pub fn a3_dictionary_count() -> i32;
    pub fn a3_dictionary_name(index: i32) -> *const c_char;
    pub fn a3_dictionary_by_name(name: *const c_char, out: *mut a3_dictionary) -> a3_status;
    pub fn a3_dictionary_mark_size(d: *const a3_dictionary) -> u8;
    pub fn a3_hamming_distance(a: u64, b: u64) -> u8;
    pub fn a3_find_nearest(d: *const a3_dictionary, bits: u64, index: *mut u64, dist: *mut u8);
    pub fn a3_try_find_nearest(d: *const a3_dictionary, bits: u64, index: *mut u64, dist: *mut u8) -> i32;
    pub fn a3_make_binary_image(d: *const a3_dictionary, marker_id: u64, bits: *mut u8, capacity: u32, n_bits: *mut u32) -> u8;

    pub fn a3_config_default(cfg: *mut a3_config);
    pub fn a3_detector_create(cfg: *const a3_config, dict: *const a3_dictionary, device: i32, out: *mut *mut a3_detector) -> a3_status;
    pub fn a3_detector_destroy(det: *mut a3_detector);
    // handle cache for plain-data `Detector` literals (reference src/aruco.rs:46-49): bracket each call
    pub fn a3_detector_acquire(cfg: *const a3_config, dict: *const a3_dictionary, device: i32, out: *mut *mut a3_detector) -> a3_status;
    pub fn a3_detector_release(det: *mut a3_detector);
    pub fn a3_detector_cache_clear();
    pub fn a3_detector_create_count() -> u64;
    pub fn a3_detector_set_host_threads(det: *mut a3_detector, threads: u32) -> a3_status;
    pub fn a3_detector_set_contour_mode(det: *mut a3_detector, mode: u32) -> a3_status;
    pub fn a3_detector_set_corner_refinement(det: *mut a3_detector, mode: u32) -> a3_status;
    pub fn a3_detect_batch(
        det: *mut a3_detector, frames: *const c_void, format: i32, mem: i32, n: u32, width: u32, height: u32, pitch: usize,
        frame_stride: usize, markers: *mut a3_marker, marker_capacity: u32, n_markers: *mut u32, outputs: *mut a3_outputs,
        stats: *mut a3_stats,
    ) -> a3_status;
    pub fn a3_gray_threshold_batch(
        det: *mut a3_detector, frames: *const c_void, format: i32, mem: i32, n: u32, width: u32, height: u32, pitch: usize,
        frame_stride: usize, grey: *mut u8, mask: *mut u8, mask_bits: *mut u32, cuda_stream: *mut c_void,
    ) -> a3_status;
    pub fn a3_quads_from_mask(
        cfg: *const a3_config, mask: *const u8, width: u32, height: u32, quads: *mut u32, quad_capacity: u32, n_quads: *mut u32,
        stats: *mut a3_stats,
    ) -> a3_status;
    pub fn a3_decode_candidates(
        det: *mut a3_detector, grey: *const u8, n_frames: u32, width: u32, height: u32, quads: *const u32, quad_frame: *const u32,
        n_quads: u32, decodes: *mut a3_decode, patches: *mut u8,
    ) -> a3_status;
    pub fn a3_refine_corners(
        det: *mut a3_detector, grey: *const u8, n_frames: u32, width: u32, height: u32, corners: *const u32, corner_frame: *const u32,
        n: u32, refined: *mut f32, ok: *mut u8,
    ) -> a3_status;

    // pose step (reference src/pose.rs, src/pinhole.rs)
    pub fn a3_detector_set_pose(det: *mut a3_detector, mode: u32, marker_size_mm: f32, k: *const a3_camera_intrinsics) -> a3_status;
    pub fn a3_solve_with_intrinsics(
        det: *mut a3_detector, corners: *const u32, n: u32, marker_size_mm: f32, k: *const a3_camera_intrinsics, best: *mut a3_pose,
        alt: *mut a3_pose,
    ) -> a3_status;
    pub fn a3_solve_with_undistorted_points(
        det: *mut a3_detector, corners: *const u32, n: u32, marker_size_mm: f32, image_width: u32, image_height: u32,
        best: *mut a3_pose, alt: *mut a3_pose,
    ) -> a3_status;
    pub fn a3_solve_with_normalized_points(
        det: *mut a3_detector, points: *const f32, n: u32, marker_size_mm: f32, best: *mut a3_pose, alt: *mut a3_pose,
    ) -> a3_status;
    // board pose (kernel K6)
    pub fn a3_detector_set_board(det: *mut a3_detector, board: *const a3_board, mode: u32, k: *const a3_camera_intrinsics) -> a3_status;
    pub fn a3_solve_board(
        det: *mut a3_detector, ids: *const u64, corners: *const f32, frame: *const u32, n: u32, n_frames: u32, image_w: u32,
        image_h: u32, out: *mut a3_board_pose,
    ) -> a3_status;
    // lens distortion (kernel K7)
    pub fn a3_detector_set_distortion(det: *mut a3_detector, d: *const a3_camera_distortion) -> a3_status;
    pub fn a3_undistort_points(
        det: *mut a3_detector, points: *const f32, n: u32, k: *const a3_camera_intrinsics, d: *const a3_camera_distortion, out: *mut f32,
        ok: *mut u8,
    ) -> a3_status;
    pub fn a3_pose_default(p: *mut a3_pose);
    pub fn a3_pose_apply_transform(p: *const a3_pose, points: *const f32, n: u32, inverse: i32, out: *mut f32);
    pub fn a3_camera_intrinsics_new(
        image_width: u32, image_height: u32, focal_x: f32, focal_y: f32, principal_x: *const f32, principal_y: *const f32,
        out: *mut a3_camera_intrinsics,
    );
    pub fn a3_camera_intrinsics_from_fov_horizontal(
        horizontal_fov_radians: f32, sensor_width_mm: f32, resolution_x: u32, resolution_y: u32, out: *mut a3_camera_intrinsics,
    );
    pub fn a3_camera_project(k: *const a3_camera_intrinsics, x: f32, y: f32, z: f32, out: *mut f32);
    pub fn a3_camera_project_culled(k: *const a3_camera_intrinsics, x: f32, y: f32, z: f32, out: *mut f32) -> i32;
    pub fn a3_camera_unproject(k: *const a3_camera_intrinsics, x: f32, y: f32, out: *mut f32);
}
