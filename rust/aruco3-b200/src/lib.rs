//! Drop-in for the detection path of `aruco3` (reference `src/aruco.rs`, `src/dictionaries.rs`): same public
//! types, field names and conventions; the work happens in libaruco3_b200.so (CUDA, sm_100a).
//! NOT COMPILED in this repository's environment (no Rust toolchain there): source only, untested.  The C++ twin of this
//! file, `aruco3::PlainDetector` in include/aruco3_b200.hpp (same lease-per-call design), is what the tests run.
use std::ffi::{CStr, CString};
use std::ptr;

use aruco3_b200_sys as sys;
use image::{DynamicImage, GrayImage};
use imageproc::point::Point;

/// reference `src/aruco.rs:8-13`
#[derive(Debug)]
pub struct Marker {
    pub id: usize,
    pub code: u64,
    pub corners: Vec<(u32, u32)>,
    pub hamming_distance: u8,
    /// Not in the reference: the sub-pixel corners in the order of `corners` (pixel-centre convention) when this thread
    /// asked for them (`set_corner_refinement(true)`) and the refinement held; `None` otherwise.
    pub corners_refined: Option<[(f32, f32); 4]>,
}

/// reference `src/aruco.rs:16-21`
#[derive(Default)]
pub struct Detection {
    pub grey: Option<GrayImage>,
    pub candidates: Vec<Vec<Point<u32>>>,
    pub homographies: Vec<GrayImage>,
    pub markers: Vec<Marker>,
    /// Not in the reference: the pose of this thread's board (`set_board`) in this frame; `None` when no board is set.
    pub board_pose: Option<pose::BoardPose>,
}

/// reference `src/aruco.rs:23-43`
pub struct DetectorConfig {
    pub threshold_window: u32,
    pub contour_simplification_epsilon: f64,
    pub min_side_length_factor: f32,
    pub min_corner_separation_factor: f32,
    pub homography_sample_size: usize,
    pub filter_high_bit_errors: bool,
}

impl Default for DetectorConfig {
    fn default() -> Self {
        DetectorConfig {
            threshold_window: 7,
            contour_simplification_epsilon: 0.05,
            min_side_length_factor: 0.2,
            min_corner_separation_factor: 0.1f32,
            homography_sample_size: 49,
            filter_high_bit_errors: true,
        }
    }
}

/// reference `src/dictionaries.rs:22-28`, field for field (no hidden state): a dictionary the reference built —
/// `ARDictionary::new_from_named_dict("ARUCO")`, or its own `code_list: &'static [u64]` table — converts with
/// `ARDictionary { num_bits: d.num_bits, tau: d.tau, code_list: d.code_list }`.
#[derive(Clone, Debug)]
pub struct ARDictionary {
    pub num_bits: u8,
    pub tau: u8,
    pub code_list: &'static [u64],
}

fn last_error() -> String {
    unsafe { CStr::from_ptr(sys::a3_last_error()).to_string_lossy().into_owned() }
}

impl ARDictionary {
    /// The C view: the table is static, so the pointer stays valid (and is part of the handle-cache key).
    fn raw(&self) -> sys::a3_dictionary {
        sys::a3_dictionary { num_bits: self.num_bits, tau: self.tau, n_codes: self.code_list.len() as u32, codes: self.code_list.as_ptr() }
    }
    /// reference `src/dictionaries.rs:140-145`: panics on an unknown name, like the reference.
    pub fn new_from_named_dict(name: &str) -> Self {
        let c = CString::new(name).expect("dictionary name");
        let mut raw = sys::a3_dictionary { num_bits: 0, tau: 0, n_codes: 0, codes: ptr::null() };
        let st = unsafe { sys::a3_dictionary_by_name(c.as_ptr(), &mut raw) };
        if st != sys::A3_OK {
            panic!("{}", last_error());
        }
        let code_list: &'static [u64] = unsafe { std::slice::from_raw_parts(raw.codes, raw.n_codes as usize) };
        ARDictionary { num_bits: raw.num_bits, tau: raw.tau, code_list }
    }
    pub fn get_mark_size(&self) -> u8 {
        unsafe { sys::a3_dictionary_mark_size(&self.raw()) }
    }
    pub fn find_nearest(&self, bits: u64) -> (usize, u8) {
        let (mut i, mut d) = (0u64, 0u8);
        unsafe { sys::a3_find_nearest(&self.raw(), bits, &mut i, &mut d) };
        (i as usize, d)
    }
    pub fn try_find_nearest(&self, bits: u64) -> Option<(usize, u8)> {
        let (mut i, mut d) = (0u64, 0u8);
        let ok = unsafe { sys::a3_try_find_nearest(&self.raw(), bits, &mut i, &mut d) };
        if ok != 0 { Some((i as usize, d)) } else { None }
    }
}

/// reference `src/aruco.rs:46-49`: plain data, built with a struct literal exactly like the reference's
/// (`benches/detect_markers.rs:17-20`).  It owns no CUDA state: every call leases a handle from the library's cache
/// (`a3_detector_acquire` / `a3_detector_release`), so a per-frame loop creates ONE handle — streams, device and pinned
/// buffers, the K3 workspace and the one-shot history stay warm between calls — and `detect` stays `&self`, `Send + Sync`.
pub struct Detector {
    pub config: DetectorConfig,
    pub dictionary: ARDictionary,
}

thread_local! {
    /// CUDA device the calling thread's detectors run on (default 0); see `set_device`.
    static DEVICE: std::cell::Cell<i32> = std::cell::Cell::new(0);
}
/// Choose the CUDA device for this thread's `detect` calls (frame-batch sharding: one thread per GPU).
pub fn set_device(device: i32) {
    DEVICE.with(|d| d.set(device));
}

thread_local! {
    /// Sub-pixel corners for this thread's `detect` calls (default off); see `set_corner_refinement`.
    static REFINE: std::cell::Cell<bool> = std::cell::Cell::new(false);
}
/// Also refine every marker's corners to sub-pixel precision (kernel K5) in this thread's `detect` calls:
/// `Marker::corners_refined`.  A wrapper-side option: the reference's `DetectorConfig` has no such field.
pub fn set_corner_refinement(on: bool) {
    REFINE.with(|r| r.set(on));
}

/// A rigid planar board (kernel K6): distinct `ids` and, per marker, its four corners `x0,y0..x3,y3` on the board plane
/// (z = 0, x right, y up, any length unit) in the order of `Marker::corners`.
#[derive(Clone, Debug)]
pub struct Board {
    pub ids: Vec<u64>,
    pub corners: Vec<[f32; 8]>,
}

impl Board {
    /// `cols` x `rows` square markers `separation` apart, centred on the origin; row 0 at the top, ids row-major from `first_id`.
    pub fn grid(cols: u32, rows: u32, marker_size: f32, separation: f32, first_id: u64) -> Board {
        let pitch = marker_size + separation;
        let w = cols as f32 * marker_size + (cols as f32 - 1.0) * separation;
        let h = rows as f32 * marker_size + (rows as f32 - 1.0) * separation;
        let (mut ids, mut corners) = (Vec::new(), Vec::new());
        for r in 0..rows {
            for c in 0..cols {
                let (x0, y0) = (-w / 2.0 + c as f32 * pitch, h / 2.0 - r as f32 * pitch);
                ids.push(first_id + (r * cols + c) as u64);
                corners.push([x0, y0, x0 + marker_size, y0, x0 + marker_size, y0 - marker_size, x0, y0 - marker_size]);
            }
        }
        Board { ids, corners }
    }
}

thread_local! {
    /// The board this thread's `detect` calls solve, with the intrinsics (`None`: undistorted at the frame size).
    static BOARD: std::cell::RefCell<Option<(Board, Option<pose::CameraIntrinsics>)>> = std::cell::RefCell::new(None);
}
/// Also solve the pose of `board` in every frame of this thread's `detect` calls (kernel K6): `Detection::board_pose`.
/// `k = None` normalises by the frame size, as `solve_with_undistorted_points`; `board = None` switches it off.  Like
/// `set_corner_refinement`, a wrapper-side option, set on each leased handle (the release resets it).
pub fn set_board(board: Option<Board>, k: Option<pose::CameraIntrinsics>) {
    BOARD.with(|b| *b.borrow_mut() = board.map(|b| (b, k)));
}

thread_local! {
    /// The lens distortion of this thread's pose and board intrinsics (`None`: the pinhole).
    static DISTORTION: std::cell::Cell<Option<sys::a3_camera_distortion>> = std::cell::Cell::new(None);
}
/// Give the intrinsics of this thread's board (`set_board`) a lens distortion, OpenCV's `k1 k2 p1 p2 k3`: the board pose
/// then solves from undistorted corners (kernel K7).  Needs intrinsics; `None` switches it off.  Like `set_board`, a
/// wrapper-side option, set on each leased handle (the release resets it).
pub fn set_distortion(d: Option<sys::a3_camera_distortion>) {
    DISTORTION.with(|x| x.set(d));
}

/// A handle out of the library's cache; goes back (warm) when dropped.
pub(crate) struct Lease(pub(crate) *mut sys::a3_detector);
impl Drop for Lease {
    fn drop(&mut self) {
        unsafe { sys::a3_detector_release(self.0) }
    }
}

/// What `detect_batch` should bring back besides the markers.
#[derive(Clone, Copy, PartialEq)]
pub enum Outputs {
    /// `Detection.markers` only: the records are assembled on the device and come back as one block.
    MarkersOnly,
    /// everything the reference's `Detection` holds: grey, candidates, homographies, markers.
    Full,
}

impl Detector {
    pub(crate) fn lease(&self) -> Lease {
        let cfg = sys::a3_config {
            threshold_window: self.config.threshold_window,
            contour_simplification_epsilon: self.config.contour_simplification_epsilon,
            min_side_length_factor: self.config.min_side_length_factor,
            min_corner_separation_factor: self.config.min_corner_separation_factor,
            homography_sample_size: self.config.homography_sample_size as u32,
            filter_high_bit_errors: self.config.filter_high_bit_errors as u8,
        };
        let mut h = ptr::null_mut();
        let st = unsafe { sys::a3_detector_acquire(&cfg, &self.dictionary.raw(), DEVICE.with(|d| d.get()), &mut h) };
        if st != sys::A3_OK {
            panic!("{}", last_error()); // threshold_window == 0 / epsilon <= 0 panic inside imageproc in the reference
        }
        if REFINE.with(|r| r.get()) {
            unsafe { sys::a3_detector_set_corner_refinement(h, sys::A3_CORNERS_REFINED) }; // the release resets it
        }
        BOARD.with(|b| {
            if let Some((board, k)) = &*b.borrow() {
                let raw = sys::a3_board { n_markers: board.ids.len() as u32, ids: board.ids.as_ptr(), corners: board.corners.as_ptr() as *const f32 };
                let (mode, kp) = match k {
                    Some(k) => (sys::A3_POSE_INTRINSICS, k as *const sys::a3_camera_intrinsics),
                    None => (sys::A3_POSE_UNDISTORTED, ptr::null()),
                };
                if unsafe { sys::a3_detector_set_board(h, &raw, mode, kp) } != sys::A3_OK {
                    unsafe { sys::a3_detector_release(h) };
                    panic!("{}", last_error());
                }
            }
        });
        if let Some(d) = DISTORTION.with(|x| x.get()) {
            if unsafe { sys::a3_detector_set_distortion(h, &d) } != sys::A3_OK {
                unsafe { sys::a3_detector_release(h) };
                panic!("{}", last_error());
            }
        }
        Lease(h)
    }

    /// reference `src/aruco.rs:52-121`.  The image's `Vec<u8>` is pageable: the library stages it through its pinned
    /// ring (`a3_stats.input_staged`), no copy is made here.
    pub fn detect(&self, image: DynamicImage) -> Detection {
        let (w, h) = (image.width(), image.height());
        let (buf, fmt, bpp): (Vec<u8>, i32, usize) = match image {
            DynamicImage::ImageLuma8(g) => (g.into_raw(), sys::A3_FMT_LUMA8, 1),
            DynamicImage::ImageRgba8(i) => (i.into_raw(), sys::A3_FMT_RGBA8, 4),
            DynamicImage::ImageRgb8(i) => (i.into_raw(), sys::A3_FMT_RGB8, 3),
            DynamicImage::ImageLumaA8(i) => (i.into_raw(), sys::A3_FMT_LUMAA8, 2),
            DynamicImage::ImageLuma16(i) => (bytes_of_u16(i.into_raw()), sys::A3_FMT_LUMA16, 2),
            DynamicImage::ImageLumaA16(i) => (bytes_of_u16(i.into_raw()), sys::A3_FMT_LUMAA16, 4),
            DynamicImage::ImageRgb16(i) => (bytes_of_u16(i.into_raw()), sys::A3_FMT_RGB16, 6),
            DynamicImage::ImageRgba16(i) => (bytes_of_u16(i.into_raw()), sys::A3_FMT_RGBA16, 8),
            // float variants: the reference's own host conversion (`image`'s into_luma8, src/aruco.rs:60), so grey is
            // identical by construction; the device then takes the Luma8 pass-through
            other => (other.into_luma8().into_raw(), sys::A3_FMT_LUMA8, 1),
        };
        self.detect_batch(&buf, fmt, 1, w, h, bpp, Outputs::Full).pop().unwrap()
    }

    /// `detect` for callers that only read `Detection.markers` (`examples/webcam_kamera.rs:59-69`): grey, candidates and
    /// homographies are left empty and never cross the bus.
    pub fn detect_markers(&self, frames: &[u8], fmt: i32, n: u32, w: u32, h: u32, bpp: usize) -> Vec<Vec<Marker>> {
        self.detect_batch(frames, fmt, n, w, h, bpp, Outputs::MarkersOnly).into_iter().map(|d| d.markers).collect()
    }

    /// `detect` over `n` equally sized, tightly packed frames (not in the reference).
    pub fn detect_batch(&self, frames: &[u8], fmt: i32, n: u32, w: u32, h: u32, bpp: usize, what: Outputs) -> Vec<Detection> {
        assert!(frames.len() >= n as usize * w as usize * h as usize * bpp);
        let hd = self.lease();
        let hs = self.config.homography_sample_size;
        let (px, np) = ((w as usize) * (h as usize), hs * hs);
        let full = what == Outputs::Full;
        let refine = REFINE.with(|r| r.get());
        let board = BOARD.with(|b| b.borrow().is_some());
        let (mut cap_m, mut cap_c) = (64 * n as usize + 1024, if full { 128 * n as usize + 2048 } else { 0 });
        loop {
            let mut markers: Vec<sys::a3_marker> = Vec::with_capacity(cap_m);
            let mut grey = vec![0u8; if full { n as usize * px } else { 0 }];
            let mut cands = vec![0u32; cap_c * 8];
            let mut cframe = vec![0u32; cap_c];
            let mut patches = vec![0u8; cap_c * np];
            let mut decs: Vec<sys::a3_decode> = Vec::with_capacity(cap_c);
            let mut refined = vec![0f32; if refine { cap_m * 8 } else { 0 }];
            let mut boards: Vec<sys::a3_board_pose> = Vec::with_capacity(if board { n as usize } else { 0 });
            let mut out = sys::a3_outputs {
                grey: grey.as_mut_ptr(), mask: ptr::null_mut(), candidates: cands.as_mut_ptr(), candidate_frame: cframe.as_mut_ptr(),
                homographies: patches.as_mut_ptr(), decodes: decs.as_mut_ptr(), cand_capacity: cap_c as u32, n_candidates: 0,
                frame_marker_offsets: ptr::null_mut(), marker_poses: ptr::null_mut(),
                marker_corners: if refine { refined.as_mut_ptr() } else { ptr::null_mut() },
                board_poses: if board { boards.as_mut_ptr() } else { ptr::null_mut() },
            };
            if !full {
                // markers only (plus their refined corners): no per-candidate output, so the device assembles the markers
                out = sys::a3_outputs { grey: ptr::null_mut(), candidates: ptr::null_mut(), candidate_frame: ptr::null_mut(),
                                        homographies: ptr::null_mut(), decodes: ptr::null_mut(), cand_capacity: 0, ..out };
            }
            let mut nm = 0u32;
            let st = unsafe {
                sys::a3_detect_batch(hd.0, frames.as_ptr() as *const _, fmt, sys::A3_MEM_HOST, n, w, h, w as usize * bpp,
                                     w as usize * bpp * h as usize, markers.as_mut_ptr(), cap_m as u32, &mut nm,
                                     if full || refine || board { &mut out } else { ptr::null_mut() }, ptr::null_mut())
            };
            if st == sys::A3_ERR_CAPACITY {
                cap_m = cap_m.max(nm as usize);
                if full {
                    cap_c = cap_c.max(out.n_candidates as usize);
                }
                continue;
            }
            if st != sys::A3_OK {
                panic!("{}", last_error());
            }
            let n_cand = if full { out.n_candidates as usize } else { 0 }; // a markers-only call reports the count only
            unsafe {
                markers.set_len(nm as usize);
                decs.set_len(n_cand);
                if board {
                    boards.set_len(n as usize);
                }
            }
            let mut dets: Vec<Detection> = (0..n).map(|_| Detection::default()).collect();
            if full {
                // one frame: the buffer becomes the GrayImage without a copy
                if n == 1 {
                    dets[0].grey = GrayImage::from_raw(w, h, grey);
                } else {
                    for f in 0..n as usize {
                        dets[f].grey = GrayImage::from_raw(w, h, grey[f * px..(f + 1) * px].to_vec());
                    }
                }
            }
            for k in 0..n_cand {
                let d = &mut dets[cframe[k] as usize];
                d.candidates.push((0..4).map(|j| Point::new(cands[k * 8 + 2 * j], cands[k * 8 + 2 * j + 1])).collect());
                d.homographies.push(if decs[k].homography_ok != 0 {
                    GrayImage::from_raw(hs as u32, hs as u32, patches[k * np..(k + 1) * np].to_vec()).unwrap()
                } else {
                    GrayImage::new(1, 1) // reference src/aruco.rs:256
                });
            }
            for (i, m) in markers.iter().enumerate() {
                let r = |k: usize| (refined[i * 8 + 2 * k], refined[i * 8 + 2 * k + 1]);
                dets[m.frame as usize].markers.push(Marker {
                    id: m.id as usize,
                    code: m.code,
                    corners: (0..4).map(|k| (m.corners[2 * k], m.corners[2 * k + 1])).collect(),
                    hamming_distance: m.hamming_distance,
                    corners_refined: if m.corners_refined != 0 { Some([r(0), r(1), r(2), r(3)]) } else { None },
                });
            }
            for (d, b) in dets.iter_mut().zip(boards.iter()) {
                d.board_pose = Some(pose::BoardPose::from_raw(b));
            }
            return dets;
        }
    }
}

/// 16-bit subpixels as the bytes the C ABI reads (native endianness, like `image`'s own `Vec<u16>`).
fn bytes_of_u16(v: Vec<u16>) -> Vec<u8> {
    let mut out = Vec::with_capacity(v.len() * 2);
    for s in v {
        out.extend_from_slice(&s.to_ne_bytes());
    }
    out
}

/// Drop-in for the reference's `pose` module (`src/pose.rs:52-81`): same function names, argument order and return
/// shape, plus the `Detector` whose device runs the solve (kernel K4).
pub mod pose {
    use super::{last_error, sys, Detector};

    /// reference `src/pose.rs:8-12`; `rotation` row-major (the reference's `na::Matrix3::new` argument order)
    #[derive(Clone, Debug)]
    pub struct MarkerPose {
        pub error: f32,
        pub rotation: [f32; 9],
        pub translation: [f32; 3],
    }

    impl Default for MarkerPose {
        /// reference `src/pose.rs:42-50`
        fn default() -> Self {
            Self { error: 1e31, rotation: [1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0], translation: [0.0; 3] }
        }
    }

    impl MarkerPose {
        fn raw(&self) -> sys::a3_pose {
            sys::a3_pose { error: self.error, rotation: self.rotation, translation: self.translation }
        }
        fn apply(&self, points: &Vec<(f32, f32, f32)>, inverse: i32) -> Vec<(f32, f32, f32)> {
            let flat: Vec<f32> = points.iter().flat_map(|p| [p.0, p.1, p.2]).collect();
            let mut out = vec![0f32; flat.len()];
            unsafe { sys::a3_pose_apply_transform(&self.raw(), flat.as_ptr(), points.len() as u32, inverse, out.as_mut_ptr()) };
            out.chunks(3).map(|c| (c[0], c[1], c[2])).collect()
        }
        /// reference `src/pose.rs:17-20`
        pub fn apply_transform_to_points(&self, points: &Vec<(f32, f32, f32)>) -> Vec<(f32, f32, f32)> {
            self.apply(points, 0)
        }
        /// reference `src/pose.rs:30-33`
        pub fn apply_inverse_transform_to_points(&self, points: &Vec<(f32, f32, f32)>) -> Vec<(f32, f32, f32)> {
            self.apply(points, 1)
        }
    }

    /// The pose of a `Board` in one frame (kernel K6): `best` has the smaller error (RMS reprojection distance over the used
    /// corners, normalised units), `alt` is the other branch of the planar ambiguity; `ok` is false when both failed or no
    /// board marker was seen.
    #[derive(Clone, Debug)]
    pub struct BoardPose {
        pub best: MarkerPose,
        pub alt: MarkerPose,
        pub n_markers: u32,
        pub ok: bool,
    }

    impl BoardPose {
        pub(crate) fn from_raw(b: &sys::a3_board_pose) -> BoardPose {
            let p = |q: &sys::a3_pose| MarkerPose { error: q.error, rotation: q.rotation, translation: q.translation };
            BoardPose { best: p(&b.best), alt: p(&b.alt), n_markers: b.n_markers, ok: b.ok != 0 }
        }
    }

    /// reference `src/pinhole.rs:11-18`
    pub type CameraIntrinsics = sys::a3_camera_intrinsics;

    /// `CameraIntrinsics::new`, reference `src/pinhole.rs:26-35`
    pub fn camera_intrinsics_new(w: u32, h: u32, fx: f32, fy: f32, px: Option<f32>, py: Option<f32>) -> CameraIntrinsics {
        let mut k = CameraIntrinsics::default();
        let (pxp, pyp) = (px.as_ref().map_or(std::ptr::null(), |v| v as *const f32), py.as_ref().map_or(std::ptr::null(), |v| v as *const f32));
        unsafe { sys::a3_camera_intrinsics_new(w, h, fx, fy, pxp, pyp, &mut k) };
        k
    }

    /// `CameraIntrinsics::new_from_fov_horizontal`, reference `src/pinhole.rs:37-60`
    pub fn camera_intrinsics_new_from_fov_horizontal(hfov: f32, sensor_width_mm: f32, rx: u32, ry: u32) -> CameraIntrinsics {
        let mut k = CameraIntrinsics::default();
        unsafe { sys::a3_camera_intrinsics_from_fov_horizontal(hfov, sensor_width_mm, rx, ry, &mut k) };
        k
    }

    fn pair(best: sys::a3_pose, alt: sys::a3_pose) -> (MarkerPose, MarkerPose) {
        let f = |p: sys::a3_pose| MarkerPose { error: p.error, rotation: p.rotation, translation: p.translation };
        (f(best), f(alt))
    }
    fn flat(points: &Vec<(u32, u32)>) -> [u32; 8] {
        assert_eq!(points.len(), 4);
        let mut c = [0u32; 8];
        for (i, p) in points.iter().enumerate() {
            c[2 * i] = p.0;
            c[2 * i + 1] = p.1;
        }
        c
    }
    const ZERO: sys::a3_pose = sys::a3_pose { error: 0.0, rotation: [0.0; 9], translation: [0.0; 3] };

    /// reference `src/pose.rs:52-55`
    pub fn solve_with_intrinsics(det: &Detector, image_points: &Vec<(u32, u32)>, marker_size_mm: f32, k: &CameraIntrinsics) -> (MarkerPose, MarkerPose) {
        let (c, mut b, mut a) = (flat(image_points), ZERO, ZERO);
        let st = unsafe { sys::a3_solve_with_intrinsics(det.lease().0, c.as_ptr(), 1, marker_size_mm, k, &mut b, &mut a) };
        if st != sys::A3_OK {
            panic!("{}", last_error());
        }
        pair(b, a)
    }

    /// reference `src/pose.rs:59-62`
    pub fn solve_with_undistorted_points(det: &Detector, image_points: &Vec<(u32, u32)>, marker_size_mm: f32, image_size: (u32, u32)) -> (MarkerPose, MarkerPose) {
        let (c, mut b, mut a) = (flat(image_points), ZERO, ZERO);
        let st = unsafe { sys::a3_solve_with_undistorted_points(det.lease().0, c.as_ptr(), 1, marker_size_mm, image_size.0, image_size.1, &mut b, &mut a) };
        if st != sys::A3_OK {
            panic!("{}", last_error());
        }
        pair(b, a)
    }

    /// reference `src/pose.rs:64-81`
    pub fn solve_with_normalized_points(det: &Detector, points: &Vec<(f32, f32)>, marker_size_mm: f32) -> (MarkerPose, MarkerPose) {
        assert_eq!(points.len(), 4);
        let c: Vec<f32> = points.iter().flat_map(|p| [p.0, p.1]).collect();
        let (mut b, mut a) = (ZERO, ZERO);
        let st = unsafe { sys::a3_solve_with_normalized_points(det.lease().0, c.as_ptr(), 1, marker_size_mm, &mut b, &mut a) };
        if st != sys::A3_OK {
            panic!("{}", last_error());
        }
        pair(b, a)
    }
}
