/*
 * aruco3_b200 — C ABI of the B200-native detection path.
 *
 * This is the boundary a Rust `-sys` crate (or any FFI) binds to replace the reference's
 * `Detector { config, dictionary }.detect(image) -> Detection`
 * (/root/reference/src/aruco.rs:46-52, re-exported at /root/reference/src/lib.rs:6-7).
 * The reference has no FFI of its own (pure Rust); every entry point below cites the Rust item it
 * stands in for.  Plain pointers and sizes only; no C++ or torch types.  See INTEGRATION.md for the
 * Rust-side binding.
 *
 * Conventions
 *   - every function returns a3_status (0 = ok) unless stated; a3_last_error() gives the text of the
 *     calling thread's last failure.  Nothing aborts or throws across this boundary (the reference
 *     panics instead: unknown dictionary name src/dictionaries.rs:144, threshold_window == 0 and
 *     epsilon <= 0 inside imageproc).
 *   - there is NO CPU fallback: the pixel and decode stages run on the CUDA device or fail with
 *     A3_ERR_CUDA.
 *   - frames are interleaved pixels, row-major (`image::RgbImage` / `RgbaImage` / `GrayImage` buffers and
 *     their 16-bit / LumaA siblings); `pitch` = bytes per row, `frame_stride` = bytes between frames.
 *   - a detector handle is thread-compatible, not thread-safe: one per (host thread, device).
 */
#ifndef ARUCO3_B200_H
#define ARUCO3_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t a3_status;
enum {
    A3_OK = 0,
    A3_ERR_INVALID_ARGUMENT = 1,   /* null pointer, zero size, threshold_window == 0, epsilon <= 0 ... */
    A3_ERR_UNKNOWN_DICTIONARY = 2, /* the reference panics here (src/dictionaries.rs:144) */
    A3_ERR_CUDA = 3,               /* no device / kernel or copy failed; text in a3_last_error() */
    A3_ERR_CAPACITY = 4,           /* caller-provided output array too small; counts are still returned */
    A3_ERR_UNSUPPORTED = 5,
    A3_ERR_OUT_OF_MEMORY = 6
};

/* DynamicImage variants accepted at the boundary (callers pass RgbImage.into() / RgbaImage.into(),
 * benches/detect_markers.rs:49, examples/webcam_kamera.rs:56); Luma8 passes through into_luma8. */
typedef enum {
    A3_FMT_RGB8 = 0,
    A3_FMT_RGBA8 = 1,
    A3_FMT_LUMA8 = 2,
    /* camera byte orders (SURVEY §8 f-4): the kernel reads B,G,R[,A] and applies the luma weights accordingly, which is
     * pixel for pixel the host swizzle into an RgbImage / RgbaImage that examples/webcam_kamera.rs:38-52 does before
     * detect.  `Detection.grey` etc. are those of the swizzled image. */
    A3_FMT_BGR8 = 3,
    A3_FMT_BGRA8 = 4,
    /* the other integer DynamicImage variants (SURVEY §8 f-4), converted on the device the way image 0.25's into_luma8
     * converts them (src/aruco.rs:60): LumaA drops alpha; 16-bit subpixels (native-endian u16, as in the crate's Vec<u16>)
     * go luma16 = (2126 R + 7152 G + 722 B) / 10000 in u32, then u8 = (luma16 + 128) / 257 (`FromPrimitive<u16> for u8`).
     * [RECALLED from the crate, not pinned by anything in the reference.]  Float variants: convert on the host. */
    A3_FMT_LUMAA8 = 5,
    A3_FMT_LUMA16 = 6,
    A3_FMT_LUMAA16 = 7,
    A3_FMT_RGB16 = 8,
    A3_FMT_RGBA16 = 9
} a3_format;
typedef enum { A3_MEM_HOST = 0, A3_MEM_DEVICE = 1 } a3_mem_kind;

/* DetectorConfig, field for field (src/aruco.rs:23-30); defaults src/aruco.rs:32-43. */
typedef struct a3_config {
    uint32_t threshold_window;              /* 7    */
    double contour_simplification_epsilon;  /* 0.05 */
    float min_side_length_factor;           /* 0.2  */
    float min_corner_separation_factor;     /* 0.1  */
    uint32_t homography_sample_size;        /* 49   */
    uint8_t filter_high_bit_errors;         /* 1    */
} a3_config;

/* ARDictionary (src/dictionaries.rs:22-28). `tau` is the effective tau (dictionaries.rs:124). */
typedef struct a3_dictionary {
    uint8_t num_bits;
    uint8_t tau;
    uint32_t n_codes;
    const uint64_t *codes; /* static storage inside the library */
} a3_dictionary;

/* Marker (src/aruco.rs:8-13) plus the frame / candidate it came from and the winning rotation.
 * corners = x0,y0,...,x3,y3 after rotate_left(rotation) (src/aruco.rs:97-103).
 * corners_refined: 1 when the detector refines corners (a3_detector_set_corner_refinement) and K5 refined this marker's,
 * 0 when refinement is off or fell back to the integer corners. */
typedef struct a3_marker {
    uint64_t id;
    uint64_t code;
    uint32_t corners[8];
    uint32_t frame;
    uint32_t candidate;
    uint8_t hamming_distance;
    uint8_t rotation;
    uint8_t corners_refined;
    uint8_t reserved[5];
} a3_marker;

/* One decoded candidate (every quad, accepted or not): the intermediates of
 * homography_to_code_permutations (src/aruco.rs:263-313) and of the match loop (src/aruco.rs:75-96). */
typedef struct a3_decode {
    uint64_t codes[4];     /* valid when has_codes */
    uint64_t id;           /* index into code_list of the best match (valid when has_codes) */
    uint8_t has_codes;     /* Some / None */
    uint8_t homography_ok; /* 0: the reference pushed a 1x1 image (src/aruco.rs:256) */
    uint8_t otsu;          /* otsu_level of the patch */
    uint8_t rotation;
    uint8_t hamming_distance;
    uint8_t accepted;      /* passed `found_any && (!filter || dist < tau)` (src/aruco.rs:96) */
    uint8_t reserved[2];
} a3_decode;

/* Counters + device-side stage times of the last call (CUDA events; host stage by steady_clock). */
typedef struct a3_stats {
    uint64_t n_frames, n_contours, n_contour_points, n_candidates_before_discard, n_candidates, n_markers;
    /* ms_h2d / ms_pixel_kernel / ms_contour_kernels / ms_mask_d2h (mask bits, or K3's quads) / ms_decode_kernel: sums of
     * CUDA-event intervals on the stream each runs on;
     * ms_host_quads: wall time the host stage was active (overlaps the others); ms_host_cpu: CPU time summed over frames */
    double ms_h2d, ms_pixel_kernel, ms_contour_kernels, ms_mask_d2h, ms_host_quads, ms_decode_kernel, ms_host_cpu, ms_total;
    uint32_t pixel_kernel_launches, decode_kernel_launches, host_threads, contour_kernel_launches;
    uint32_t host_fallback_frames; /* device contour stage: frames it handed back to the host stage */
    uint32_t pose_kernel_launches; /* K4 launches (a3_detector_set_pose) */
    /* one-shot route (device contour stage, one K3 launch per call): K3's second half, K2 and K4 queued without a host
     * synchronisation, sized from the previous call of the same geometry.  one_shot = 1 when this call's results came
     * from it; one_shot_retry = 1 when its sizes did not hold and the ordinary route finished the call instead. */
    uint32_t one_shot, one_shot_retry;
    /* pageable memory at the boundary: 1 when this call's host frames (input) / Detection.grey (output) were not page-locked and
     * went through the library's pinned staging rings (copy threads), 0 when the DMA used the caller's memory directly */
    uint32_t input_staged, output_staged;
    /* corner refinement (K5, a3_detector_set_corner_refinement): launches, and the sum of its CUDA-event intervals */
    uint32_t refine_kernel_launches;
    double ms_refine_kernel;
    /* board pose (K6, a3_detector_set_board): launches, and the sum of its CUDA-event intervals */
    uint32_t board_kernel_launches;
    double ms_board_kernel;
    /* corner undistortion (K7, a3_detector_set_distortion): launches, and the sum of its CUDA-event intervals */
    uint32_t undistort_kernel_launches;
    double ms_undistort_kernel;
} a3_stats;

/* MarkerPose (src/pose.rs:8-12): scene-from-marker transform in OpenCV chirality (+Z forward, +Y down, +X right).
 * rotation is row-major (m11 m12 m13 m21 ...).  Default (src/pose.rs:42-50): error 1e31, identity, zero. */
typedef struct a3_pose {
    float error;
    float rotation[9];
    float translation[3];
} a3_pose;

/* CameraIntrinsics, field for field (src/pinhole.rs:11-18). */
typedef struct a3_camera_intrinsics {
    uint32_t image_width, image_height;
    float focal_x, focal_y, principal_x, principal_y;
} a3_camera_intrinsics;

/* Lens distortion: OpenCV's five-coefficient Brown-Conrady model, in OpenCV's order (calibrateCamera's distCoeffs), on the
 * normalised coordinates of a3_camera_intrinsics: with r2 = x^2 + y^2, a normalised undistorted point (x, y) is seen at
 *     x (1 + k1 r2 + k2 r2^2 + k3 r2^3) + 2 p1 x y + p2 (r2 + 2 x^2),   y (1 + k1 r2 + k2 r2^2 + k3 r2^3) + p1 (r2 + 2 y^2) + 2 p2 x y.
 * Not part of the reference's pinhole model. */
typedef struct a3_camera_distortion {
    float k1, k2, p1, p2, k3;
} a3_camera_distortion;

/* How image corners become the normalised points the pose solver works on. */
enum {
    A3_POSE_OFF = 0,
    A3_POSE_UNDISTORTED = 1, /* solve_with_undistorted_points: (x / image_w, y / image_h), src/pose.rs:59-62 */
    A3_POSE_INTRINSICS = 2,  /* solve_with_intrinsics: CameraIntrinsics::unproject, src/pose.rs:52-55           */
    A3_POSE_NORMALIZED = 3   /* solve_with_normalized_points: f32 points used as they are, src/pose.rs:64-81   */
};

/* Optional per-call outputs of a3_detect_batch (all may be NULL). Host pointers; tightly packed. */
typedef struct a3_outputs {
    uint8_t *grey;              /* n*h*w      Detection.grey                              */
    uint8_t *mask;              /* n*h*w      the thresholded image (0/255)               */
    uint32_t *candidates;       /* cand_capacity*8  Detection.candidates, frame-major     */
    uint32_t *candidate_frame;  /* cand_capacity    frame index of each candidate         */
    uint8_t *homographies;      /* cand_capacity*hs*hs  Detection.homographies (zeros when !homography_ok) */
    a3_decode *decodes;         /* cand_capacity                                          */
    uint32_t cand_capacity;
    uint32_t n_candidates;      /* out */
    uint32_t *frame_marker_offsets; /* n+1: markers of frame f are [off[f], off[f+1]) (may be NULL) */
    a3_pose *marker_poses;      /* marker_capacity*2: [2i] best and [2i+1] alternative pose of markers[i]; filled when
                                 * the detector has a pose mode (a3_detector_set_pose), may be NULL */
    float *marker_corners;      /* marker_capacity*8: x0,y0..x3,y3 of markers[i] in f32, the order of a3_marker.corners; filled
                                 * when the detector refines corners (A3_CORNERS_REFINED), may be NULL.  Where a marker's
                                 * corners_refined is 0 these are its integer corners. */
    struct a3_board_pose *board_poses; /* n: the board's pose in each frame; filled when the detector has a board
                                        * (a3_detector_set_board), may be NULL */
} a3_outputs;

typedef struct a3_detector a3_detector;

/* ---- library ---- */
const char *a3_version(void);
const char *a3_last_error(void);
const char *a3_status_string(a3_status s);
int32_t a3_device_count(void); /* 0 when no CUDA device is usable */

/* ---- dictionaries (src/dictionaries.rs) ---- */
int32_t a3_dictionary_count(void);
const char *a3_dictionary_name(int32_t index);                                    /* get_dictionary_names :147-149 */
a3_status a3_dictionary_by_name(const char *name, a3_dictionary *out);             /* new_from_named_dict :140-145  */
uint8_t a3_dictionary_mark_size(const a3_dictionary *d);                           /* get_mark_size :154-156        */
uint8_t a3_hamming_distance(uint64_t a, uint64_t b);                               /* src/lib.rs:11-21              */
void a3_find_nearest(const a3_dictionary *d, uint64_t bits, uint64_t *index, uint8_t *dist); /* :160-196            */
int32_t a3_try_find_nearest(const a3_dictionary *d, uint64_t bits, uint64_t *index, uint8_t *dist); /* :200-207      */
uint8_t a3_make_binary_image(const a3_dictionary *d, uint64_t marker_id, uint8_t *bits, uint32_t capacity,
                             uint32_t *n_bits);                                    /* make_binary_image :212-232    */

/* ---- detector ---- */
void a3_config_default(a3_config *cfg);                                            /* Default, src/aruco.rs:32-43   */
a3_status a3_detector_create(const a3_config *cfg, const a3_dictionary *dict, int32_t device, a3_detector **out);
void a3_detector_destroy(a3_detector *det);
/* Handle cache for bindings whose `Detector` is plain data built with a struct literal, as in the reference
 * (src/aruco.rs:46-49, benches/detect_markers.rs:17-20, README.md:14-17), and so cannot own a handle: bracket each
 * detect with acquire / release.  acquire returns an idle cached handle created with exactly this config, dictionary
 * (same `codes` pointer, sizes and tau) and device — warm: streams, device / pinned buffers and the one-shot history
 * survive — and creates one only when none is idle; release puts it back (pose / contour / corner mode, tuning reset to the
 * defaults) and never blocks on the GPU.  A handle is held by one caller at a time; the cache itself is thread-safe and
 * keeps at most 16 idle handles (oldest destroyed).  a3_detector_cache_clear destroys the idle ones (call before unloading).
 * a3_detector_create_count: successful a3_detector_create calls of this process so far (diagnostic: a per-frame loop over
 * one Detector must not make it grow). */
a3_status a3_detector_acquire(const a3_config *cfg, const a3_dictionary *dict, int32_t device, a3_detector **out);
void a3_detector_release(a3_detector *det);
void a3_detector_cache_clear(void);
uint64_t a3_detector_create_count(void);
/* number of host threads used for the contour / quad stage (default: all cores, capped at 64) */
a3_status a3_detector_set_host_threads(a3_detector *det, uint32_t threads);

/* Where find_contours + the quad filters (src/aruco.rs:64-69) run.  A3_CONTOURS_DEVICE (default): kernel K3; frames
 * it cannot prove identical to the sequential algorithm (a border whose natural start is barred by the reference's
 * `x > 0` guard, > 1024 quads, pathological polygon recursion) are redone by the host stage, so results never depend on
 * the mode.  A3_CONTOURS_HOST: always the host stage (C++ threads), as BASELINE.json's north_star describes it. */
enum { A3_CONTOURS_HOST = 0, A3_CONTOURS_DEVICE = 1 };
a3_status a3_detector_set_contour_mode(a3_detector *det, uint32_t mode);

/* Sub-pixel marker corners (kernel K5, queued behind the decode kernel).  A3_CORNERS_INTEGER (default): the corners are
 * the contour pixels the reference returns, and nothing else runs.  A3_CORNERS_REFINED: a3_detect_batch also fits a line
 * to the grey image's edge profile along each side of every marker and returns the four intersections in
 * a3_outputs.marker_corners, in the pixel-centre convention (grey pixel (x, y) is the point (x, y)); a3_marker.corners
 * stay the integer corners.  Where the fit is not trustworthy (too few edge samples, near-parallel sides, a quad that is
 * not convex and clockwise, a corner moved by more than a quarter of the shortest side) the marker keeps its integer
 * corners and corners_refined = 0.  With a pose mode set, K4 solves from these corners.  Not a field of the reference's
 * DetectorConfig; a3_detector_release resets it. */
enum { A3_CORNERS_INTEGER = 0, A3_CORNERS_REFINED = 1 };
a3_status a3_detector_set_corner_refinement(a3_detector *det, uint32_t mode);

/* Launch-shape knobs of the pixel kernel (benchmark sweeps and tests; results never depend on them). 0 = automatic. */
typedef struct a3_k1_tuning {
    uint32_t strip_cols;    /* generic kernel: output columns per CTA strip */
    uint32_t seg_rows;      /* output rows per row segment (both kernels) */
    uint32_t force_no_tma;  /* generic kernel: plain loads instead of bulk copies */
    uint32_t force_generic; /* never take the warp-strip kernel (k1_strips.cu) */
    uint32_t chunk_frames;  /* a3_detect_batch: frames per front-end chunk (copy / event granularity) */
    uint32_t reserved[3];
} a3_k1_tuning;
a3_status a3_detector_set_k1_tuning(a3_detector *det, const a3_k1_tuning *tuning); /* NULL restores the defaults */

/* Detector::detect over a batch of n equally sized frames (src/aruco.rs:52-121 per frame).
 * markers are written frame-major, in candidate order within a frame (the order of Detection.markers).
 * Returns A3_ERR_CAPACITY (with *n_markers = the number found) when marker_capacity is too small. */
a3_status a3_detect_batch(a3_detector *det, const void *frames, a3_format format, a3_mem_kind mem, uint32_t n,
                          uint32_t width, uint32_t height, size_t pitch, size_t frame_stride, a3_marker *markers,
                          uint32_t marker_capacity, uint32_t *n_markers, a3_outputs *outputs, a3_stats *stats);

/* ---- stage entry points (parity probes; the same kernels a3_detect_batch launches) ---- */

/* into_luma8 + adaptive_threshold (src/aruco.rs:60-61). All pointers are DEVICE pointers when
 * mem == A3_MEM_DEVICE (no copies, launches on `cuda_stream`, a cudaStream_t or NULL, and returns
 * without synchronising), HOST pointers otherwise (copies in and out, synchronous).
 * grey / mask: n*h*w bytes each; mask_bits: n*h*ceil(w/32) little-endian words, bit (x&31) of word x>>5.
 * Any of the three outputs may be NULL. */
a3_status a3_gray_threshold_batch(a3_detector *det, const void *frames, a3_format format, a3_mem_kind mem,
                                  uint32_t n, uint32_t width, uint32_t height, size_t pitch, size_t frame_stride,
                                  uint8_t *grey, uint8_t *mask, uint32_t *mask_bits, void *cuda_stream);

/* find_contours + contours_to_candidates + enforce_clockwise_corners + discard_too_near
 * (src/aruco.rs:64-69) on one host mask (0 / non-zero bytes). Host stage of the product. */
a3_status a3_quads_from_mask(const a3_config *cfg, const uint8_t *mask, uint32_t width, uint32_t height,
                             uint32_t *quads, uint32_t quad_capacity, uint32_t *n_quads, a3_stats *stats);

/* The same stage on the device (kernel K3) for n host masks of w*h bytes each (0 / non-zero), as a parity probe:
 * quads n*quad_capacity*8, counts n, flags n (non-zero: K3 hands this frame back to the host stage and its quads are
 * not meaningful), contours n and points n (borders followed and their total points; may be NULL). */
a3_status a3_quads_from_masks_device(a3_detector *det, const uint8_t *masks, uint32_t n, uint32_t width, uint32_t height,
                                     uint32_t *quads, uint32_t quad_capacity, uint32_t *counts, uint32_t *flags,
                                     uint32_t *contours, uint64_t *points);

/* extract_homographies + homography_to_code_permutations + the match loop (src/aruco.rs:72-113) for
 * n_quads candidates over grey frames. HOST pointers; quads n_quads*8, quad_frame n_quads (frame index of
 * each quad; NULL = all frame 0); patches (optional) n_quads*hs*hs. */
a3_status a3_decode_candidates(a3_detector *det, const uint8_t *grey, uint32_t n_frames, uint32_t width,
                               uint32_t height, const uint32_t *quads, const uint32_t *quad_frame, uint32_t n_quads,
                               a3_decode *decodes, uint8_t *patches);

/* The corner refinement (kernel K5) for n sets of four integer corners over grey frames, as a probe.  HOST pointers;
 * corners n*8 (x0,y0..x3,y3, screen-clockwise: a3_marker.corners), corner_frame n (NULL = all frame 0); refined n*8 f32
 * in the same corner order, ok n (1 refined, 0 fell back to the integer corners). */
a3_status a3_refine_corners(a3_detector *det, const uint8_t *grey, uint32_t n_frames, uint32_t width, uint32_t height,
                            const uint32_t *corners, const uint32_t *corner_frame, uint32_t n, float *refined, uint8_t *ok);

/* ---- pose (src/pose.rs, src/pinhole.rs): the step after detect in the reference's examples ---- */

/* Make a3_detect_batch also solve the pose pair of every marker on the device (kernel K4, queued behind K2) into
 * a3_outputs.marker_poses.  mode: A3_POSE_OFF, A3_POSE_UNDISTORTED (image size = the frame size, as
 * examples/webcam_kamera.rs:68 calls it) or A3_POSE_INTRINSICS (k required, examples/macroquad_detect.rs:150). */
a3_status a3_detector_set_pose(a3_detector *det, uint32_t mode, float marker_size_mm, const a3_camera_intrinsics *k);

/* pose::solve_with_intrinsics / solve_with_undistorted_points / solve_with_normalized_points over n markers at once
 * (src/pose.rs:52-81).  HOST pointers; corners n*8 u32 (x0,y0..x3,y3, clockwise from the marker's top-left, i.e.
 * a3_marker.corners), points n*8 f32; best / alt: n poses each, best has the smaller reprojection error. */
a3_status a3_solve_with_intrinsics(a3_detector *det, const uint32_t *corners, uint32_t n, float marker_size_mm,
                                   const a3_camera_intrinsics *k, a3_pose *best, a3_pose *alt);
a3_status a3_solve_with_undistorted_points(a3_detector *det, const uint32_t *corners, uint32_t n, float marker_size_mm,
                                           uint32_t image_width, uint32_t image_height, a3_pose *best, a3_pose *alt);
a3_status a3_solve_with_normalized_points(a3_detector *det, const float *points, uint32_t n, float marker_size_mm,
                                          a3_pose *best, a3_pose *alt);

/* ---- board pose: one pose per frame from every visible marker of a planar board (kernel K6) ---- */

/* A rigid planar board: n_markers (1..1024) distinct ids below the dictionary's code count, and for each marker its four
 * corners (x, y) on the board plane (z = 0), in any length unit, in the order of a3_marker.corners (the marker's own TL, TR,
 * BR, BL).  x to the right and y up on the board's face: one marker of side L centred at the origin has TL = (-L/2, +L/2),
 * the square the single-marker solve uses. */
typedef struct a3_board {
    uint32_t n_markers;
    const uint64_t *ids;   /* n_markers */
    const float *corners;  /* n_markers*8: x0,y0..x3,y3 */
} a3_board;

/* The board's pose in one frame: the map from board points (x, y, 0) to camera coordinates, in the chirality and row-major
 * layout of a3_pose.  best has the smaller error, alt is the other branch of the planar ambiguity.  error = RMS reprojection
 * distance over the used corners in normalised units (unlike a3_pose.error of one marker, a sum over its 4 corners).  A
 * branch that failed (non-finite value, singular system, translation z <= 0) is a3_pose_default (error 1e31).  n_markers =
 * markers the solve used; ok = 0 when both branches failed or no board marker was seen (then both are the default). */
typedef struct a3_board_pose {
    a3_pose best, alt;
    uint32_t n_markers;
    uint8_t ok;
    uint8_t reserved[3];
} a3_board_pose;

/* Make a3_detect_batch also solve the board's pose in every frame (kernel K6, queued behind the decode kernel and K5) into
 * a3_outputs.board_poses.  Every accepted marker whose id is on the board contributes its four corners, in candidate
 * order: K5's corners when the detector refines corners (A3_CORNERS_REFINED), else the integer corners.  An id detected more
 * than once in a frame is skipped there.  mode: A3_POSE_UNDISTORTED (image size = the frame size) or A3_POSE_INTRINSICS (k
 * required).  The board is copied to the device.  board = NULL switches it off; a3_detector_release resets it.  Invalid: duplicate ids, an
 * id >= the dictionary's code count, 0 or more than 1024 markers, a non-finite coordinate, mode OFF or NORMALIZED. */
a3_status a3_detector_set_board(a3_detector *det, const a3_board *board, uint32_t mode, const a3_camera_intrinsics *k);

/* The board solve (kernel K6) as a probe, with the detector's board and mode, over n markers: ids n, corners n*8 f32 (the
 * order of a3_marker.corners, image pixels), frame n (non-decreasing frame index of each marker, < n_frames; NULL = all
 * frame 0).  HOST pointers; out: n_frames board poses.  image_w / image_h: the frame size (A3_POSE_UNDISTORTED). */
a3_status a3_solve_board(a3_detector *det, const uint64_t *ids, const float *corners, const uint32_t *frame, uint32_t n,
                         uint32_t n_frames, uint32_t image_w, uint32_t image_h, a3_board_pose *out);

/* ---- lens distortion: undistorted marker corners for the pose kernels (kernel K7) ---- */

/* Give the detector's intrinsics a lens distortion.  It applies exactly where A3_POSE_INTRINSICS is used: the marker pose
 * (a3_detector_set_pose), the board pose (a3_detector_set_board) and a3_solve_board.  a3_detect_batch then undistorts every
 * corner those kernels read once (kernel K7, queued behind the decode kernel and K5: K5's corners when the detector refines
 * corners, else the integer corners), by Newton's method on the model (k7_undistort_spec.h), and K4 / K6 solve from the
 * normalised undistorted points.  A marker with a corner that does not undistort (the model folds there, no convergence, a
 * non-finite value) gets two a3_pose_default poses and is left out of the board solve as if it had not been detected.
 * d = NULL, or all five coefficients zero, switches it off: nothing more runs.  a3_detector_release resets it.  Invalid:
 * a non-finite coefficient; distortion together with an A3_POSE_UNDISTORTED or A3_POSE_NORMALIZED pose or board mode,
 * whichever of the setters is called last.  a3_solve_with_intrinsics stays the reference's pinhole solve. */
a3_status a3_detector_set_distortion(a3_detector *det, const a3_camera_distortion *d);

/* The undistortion (K7's device function) as a probe.  HOST pointers; points n*2 pixel coordinates (pixel-centre
 * convention), out n*2 normalised undistorted coordinates, ok n (1 converged, 0 failed).  Followed by
 * a3_solve_with_normalized_points, this is what the marker pose with distortion computes. */
a3_status a3_undistort_points(a3_detector *det, const float *points, uint32_t n, const a3_camera_intrinsics *k,
                              const a3_camera_distortion *d, float *out, uint8_t *ok);

/* Plain host helpers (constructors and one-point conversions; nothing here is on the hot path). */
void a3_pose_default(a3_pose *p);                                                   /* src/pose.rs:42-50        */
/* apply_transform_to_points / apply_inverse_transform_to_points (src/pose.rs:17-39); points and out: n*3 f32 */
void a3_pose_apply_transform(const a3_pose *p, const float *points, uint32_t n, int32_t inverse, float *out);
/* CameraIntrinsics::new (src/pinhole.rs:26-35); principal_x / principal_y may be NULL (= image centre) */
void a3_camera_intrinsics_new(uint32_t image_width, uint32_t image_height, float focal_x, float focal_y,
                              const float *principal_x, const float *principal_y, a3_camera_intrinsics *out);
/* CameraIntrinsics::new_from_fov_horizontal (src/pinhole.rs:37-60) */
void a3_camera_intrinsics_from_fov_horizontal(float horizontal_fov_radians, float sensor_width_mm, uint32_t resolution_x,
                                              uint32_t resolution_y, a3_camera_intrinsics *out);
void a3_camera_project(const a3_camera_intrinsics *k, float x, float y, float z, float out[3]);        /* :65-71 */
int32_t a3_camera_project_culled(const a3_camera_intrinsics *k, float x, float y, float z, float out[2]); /* :76-84 */
void a3_camera_unproject(const a3_camera_intrinsics *k, float x, float y, float out[2]);               /* :88-93 */

#ifdef __cplusplus
}
#endif
#endif /* ARUCO3_B200_H */
