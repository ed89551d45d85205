// Internal declarations shared by the CUDA kernels, the host quad stage and the C ABI.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <memory>
#include <string>
#include <vector>

#include "../../include/aruco3_b200.h"

namespace a3 {

// ---- pixel formats (a3_format) ----------------------------------------------------------------------------
__host__ __device__ constexpr int fmt_bpp(int f) {
    return (f == A3_FMT_RGB8 || f == A3_FMT_BGR8) ? 3
           : (f == A3_FMT_RGBA8 || f == A3_FMT_BGRA8 || f == A3_FMT_LUMAA16) ? 4
           : (f == A3_FMT_LUMAA8 || f == A3_FMT_LUMA16) ? 2
           : f == A3_FMT_RGB16 ? 6
           : f == A3_FMT_RGBA16 ? 8 : 1;
}
__host__ __device__ constexpr bool fmt_bgr(int f) { return f == A3_FMT_BGR8 || f == A3_FMT_BGRA8; }  // byte 0 is blue
__host__ __device__ constexpr bool fmt_valid(int f) { return f >= 0 && f <= A3_FMT_RGBA16; }
// LumaA8 and the 16-bit variants: brought to Luma8 by k0_to_luma8 first, K1 then takes the Luma8 pass-through
__host__ __device__ constexpr bool fmt_wide(int f) { return f >= A3_FMT_LUMAA8 && f <= A3_FMT_RGBA16; }

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const std::string &msg);
a3_status fail(a3_status s, const std::string &msg);
a3_status cuda_fail(cudaError_t e, const char *what);
#define A3_CUDA(expr)                                                    \
    do {                                                                 \
        cudaError_t e__ = (expr);                                        \
        if (e__ != cudaSuccess) return ::a3::cuda_fail(e__, #expr);      \
    } while (0)

// Device / pinned buffers that only grow; freed with their owner (the owner's device must be current then).
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
};
template <typename T>
struct PinBuf {
    T *p = nullptr;
    size_t cap = 0;
    PinBuf() = default;
    PinBuf(const PinBuf &) = delete;
    PinBuf &operator=(const PinBuf &) = delete;
    ~PinBuf() { if (p) cudaFreeHost(p); }
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaHostAlloc(&p, n * sizeof(T), cudaHostAllocDefault);
        if (e == cudaSuccess) cap = n;
        return e;
    }
};

// ---- K1: fused into_luma8 + adaptive_threshold (k1_threshold.cu) -------------------------------
struct K1Params {
    const uint8_t *src;   // device, n frames
    int format;           // a3_format
    uint32_t n, w, h;
    size_t pitch, frame_stride;
    uint8_t *grey;        // device n*h*w or null
    uint8_t *mask;        // device n*h*w or null
    uint32_t *bits;       // device 1-bit mask or null: word of pixel (x, y) of frame f =
                          //   bits[f * bits_frame_words + y * bits_row_words + (x >> 5) * bits_col_words]
    uint32_t radius;      // threshold_window
    size_t bits_row_words = 0;    // 0 = ceil(w/32) (row-major, tightly packed rows)
    size_t bits_col_words = 0;    // 0 = 1
    size_t bits_frame_words = 0;  // 0 = h * ceil(w/32)
};
struct K1Tuning {
    uint32_t strip_cols;  // generic kernel: core columns per strip (multiple of 32); 0 = auto
    uint32_t seg_rows;    // output rows per row segment; 0 = auto
    int force_no_tma;     // generic kernel: 1 = plain loads even when the bulk-copy path is legal (tests)
    int force_generic;    // 1 = never take the warp-strip kernel (k1_strips.cu)
};
struct K1LaunchInfo {
    uint32_t grid, block, smem_bytes, strips, segs, strip_cols, seg_rows;
    int tma, specialised_radius;
};
cudaError_t k1_gray_threshold(const K1Params &p, const K1Tuning *tuning, cudaStream_t stream, K1LaunchInfo *info);
// K0: image 0.25's into_luma8 for LumaA8 / Luma16 / LumaA16 / Rgb16 / Rgba16 frames -> Luma8 frames (dst_pitch bytes per row)
cudaError_t k0_to_luma8(const uint8_t *src, int format, uint32_t n, uint32_t w, uint32_t h, size_t pitch, size_t frame_stride, uint8_t *dst,
                        size_t dst_pitch, size_t dst_frame_stride, cudaStream_t stream);
// warp-strip fast path (k1_strips.cu): radius 7, 16-byte aligned rows, width % 4 == 0
bool k1_strips_eligible(const K1Params &p);
cudaError_t k1_strips(const K1Params &p, const K1Tuning *tuning, cudaStream_t stream, K1LaunchInfo *info);

// ---- K2: per-candidate homography + warp + otsu + resize + bits + dictionary match (k2_decode.cu) ----
struct K2Params {
    const uint8_t *grey;        // device, n_frames*h*w
    uint32_t w, h;
    const uint32_t *quads;      // device n_quads*8
    const uint32_t *quad_frame; // device n_quads or null (all frame 0)
    uint32_t n_quads;
    const uint32_t *n_quads_dev = nullptr;  // device, optional: the real number of quads (<= n_quads, which then only sizes the launch)
    uint32_t *queue = nullptr;  // device, optional, zero at launch: warps take quads from this counter instead of a fixed stride, so
                                // the last, partial wave of quads spreads over all resident warps
    uint32_t *accept_counts = nullptr;  // device, optional, zero at launch: [q >> 10] += 1 for every accepted quad q (marker assembly)
    uint32_t patch_size;        // homography_sample_size
    uint32_t mark_size;         // get_mark_size()
    const uint64_t *codes;      // device dictionary
    uint32_t n_codes;
    uint32_t tau;
    int filter_high_bit_errors;
    const float *resize_w;      // device: resize tap weights (see ResizeTaps)
    const int *resize_meta;     // device: per output index {left, count}, then for the 1x1 source
    a3_decode *decodes;         // device n_quads
    uint8_t *patches;           // device n_quads*ps*ps or null
};
cudaError_t k2_decode(const K2Params &p, cudaStream_t stream);
size_t k2_smem_bytes(uint32_t patch_size, uint32_t mark_size, uint32_t n_codes);
// whether K2 can decode with this homography_sample_size / dictionary at all (at least one patch + the dictionary in shared memory)
bool k2_supported(uint32_t patch_size, uint32_t mark_size, uint32_t n_codes);

// image::imageops::resize(Triangle) tap table for n_in -> n_out, computed on the host in f32 with the
// reference's expression order (SURVEY A.10).  weights[o*max_taps + i], meta[2*o] = left, meta[2*o+1] = count.
struct ResizeTaps {
    uint32_t n_in, n_out, max_taps;
    std::vector<float> weights;
    std::vector<int> meta;
};
ResizeTaps make_resize_taps(uint32_t n_in, uint32_t n_out);

// ---- K3: border following + quad filters on the device (k3_contours.cu) ----------------------------------------
// Guarded bit planes, COLUMN-major: per frame ceil(w/32) + 2 word columns of Hp = h + 2 words, all guard words zero;
// pixel (x, y) is bit x & 31 of word ((x >> 5) + 1) * Hp + (y + 1).  Vertically adjacent pixels are adjacent words, so a
// border walk stays inside a 32-byte sector for 8 rows and inside a word for 32 columns.  K1 writes straight into this
// layout (bits_col_words = Hp, bits_row_words = 1, bits_frame_words = (ceil(w/32) + 2) * Hp, bits = plane + Hp + 1).
struct K3Params {
    const uint32_t *planes;       // device, n guarded planes
    uint32_t n, w, h;
    double eps_factor;            // contour_simplification_epsilon
    uint32_t min_edge_length;     // (min(w,h) as f32 * min_side_length_factor) as u32
    float min_corner_separation;  // min(w,h) as f32 * min_corner_separation_factor
    uint32_t min_points;          // borders shorter than this cannot pass the edge test (see host_quads.cpp)
    uint32_t quad_cap;            // quads per frame the output can hold
    uint32_t *quads;              // device out: n * quad_cap * 8
    uint32_t *quad_counts;        // device out: n (after discard_too_near)
    uint32_t *before_discard;     // device out: n
    uint32_t *frame_flags;        // device out: n; non-zero = redo this frame with the host stage
    uint32_t *frame_contours;     // device out: n (borders followed) or null
    unsigned long long *frame_points;  // device out: n or null
};
struct K3Workspace {
    struct Impl;
    std::unique_ptr<Impl> impl;
    K3Workspace();
    ~K3Workspace();
};
cudaError_t k3_quads(K3Workspace &ws, const K3Params &p, cudaStream_t stream);  // k3_begin + k3_finish
// The two halves, so that several batches (each with its own workspace and stream) can be in flight: k3_begin only
// enqueues; k3_finish synchronises the stream once (buffer sizing) and enqueues the rest.
cudaError_t k3_begin(K3Workspace &ws, const K3Params &p, cudaStream_t stream);
cudaError_t k3_finish(K3Workspace &ws, const K3Params &p, cudaStream_t stream);
// k3_finish without the synchronisation: launches sized from the previous call of this geometry, real sizes read on the
// device.  After the caller's own synchronisation of the stream k3_speculation_held() says whether the sizes fitted; if
// not (or if *speculated came back false), k3_finish does the second half exactly.
cudaError_t k3_finish_speculative(K3Workspace &ws, const K3Params &p, cudaStream_t stream, bool *speculated);
bool k3_speculation_held(K3Workspace &ws, const K3Params &p);
const uint32_t *k3_speculation_failed_flag(K3Workspace &ws);  // device word, non-zero = the speculative finish in flight gave up

// ---- K4: marker pose from four corners (k4_pose.cu) --------------------------------------------------------------
struct K4Params {
    uint32_t mode;               // A3_POSE_UNDISTORTED / A3_POSE_INTRINSICS (corners) or A3_POSE_NORMALIZED (points)
    const float *points;         // device n*8 (NORMALIZED)
    const uint32_t *corners;     // device n*8 (other modes)
    const float *corners_f32 = nullptr;  // device n*8 or null: f32 corners (K5's), already rotate_left(rotation), read instead of `corners`
    const uint8_t *points_ok = nullptr;  // device n or null (NORMALIZED): K7's flags; an item with 0 gets two default poses
    const a3_decode *decodes;    // device n or null; when set: only accepted items, corners.rotate_left(rotation)
    uint32_t n;
    const uint32_t *n_dev = nullptr;  // device, optional: the real number of items (<= n, which then only sizes the launch)
    float marker_size;
    uint32_t image_w, image_h;   // UNDISTORTED
    a3_camera_intrinsics k;      // INTRINSICS
    a3_pose *poses;              // device n*2: [2i] best, [2i+1] alternative
};
cudaError_t k4_pose(const K4Params &p, cudaStream_t stream);

// ---- K5: sub-pixel marker corners (k5_corners.cu; specification oracle/a3ref_refine.c) ---------------------------------
struct K5Params {
    const uint8_t *grey;         // device, n_frames*h*w
    uint32_t w, h;
    const uint32_t *quads;       // device n*8 integer corners, screen-clockwise
    const uint32_t *quad_frame;  // device n or null (all frame 0)
    const a3_decode *decodes;    // device n or null; when set: only accepted items, output corners.rotate_left(rotation)
    uint32_t n;
    const uint32_t *n_dev = nullptr;  // device, optional: the real number of items (<= n, which then only sizes the launch)
    float *corners;              // device out n*8: refined corners, or the integer corners as f32 where it fell back
    uint8_t *ok;                 // device out n: 1 refined, 0 fell back
};
cudaError_t k5_corners(const K5Params &p, cudaStream_t stream);

// ---- K6: one pose per frame from every visible marker of a planar board (k6_board.cu; specification oracle/a3ref_board.c)
struct K6Params {
    const a3_decode *decodes = nullptr;     // device n or null; when set: accepted items only, id from the record, integer corners
                                            //   rotate_left(rotation)
    const uint64_t *ids = nullptr;          // device n: the items' ids when decodes is null (probe; every item counts)
    const uint32_t *quads = nullptr;        // device n*8 integer corners (screen order), read when corners_f32 is null
    const float *corners_f32 = nullptr;     // device n*8 or null: f32 corners already in marker order (K5's, or the probe's)
    const float *norm = nullptr;            // device n*8 or null: K7's normalised undistorted corners (K7's layout), read instead of
                                            //   both corner sources and of the mode's normalisation
    const uint8_t *norm_ok = nullptr;       // device n, with norm: K7's flags; an item with 0 is left out as if not detected
    const uint32_t *offsets = nullptr;      // device n_frames + 1: items of frame f are [offsets[f], offsets[f + 1])
    const uint32_t *skip = nullptr;         // device flag or null: non-zero = the launch writes nothing (a one-shot route that did not hold)
    uint32_t n_frames = 0;
    const uint16_t *slots = nullptr;        // device n_codes: board slot of each id, A3_K6_NO_SLOT when the id is not on the board
    uint32_t n_codes = 0;
    const float *board = nullptr;           // device n_board*8: board points of each slot, the order of a3_marker.corners
    uint32_t n_board = 0;
    uint32_t mode = 0;                      // A3_POSE_UNDISTORTED / A3_POSE_INTRINSICS
    uint32_t image_w = 0, image_h = 0;
    a3_camera_intrinsics k{};
    a3_board_pose *out = nullptr;           // device n_frames
};
cudaError_t k6_board(const K6Params &p, cudaStream_t stream);

// ---- K7: lens undistortion of marker corners (k7_undistort.cu; specification k7_undistort_spec.h, oracle/a3ref_distort.c)
struct K7Params {
    const uint32_t *quads = nullptr;        // device n*8 integer corners (screen order), read when corners_f32 is null
    const float *corners_f32 = nullptr;     // device n*8 or null: f32 corners already in marker order (K5's, or the probe's)
    const a3_decode *decodes = nullptr;     // device n or null; when set: accepted items only, rotation from the record
    uint32_t n = 0;
    const uint32_t *n_dev = nullptr;        // device, optional: the real number of items (<= n, which then only sizes the launch)
    a3_camera_intrinsics k{};
    a3_camera_distortion dist{};
    float *out = nullptr;                   // device out n*8: marker corner c at [8 i + 2 ((c + rotation) & 3)], the slot K4's
                                            //   A3_POSE_NORMALIZED read and K6 take it from
    uint8_t *ok = nullptr;                  // device out n: 1 when all four corners undistorted
};
cudaError_t k7_undistort(const K7Params &p, cudaStream_t stream);
// the probe: n points (x, y) -> n normalised undistorted points and their flags
cudaError_t k7_undistort_points(const float *pts, uint32_t n, const a3_camera_intrinsics &k, const a3_camera_distortion &dist, float *out,
                                uint8_t *ok, cudaStream_t stream);

// ---- host quad stage (host_quads.cpp) ---------------------------------------------------------------
struct QuadStats {
    uint64_t n_contours = 0, n_contour_points = 0, n_before_discard = 0;
};
// mask bits: h rows of `words_per_row` little-endian 32-bit words (bit x&31 of word x>>5), zero beyond w.
// Appends 8 uint32 per surviving quad (x0,y0..x3,y3) to `quads`.
void quads_from_bits(const uint32_t *bits, uint32_t words_per_row, uint32_t w, uint32_t h, const a3_config &cfg,
                     std::vector<uint32_t> &quads, QuadStats *stats, size_t row_stride_words = 0);
void bits_from_mask(const uint8_t *mask, uint32_t w, uint32_t h, std::vector<uint32_t> &bits, uint32_t *words_per_row);

// ---- dictionaries (a3_dictionary.cpp) ---------------------------------------------------------------
uint8_t mark_size_of(uint8_t num_bits);

}  // namespace a3
