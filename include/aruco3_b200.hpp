// aruco3_b200.hpp — header-only C++ mirror of the reference's detection API over the C ABI (aruco3_b200.h).
//
// The reference is a Rust crate; Rust is not available in this build environment, so the host side above the C ABI is
// C++ with the reference's names, argument meaning and error behaviour:
//   DetectorConfig   /root/reference/src/aruco.rs:23-43        Detector    /root/reference/src/aruco.rs:46-52
//   Detection        /root/reference/src/aruco.rs:16-21        Marker      /root/reference/src/aruco.rs:8-13
//   ARDictionary     /root/reference/src/dictionaries.rs:22-28, 115-232
//   MarkerPose, pose::solve_with_*   /root/reference/src/pose.rs:8-81     CameraIntrinsics  /root/reference/src/pinhole.rs:11-94
// Where the reference panics (unknown dictionary name, threshold_window == 0, epsilon <= 0) this mirror throws
// aruco3::Error.  Link with -laruco3_b200.  No CPU fallback: constructing a Detector without a CUDA device throws.
#ifndef ARUCO3_B200_HPP
#define ARUCO3_B200_HPP

#include <array>
#include <cstdint>
#include <exception>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "aruco3_b200.h"

namespace aruco3 {

struct Error : std::runtime_error {
    a3_status status;
    Error(a3_status s, const std::string &what) : std::runtime_error(what), status(s) {}
};
inline void check(a3_status s) {
    if (s != A3_OK) throw Error(s, std::string(a3_status_string(s)) + ": " + a3_last_error());
}

// src/lib.rs:11-21
inline uint8_t hamming_distance(uint64_t a, uint64_t b) { return a3_hamming_distance(a, b); }

// src/dictionaries.rs:22-28
class ARDictionary {
public:
    uint8_t num_bits = 0;
    uint8_t tau = 0;
    const uint64_t *code_list = nullptr;  // static storage inside the library
    size_t code_count = 0;

    // src/dictionaries.rs:140-145 (case-insensitive; the reference panics on an unknown name)
    static ARDictionary new_from_named_dict(const std::string &name) {
        ARDictionary d;
        check(a3_dictionary_by_name(name.c_str(), &d.c_));
        d.num_bits = d.c_.num_bits; d.tau = d.c_.tau; d.code_list = d.c_.codes; d.code_count = d.c_.n_codes;
        return d;
    }
    // src/dictionaries.rs:147-149
    static std::vector<std::string> get_dictionary_names() {
        std::vector<std::string> v;
        for (int32_t i = 0; i < a3_dictionary_count(); i++) v.emplace_back(a3_dictionary_name(i));
        return v;
    }
    uint8_t get_mark_size() const { return a3_dictionary_mark_size(&c_); }  // :154-156
    std::pair<size_t, uint8_t> find_nearest(uint64_t bits) const {          // :160-196
        uint64_t i; uint8_t dist;
        a3_find_nearest(&c_, bits, &i, &dist);
        return {(size_t)i, dist};
    }
    bool try_find_nearest(uint64_t bits, size_t *index, uint8_t *dist) const {  // :200-207 (Option -> bool)
        uint64_t i; uint8_t dd;
        const bool ok = a3_try_find_nearest(&c_, bits, &i, &dd) != 0;
        if (index) *index = (size_t)i;
        if (dist) *dist = dd;
        return ok;
    }
    std::pair<uint8_t, std::vector<bool>> make_binary_image(size_t marker_id) const {  // :212-232, (width, bits) as there
        uint8_t buf[256]; uint32_t n = 0;
        const uint8_t w = a3_make_binary_image(&c_, marker_id, buf, sizeof(buf), &n);
        return {w, std::vector<bool>(buf, buf + (n < sizeof(buf) ? n : sizeof(buf)))};
    }
    const a3_dictionary &c() const { return c_; }

private:
    a3_dictionary c_{};
};

// src/aruco.rs:23-30; defaults :32-43
struct DetectorConfig {
    uint32_t threshold_window = 7;
    double contour_simplification_epsilon = 0.05;
    float min_side_length_factor = 0.2f;
    float min_corner_separation_factor = 0.1f;
    size_t homography_sample_size = 49;
    bool filter_high_bit_errors = true;
};

// src/pinhole.rs:11-18
struct CameraIntrinsics {
    uint32_t image_width = 0, image_height = 0;
    float focal_x = 0, focal_y = 0, principal_x = 0, principal_y = 0;

    CameraIntrinsics() = default;
    // CameraIntrinsics::new (src/pinhole.rs:26-35); a null principal point is the image centre (Option::None)
    CameraIntrinsics(uint32_t w, uint32_t h, float fx, float fy, const float *px = nullptr, const float *py = nullptr) {
        a3_camera_intrinsics k;
        a3_camera_intrinsics_new(w, h, fx, fy, px, py, &k);
        *this = from_c(k);
    }
    // src/pinhole.rs:37-60
    static CameraIntrinsics new_from_fov_horizontal(float horizontal_fov_radians, float sensor_width_mm, uint32_t resolution_x, uint32_t resolution_y) {
        a3_camera_intrinsics k;
        a3_camera_intrinsics_from_fov_horizontal(horizontal_fov_radians, sensor_width_mm, resolution_x, resolution_y, &k);
        return from_c(k);
    }
    std::array<float, 3> project(float x, float y, float z) const {  // :65-71
        std::array<float, 3> o{};
        const a3_camera_intrinsics k = c();
        a3_camera_project(&k, x, y, z, o.data());
        return o;
    }
    bool project_culled(float x, float y, float z, std::pair<float, float> *out) const {  // :76-84 (Option -> bool)
        float o[2];
        const a3_camera_intrinsics k = c();
        if (!a3_camera_project_culled(&k, x, y, z, o)) return false;
        if (out) *out = {o[0], o[1]};
        return true;
    }
    std::pair<float, float> unproject(float x, float y) const {  // :88-93
        float o[2];
        const a3_camera_intrinsics k = c();
        a3_camera_unproject(&k, x, y, o);
        return {o[0], o[1]};
    }
    a3_camera_intrinsics c() const { return a3_camera_intrinsics{image_width, image_height, focal_x, focal_y, principal_x, principal_y}; }
    static CameraIntrinsics from_c(const a3_camera_intrinsics &k) {
        CameraIntrinsics r;
        r.image_width = k.image_width; r.image_height = k.image_height; r.focal_x = k.focal_x; r.focal_y = k.focal_y;
        r.principal_x = k.principal_x; r.principal_y = k.principal_y;
        return r;
    }
};

// src/pose.rs:8-12; Default src/pose.rs:42-50.  rotation is row-major.
struct MarkerPose {
    float error = 1e31f;
    std::array<float, 9> rotation{{1, 0, 0, 0, 1, 0, 0, 0, 1}};
    std::array<float, 3> translation{{0, 0, 0}};

    using Point3 = std::array<float, 3>;
    std::vector<Point3> apply_transform_to_points(const std::vector<Point3> &points) const { return apply(points, 0); }          // :17-28
    std::vector<Point3> apply_inverse_transform_to_points(const std::vector<Point3> &points) const { return apply(points, 1); }  // :30-39
    static MarkerPose from_c(const a3_pose &p) {
        MarkerPose m;
        m.error = p.error;
        for (int i = 0; i < 9; i++) m.rotation[i] = p.rotation[i];
        for (int i = 0; i < 3; i++) m.translation[i] = p.translation[i];
        return m;
    }

private:
    std::vector<Point3> apply(const std::vector<Point3> &points, int inverse) const {
        a3_pose p;
        p.error = error;
        for (int i = 0; i < 9; i++) p.rotation[i] = rotation[i];
        for (int i = 0; i < 3; i++) p.translation[i] = translation[i];
        std::vector<Point3> out(points.size());
        if (!points.empty()) a3_pose_apply_transform(&p, points[0].data(), (uint32_t)points.size(), inverse, out[0].data());
        return out;
    }
};

// The pose of a Board in one frame (kernel K6): board points (x, y, 0) -> camera.  `best` has the smaller error (RMS
// reprojection distance over the used corners, normalised units), `alt` is the other branch of the planar ambiguity;
// `ok` is false when both failed or no board marker was seen.
struct BoardPose {
    MarkerPose best, alt;
    uint32_t n_markers = 0;
    bool ok = false;
    static BoardPose from_c(const a3_board_pose &p) {
        BoardPose b;
        b.best = MarkerPose::from_c(p.best); b.alt = MarkerPose::from_c(p.alt); b.n_markers = p.n_markers; b.ok = p.ok != 0;
        return b;
    }
};

// A rigid planar board (a3_board): distinct ids and, per marker, its four corners x0,y0..x3,y3 on the board plane (z = 0,
// x right, y up, any length unit) in the order of Marker::corners.
struct Board {
    std::vector<uint64_t> ids;
    std::vector<std::array<float, 8>> corners;

    // cols x rows square markers `separation` apart, centred on the origin; row 0 at the top, ids row-major from first_id
    static Board grid(uint32_t cols, uint32_t rows, float marker_size, float separation, uint64_t first_id = 0) {
        const float pitch = marker_size + separation;
        const float w = (float)cols * marker_size + (float)(cols - 1) * separation, h = (float)rows * marker_size + (float)(rows - 1) * separation;
        Board b;
        for (uint32_t r = 0; r < rows; r++)
            for (uint32_t c = 0; c < cols; c++) {
                const float x0 = -w / 2 + (float)c * pitch, y0 = h / 2 - (float)r * pitch;
                b.ids.push_back(first_id + (uint64_t)r * cols + c);
                b.corners.push_back({x0, y0, x0 + marker_size, y0, x0 + marker_size, y0 - marker_size, x0, y0 - marker_size});
            }
        return b;
    }
    // the C view; it points into this object
    a3_board c() const { return a3_board{(uint32_t)ids.size(), ids.data(), corners.empty() ? nullptr : corners[0].data()}; }
};

// A lens distortion of the intrinsics (a3_camera_distortion): OpenCV's k1 k2 p1 p2 k3.  With it the pose kernels solve
// from undistorted corners (kernel K7); only with intrinsics modes.
struct CameraDistortion {
    float k1 = 0, k2 = 0, p1 = 0, p2 = 0, k3 = 0;
    a3_camera_distortion c() const { return a3_camera_distortion{k1, k2, p1, p2, k3}; }
};

// a3_detector_set_distortion on `h` (nullptr = off)
inline void set_distortion_on(a3_detector *h, const CameraDistortion *d) {
    if (!d) {
        check(a3_detector_set_distortion(h, nullptr));
        return;
    }
    const a3_camera_distortion c = d->c();
    check(a3_detector_set_distortion(h, &c));
}

// a3_detector_set_board on `h` (nullptr board = off; nullptr k = undistorted at the frame size)
inline void set_board_on(a3_detector *h, const Board *board, const CameraIntrinsics *k) {
    if (!board) {
        check(a3_detector_set_board(h, nullptr, A3_POSE_OFF, nullptr));
        return;
    }
    const a3_board b = board->c();
    const a3_camera_intrinsics kc = k ? k->c() : a3_camera_intrinsics{};
    check(a3_detector_set_board(h, &b, k ? A3_POSE_INTRINSICS : A3_POSE_UNDISTORTED, k ? &kc : nullptr));
}

// src/aruco.rs:8-13
struct Marker {
    size_t id = 0;
    uint64_t code = 0;
    std::vector<std::pair<uint32_t, uint32_t>> corners;  // 4, already rotate_left(rotation)
    uint8_t hamming_distance = 0;
    // Detector::set_corner_refinement(true): the 4 sub-pixel corners in the order of `corners` (pixel-centre convention),
    // empty otherwise; `refined` is false where the refinement fell back to the integer corners
    std::vector<std::pair<float, float>> corners_refined;
    bool refined = false;
};

struct GrayImage {  // image::GrayImage: tightly packed, row-major
    uint32_t width = 0, height = 0;
    std::vector<uint8_t> data;
};

// src/aruco.rs:16-21
struct Detection {
    GrayImage grey;                                                    // always present, like Some(grey)
    std::vector<std::vector<std::pair<uint32_t, uint32_t>>> candidates;
    std::vector<GrayImage> homographies;                               // 1x1 when the projection failed (src/aruco.rs:256)
    std::vector<Marker> markers;
    std::optional<BoardPose> board_pose;                               // the detector's board (set_board), else empty
};

enum class PixelFormat { Rgb8 = A3_FMT_RGB8, Rgba8 = A3_FMT_RGBA8, Luma8 = A3_FMT_LUMA8, Bgr8 = A3_FMT_BGR8, Bgra8 = A3_FMT_BGRA8 };

inline a3_config to_c(const DetectorConfig &config) {
    a3_config c;
    c.threshold_window = config.threshold_window;
    c.contour_simplification_epsilon = config.contour_simplification_epsilon;
    c.min_side_length_factor = config.min_side_length_factor;
    c.min_corner_separation_factor = config.min_corner_separation_factor;
    c.homography_sample_size = (uint32_t)config.homography_sample_size;
    c.filter_high_bit_errors = config.filter_high_bit_errors ? 1 : 0;
    return c;
}

// a3_detect_batch on handle `h` (host frames) unpacked into Detections; `full` fills grey / candidates / homographies,
// otherwise only markers.
inline std::vector<Detection> detect_batch_on(a3_detector *h_, const DetectorConfig &config, const uint8_t *frames, uint32_t n, uint32_t width,
                                              uint32_t height, PixelFormat fmt, bool full, a3_stats *stats, bool refined = false,
                                              bool board = false) {
    const uint32_t bpp = (fmt == PixelFormat::Rgb8 || fmt == PixelFormat::Bgr8) ? 3 : (fmt == PixelFormat::Luma8 ? 1 : 4);
    const size_t pitch = (size_t)width * bpp, stride = pitch * height, px = (size_t)width * height;
    const size_t hs = config.homography_sample_size, np = hs * hs;
    std::vector<Detection> out(n);
    uint32_t cap_m = 64 * n + 1024, cap_c = 128 * n + 2048;
    for (;;) {
        std::vector<a3_marker> markers(cap_m);
        std::vector<uint8_t> grey, patches;
        std::vector<uint32_t> cands, cframe, offsets(n + 1);
        std::vector<a3_decode> decs;
        std::vector<float> mcorners(refined ? (size_t)cap_m * 8 : 0);
        std::vector<a3_board_pose> bposes(board ? n : 0);
        a3_outputs o{};
        if (board) o.board_poses = bposes.data();
        o.frame_marker_offsets = offsets.data();
        if (refined) o.marker_corners = mcorners.data();
        if (full) {
            grey.resize(n * px); cands.resize((size_t)cap_c * 8); cframe.resize(cap_c); patches.resize((size_t)cap_c * np); decs.resize(cap_c);
            o.grey = grey.data(); o.candidates = cands.data(); o.candidate_frame = cframe.data();
            o.homographies = patches.data(); o.decodes = decs.data(); o.cand_capacity = cap_c;
        }
        uint32_t nm = 0;
        const a3_status s = a3_detect_batch(h_, frames, (a3_format)fmt, A3_MEM_HOST, n, width, height, pitch, stride, markers.data(),
                                            cap_m, &nm, &o, stats);
        if (s == A3_ERR_CAPACITY) {  // counts are valid: size once more
            cap_m = nm > cap_m ? nm : cap_m;
            cap_c = o.n_candidates > cap_c ? o.n_candidates : cap_c;
            continue;
        }
        check(s);
        for (uint32_t i = 0; i < nm; i++) {
            const a3_marker &m = markers[i];
            Marker mk;
            mk.id = (size_t)m.id; mk.code = m.code; mk.hamming_distance = m.hamming_distance;
            for (int k = 0; k < 4; k++) mk.corners.emplace_back(m.corners[2 * k], m.corners[2 * k + 1]);
            if (refined) {
                for (int k = 0; k < 4; k++) mk.corners_refined.emplace_back(mcorners[(size_t)i * 8 + 2 * k], mcorners[(size_t)i * 8 + 2 * k + 1]);
                mk.refined = m.corners_refined != 0;
            }
            out[m.frame].markers.push_back(std::move(mk));
        }
        for (uint32_t f = 0; board && f < n; f++) out[f].board_pose = BoardPose::from_c(bposes[f]);
        if (full) {
            for (uint32_t f = 0; f < n; f++) {
                out[f].grey.width = width; out[f].grey.height = height;
                out[f].grey.data.assign(grey.begin() + f * px, grey.begin() + (f + 1) * px);
            }
            for (uint32_t k = 0; k < o.n_candidates; k++) {
                Detection &d = out[cframe[k]];
                std::vector<std::pair<uint32_t, uint32_t>> poly;
                for (int j = 0; j < 4; j++) poly.emplace_back(cands[(size_t)k * 8 + 2 * j], cands[(size_t)k * 8 + 2 * j + 1]);
                d.candidates.push_back(std::move(poly));
                GrayImage g;
                if (decs[k].homography_ok) {
                    g.width = g.height = (uint32_t)hs;
                    g.data.assign(patches.begin() + (size_t)k * np, patches.begin() + (size_t)(k + 1) * np);
                } else {
                    g.width = g.height = 1;
                    g.data.assign(1, 0);
                }
                d.homographies.push_back(std::move(g));
            }
        }
        return out;
    }
}


// `Detector { config, dictionary }` (src/aruco.rs:46-49) bound to one CUDA device.  Thread-compatible: one per
// (host thread, device).  Public fields are read at construction; call rebuild() after changing them.
class Detector {
public:
    DetectorConfig config;
    ARDictionary dictionary;

    Detector(const DetectorConfig &cfg, const ARDictionary &dict, int device = 0) : config(cfg), dictionary(dict), device_(device) { rebuild(); }
    ~Detector() { a3_detector_destroy(h_); }
    Detector(const Detector &) = delete;
    Detector &operator=(const Detector &) = delete;

    void rebuild() {
        a3_detector_destroy(h_);
        h_ = nullptr;
        const a3_config c = to_c(config);
        check(a3_detector_create(&c, &dictionary.c(), device_, &h_));
        if (refine_) check(a3_detector_set_corner_refinement(h_, A3_CORNERS_REFINED));
        if (board_) set_board_on(h_, &*board_, board_k_ ? &*board_k_ : nullptr);
        if (dist_) set_distortion_on(h_, &*dist_);
    }

    // Detector::detect(&self, image: DynamicImage) -> Detection (src/aruco.rs:52-121): one tightly packed image.
    Detection detect(const uint8_t *pixels, uint32_t width, uint32_t height, PixelFormat fmt = PixelFormat::Rgb8) const {
        std::vector<Detection> v = detect_batch(pixels, 1, width, height, fmt, /*full=*/true);
        return std::move(v[0]);
    }

    // The same over n equally sized frames; `full` fills grey / candidates / homographies, otherwise only markers.
    std::vector<Detection> detect_batch(const uint8_t *frames, uint32_t n, uint32_t width, uint32_t height,
                                        PixelFormat fmt = PixelFormat::Rgb8, bool full = false, a3_stats *stats = nullptr) const {
        return detect_batch_on(h_, config, frames, n, width, height, fmt, full, stats, refine_, board_.has_value());
    }

    // Sub-pixel corners (kernel K5) in Marker::corners_refined, and poses from them; off by default.  Kept across rebuild().
    void set_corner_refinement(bool on) {
        check(a3_detector_set_corner_refinement(h_, on ? A3_CORNERS_REFINED : A3_CORNERS_INTEGER));
        refine_ = on;
    }

    // The pose of a planar board in every frame (kernel K6) in Detection::board_pose; `k` = nullptr normalises by the frame
    // size (undistorted), `board` = nullptr switches it off.  Both are copied and kept across rebuild().
    void set_board(const Board *board, const CameraIntrinsics *k = nullptr) {
        set_board_on(h_, board, k);
        board_ = board ? std::optional<Board>(*board) : std::nullopt;
        board_k_ = k ? std::optional<CameraIntrinsics>(*k) : std::nullopt;
    }

    // A lens distortion of the board's intrinsics (kernel K7 undistorts the corners K6 reads); nullptr switches it off.
    // Copied and kept across rebuild().
    void set_distortion(const CameraDistortion *d) {
        set_distortion_on(h_, d);
        dist_ = d ? std::optional<CameraDistortion>(*d) : std::nullopt;
    }

    a3_detector *handle() const { return h_; }

private:
    int device_ = 0;
    a3_detector *h_ = nullptr;
    bool refine_ = false;
    std::optional<Board> board_;
    std::optional<CameraIntrinsics> board_k_;
    std::optional<CameraDistortion> dist_;
};

// The reference's own shape: `Detector { config, dictionary }` is plain data built with a literal (src/aruco.rs:46-49,
// benches/detect_markers.rs:17-20) and `detect` takes `&self`, so there is nowhere to keep a handle.  Every call leases
// one from the library's cache (a3_detector_acquire / a3_detector_release): the first call creates it, later calls —
// from any PlainDetector with the same config, dictionary and device — get it back warm.  This is what the Rust wrapper
// in rust/aruco3-b200 does.
struct PlainDetector {
    DetectorConfig config;
    ARDictionary dictionary;
    int device = 0;
    bool refine_corners = false;  // wrapper-side option (not in the reference's DetectorConfig): set on the leased handle per call
    std::optional<Board> board;   // likewise: the board whose pose every frame gets (kernel K6)
    std::optional<CameraIntrinsics> board_intrinsics;  // empty: undistorted at the frame size
    std::optional<CameraDistortion> distortion;        // likewise: the lens of board_intrinsics (kernel K7)

    Detection detect(const uint8_t *pixels, uint32_t width, uint32_t height, PixelFormat fmt = PixelFormat::Rgb8) const {
        std::vector<Detection> v = detect_batch(pixels, 1, width, height, fmt, /*full=*/true);
        return std::move(v[0]);
    }
    std::vector<Detection> detect_batch(const uint8_t *frames, uint32_t n, uint32_t width, uint32_t height,
                                        PixelFormat fmt = PixelFormat::Rgb8, bool full = false, a3_stats *stats = nullptr) const {
        struct Lease {
            a3_detector *h = nullptr;
            ~Lease() { a3_detector_release(h); }
        } lease;
        const a3_config c = to_c(config);
        check(a3_detector_acquire(&c, &dictionary.c(), device, &lease.h));
        if (refine_corners) check(a3_detector_set_corner_refinement(lease.h, A3_CORNERS_REFINED));
        if (board) set_board_on(lease.h, &*board, board_intrinsics ? &*board_intrinsics : nullptr);  // the release resets it
        if (distortion) set_distortion_on(lease.h, &*distortion);                                      // and this
        return detect_batch_on(lease.h, config, frames, n, width, height, fmt, full, stats, refine_corners, board.has_value());
    }
};

// Frame-batch sharding over several GPUs (SURVEY 8e): frames are independent, so a batch is cut into contiguous blocks,
// one per device (block sizes differ by at most one frame, earlier devices take the extras — the rule of
// aruco3_b200/sharding.py), each block goes through its own Detector on its own host thread, and the per-frame results
// are concatenated in frame order.  No collective, no peer traffic.  The same device may be listed more than once.
class ShardedDetector {
public:
    ShardedDetector(const DetectorConfig &cfg, const ARDictionary &dict, const std::vector<int> &devices) {
        if (devices.empty()) throw Error(A3_ERR_INVALID_ARGUMENT, "ShardedDetector: no devices");
        for (int dev : devices) shards_.emplace_back(new Detector(cfg, dict, dev));
    }
    size_t size() const { return shards_.size(); }
    void set_corner_refinement(bool on) {
        for (auto &d : shards_) d->set_corner_refinement(on);
    }
    void set_board(const Board *board, const CameraIntrinsics *k = nullptr) {
        for (auto &d : shards_) d->set_board(board, k);
    }
    void set_distortion(const CameraDistortion *dist) {
        for (auto &d : shards_) d->set_distortion(dist);
    }
    static std::pair<uint32_t, uint32_t> shard_range(uint32_t n_frames, uint32_t rank, uint32_t world) {
        const uint32_t base = n_frames / world, extra = n_frames % world;
        const uint32_t lo = rank * base + (rank < extra ? rank : extra);
        return {lo, lo + base + (rank < extra ? 1u : 0u)};
    }
    std::vector<Detection> detect_batch(const uint8_t *frames, uint32_t n, uint32_t width, uint32_t height,
                                        PixelFormat fmt = PixelFormat::Rgb8, bool full = false) const {
        const uint32_t bpp = (fmt == PixelFormat::Rgb8 || fmt == PixelFormat::Bgr8) ? 3 : (fmt == PixelFormat::Luma8 ? 1 : 4);
        const size_t stride = (size_t)width * bpp * height;
        const uint32_t world = (uint32_t)shards_.size();
        std::vector<std::vector<Detection>> parts(world);
        std::vector<std::exception_ptr> errors(world);
        std::vector<std::thread> threads;
        for (uint32_t r = 0; r < world; r++)
            threads.emplace_back([&, r] {
                try {
                    const auto range = shard_range(n, r, world);
                    if (range.second > range.first)
                        parts[r] = shards_[r]->detect_batch(frames + (size_t)range.first * stride, range.second - range.first, width, height, fmt, full);
                } catch (...) {
                    errors[r] = std::current_exception();
                }
            });
        for (auto &t : threads) t.join();
        for (auto &e : errors)
            if (e) std::rethrow_exception(e);
        std::vector<Detection> out;
        out.reserve(n);
        for (auto &part : parts)
            for (auto &d : part) out.push_back(std::move(d));
        return out;
    }

private:
    std::vector<std::unique_ptr<Detector>> shards_;
};

// src/pose.rs:52-81.  The solvers run on the detector's device (kernel K4); (best, alt) as in the reference.
namespace pose {
using Corners = std::vector<std::pair<uint32_t, uint32_t>>;  // Marker::corners

inline std::pair<MarkerPose, MarkerPose> solve_with_intrinsics(const Detector &det, const Corners &image_points, float marker_size_mm,
                                                               const CameraIntrinsics &camera_intrinsics) {
    if (image_points.size() != 4) throw Error(A3_ERR_INVALID_ARGUMENT, "solve_with_intrinsics: four corners expected");
    uint32_t c[8];
    for (int i = 0; i < 4; i++) { c[2 * i] = image_points[i].first; c[2 * i + 1] = image_points[i].second; }
    const a3_camera_intrinsics k = camera_intrinsics.c();
    a3_pose best, alt;
    check(a3_solve_with_intrinsics(det.handle(), c, 1, marker_size_mm, &k, &best, &alt));
    return {MarkerPose::from_c(best), MarkerPose::from_c(alt)};
}
inline std::pair<MarkerPose, MarkerPose> solve_with_undistorted_points(const Detector &det, const Corners &image_points, float marker_size_mm,
                                                                       std::pair<uint32_t, uint32_t> image_size) {
    if (image_points.size() != 4) throw Error(A3_ERR_INVALID_ARGUMENT, "solve_with_undistorted_points: four corners expected");
    uint32_t c[8];
    for (int i = 0; i < 4; i++) { c[2 * i] = image_points[i].first; c[2 * i + 1] = image_points[i].second; }
    a3_pose best, alt;
    check(a3_solve_with_undistorted_points(det.handle(), c, 1, marker_size_mm, image_size.first, image_size.second, &best, &alt));
    return {MarkerPose::from_c(best), MarkerPose::from_c(alt)};
}
inline std::pair<MarkerPose, MarkerPose> solve_with_normalized_points(const Detector &det, const std::vector<std::pair<float, float>> &points,
                                                                      float marker_size_mm) {
    if (points.size() != 4) throw Error(A3_ERR_INVALID_ARGUMENT, "solve_with_normalized_points: four points expected");
    float c[8];
    for (int i = 0; i < 4; i++) { c[2 * i] = points[i].first; c[2 * i + 1] = points[i].second; }
    a3_pose best, alt;
    check(a3_solve_with_normalized_points(det.handle(), c, 1, marker_size_mm, &best, &alt));
    return {MarkerPose::from_c(best), MarkerPose::from_c(alt)};
}
}  // namespace pose

}  // namespace aruco3
#endif  // ARUCO3_B200_HPP
