// C ABI of the detection path (include/aruco3_b200.h): detector handle, the batched pipeline and the stage probes.
//
// Pipeline of a3_detect_batch (frames are independent — src/aruco.rs:52-121 is a pure function of one image — so
// frames, chunks and GPUs never exchange data):
//
//   copy stream     H2D of front-end chunk j into a staging ring            (host input only)
//   pixel stream    K1 (grey + 1-bit mask, k1_strips.cu) -> D2H of the mask bits -> event[j]
//   host pool       persistent threads; frame f becomes runnable when event[chunk of f] has fired; one task = border
//                   following + quad filters of one frame (host_quads.cpp)
//   decode stream   per group of frames whose quads are ready: H2D quads -> K2 (k2_decode.cu) -> D2H decode records
//   caller thread   feeds the pool, launches decode groups, finally assembles markers in frame / candidate order
//
// Device input runs K1 once over the whole (super-)batch; host input runs it per front-end chunk right behind the
// copy, so the PCIe transfer, the host stage and the decode kernel all overlap.
// There is no CPU fallback: without a CUDA device every compute entry point returns A3_ERR_CUDA.
#include <immintrin.h>
#include <math.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "a3_internal.h"
#include "k6_board_spec.h"

namespace a3 {

static thread_local std::string g_error;
void set_error(const std::string &msg) { g_error = msg; }
a3_status fail(a3_status s, const std::string &msg) { g_error = msg; return s; }
a3_status cuda_fail(cudaError_t e, const char *what) {
    g_error = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
    cudaGetLastError();
    return A3_ERR_CUDA;
}

namespace {

// Persistent host threads.  A job is a function of a frame index; indices [0, ready) may be claimed.
class WorkerPool {
public:
    ~WorkerPool() { stop(); }
    void resize(uint32_t threads) {
        if (threads == workers_.size()) return;
        stop();
        quit_ = false;
        for (uint32_t t = 0; t < threads; t++) workers_.emplace_back([this] { loop(); });
    }
    uint32_t size() const { return (uint32_t)workers_.size(); }
    void begin(std::function<void(uint32_t)> fn, uint32_t total) {
        std::lock_guard<std::mutex> lk(mu_);
        fn_ = std::move(fn); total_ = total; next_ = 0; ready_ = 0; done_ = 0;
    }
    void publish(uint32_t upto) {
        { std::lock_guard<std::mutex> lk(mu_); if (upto > ready_) ready_ = upto; }
        cv_.notify_all();
    }
    // Tasks do not finish in index order; callers keep their own counters inside the job function and sleep on them
    // with wait_caller(); the job calls notify_caller() when a counter reaches its goal.
    void notify_caller() { { std::lock_guard<std::mutex> lk(mu_); } cv_done_.notify_all(); }
    template <typename Pred>
    void wait_caller(Pred pred) {
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, pred);
    }
    void finish() {  // block until all `total` tasks are done
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, [this] { return done_ >= total_; });
        fn_ = nullptr;
    }

private:
    void loop() {
        std::unique_lock<std::mutex> lk(mu_);
        for (;;) {
            cv_.wait(lk, [this] { return quit_ || (fn_ && next_ < ready_); });
            if (quit_) return;
            const uint32_t i = next_++;
            lk.unlock();
            fn_(i);  // fn_ stays alive until finish(), which waits for this task
            lk.lock();
            if (++done_ >= total_) cv_done_.notify_all();
        }
    }
    void stop() {
        { std::lock_guard<std::mutex> lk(mu_); quit_ = true; }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
        workers_.clear();
    }
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_, cv_done_;
    std::function<void(uint32_t)> fn_;
    uint32_t total_ = 0, next_ = 0, ready_ = 0, done_ = 0;
    bool quit_ = false;
};

// Host threads that move bytes between the caller's pageable memory and the pinned staging rings (a3_detect_batch with
// A3_MEM_HOST frames that are not page-locked, and `Detection.grey` into a pageable buffer): a FIFO of small tasks.  Callers
// keep their own completion counters (atomics) and sleep on them with wait(); a task calls notify() when a counter reaches
// its goal.
class CopyPool {
public:
    ~CopyPool() { stop(); }
    void start(uint32_t threads, int device) {
        if (!workers_.empty()) return;
        quit_ = false;
        for (uint32_t t = 0; t < threads; t++)
            workers_.emplace_back([this, device] {
                cudaSetDevice(device);  // tasks wait on CUDA events of the detector's device
                loop();
            });
    }
    void submit(std::function<void()> fn) {
        { std::lock_guard<std::mutex> lk(mu_); q_.push_back(std::move(fn)); }
        cv_.notify_one();
    }
    void notify() { { std::lock_guard<std::mutex> lk(mu_); } cv_done_.notify_all(); }
    template <typename Pred>
    void wait(Pred pred) {
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, pred);
    }
    void drain() {  // until the queue is empty and no task is running
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, [this] { return q_.empty() && running_ == 0; });
    }
    void stop() {
        { std::lock_guard<std::mutex> lk(mu_); quit_ = true; }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
        workers_.clear();
    }

private:
    void loop() {
        std::unique_lock<std::mutex> lk(mu_);
        for (;;) {
            cv_.wait(lk, [this] { return quit_ || !q_.empty(); });
            if (quit_) return;
            std::function<void()> fn = std::move(q_.front());
            q_.pop_front();
            running_++;
            lk.unlock();
            fn();
            lk.lock();
            running_--;
            if (q_.empty() && running_ == 0) cv_done_.notify_all();
        }
    }
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_, cv_done_;
    std::deque<std::function<void()>> q_;
    uint32_t running_ = 0;
    bool quit_ = false;
};

// memcpy for the staging rings: the destination is written once and read next by the DMA engine (input ring) or by nobody
// soon (the caller's grey buffer), so streaming stores keep it out of the caches and spare the read-for-ownership of every
// destination line — a third of the DRAM traffic of a plain copy, and the copy threads share the memory bus with the DMA.
__attribute__((target("avx2"))) void copy_stream_avx2(uint8_t *dst, const uint8_t *src, size_t len) {
    while (len && ((uintptr_t)dst & 31)) { *dst++ = *src++; len--; }
    size_t i = 0;
    for (; i + 128 <= len; i += 128) {
        const __m256i a = _mm256_loadu_si256((const __m256i *)(src + i)), b = _mm256_loadu_si256((const __m256i *)(src + i + 32));
        const __m256i c = _mm256_loadu_si256((const __m256i *)(src + i + 64)), d = _mm256_loadu_si256((const __m256i *)(src + i + 96));
        _mm256_stream_si256((__m256i *)(dst + i), a); _mm256_stream_si256((__m256i *)(dst + i + 32), b);
        _mm256_stream_si256((__m256i *)(dst + i + 64), c); _mm256_stream_si256((__m256i *)(dst + i + 96), d);
    }
    _mm_sfence();
    if (i < len) memcpy(dst + i, src + i, len - i);
}
void copy_stream(uint8_t *dst, const uint8_t *src, size_t len) {
    static const bool avx2 = __builtin_cpu_supports("avx2") && !getenv("A3_PLAIN_MEMCPY");
    if (avx2 && len >= 4096) copy_stream_avx2(dst, src, len);
    else memcpy(dst, src, len);
}

// Shared between a call and the copy tasks it has in flight (kept alive by the tasks, so an early error return cannot
// leave a task with a dangling reference).
struct StageState {
    std::unique_ptr<std::atomic<uint32_t>[]> in_left;   // per front-end chunk: pieces of its stage-in copy still to do
    struct Out { cudaEvent_t ev; std::atomic<uint32_t> left; };
    std::deque<Out> out;                                // per grey sub-chunk, in issue order (deque: stable addresses)
};

// The post-decode stages a call runs, in this order behind K2: K5 (refine), K7 (und_sets sets of undistorted corners), K4
// (poses), K6 (board).  K7 writes one set for K4 (the pose intrinsics) and one for K6 (the board intrinsics), shared when the
// two intrinsics are the same; the setters allow distortion only with INTRINSICS modes.
struct StagePlan {
    bool poses = false, refine = false, board = false;
    bool und_pose = false, und_board = false;  // K4 / K6 read K7's points
    uint32_t und_sets = 0, und_board_set = 0;  // corner sets (0 = K7 does not run), and the one K6 reads
    void count(a3_stats &st) const {  // the chain's launches
        st.decode_kernel_launches++;
        if (refine) st.refine_kernel_launches++;
        st.undistort_kernel_launches += und_sets;
        if (poses) st.pose_kernel_launches++;
        if (board) st.board_kernel_launches++;
    }
};

size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// Byte offsets of a decode group's outputs in one buffer, for `cap` candidates of `n_frames` frames: K6's board pose per frame,
// K2's records, K4's two poses, K5's corners and flags (accepted candidates only), then K7's points and flags, set j at
// norm + 32 cap j and nok + cap j.  The board comes first so that [board, dec) is the per-frame part alone, and K7's points last
// so that [0, host_end) is everything the host reads.
struct OutLayout {
    size_t board = 0, dec, pose, ref, refok, host_end, norm, nok, bytes;
};
OutLayout out_layout(const StagePlan &sp, uint32_t cap, uint32_t n_frames) {
    OutLayout l;
    l.dec = align16(sp.board ? (size_t)n_frames * sizeof(a3_board_pose) : 0);
    l.pose = l.dec + (size_t)cap * sizeof(a3_decode);
    l.ref = l.pose + (sp.poses ? (size_t)cap * 2 * sizeof(a3_pose) : 0);
    l.refok = l.ref + (sp.refine ? (size_t)cap * 32 : 0);
    l.host_end = l.refok + (sp.refine ? cap : 0);
    l.norm = sp.und_sets ? align16(l.host_end) : l.host_end;
    l.nok = l.norm + (size_t)sp.und_sets * cap * 32;
    l.bytes = l.nok + (size_t)sp.und_sets * cap;
    return l;
}

// Timed stages of the chain (K4 is not timed), and the a3_stats field of each one's time
enum Stage { kDecode, kRefine, kUndistort, kBoard, kStages };
using StatsMs = double a3_stats::*;
constexpr StatsMs kStageMs[kStages] = {&a3_stats::ms_decode_kernel, &a3_stats::ms_refine_kernel, &a3_stats::ms_undistort_kernel,
                                       &a3_stats::ms_board_kernel};

// Buffers of one decode group (the quads of a few frames); kept for reuse across calls.
struct DecodeBlock {
    PinBuf<uint32_t> h_quads, h_qframe;
    PinBuf<uint32_t> h_qoff;  // K6: per-frame quad offsets of a group whose quads came from the host
    DevBuf<uint32_t> d_quads, d_qframe, d_info, d_qoff;  // d_info / d_qoff: the device-side gather of K3's quads for this group
    DevBuf<uint8_t> d_patches;
    DevBuf<uint8_t> d_out;  // the group's outputs (OutLayout), and their host copy
    PinBuf<uint8_t> h_out;
    cudaEvent_t ev[kStages][2] = {};  // around each timed stage; created with the block
    uint32_t timed = 0;               // bit per Stage: its pair was recorded in this call
    uint32_t n_quads = 0;
    // where the host reads this group's records: h_out, or the one-shot arena
    const a3_decode *dec_view = nullptr;
    const a3_pose *pose_view = nullptr;
    const float *ref_view = nullptr;
    const uint8_t *refok_view = nullptr;
    const a3_board_pose *board_view = nullptr;
    void set_views(const uint8_t *base, const OutLayout &l) {
        dec_view = reinterpret_cast<const a3_decode *>(base + l.dec);
        pose_view = reinterpret_cast<const a3_pose *>(base + l.pose);
        ref_view = reinterpret_cast<const float *>(base + l.ref);
        refok_view = base + l.refok;
        board_view = reinterpret_cast<const a3_board_pose *>(base + l.board);
    }
    ~DecodeBlock() {
        for (auto &pair : ev)
            for (cudaEvent_t e : pair) if (e) cudaEventDestroy(e);
    }
};

struct EventPool {
    std::vector<cudaEvent_t> ev;
    size_t used = 0;
    EventPool() = default;
    EventPool(const EventPool &) = delete;
    EventPool &operator=(const EventPool &) = delete;
    ~EventPool() { for (auto e : ev) cudaEventDestroy(e); }
    cudaError_t get(cudaEvent_t *out) {
        if (used == ev.size()) {
            cudaEvent_t e;
            cudaError_t r = cudaEventCreate(&e);
            if (r != cudaSuccess) return r;
            ev.push_back(e);
        }
        *out = ev[used++];
        return cudaSuccess;
    }
    void reset() { used = 0; }
};

// The options a handle's setters change; a3_detector_release puts back these defaults, the state a3_detector_create leaves.
struct Options {
    uint32_t contour_mode = A3_CONTOURS_DEVICE;
    // pose step (K4)
    uint32_t pose_mode = A3_POSE_OFF;
    float pose_marker_size = 0.0f;
    a3_camera_intrinsics pose_k{};
    // corner refinement (K5)
    uint32_t corner_mode = A3_CORNERS_INTEGER;
    // board pose (K6): board_n = 0 is off; the board itself is in the detector's d_board_slots / d_board_pts
    uint32_t board_n = 0, board_mode = A3_POSE_OFF;
    a3_camera_intrinsics board_k{};
    // lens distortion (K7) of the intrinsics of the pose and board modes; off unless set
    bool dist_on = false;
    a3_camera_distortion dist{};
    // K1 launch tuning and the front-end chunk size (a3_detector_set_k1_tuning)
    bool has_tuning = false;
    K1Tuning k1_tuning{};
    uint32_t chunk_override = 0;
};

}  // namespace
}  // namespace a3

struct a3_detector {
    a3_config cfg;
    a3_dictionary dict;
    int device = 0;
    uint32_t host_threads = 1;
    uint32_t mark_size = 0;
    uint32_t max_taps = 0;
    a3::Options opt;
    cudaStream_t s_copy = nullptr, s_pixel = nullptr, s_decode = nullptr;
    a3::DevBuf<uint8_t> d_src, d_grey, d_mask, d_patches, d_luma;  // d_luma: K0's Luma8 copy of LumaA8 / 16-bit frames
    a3::DevBuf<uint32_t> d_bits, d_quads, d_qframe;
    a3::DevBuf<a3_decode> d_dec;
    a3::PinBuf<uint32_t> h_bits;
    a3::DevBuf<uint64_t> d_codes;
    a3::DevBuf<float> d_taps;
    a3::DevBuf<int> d_meta;
    a3::EventPool events;
    std::vector<std::unique_ptr<a3::DecodeBlock>> blocks;
    a3::WorkerPool pool;
    // pageable host memory at the boundary: pinned rings + copy threads (created on first use)
    a3::CopyPool copy_pool;
    a3::PinBuf<uint8_t> h_stage_in, h_stage_out;
    // GPU contour stage (K3)
    a3::K3Workspace k3;
    a3::DevBuf<uint32_t> d_planes, d_k3quads;
    a3::PinBuf<uint32_t> h_k3quads, h_plane;
    a3::DevBuf<uint8_t> d_k3frames;  // K3's per-frame outputs (K3Frames) outside the one-shot arena, and their host copy
    a3::PinBuf<uint8_t> h_k3frames;
    size_t planes_zeroed_words = 0;
    uint32_t planes_w = 0, planes_h = 0;
    std::vector<std::vector<uint32_t>> frame_quads;  // per-frame quads of the batch in flight (capacity reused across calls)
    // one-shot route (pack_quads): K3's quads go to K2 on the device; launch and copy sizes come from the previous call
    a3::DevBuf<uint32_t> d_qoff;
    a3::DevBuf<uint32_t> d_k2queue;  // K2's work counter where the one-shot arena does not provide it
    // arena of the one-shot route, one device-to-host copy per call: [0] quads in total, [1] route unusable; K3's per-frame
    // counters; the markers (lean calls); the decode group's outputs (OutLayout); the gathered quads
    a3::DevBuf<uint8_t> d_shot;
    a3::PinBuf<uint8_t> h_shot;
    uint32_t hist_nq = 0, hist_nq_n = 0, hist_nq_w = 0, hist_nq_h = 0;  // quads of the previous call with this geometry (0 = none)
    a3::DevBuf<float> d_pose_in;      // standalone solve entry points: 8 x 4 bytes per marker (f32 points or u32 corners)
    a3::DevBuf<a3_pose> d_pose_out;
    a3::PinBuf<a3_pose> h_pose_out;
    a3::DevBuf<float> d_refined;      // a3_refine_corners: refined corners and their flags
    a3::DevBuf<uint8_t> d_refined_ok;
    // board pose (K6): the board as its id -> slot table and points on the device
    a3::DevBuf<uint16_t> d_board_slots;
    a3::DevBuf<float> d_board_pts;
    a3::DevBuf<uint64_t> d_probe_ids;  // a3_solve_board
    a3::DevBuf<uint32_t> d_probe_off;
    a3::DevBuf<a3_board_pose> d_probe_out;
    a3::DevBuf<float> d_und_in, d_und_out;  // a3_undistort_points, and K7's points for a3_solve_board
    a3::DevBuf<uint8_t> d_und_ok;
};

namespace a3 {
namespace {

a3_status check_config(const a3_config &c) {
    if (c.threshold_window == 0) return fail(A3_ERR_INVALID_ARGUMENT, "threshold_window must be > 0 (imageproc asserts block_radius > 0)");
    if (c.threshold_window > 127) return fail(A3_ERR_UNSUPPORTED, "threshold_window > 127 is not supported by the CUDA path (16-bit column sums)");
    if (!(c.contour_simplification_epsilon > 0.0))
        return fail(A3_ERR_INVALID_ARGUMENT, "contour_simplification_epsilon must be > 0 (approximate_polygon_dp panics otherwise)");
    if (c.homography_sample_size == 0) return fail(A3_ERR_INVALID_ARGUMENT, "homography_sample_size must be > 0");
    if (c.homography_sample_size > 4096) return fail(A3_ERR_UNSUPPORTED, "homography_sample_size > 4096 is not supported by the CUDA path");
    return A3_OK;
}

uint32_t bytes_per_pixel(a3_format f) { return (uint32_t)fmt_bpp((int)f); }

// Bytes of caller memory that `cn` consecutive frames cover: from the first frame's first pixel to the last frame's last
// pixel.  Host input copies move exactly this much; the rest of the last frame's stride (the parent image's row tail when the
// frames are crops, a gap after the frame) is memory the caller never passed.  The device slots stay frame_stride apart.
size_t input_span(size_t cn, uint32_t w, uint32_t h, uint32_t bpp, size_t pitch, size_t frame_stride) {
    return (cn - 1) * frame_stride + (size_t)(h - 1) * pitch + (size_t)w * bpp;
}

double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// K3's per-frame outputs of n frames in one block of bytes(n): counts, before-discard, flags and contours as c-word sections
// (c = n rounded up to even), then the points (u64) at word 4c.
struct K3Frames {
    uint32_t *counts, *before, *flags, *contours;
    unsigned long long *points;
    static size_t words(uint32_t n) { return ((size_t)n + 1) & ~(size_t)1; }
    static size_t bytes(uint32_t n) { return 24 * words(n); }
    K3Frames(void *base, uint32_t n) {
        uint32_t *q = static_cast<uint32_t *>(base);
        const size_t c = words(n);
        counts = q; before = q + c; flags = q + 2 * c; contours = q + 3 * c; points = reinterpret_cast<unsigned long long *>(q + 4 * c);
    }
    void stats(uint32_t i, QuadStats &qs) const {
        qs.n_contours = contours[i]; qs.n_contour_points = points[i]; qs.n_before_discard = before[i];
    }
};

// K3's parameters for frames [f0, f0 + n) of guarded planes, quads and per-frame outputs that start at frame 0
K3Params k3_params(const a3_config &cfg, const uint32_t *planes, uint32_t w, uint32_t h, uint32_t f0, uint32_t n, uint32_t *quads,
                   uint32_t quad_cap, const K3Frames &out) {
    const uint32_t mn = w < h ? w : h;
    K3Params kp;
    kp.planes = planes + (size_t)f0 * ((w + 31) / 32 + 2) * (h + 2); kp.n = n; kp.w = w; kp.h = h;
    kp.eps_factor = cfg.contour_simplification_epsilon;
    kp.min_edge_length = (uint32_t)((float)mn * cfg.min_side_length_factor);  // src/aruco.rs:55
    kp.min_corner_separation = (float)mn * cfg.min_corner_separation_factor;   // src/aruco.rs:56
    kp.min_points = (uint32_t)floor(sqrt(2.0 * (double)kp.min_edge_length));
    kp.quad_cap = quad_cap; kp.quads = quads + (size_t)f0 * quad_cap * 8;
    kp.quad_counts = out.counts + f0; kp.before_discard = out.before + f0; kp.frame_flags = out.flags + f0;
    kp.frame_contours = out.contours + f0; kp.frame_points = out.points + f0;
    return kp;
}

// ---- K3 -> K2 on the device -----------------------------------------------------------------------------------------
// K3 leaves each frame's quads in its own block of quad_cap slots.  These two kernels gather them into the dense list in
// frame / candidate order that K2, K4 and the marker assembly use, so the quads need not visit the host between the
// contour stage and the decode.  info[0] = quads in total, info[2] = 0 (K2's work counter), info[1] = 1 when that route cannot be used for this call (the
// speculative K3 finish gave up, a frame is flagged for the host stage, or the list does not fit `cap`): the host then takes
// the ordinary route.
__global__ void __launch_bounds__(1024) pack_offsets_kernel(const uint32_t *counts, const uint32_t *flags, uint32_t n_frames, uint32_t quad_cap,
                                                            uint32_t cap, const uint32_t *k3_failed, uint32_t *offsets, uint32_t *info,
                                                            uint32_t *chunk_end, uint32_t n_chunks) {
    for (uint32_t i = threadIdx.x; i < n_chunks; i += blockDim.x) chunk_end[i] = 0;  // K2's accepted counts per 1024 quads (assemble_markers_kernel)
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t base_s, bad_s;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) info[2] = 0;  // K2's work counter
    if (k3_failed && *k3_failed) {
        if (threadIdx.x == 0) { info[0] = 0; info[1] = 1; }
        return;
    }
    if (threadIdx.x == 0) { base_s = 0; bad_s = 0; }
    __syncthreads();
    for (uint32_t f0 = 0; f0 < n_frames; f0 += 1024) {
        const uint32_t f = f0 + threadIdx.x;
        uint32_t m = 0;
        if (f < n_frames) {
            m = counts[f] < quad_cap ? counts[f] : quad_cap;
            if (flags[f]) { m = 0; bad_s = 1; }
        }
        uint32_t incl = m;
        for (uint32_t o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const uint32_t ws = warp_sums[lane];
            uint32_t wi = ws;
            for (uint32_t o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += v;
            }
            warp_sums[lane] = wi - ws;
        }
        __syncthreads();
        const uint32_t off = base_s + warp_sums[warp] + incl - m;
        if (f < n_frames) offsets[f] = off;
        __syncthreads();
        if (threadIdx.x == 1023) base_s = off + m;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        offsets[n_frames] = base_s;
        const bool bad = bad_s || base_s > cap;
        info[0] = bad ? 0u : base_s;
        info[1] = bad ? 1u : 0u;
    }
}
__global__ void __launch_bounds__(128) pack_quads_kernel(const uint32_t *quads, const uint32_t *offsets, uint32_t quad_cap, uint32_t cap,
                                                         const uint32_t *info, uint32_t *out_quads, uint32_t *out_frame, uint32_t frame_base) {
    if (info[1]) return;
    const uint32_t f = blockIdx.x, o0 = offsets[f], m = offsets[f + 1] - o0;
    const uint32_t *src = quads + (size_t)f * quad_cap * 8;
    for (uint32_t i = threadIdx.x; i < m * 8; i += blockDim.x)
        if (o0 + (i >> 3) < cap) out_quads[(size_t)o0 * 8 + i] = src[i];
    for (uint32_t i = threadIdx.x; i < m; i += blockDim.x)
        if (o0 + i < cap) out_frame[o0 + i] = frame_base + f;
}

// Marker assembly on the device (src/aruco.rs:96-111) for callers that want markers only: the accepted candidates, in
// frame / candidate order, as finished a3_marker records (corners.rotate_left(rotation), the observed code of the winning
// rotation) with their poses beside them, so the host copies one block instead of walking every candidate.
// info[3] = number of markers.
__global__ void __launch_bounds__(1024) assemble_markers_kernel(const a3_decode *dec, const uint32_t *quads, const uint32_t *qframe,
                                                                const uint32_t *qoff, const a3_pose *poses, const float *refined,
                                                                const uint8_t *refined_ok, uint32_t cap, uint32_t *info,
                                                                const uint32_t *chunk_accepted, a3_marker *markers, a3_pose *mposes,
                                                                float *mcorners) {
    // One CTA per 1024 quads.  The number of markers before a chunk is the sum of the accepted counts of the chunks before
    // it, which K2 accumulated while it decoded (K2Params::accept_counts; zeroed by pack_offsets_kernel): no CTA waits for
    // another, so the kernel needs no co-residency and any number of chunks is fine.
    __shared__ uint32_t warp_sums[32], warp_before[32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, c = blockIdx.x;
    const bool bad = info[1] != 0;
    const uint32_t nq = bad ? 0u : (info[0] < cap ? info[0] : cap);
    const uint32_t k = c * 1024 + threadIdx.x;
    const uint32_t acc = (k < nq && dec[k].accepted) ? 1u : 0u;
    const uint32_t bal = __ballot_sync(0xffffffffu, acc);
    uint32_t before = 0;
    if (!bad)
        for (uint32_t i = threadIdx.x; i < c; i += 1024) before += chunk_accepted[i];
    for (uint32_t o = 16; o; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (lane == 0) { warp_sums[warp] = __popc(bal); warp_before[warp] = before; }
    __syncthreads();
    uint32_t base = 0, idx = 0;
    for (uint32_t i = 0; i < 32; i++) {
        base += warp_before[i];
        if (i < warp) idx += warp_sums[i];
    }
    if (c == gridDim.x - 1 && threadIdx.x == 0) {
        uint32_t total = base;
        for (uint32_t i = 0; i < 32; i++) total += warp_sums[i];
        info[3] = total;
    }
    if (!acc) return;
    idx += base + __popc(bal & ((1u << lane) - 1u));
    const a3_decode dc = dec[k];
    const uint32_t frame = qframe[k], rot = dc.rotation & 3u;
    const uint32_t *q = quads + (size_t)k * 8;
    a3_marker m;
    m.id = dc.id;
    m.code = dc.codes[rot];
    for (uint32_t cc = 0; cc < 4; cc++) {  // corners.rotate_left(min_rotation)
        const uint32_t sidx = (cc + rot) & 3u;
        m.corners[2 * cc] = q[2 * sidx];
        m.corners[2 * cc + 1] = q[2 * sidx + 1];
    }
    m.frame = frame;
    m.candidate = k - qoff[frame];
    m.hamming_distance = dc.hamming_distance;
    m.rotation = dc.rotation;
    m.corners_refined = refined ? refined_ok[k] : 0;
    for (int i = 0; i < 5; i++) m.reserved[i] = 0;
    markers[idx] = m;
    if (poses) { mposes[2 * (size_t)idx] = poses[2 * (size_t)k]; mposes[2 * (size_t)idx + 1] = poses[2 * (size_t)k + 1]; }
    if (refined)  // K5 wrote them in marker order already
        for (int i = 0; i < 8; i++) mcorners[8 * (size_t)idx + i] = refined[8 * (size_t)k + i];
}

// K1 over `p`.  LumaA8 / 16-bit frames first go through K0 (image's into_luma8 for those variants) into the detector's Luma8
// scratch, rows padded to 16 bytes so that the warp-strip kernel stays eligible, and K1 then takes its Luma8 pass-through.
cudaError_t run_k1(a3_detector *d, K1Params p, const K1Tuning *tune, cudaStream_t s) {
    if (fmt_wide(p.format)) {
        const size_t lp = ((size_t)p.w + 15) & ~(size_t)15, lf = lp * p.h;
        cudaError_t e = d->d_luma.reserve(lf * p.n);
        if (e == cudaSuccess) e = k0_to_luma8(p.src, p.format, p.n, p.w, p.h, p.pitch, p.frame_stride, d->d_luma.p, lp, lf, s);
        if (e != cudaSuccess) return e;
        p.src = d->d_luma.p; p.format = A3_FMT_LUMA8; p.pitch = lp; p.frame_stride = lf;
    }
    return k1_gray_threshold(p, tune, s, nullptr);
}

K2Params k2_params(const a3_detector *d, const uint8_t *grey, uint32_t w, uint32_t h) {
    K2Params p;
    p.grey = grey; p.w = w; p.h = h; p.quads = nullptr; p.quad_frame = nullptr; p.n_quads = 0;
    p.patch_size = d->cfg.homography_sample_size; p.mark_size = d->mark_size; p.codes = d->d_codes.p;
    p.n_codes = d->dict.n_codes; p.tau = d->dict.tau; p.filter_high_bit_errors = d->cfg.filter_high_bit_errors;
    p.resize_w = d->d_taps.p; p.resize_meta = d->d_meta.p; p.decodes = nullptr; p.patches = nullptr;
    return p;
}

StagePlan plan_stages(const a3_detector *d, bool poses, bool refine, bool board) {
    StagePlan sp;
    sp.poses = poses; sp.refine = refine; sp.board = board;
    if (!d->opt.dist_on) return sp;
    sp.und_pose = poses;
    sp.und_board = board;
    const bool shared = poses && board && memcmp(&d->opt.pose_k, &d->opt.board_k, sizeof(a3_camera_intrinsics)) == 0;
    sp.und_sets = (poses ? 1u : 0u) + ((board && !shared) ? 1u : 0u);
    sp.und_board_set = (poses && !shared) ? 1u : 0u;
    return sp;
}

// K2's work counter: beyond one wave of warps (2048 quads) the warps share the quads out through a counter that is zero at
// launch: `zeroed` when the caller has one, else the detector's own after a memset on `s`.  Null below that.
cudaError_t k2_queue(a3_detector *d, uint32_t n_quads, uint32_t *zeroed, cudaStream_t s, uint32_t **queue) {
    *queue = nullptr;
    if (n_quads <= 2048) return cudaSuccess;
    if (zeroed) { *queue = zeroed; return cudaSuccess; }
    cudaError_t e = d->d_k2queue.reserve(1);
    if (e == cudaSuccess) e = cudaMemsetAsync(d->d_k2queue.p, 0, 4, s);
    if (e == cudaSuccess) *queue = d->d_k2queue.p;
    return e;
}

// What the post-decode chain reads: n candidates (quads, their frames) on the grey frames, and per-route extras
struct ChainIn {
    const uint8_t *grey = nullptr;
    uint32_t w = 0, h = 0;
    const uint32_t *quads = nullptr, *qframe = nullptr;
    uint32_t n = 0;                       // launch size
    const uint32_t *n_dev = nullptr;      // device, optional: the real number of candidates
    uint32_t *queue = nullptr;            // K2's work counter (k2_queue) or null
    uint32_t *accept_counts = nullptr;    // K2's accepted count per 1024 quads (assemble_markers_kernel) or null
    uint8_t *patches = nullptr;           // K2's sampled patches or null
    const uint32_t *offsets = nullptr;    // K6: candidates of frame f are [offsets[f], offsets[f + 1])
    const uint32_t *skip = nullptr;       // K6: device flag or null, non-zero = write nothing
    uint32_t n_frames = 0;
};

// The post-decode stages of one decode group on stream s: K2 -> K5 -> K7 (each set) -> K4 -> K6, into `out` laid out by `l`.
// Each timed stage is bracketed by the block's pair of events and marked as recorded.
cudaError_t enqueue_chain(const a3_detector *d, const StagePlan &sp, const ChainIn &in, uint8_t *out, const OutLayout &l, DecodeBlock &b,
                          cudaStream_t s) {
    const Options &o = d->opt;
    a3_decode *dec = reinterpret_cast<a3_decode *>(out + l.dec);
    float *ref = sp.refine ? reinterpret_cast<float *>(out + l.ref) : nullptr;
    float *norm = reinterpret_cast<float *>(out + l.norm);
    uint8_t *nok = out + l.nok;
    auto timed = [&](Stage st, auto &&launch) {
        cudaError_t e = cudaEventRecord(b.ev[st][0], s);
        if (e == cudaSuccess) e = launch();
        if (e == cudaSuccess) e = cudaEventRecord(b.ev[st][1], s);
        if (e == cudaSuccess) b.timed |= 1u << st;
        return e;
    };
    K2Params p2 = k2_params(d, in.grey, in.w, in.h);
    p2.quads = in.quads; p2.quad_frame = in.qframe; p2.n_quads = in.n; p2.n_quads_dev = in.n_dev; p2.queue = in.queue;
    p2.accept_counts = in.accept_counts; p2.decodes = dec; p2.patches = in.patches;
    cudaError_t e = timed(kDecode, [&] { return k2_decode(p2, s); });
    if (e == cudaSuccess && sp.refine) {  // on K2's accepted candidates
        K5Params p5{};
        p5.grey = in.grey; p5.w = in.w; p5.h = in.h; p5.quads = in.quads; p5.quad_frame = in.qframe; p5.decodes = dec;
        p5.n = in.n; p5.n_dev = in.n_dev; p5.corners = ref; p5.ok = out + l.refok;
        e = timed(kRefine, [&] { return k5_corners(p5, s); });
    }
    if (e == cudaSuccess && sp.und_sets)  // the corners K4 and K6 read
        e = timed(kUndistort, [&] {
            cudaError_t r = cudaSuccess;
            for (uint32_t j = 0; j < sp.und_sets && r == cudaSuccess; j++) {
                K7Params p7;
                p7.quads = in.quads; p7.corners_f32 = ref; p7.decodes = dec; p7.n = in.n; p7.n_dev = in.n_dev;
                p7.k = (j == 0 && sp.und_pose) ? o.pose_k : o.board_k; p7.dist = o.dist;
                p7.out = norm + (size_t)in.n * 8 * j; p7.ok = nok + (size_t)in.n * j;
                r = k7_undistort(p7, s);
            }
            return r;
        });
    if (e == cudaSuccess && sp.poses) {
        K4Params p4{};
        p4.mode = o.pose_mode; p4.corners = in.quads; p4.corners_f32 = ref; p4.decodes = dec; p4.n = in.n; p4.n_dev = in.n_dev;
        p4.marker_size = o.pose_marker_size; p4.image_w = in.w; p4.image_h = in.h; p4.k = o.pose_k;
        p4.poses = reinterpret_cast<a3_pose *>(out + l.pose);
        if (sp.und_pose) { p4.mode = A3_POSE_NORMALIZED; p4.points = norm; p4.points_ok = nok; }
        e = k4_pose(p4, s);
    }
    if (e == cudaSuccess && sp.board) {
        K6Params p6;
        p6.decodes = dec; p6.quads = in.quads; p6.corners_f32 = ref; p6.offsets = in.offsets; p6.skip = in.skip; p6.n_frames = in.n_frames;
        p6.slots = d->d_board_slots.p; p6.n_codes = d->dict.n_codes; p6.board = d->d_board_pts.p; p6.n_board = o.board_n;
        p6.mode = o.board_mode; p6.image_w = in.w; p6.image_h = in.h; p6.k = o.board_k;
        p6.out = reinterpret_cast<a3_board_pose *>(out + l.board);
        if (sp.und_board) { p6.norm = norm + (size_t)in.n * 8 * sp.und_board_set; p6.norm_ok = nok + (size_t)in.n * sp.und_board_set; }
        e = timed(kBoard, [&] { return k6_board(p6, s); });
    }
    return e;
}

// The stage times the block recorded in this call, summed; each is also added to its a3_stats field when `st` is given
double stage_ms(const DecodeBlock &b, a3_stats *st) {
    double sum = 0;
    for (int i = 0; i < kStages; i++) {
        if (!(b.timed >> i & 1u)) continue;
        float ms = 0;
        cudaEventElapsedTime(&ms, b.ev[i][0], b.ev[i][1]);
        sum += ms;
        if (st) st->*kStageMs[i] += ms;
    }
    return sum;
}

}  // namespace
}  // namespace a3

using namespace a3;

static std::atomic<uint64_t> g_created{0};        // successful a3_detector_create calls (a3_detector_create_count)
static std::mutex g_cache_mu;                     // idle handles of a3_detector_acquire / a3_detector_release, oldest first
static std::vector<a3_detector *> g_cache;
static constexpr size_t kCacheMax = 16;

extern "C" {

const char *a3_version(void) { return "aruco3_b200 0.1.0 (sm_100a)"; }
const char *a3_last_error(void) { return g_error.c_str(); }
const char *a3_status_string(a3_status s) {
    switch (s) {
        case A3_OK: return "ok";
        case A3_ERR_INVALID_ARGUMENT: return "invalid argument";
        case A3_ERR_UNKNOWN_DICTIONARY: return "unknown dictionary";
        case A3_ERR_CUDA: return "CUDA error";
        case A3_ERR_CAPACITY: return "output capacity too small";
        case A3_ERR_UNSUPPORTED: return "unsupported";
        case A3_ERR_OUT_OF_MEMORY: return "out of memory";
        default: return "unknown status";
    }
}
int32_t a3_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void a3_config_default(a3_config *c) {
    if (!c) return;
    c->threshold_window = 7;
    c->contour_simplification_epsilon = 0.05;
    c->min_side_length_factor = 0.2f;
    c->min_corner_separation_factor = 0.1f;
    c->homography_sample_size = 49;
    c->filter_high_bit_errors = 1;
}

a3_status a3_detector_create(const a3_config *cfg, const a3_dictionary *dict, int32_t device, a3_detector **out) {
    if (!cfg || !dict || !out || !dict->codes) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_create: null argument");
    if (a3_status s = check_config(*cfg)) return s;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(A3_ERR_CUDA, "no CUDA device: aruco3_b200 has no CPU fallback");
    }
    if (device < 0 || device >= ndev) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_create: bad device index");
    A3_CUDA(cudaSetDevice(device));
    a3_detector *d = new a3_detector();
    d->cfg = *cfg;
    d->dict = *dict;
    d->device = device;
    d->mark_size = mark_size_of(dict->num_bits);
    uint32_t hc = std::thread::hardware_concurrency();
    d->host_threads = hc ? (hc > 64 ? 64 : hc) : 1;
    if (!k2_supported(cfg->homography_sample_size, d->mark_size, dict->n_codes)) {
        a3_detector_destroy(d);
        return fail(A3_ERR_UNSUPPORTED, "homography_sample_size is too large for the CUDA path: one sampled patch (size^2 bytes) and the dictionary "
                                        "must fit the 220 KB of shared memory of an SM (about 400 with the shipped dictionaries)");
    }
    ResizeTaps tp = make_resize_taps(cfg->homography_sample_size, d->mark_size);
    d->max_taps = tp.max_taps;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = d->d_codes.reserve(dict->n_codes ? dict->n_codes : 1);
    if (e == cudaSuccess && dict->n_codes) e = cudaMemcpy(d->d_codes.p, dict->codes, (size_t)dict->n_codes * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = d->d_taps.reserve(tp.weights.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_taps.p, tp.weights.data(), tp.weights.size() * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = d->d_meta.reserve(tp.meta.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_meta.p, tp.meta.data(), tp.meta.size() * 4, cudaMemcpyHostToDevice);
    for (cudaStream_t *s : {&d->s_copy, &d->s_pixel, &d->s_decode})
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        a3_detector_destroy(d);
        return cuda_fail(e, "a3_detector_create");
    }
    g_created.fetch_add(1);
    *out = d;
    return A3_OK;
}

uint64_t a3_detector_create_count(void) { return g_created.load(); }

// ---- handle cache -------------------------------------------------------------------------------------------------
// The reference's `Detector` is plain data built with a struct literal (src/aruco.rs:46-49, benches/detect_markers.rs:17-20),
// so a binding that keeps that shape has nowhere to store a handle.  It brackets every call with acquire / release instead:
// an idle handle with exactly this config, dictionary and device comes out of the cache warm (streams, device and pinned
// buffers, K3 workspace and the one-shot history all survive), and a new one is created only when none is idle.
a3_status a3_detector_acquire(const a3_config *cfg, const a3_dictionary *dict, int32_t device, a3_detector **out) {
    if (!cfg || !dict || !out) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_acquire: null argument");
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        for (size_t i = g_cache.size(); i-- > 0;) {  // most recently released first
            a3_detector *d = g_cache[i];
            const a3_config &c = d->cfg;
            if (d->device == device && c.threshold_window == cfg->threshold_window &&
                c.contour_simplification_epsilon == cfg->contour_simplification_epsilon &&
                c.min_side_length_factor == cfg->min_side_length_factor && c.min_corner_separation_factor == cfg->min_corner_separation_factor &&
                c.homography_sample_size == cfg->homography_sample_size && (c.filter_high_bit_errors != 0) == (cfg->filter_high_bit_errors != 0) &&
                d->dict.codes == dict->codes && d->dict.n_codes == dict->n_codes && d->dict.num_bits == dict->num_bits && d->dict.tau == dict->tau) {
                g_cache.erase(g_cache.begin() + (long)i);
                *out = d;
                return A3_OK;
            }
        }
    }
    return a3_detector_create(cfg, dict, device, out);
}

void a3_detector_release(a3_detector *d) {
    if (!d) return;
    d->opt = Options{};  // back to the state a3_detector_create leaves a handle in (the buffers stay)
    a3_detector *evict = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        g_cache.push_back(d);
        if (g_cache.size() > kCacheMax) { evict = g_cache.front(); g_cache.erase(g_cache.begin()); }
    }
    if (evict) a3_detector_destroy(evict);
}

void a3_detector_cache_clear(void) {
    std::vector<a3_detector *> all;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        all.swap(g_cache);
    }
    for (a3_detector *d : all) a3_detector_destroy(d);
}

void a3_detector_destroy(a3_detector *d) {
    if (!d) return;
    cudaSetDevice(d->device);
    for (cudaStream_t s : {d->s_copy, d->s_pixel, d->s_decode})
        if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
    d->copy_pool.stop();  // its tasks use the staging rings, which go with the handle
    delete d;             // buffers and events free themselves, on the device set above
}

a3_status a3_detector_set_host_threads(a3_detector *d, uint32_t threads) {
    if (!d || threads == 0) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_host_threads: bad argument");
    d->host_threads = threads > 256 ? 256 : threads;
    return A3_OK;
}

a3_status a3_detector_set_contour_mode(a3_detector *d, uint32_t mode) {
    if (!d || mode > A3_CONTOURS_DEVICE) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_contour_mode: bad argument");
    d->opt.contour_mode = mode;
    return A3_OK;
}

a3_status a3_detector_set_corner_refinement(a3_detector *d, uint32_t mode) {
    if (!d || mode > A3_CORNERS_REFINED) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_corner_refinement: bad argument");
    d->opt.corner_mode = mode;
    return A3_OK;
}

a3_status a3_detector_set_k1_tuning(a3_detector *d, const a3_k1_tuning *t) {
    if (!d) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_k1_tuning: null detector");
    d->opt.has_tuning = t != nullptr;
    d->opt.k1_tuning = K1Tuning{};
    d->opt.chunk_override = 0;
    if (t) {
        d->opt.k1_tuning.strip_cols = t->strip_cols; d->opt.k1_tuning.seg_rows = t->seg_rows; d->opt.k1_tuning.force_no_tma = (int)t->force_no_tma;
        d->opt.k1_tuning.force_generic = (int)t->force_generic;
        d->opt.chunk_override = t->chunk_frames;
    }
    return A3_OK;
}

a3_status a3_gray_threshold_batch(a3_detector *d, const void *frames, a3_format format, a3_mem_kind mem, uint32_t n,
                                  uint32_t w, uint32_t h, size_t pitch, size_t frame_stride, uint8_t *grey, uint8_t *mask,
                                  uint32_t *mask_bits, void *cuda_stream) {
    if (!d || !frames) return fail(A3_ERR_INVALID_ARGUMENT, "a3_gray_threshold_batch: null argument");
    if (!fmt_valid((int)format)) return fail(A3_ERR_INVALID_ARGUMENT, "bad format");
    if (n == 0 || w == 0 || h == 0) return A3_OK;
    const uint32_t bpp = bytes_per_pixel(format);
    if (pitch < (size_t)w * bpp || frame_stride < pitch * h) return fail(A3_ERR_INVALID_ARGUMENT, "pitch / frame_stride too small");
    A3_CUDA(cudaSetDevice(d->device));
    const K1Tuning *tune = d->opt.has_tuning ? &d->opt.k1_tuning : nullptr;
    K1Params p;
    p.format = format; p.n = n; p.w = w; p.h = h; p.pitch = pitch; p.frame_stride = frame_stride; p.radius = d->cfg.threshold_window;
    if (mem == A3_MEM_DEVICE) {
        p.src = static_cast<const uint8_t *>(frames); p.grey = grey; p.mask = mask; p.bits = mask_bits;
        A3_CUDA(run_k1(d, p, tune, static_cast<cudaStream_t>(cuda_stream)));
        return A3_OK;
    }
    // host pointers: stage chunk by chunk, synchronously
    cudaStream_t s = d->s_pixel;
    const size_t px = (size_t)w * h, wpr = (w + 31) / 32;
    size_t chunk = ((size_t)512 << 20) / (frame_stride + 2 * px + 1);
    if (chunk < 1) chunk = 1;
    if (chunk > n) chunk = n;
    for (uint32_t f0 = 0; f0 < n; f0 += (uint32_t)chunk) {
        const uint32_t c = n - f0 < chunk ? n - f0 : (uint32_t)chunk;
        A3_CUDA(d->d_src.reserve((size_t)c * frame_stride));
        A3_CUDA(cudaMemcpyAsync(d->d_src.p, static_cast<const uint8_t *>(frames) + (size_t)f0 * frame_stride,
                                input_span(c, w, h, bpp, pitch, frame_stride), cudaMemcpyHostToDevice, s));
        if (grey) A3_CUDA(d->d_grey.reserve(c * px));
        if (mask) A3_CUDA(d->d_mask.reserve(c * px));
        if (mask_bits) A3_CUDA(d->d_bits.reserve(c * wpr * h));
        p.src = d->d_src.p; p.n = c;
        p.grey = grey ? d->d_grey.p : nullptr; p.mask = mask ? d->d_mask.p : nullptr; p.bits = mask_bits ? d->d_bits.p : nullptr;
        A3_CUDA(run_k1(d, p, tune, s));
        if (grey) A3_CUDA(cudaMemcpyAsync(grey + f0 * px, d->d_grey.p, c * px, cudaMemcpyDeviceToHost, s));
        if (mask) A3_CUDA(cudaMemcpyAsync(mask + f0 * px, d->d_mask.p, c * px, cudaMemcpyDeviceToHost, s));
        if (mask_bits) A3_CUDA(cudaMemcpyAsync(mask_bits + f0 * wpr * h, d->d_bits.p, c * wpr * h * 4, cudaMemcpyDeviceToHost, s));
        A3_CUDA(cudaStreamSynchronize(s));
    }
    return A3_OK;
}

a3_status a3_quads_from_mask(const a3_config *cfg, const uint8_t *mask, uint32_t w, uint32_t h, uint32_t *quads,
                             uint32_t quad_capacity, uint32_t *n_quads, a3_stats *stats) {
    if (!cfg || !mask || !n_quads) return fail(A3_ERR_INVALID_ARGUMENT, "a3_quads_from_mask: null argument");
    if (a3_status s = check_config(*cfg)) return s;
    std::vector<uint32_t> bits, q;
    uint32_t wpr = 0;
    bits_from_mask(mask, w, h, bits, &wpr);
    QuadStats qs;
    quads_from_bits(bits.data(), wpr, w, h, *cfg, q, &qs);
    *n_quads = (uint32_t)(q.size() / 8);
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->n_frames = 1; stats->n_contours = qs.n_contours; stats->n_contour_points = qs.n_contour_points;
        stats->n_candidates_before_discard = qs.n_before_discard; stats->n_candidates = *n_quads;
    }
    if (*n_quads > quad_capacity || (!quads && *n_quads)) return fail(A3_ERR_CAPACITY, "a3_quads_from_mask: quad_capacity too small");
    if (*n_quads) memcpy(quads, q.data(), q.size() * 4);
    return A3_OK;
}

a3_status a3_quads_from_masks_device(a3_detector *d, const uint8_t *masks, uint32_t n, uint32_t w, uint32_t h, uint32_t *quads,
                                     uint32_t quad_capacity, uint32_t *counts, uint32_t *flags, uint32_t *contours, uint64_t *points) {
    if (!d || !masks || !quads || !counts || !flags || quad_capacity == 0)
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_quads_from_masks_device: null argument");
    if (n == 0 || w == 0 || h == 0) return A3_OK;
    if (w > 65535 || h > 65535 || (uint64_t)w * h >= (1ull << 29))
        return fail(A3_ERR_UNSUPPORTED, "a3_quads_from_masks_device: frames larger than 65535 pixels a side or 2^29 pixels");
    A3_CUDA(cudaSetDevice(d->device));
    const uint32_t wpr = (w + 31) / 32, Hp = h + 2;
    const size_t plane_words = (size_t)(wpr + 2) * Hp;
    std::vector<uint32_t> planes((size_t)n * plane_words, 0u);
    for (uint32_t f = 0; f < n; f++)
        for (uint32_t y = 0; y < h; y++)
            for (uint32_t x = 0; x < w; x++)
                if (masks[((size_t)f * h + y) * w + x]) planes[(size_t)f * plane_words + (size_t)((x >> 5) + 1) * Hp + (y + 1)] |= 1u << (x & 31);
    cudaStream_t s = d->s_pixel;
    d->planes_zeroed_words = 0;  // the pipeline's guard words are overwritten below
    A3_CUDA(d->d_planes.reserve(planes.size()));
    A3_CUDA(d->d_k3quads.reserve((size_t)n * quad_capacity * 8));
    A3_CUDA(d->d_k3frames.reserve(K3Frames::bytes(n)));
    A3_CUDA(cudaMemcpyAsync(d->d_planes.p, planes.data(), planes.size() * 4, cudaMemcpyHostToDevice, s));
    const K3Frames k3f(d->d_k3frames.p, n);
    A3_CUDA(k3_quads(d->k3, k3_params(d->cfg, d->d_planes.p, w, h, 0, n, d->d_k3quads.p, quad_capacity, k3f), s));
    A3_CUDA(cudaMemcpyAsync(quads, d->d_k3quads.p, (size_t)n * quad_capacity * 32, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaMemcpyAsync(counts, k3f.counts, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaMemcpyAsync(flags, k3f.flags, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    if (contours) A3_CUDA(cudaMemcpyAsync(contours, k3f.contours, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    if (points) A3_CUDA(cudaMemcpyAsync(points, k3f.points, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaStreamSynchronize(s));
    return A3_OK;
}

a3_status a3_decode_candidates(a3_detector *d, const uint8_t *grey, uint32_t n_frames, uint32_t w, uint32_t h,
                               const uint32_t *quads, const uint32_t *quad_frame, uint32_t n_quads, a3_decode *decodes,
                               uint8_t *patches) {
    if (!d || !grey || (!quads && n_quads) || (!decodes && n_quads)) return fail(A3_ERR_INVALID_ARGUMENT, "a3_decode_candidates: null argument");
    if (n_quads == 0) return A3_OK;
    for (uint32_t i = 0; quad_frame && i < n_quads; i++)
        if (quad_frame[i] >= n_frames) return fail(A3_ERR_INVALID_ARGUMENT, "a3_decode_candidates: quad_frame out of range");
    A3_CUDA(cudaSetDevice(d->device));
    cudaStream_t s = d->s_decode;
    const size_t px = (size_t)w * h, np = (size_t)d->cfg.homography_sample_size * d->cfg.homography_sample_size;
    A3_CUDA(d->d_grey.reserve(px * n_frames));
    A3_CUDA(d->d_quads.reserve((size_t)n_quads * 8));
    A3_CUDA(d->d_qframe.reserve(n_quads));
    A3_CUDA(d->d_dec.reserve(n_quads));
    if (patches) A3_CUDA(d->d_patches.reserve(n_quads * np));
    A3_CUDA(cudaMemcpyAsync(d->d_grey.p, grey, px * n_frames, cudaMemcpyHostToDevice, s));
    A3_CUDA(cudaMemcpyAsync(d->d_quads.p, quads, (size_t)n_quads * 32, cudaMemcpyHostToDevice, s));
    if (quad_frame) A3_CUDA(cudaMemcpyAsync(d->d_qframe.p, quad_frame, (size_t)n_quads * 4, cudaMemcpyHostToDevice, s));
    K2Params p = k2_params(d, d->d_grey.p, w, h);
    p.quads = d->d_quads.p; p.quad_frame = quad_frame ? d->d_qframe.p : nullptr; p.n_quads = n_quads;
    p.decodes = d->d_dec.p; p.patches = patches ? d->d_patches.p : nullptr;
    A3_CUDA(k2_queue(d, n_quads, nullptr, s, &p.queue));
    A3_CUDA(k2_decode(p, s));
    A3_CUDA(cudaMemcpyAsync(decodes, d->d_dec.p, (size_t)n_quads * sizeof(a3_decode), cudaMemcpyDeviceToHost, s));
    if (patches) A3_CUDA(cudaMemcpyAsync(patches, d->d_patches.p, n_quads * np, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaStreamSynchronize(s));
    return A3_OK;
}

a3_status a3_refine_corners(a3_detector *d, const uint8_t *grey, uint32_t n_frames, uint32_t w, uint32_t h, const uint32_t *corners,
                            const uint32_t *corner_frame, uint32_t n, float *refined, uint8_t *ok) {
    if (!d || !grey || (n && (!corners || !refined || !ok))) return fail(A3_ERR_INVALID_ARGUMENT, "a3_refine_corners: null argument");
    if (n == 0) return A3_OK;
    if (n_frames == 0 || w == 0 || h == 0) return fail(A3_ERR_INVALID_ARGUMENT, "a3_refine_corners: empty grey frames");
    for (uint32_t i = 0; corner_frame && i < n; i++)
        if (corner_frame[i] >= n_frames) return fail(A3_ERR_INVALID_ARGUMENT, "a3_refine_corners: corner_frame out of range");
    A3_CUDA(cudaSetDevice(d->device));
    cudaStream_t s = d->s_decode;
    const size_t px = (size_t)w * h;
    A3_CUDA(d->d_grey.reserve(px * n_frames));
    A3_CUDA(d->d_quads.reserve((size_t)n * 8));
    A3_CUDA(d->d_qframe.reserve(n));
    A3_CUDA(d->d_refined.reserve((size_t)n * 8));
    A3_CUDA(d->d_refined_ok.reserve(n));
    A3_CUDA(cudaMemcpyAsync(d->d_grey.p, grey, px * n_frames, cudaMemcpyHostToDevice, s));
    A3_CUDA(cudaMemcpyAsync(d->d_quads.p, corners, (size_t)n * 32, cudaMemcpyHostToDevice, s));
    if (corner_frame) A3_CUDA(cudaMemcpyAsync(d->d_qframe.p, corner_frame, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    K5Params kp{};
    kp.grey = d->d_grey.p; kp.w = w; kp.h = h; kp.quads = d->d_quads.p; kp.quad_frame = corner_frame ? d->d_qframe.p : nullptr;
    kp.decodes = nullptr; kp.n = n; kp.corners = d->d_refined.p; kp.ok = d->d_refined_ok.p;
    A3_CUDA(k5_corners(kp, s));
    A3_CUDA(cudaMemcpyAsync(refined, d->d_refined.p, (size_t)n * 32, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaMemcpyAsync(ok, d->d_refined_ok.p, n, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaStreamSynchronize(s));
    return A3_OK;
}

a3_status a3_detect_batch(a3_detector *d, const void *frames, a3_format format, a3_mem_kind mem, uint32_t n, uint32_t w,
                          uint32_t h, size_t pitch, size_t frame_stride, a3_marker *markers, uint32_t marker_capacity,
                          uint32_t *n_markers, a3_outputs *outs, a3_stats *stats) {
    if (!d || !frames || !n_markers) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detect_batch: null argument");
    if (!fmt_valid((int)format)) return fail(A3_ERR_INVALID_ARGUMENT, "bad format");
    *n_markers = 0;
    if (outs) outs->n_candidates = 0;
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n == 0 || w == 0 || h == 0) {
        if (outs && outs->frame_marker_offsets) memset(outs->frame_marker_offsets, 0, ((size_t)n + 1) * 4);
        return A3_OK;
    }
    const uint32_t bpp = bytes_per_pixel(format);
    if (pitch < (size_t)w * bpp || frame_stride < pitch * h) return fail(A3_ERR_INVALID_ARGUMENT, "pitch / frame_stride too small");
    A3_CUDA(cudaSetDevice(d->device));
    const double t_begin = now_ms();
    const size_t px = (size_t)w * h, wpr = (w + 31) / 32, bits_words = wpr * h;
    const size_t np = (size_t)d->cfg.homography_sample_size * d->cfg.homography_sample_size;
    const bool want_mask = outs && outs->mask, want_grey = outs && outs->grey, want_patches = outs && outs->homographies;
    const bool want_poses = outs && outs->marker_poses && markers && d->opt.pose_mode != A3_POSE_OFF;
    // K6 solves the board's pose per frame (a3_outputs.board_poses), whatever else the caller asked for
    const bool want_board = d->opt.board_n > 0 && outs && outs->board_poses;  // no board: the field is never read
    // K5 refines the markers' corners (a3_marker.corners_refined, a3_outputs.marker_corners); K4 and K6 then solve from them
    const bool want_refine = (markers || want_board) && d->opt.corner_mode == A3_CORNERS_REFINED;
    float *const out_corners = want_refine && markers && outs ? outs->marker_corners : nullptr;
    // K7 undistorts the corners K4 and K6 read when their intrinsics have a distortion
    const StagePlan plan = plan_stages(d, want_poses, want_refine, want_board);
    const K1Tuning *tune = d->opt.has_tuning ? &d->opt.k1_tuning : nullptr;
    const uint8_t *src_all = static_cast<const uint8_t *>(frames);
    a3_stats st;
    memset(&st, 0, sizeof(st));
    st.n_frames = n;
    st.host_threads = d->host_threads;
    if (d->pool.size() != d->host_threads) d->pool.resize(d->host_threads);
    // Pageable host memory at the boundary (the Vec<u8> of a `DynamicImage`, a `Detection.grey` the caller got from malloc): a
    // cudaMemcpyAsync on it is neither asynchronous nor fast, so such buffers go through pinned rings that the copy threads
    // fill (input) or empty (grey) one front-end chunk ahead of / behind the DMA.
    auto is_pageable = [](const void *ptr) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) { cudaGetLastError(); return true; }
        return at.type == cudaMemoryTypeUnregistered;
    };
    static const bool no_staging = getenv("A3_NO_HOST_STAGING") != nullptr;
    const bool stage_in = mem == A3_MEM_HOST && !no_staging && (size_t)n * frame_stride >= ((size_t)1 << 20) && is_pageable(frames);
    const bool stage_out = want_grey && !no_staging && (size_t)n * px >= ((size_t)1 << 20) && is_pageable(outs->grey);
    if (stage_in || stage_out) d->copy_pool.start(d->host_threads < 16u ? d->host_threads : 16u, d->device);
    st.input_staged = stage_in ? 1u : 0u;
    st.output_staged = stage_out ? 1u : 0u;

    // ---- sizes: super-batch (device footprint), front-end chunk (copy / event granularity), decode group ----
    size_t sb = ((size_t)3 << 30) / (px + bits_words * 4 + (want_mask ? px : 0));  // grey + bits (+ mask) stay resident per frame
    if (sb < 1) sb = 1;
    if (sb > n) sb = n;
    size_t fe = ((size_t)96 << 20) / (frame_stride ? frame_stride : 1);           // ~96 MB of input per front-end chunk
    if (d->opt.chunk_override) fe = d->opt.chunk_override;
    if (fe < 1) fe = 1;
    if (fe > 64) fe = 64;
    if (fe > sb) fe = sb;
    uint32_t group = 32;          // frames per decode launch
    const uint32_t kStaging = 3;  // staging ring depth (host input)
    // contour stage on the device (K3) unless the caller asked for the host stage or the frame is too large for K3's 16-bit points
    const bool gpu_contours = d->opt.contour_mode == A3_CONTOURS_DEVICE && w <= 65535 && h <= 65535 && (uint64_t)w * h < (1ull << 29);
    // resident input + device contours: every quad of the super-batch is known at once, so one decode launch keeps the
    // whole GPU busy (K2 is latency-bound: what counts is candidates in flight)
    if (gpu_contours && mem == A3_MEM_DEVICE) {
        group = (uint32_t)sb;
        fe = sb;  // nothing to stage and one K3 launch: one front-end unit per super-batch
    }
    // One-shot route: when one K3 launch covers the whole (super-)batch — resident input, or host input that fits one
    // front-end chunk, e.g. a single frame — the second half of K3, the gather of its quads, K2 and K4 are all queued behind
    // K1 without a host synchronisation, sized from the previous call of the same geometry; the host synchronises once at the
    // end, checks that the sizes held and otherwise takes the ordinary route from where the speculation stopped.
    const bool one_shot = gpu_contours && (mem == A3_MEM_DEVICE || n <= fe) && !getenv("A3_NO_ONE_SHOT");
    if (one_shot) group = (uint32_t)sb;
    const uint32_t Hp = h + 2;                               // guarded column-major plane: words per 32-pixel column
    const size_t plane_words = (size_t)(wpr + 2) * Hp;       // words per frame
    const uint32_t quad_cap = 1024;                          // quads per frame K3 can return (more -> host stage)
    const uint32_t quad_head = 64;                           // quads per frame copied back unconditionally

    uint32_t total_markers = 0, total_cands = 0;
    bool overflow = false;
    std::vector<std::vector<uint32_t>> &frame_quads = d->frame_quads;  // kept in the handle: no allocation per call once warm
    std::vector<QuadStats> frame_stats;
    std::vector<double> frame_ms;

    for (uint32_t s0 = 0; s0 < n; s0 += (uint32_t)sb) {
        const uint32_t sn = n - s0 < sb ? n - s0 : (uint32_t)sb;
        const uint32_t nfe = (sn + (uint32_t)fe - 1) / (uint32_t)fe, ngroups = (sn + group - 1) / group;
        A3_CUDA(d->d_grey.reserve(sn * px));
        if (gpu_contours) {
            const size_t need = (size_t)sn * plane_words;
            const bool fresh = need > d->d_planes.cap || d->planes_w != w || d->planes_h != h || need > d->planes_zeroed_words;
            A3_CUDA(d->d_planes.reserve(need));
            if (fresh) {  // guard words are written once and never touched by K1
                A3_CUDA(cudaMemsetAsync(d->d_planes.p, 0, d->d_planes.cap * 4, d->s_pixel));
                d->planes_zeroed_words = d->d_planes.cap; d->planes_w = w; d->planes_h = h;
            }
            A3_CUDA(d->d_k3quads.reserve((size_t)sn * quad_cap * 8)); A3_CUDA(d->h_k3quads.reserve((size_t)sn * quad_cap * 8));
            A3_CUDA(d->d_k3frames.reserve(K3Frames::bytes(sn))); A3_CUDA(d->h_k3frames.reserve(K3Frames::bytes(sn)));
            A3_CUDA(d->h_plane.reserve(plane_words));
        } else {
            A3_CUDA(d->d_bits.reserve(sn * bits_words));
            A3_CUDA(d->h_bits.reserve(sn * bits_words));
        }
        if (want_mask) A3_CUDA(d->d_mask.reserve(sn * px));
        if (mem == A3_MEM_HOST) A3_CUDA(d->d_src.reserve((size_t)kStaging * fe * frame_stride));
        while (d->blocks.size() < ngroups) {
            std::unique_ptr<DecodeBlock> b(new DecodeBlock());
            for (auto &pair : b->ev)
                for (cudaEvent_t &e : pair) A3_CUDA(cudaEventCreate(&e));
            d->blocks.push_back(std::move(b));
        }
        for (uint32_t g = 0; g < ngroups; g++) d->blocks[g]->timed = 0;
        // pinned rings for pageable memory: kHostRing front-end chunks of input, kOutRing sub-chunks (<= 32 MB) of grey
        constexpr uint32_t kHostRing = 6, kOutRing = 4;
        const size_t kPiece = (size_t)1 << 20;  // bytes per copy task
        const size_t in_slot_bytes = fe * frame_stride;
        const size_t out_slot_frames = ((size_t)32 << 20) / px ? ((size_t)32 << 20) / px : 1, out_slot_bytes = out_slot_frames * px;
        if (stage_in) A3_CUDA(d->h_stage_in.reserve((nfe < kHostRing ? nfe : kHostRing) * in_slot_bytes));
        if (stage_out) A3_CUDA(d->h_stage_out.reserve(kOutRing * out_slot_bytes));
        auto stg = std::make_shared<StageState>();
        if (stage_in) {
            stg->in_left.reset(new std::atomic<uint32_t>[nfe]);
            for (uint32_t j = 0; j < nfe; j++) stg->in_left[j].store(0);
        }
        uint32_t stage_submitted = 0;  // front-end chunks whose stage-in tasks are in the copy pool
        const bool shot = one_shot && s0 == 0 && sn == n;
        const bool shot_hist = shot && d->hist_nq && d->hist_nq_n == n && d->hist_nq_w == w && d->hist_nq_h == h;
        const uint32_t shot_cap = shot_hist ? d->hist_nq + d->hist_nq / 8 + 256 : 0;  // quads the arena holds
        // markers only (no per-candidate outputs requested): the device also assembles the markers, and the copy stops after them
        const bool lean = shot && markers && !(outs && (outs->candidates || outs->candidate_frame || outs->decodes || outs->homographies));
        const size_t off_stats = 16, off_markers = align16(off_stats + K3Frames::bytes(sn));
        const size_t off_mposes = off_markers + (lean ? (size_t)shot_cap * sizeof(a3_marker) : 0);
        const size_t off_mcorners = off_mposes + ((lean && want_poses) ? (size_t)shot_cap * 2 * sizeof(a3_pose) : 0);  // K5's, per marker
        const size_t off_out = align16(off_mcorners + ((lean && want_refine) ? (size_t)shot_cap * 32 : 0));  // the decode group's outputs
        const OutLayout shot_out = out_layout(plan, shot_cap, sn);
        const size_t off_quads = align16(off_out + shot_out.bytes);
        const size_t shot_bytes = off_quads + (size_t)shot_cap * 32;
        // what goes back to the host: lean calls stop before the per-candidate outputs, after the board poses
        const size_t shot_copy_bytes = lean ? off_out + shot_out.dec : shot_bytes;
        if (shot) {
            A3_CUDA(d->d_shot.reserve(shot_bytes)); A3_CUDA(d->h_shot.reserve(shot_bytes));
        }
        // K3's per-frame outputs: their own block, or (one-shot route) a section of the arena that goes back in one copy
        uint8_t *const ds_base = shot ? d->d_shot.p + off_stats : d->d_k3frames.p;
        uint8_t *const hs_base = shot ? d->h_shot.p + off_stats : d->h_k3frames.p;
        const K3Frames ds(ds_base, sn), hs(hs_base, sn);
        uint32_t *const d_info = reinterpret_cast<uint32_t *>(d->d_shot.p);
        const uint32_t *const h_info = reinterpret_cast<const uint32_t *>(d->h_shot.p);
        d->events.reset();
        std::vector<cudaEvent_t> ev_fe(nfe), ev_k1a(nfe), ev_k1b(nfe), ev_h2da(nfe), ev_h2db(nfe), ev_k3(nfe);
        for (uint32_t j = 0; j < nfe; j++) {
            A3_CUDA(d->events.get(&ev_fe[j])); A3_CUDA(d->events.get(&ev_k1a[j])); A3_CUDA(d->events.get(&ev_k1b[j]));
            A3_CUDA(d->events.get(&ev_h2da[j])); A3_CUDA(d->events.get(&ev_h2db[j])); A3_CUDA(d->events.get(&ev_k3[j]));
        }
        if (frame_quads.size() < sn) frame_quads.resize(sn);
        for (uint32_t i = 0; i < sn; i++) frame_quads[i].clear();
        frame_stats.assign(sn, QuadStats());
        frame_ms.assign(sn, 0.0);
        std::unique_ptr<std::atomic<uint32_t>[]> group_done(new std::atomic<uint32_t>[ngroups]);
        for (uint32_t g = 0; g < ngroups; g++) group_done[g].store(0);
        auto group_size = [&](uint32_t g) { return (g + 1) * group <= sn ? group : sn - g * group; };

        // ---- device front end of chunk j (asynchronous) ----
        auto k1_launch = [&](const uint8_t *src, uint32_t f0, uint32_t cn, uint32_t j) -> a3_status {
            K1Params p;
            p.src = src; p.format = format; p.n = cn; p.w = w; p.h = h; p.pitch = pitch; p.frame_stride = frame_stride;
            p.grey = d->d_grey.p + (size_t)f0 * px; p.mask = want_mask ? d->d_mask.p + (size_t)f0 * px : nullptr;
            p.radius = d->cfg.threshold_window;
            if (gpu_contours) {  // straight into the guarded planes K3 reads
                p.bits = d->d_planes.p + (size_t)f0 * plane_words + Hp + 1;
                p.bits_col_words = Hp; p.bits_row_words = 1; p.bits_frame_words = plane_words;
            } else {
                p.bits = d->d_bits.p + (size_t)f0 * bits_words;
            }
            A3_CUDA(cudaEventRecord(ev_k1a[j], d->s_pixel));
            A3_CUDA(run_k1(d, p, tune, d->s_pixel));
            A3_CUDA(cudaEventRecord(ev_k1b[j], d->s_pixel));
            st.pixel_kernel_launches++;
            return A3_OK;
        };
        // ---- device contour stage: copies of K3's results, and the one-shot route behind a speculative K3 finish ----
        K3Params k3_last{};
        bool k3_spec_inflight = false, one_shot_enqueued = false, one_shot_done = false, lean_done = false;
        uint32_t one_shot_cap = 0;
        auto k3_stats_d2h = [&](uint32_t f0, uint32_t kn) -> a3_status {
            if (kn == sn) {  // K3 covered the whole super-batch (every one-shot call, resident input): the block in one copy
                A3_CUDA(cudaMemcpyAsync(hs_base, ds_base, K3Frames::bytes(sn), cudaMemcpyDeviceToHost, d->s_pixel));
                return A3_OK;
            }
            A3_CUDA(cudaMemcpyAsync(hs.counts + f0, ds.counts + f0, (size_t)kn * 4, cudaMemcpyDeviceToHost, d->s_pixel));
            A3_CUDA(cudaMemcpyAsync(hs.before + f0, ds.before + f0, (size_t)kn * 4, cudaMemcpyDeviceToHost, d->s_pixel));
            A3_CUDA(cudaMemcpyAsync(hs.flags + f0, ds.flags + f0, (size_t)kn * 4, cudaMemcpyDeviceToHost, d->s_pixel));
            A3_CUDA(cudaMemcpyAsync(hs.contours + f0, ds.contours + f0, (size_t)kn * 4, cudaMemcpyDeviceToHost, d->s_pixel));
            A3_CUDA(cudaMemcpyAsync(hs.points + f0, ds.points + f0, (size_t)kn * 8, cudaMemcpyDeviceToHost, d->s_pixel));
            return A3_OK;
        };
        auto k3_head_d2h = [&](uint32_t f0, uint32_t kn) -> a3_status {
            // the first `quad_head` quads of every frame in one strided copy; a frame with more fetches the rest itself
            A3_CUDA(cudaMemcpy2DAsync(d->h_k3quads.p + (size_t)f0 * quad_cap * 8, (size_t)quad_cap * 32,
                                      d->d_k3quads.p + (size_t)f0 * quad_cap * 8, (size_t)quad_cap * 32, (size_t)quad_head * 32, kn,
                                      cudaMemcpyDeviceToHost, d->s_pixel));
            return A3_OK;
        };
        // gather K3's quads on the device, run the decode chain on them and copy everything back, all on the pixel stream
        auto enqueue_one_shot = [&]() -> a3_status {
            DecodeBlock &b = *d->blocks[0];
            const uint32_t cap = shot_cap, n_chunks = (cap + 1023) / 1024;
            uint32_t *d_quads = reinterpret_cast<uint32_t *>(d->d_shot.p + off_quads);
            uint8_t *d_out = d->d_shot.p + off_out;
            A3_CUDA(d->d_qoff.reserve((size_t)sn + 1 + n_chunks));  // frame offsets of the quads, then the accepted count of every 1024 quads
            uint32_t *d_accepted = d->d_qoff.p + sn + 1;
            A3_CUDA(b.d_qframe.reserve(cap));
            if (want_patches) A3_CUDA(b.d_patches.reserve(cap * np));
            pack_offsets_kernel<<<1, 1024, 0, d->s_pixel>>>(ds.counts, ds.flags, sn, quad_cap, cap, k3_speculation_failed_flag(d->k3), d->d_qoff.p, d_info,
                                                            d_accepted, n_chunks);
            A3_CUDA(cudaGetLastError());
            pack_quads_kernel<<<sn, 128, 0, d->s_pixel>>>(d->d_k3quads.p, d->d_qoff.p, quad_cap, cap, d_info, d_quads, b.d_qframe.p, 0u);
            A3_CUDA(cudaGetLastError());
            ChainIn in;
            in.grey = d->d_grey.p; in.w = w; in.h = h; in.quads = d_quads; in.qframe = b.d_qframe.p; in.n = cap; in.n_dev = d_info;
            in.queue = d_info + 2; in.accept_counts = lean ? d_accepted : nullptr; in.patches = want_patches ? b.d_patches.p : nullptr;
            in.offsets = d->d_qoff.p; in.skip = d_info + 1; in.n_frames = sn;
            A3_CUDA(enqueue_chain(d, plan, in, d_out, shot_out, b, d->s_pixel));
            if (lean) {
                assemble_markers_kernel<<<n_chunks, 1024, 0, d->s_pixel>>>(
                    reinterpret_cast<const a3_decode *>(d_out + shot_out.dec), d_quads, b.d_qframe.p, d->d_qoff.p,
                    want_poses ? reinterpret_cast<const a3_pose *>(d_out + shot_out.pose) : nullptr,
                    want_refine ? reinterpret_cast<const float *>(d_out + shot_out.ref) : nullptr, want_refine ? d_out + shot_out.refok : nullptr, cap,
                    d_info, d_accepted, reinterpret_cast<a3_marker *>(d->d_shot.p + off_markers), reinterpret_cast<a3_pose *>(d->d_shot.p + off_mposes),
                    reinterpret_cast<float *>(d->d_shot.p + off_mcorners));
                A3_CUDA(cudaGetLastError());
            }
            // everything the host needs in one copy: route info, K3's counters, then either the finished markers (+ poses) and
            // the board poses, or the group's outputs and the quads
            A3_CUDA(cudaMemcpyAsync(d->h_shot.p, d->d_shot.p, shot_copy_bytes, cudaMemcpyDeviceToHost, d->s_pixel));
            one_shot_enqueued = true; one_shot_cap = cap;
            return A3_OK;
        };
        // after the synchronisation: did every speculated size hold?  Then the frames' quads and the decode records are already
        // on the host.  Otherwise finish K3 exactly (if that was what failed) and fetch its quads the ordinary way.
        auto settle_one_shot = [&]() -> a3_status {
            const bool held = k3_speculation_held(d->k3, k3_last);
            k3_spec_inflight = false;
            if (held && one_shot_enqueued && h_info[1] == 0 && h_info[0] <= one_shot_cap) {
                DecodeBlock &b = *d->blocks[0];
                b.n_quads = h_info[0];
                b.set_views(d->h_shot.p + off_out, shot_out);
                const uint32_t *h_quads = reinterpret_cast<const uint32_t *>(d->h_shot.p + off_quads);
                uint32_t k = 0;
                for (uint32_t i = 0; i < sn; i++) {
                    const uint32_t m = hs.counts[i] < quad_cap ? hs.counts[i] : quad_cap;
                    if (!lean) frame_quads[i].assign(h_quads + (size_t)k * 8, h_quads + (size_t)(k + m) * 8);
                    hs.stats(i, frame_stats[i]);
                    k += m;
                }
                group_done[0].store(sn);
                d->hist_nq = b.n_quads ? b.n_quads : 1;
                plan.count(st);
                st.one_shot = 1;
                one_shot_done = true;
                lean_done = lean;
                return A3_OK;
            }
            if (!held || one_shot_enqueued) st.one_shot_retry = 1;
            one_shot_enqueued = false;
            d->blocks[0]->timed = 0;  // the ordinary route times its own chain
            if (!held) {
                A3_CUDA(k3_finish(d->k3, k3_last, d->s_pixel));
                if (a3_status s = k3_stats_d2h(0, sn)) return s;
            }
            if (a3_status s = k3_head_d2h(0, sn)) return s;
            A3_CUDA(cudaStreamSynchronize(d->s_pixel));
            return A3_OK;
        };
        // Detection.grey of frames [f0, f0 + cn): straight into page-locked memory, or through the pinned ring (the copy tasks
        // wait for the sub-chunk's event and move it on to the caller's buffer)
        auto grey_d2h = [&](uint32_t f0, uint32_t cn) -> a3_status {
            if (!stage_out) {
                A3_CUDA(cudaMemcpyAsync(outs->grey + (size_t)(s0 + f0) * px, d->d_grey.p + (size_t)f0 * px, (size_t)cn * px, cudaMemcpyDeviceToHost, d->s_pixel));
                return A3_OK;
            }
            CopyPool *cp = &d->copy_pool;
            for (uint32_t sub = 0; sub < cn; sub += (uint32_t)out_slot_frames) {
                const uint32_t m = cn - sub < out_slot_frames ? cn - sub : (uint32_t)out_slot_frames;
                const size_t q = stg->out.size(), bytes = (size_t)m * px;
                if (q >= kOutRing) {  // the slot's previous tenant must have left for the caller's buffer
                    StageState::Out *prev = &stg->out[q - kOutRing];
                    cp->wait([prev] { return prev->left.load() == 0; });
                }
                uint8_t *slot = d->h_stage_out.p + (q % kOutRing) * out_slot_bytes;
                A3_CUDA(cudaMemcpyAsync(slot, d->d_grey.p + (size_t)(f0 + sub) * px, bytes, cudaMemcpyDeviceToHost, d->s_pixel));
                cudaEvent_t ev;
                A3_CUDA(d->events.get(&ev));
                A3_CUDA(cudaEventRecord(ev, d->s_pixel));
                const uint32_t pieces = (uint32_t)((bytes + kPiece - 1) / kPiece);
                stg->out.emplace_back();
                StageState::Out *o = &stg->out.back();
                o->ev = ev; o->left.store(pieces);
                uint8_t *dst = outs->grey + (size_t)(s0 + f0 + sub) * px;
                for (uint32_t k = 0; k < pieces; k++) {
                    const size_t off = (size_t)k * kPiece, len = bytes - off < kPiece ? bytes - off : kPiece;
                    cp->submit([stg, o, cp, dst, slot, off, len] {
                        cudaEventSynchronize(o->ev);
                        copy_stream(dst + off, slot + off, len);
                        if (o->left.fetch_sub(1) == 1) cp->notify();
                    });
                }
            }
            return A3_OK;
        };
        auto bits_d2h = [&](uint32_t f0, uint32_t cn, uint32_t j) -> a3_status {
            if (gpu_contours) {
                if (mem == A3_MEM_HOST || j == 0) {  // K3 over the frames K1 just produced (everything for resident input)
                    const uint32_t kn = mem == A3_MEM_HOST ? cn : sn;
                    const K3Params kp = k3_params(d->cfg, d->d_planes.p, w, h, f0, kn, d->d_k3quads.p, quad_cap, ds);
                    A3_CUDA(k3_begin(d->k3, kp, d->s_pixel));
                    bool spec = false;
                    if (shot) A3_CUDA(k3_finish_speculative(d->k3, kp, d->s_pixel, &spec));
                    if (!spec) A3_CUDA(k3_finish(d->k3, kp, d->s_pixel));
                    A3_CUDA(cudaEventRecord(ev_k3[j], d->s_pixel));
                    st.contour_kernel_launches++;
                    k3_last = kp; k3_spec_inflight = spec;
                    if (spec && shot_cap) {
                        if (a3_status s = enqueue_one_shot()) return s;  // its single copy carries the counters too
                    } else {
                        if (a3_status s = k3_stats_d2h(f0, kn)) return s;
                        if (!spec)
                            if (a3_status s = k3_head_d2h(f0, kn)) return s;
                    }
                }
            } else {
                A3_CUDA(cudaMemcpyAsync(d->h_bits.p + (size_t)f0 * bits_words, d->d_bits.p + (size_t)f0 * bits_words, (size_t)cn * bits_words * 4,
                                        cudaMemcpyDeviceToHost, d->s_pixel));
            }
            A3_CUDA(cudaEventRecord(ev_fe[j], d->s_pixel));
            if (want_grey)
                if (a3_status s = grey_d2h(f0, cn)) return s;
            if (want_mask)
                A3_CUDA(cudaMemcpyAsync(outs->mask + (size_t)(s0 + f0) * px, d->d_mask.p + (size_t)f0 * px, (size_t)cn * px, cudaMemcpyDeviceToHost, d->s_pixel));
            return A3_OK;
        };
        // the copy of chunk j (host input) is queued `kStaging` chunks ahead of its compute, so the PCIe link never idles
        // even though K3 synchronises the pixel stream once per chunk
        uint32_t copies_issued = 0, issued = 0;
        const uint32_t lookahead = gpu_contours ? 1 : kStaging;  // chunks whose compute is queued ahead of the one being consumed
        // Pageable input: the copy threads move chunk c into pinned slot c % kHostRing; the slot is free once the H2D of chunk
        // c - kHostRing has completed.  Chunks are handed to the threads as early as that allows (without blocking), and the
        // caller only ever blocks for the chunk it is about to send (`must`).
        auto advance_stage_in = [&](uint32_t must) -> a3_status {
            CopyPool *cp = &d->copy_pool;
            while (stage_submitted < nfe) {
                const uint32_t c = stage_submitted;
                if (c >= kHostRing) {
                    const uint32_t prev = c - kHostRing;
                    if (prev >= copies_issued) break;  // its H2D is not even queued yet
                    if (c <= must) {
                        A3_CUDA(cudaEventSynchronize(ev_h2db[prev]));
                    } else if (cudaEventQuery(ev_h2db[prev]) != cudaSuccess) {
                        cudaGetLastError();  // cudaErrorNotReady is not an error
                        break;
                    }
                }
                const uint32_t f0 = c * (uint32_t)fe, cn = sn - f0 < fe ? sn - f0 : (uint32_t)fe;
                const size_t bytes = input_span(cn, w, h, bpp, pitch, frame_stride);
                const uint32_t pieces = (uint32_t)((bytes + kPiece - 1) / kPiece);
                const uint8_t *src = src_all + (size_t)(s0 + f0) * frame_stride;
                uint8_t *dst = d->h_stage_in.p + (size_t)(c % kHostRing) * in_slot_bytes;
                stg->in_left[c].store(pieces);
                for (uint32_t k = 0; k < pieces; k++) {
                    const size_t off = (size_t)k * kPiece, len = bytes - off < kPiece ? bytes - off : kPiece;
                    cp->submit([stg, cp, c, dst, src, off, len] {
                        copy_stream(dst + off, src + off, len);
                        if (stg->in_left[c].fetch_sub(1) == 1) cp->notify();
                    });
                }
                stage_submitted++;
            }
            return A3_OK;
        };
        auto issue_copy = [&](uint32_t j) -> a3_status {
            const uint32_t f0 = j * (uint32_t)fe, cn = sn - f0 < fe ? sn - f0 : (uint32_t)fe;
            uint8_t *slot = d->d_src.p + (size_t)(j % kStaging) * fe * frame_stride;
            const uint8_t *from = src_all + (size_t)(s0 + f0) * frame_stride;
            if (stage_in) {
                if (a3_status s = advance_stage_in(j)) return s;
                StageState *sp = stg.get();
                d->copy_pool.wait([sp, j] { return sp->in_left[j].load() == 0; });
                from = d->h_stage_in.p + (size_t)(j % kHostRing) * in_slot_bytes;
            }
            if (j >= kStaging) A3_CUDA(cudaStreamWaitEvent(d->s_copy, ev_k1b[j - kStaging], 0));  // the slot's previous K1 is done
            A3_CUDA(cudaEventRecord(ev_h2da[j], d->s_copy));
            A3_CUDA(cudaMemcpyAsync(slot, from, input_span(cn, w, h, bpp, pitch, frame_stride), cudaMemcpyHostToDevice, d->s_copy));
            A3_CUDA(cudaEventRecord(ev_h2db[j], d->s_copy));
            return A3_OK;
        };
        auto issue = [&](uint32_t j) -> a3_status {
            const uint32_t f0 = j * (uint32_t)fe, cn = sn - f0 < fe ? sn - f0 : (uint32_t)fe;
            if (mem == A3_MEM_HOST) {
                // copy c reuses the slot of chunk c - kStaging and waits for that chunk's K1, whose event exists once
                // issue(c - kStaging) has run: c < j + kStaging
                while (copies_issued < nfe && copies_issued < j + kStaging) {
                    if (a3_status s = issue_copy(copies_issued)) return s;
                    copies_issued++;
                }
                uint8_t *slot = d->d_src.p + (size_t)(j % kStaging) * fe * frame_stride;
                A3_CUDA(cudaStreamWaitEvent(d->s_pixel, ev_h2db[j], 0));
                if (a3_status s = k1_launch(slot, f0, cn, j)) return s;
            } else if (j == 0) {
                // resident input: one K1 launch over the whole super-batch
                if (a3_status s = k1_launch(src_all + (size_t)s0 * frame_stride, 0, sn, 0)) return s;
            }
            return bits_d2h(f0, cn, j);
        };

        // ---- host stage: one task per frame (host-contour mode; in device-contour mode only flagged frames, inline) ----
        const a3_config cfg = d->cfg;
        uint32_t *h_bits = d->h_bits.p;
        a3_detector *det = d;
        if (!gpu_contours) {
            d->pool.begin([&, h_bits, cfg, det](uint32_t i) {
                const double t0 = now_ms();
                quads_from_bits(h_bits + (size_t)i * bits_words, (uint32_t)wpr, w, h, cfg, frame_quads[i], &frame_stats[i]);
                frame_ms[i] = now_ms() - t0;
                const uint32_t g = i / group;
                if (group_done[g].fetch_add(1) + 1 == group_size(g)) det->pool.notify_caller();
            }, sn);
        }
        // device-contour mode: take frame i's quads from K3's output, or redo the frame on the host when K3 flagged it
        auto take_k3_frame = [&](uint32_t i) -> a3_status {
            if (hs.flags[i] == 0) {
                const uint32_t m = hs.counts[i];
                if (m > quad_head) {  // rare (decode-stress scenes): the tail of this frame's quads
                    A3_CUDA(cudaMemcpyAsync(d->h_k3quads.p + ((size_t)i * quad_cap + quad_head) * 8, d->d_k3quads.p + ((size_t)i * quad_cap + quad_head) * 8,
                                            (size_t)(m - quad_head) * 32, cudaMemcpyDeviceToHost, d->s_decode));
                    A3_CUDA(cudaStreamSynchronize(d->s_decode));
                }
                frame_quads[i].assign(d->h_k3quads.p + (size_t)i * quad_cap * 8, d->h_k3quads.p + (size_t)i * quad_cap * 8 + (size_t)m * 8);
                hs.stats(i, frame_stats[i]);
            } else {
                const double t0 = now_ms();
                A3_CUDA(cudaMemcpyAsync(d->h_plane.p, d->d_planes.p + (size_t)i * plane_words, plane_words * 4, cudaMemcpyDeviceToHost, d->s_decode));
                A3_CUDA(cudaStreamSynchronize(d->s_decode));
                std::vector<uint32_t> rows(bits_words);  // back to the row-major mask the host stage reads
                for (uint32_t k = 0; k < wpr; k++)
                    for (uint32_t y = 0; y < h; y++) rows[(size_t)y * wpr + k] = d->h_plane.p[(size_t)(k + 1) * Hp + (y + 1)];
                quads_from_bits(rows.data(), (uint32_t)wpr, w, h, cfg, frame_quads[i], &frame_stats[i]);
                frame_ms[i] = now_ms() - t0;
                st.host_fallback_frames++;
            }
            group_done[i / group].fetch_add(1);
            return A3_OK;
        };

        // ---- decode of group g (asynchronous) ----
        auto launch_group = [&](uint32_t g) -> a3_status {
            DecodeBlock &b = *d->blocks[g];
            if (one_shot_done && g == 0) return A3_OK;  // decoded on the device behind K3 already
            const uint32_t f0 = g * group, f1 = f0 + group_size(g), gn = f1 - f0;
            uint32_t nq = 0;
            for (uint32_t i = f0; i < f1; i++) nq += (uint32_t)(frame_quads[i].size() / 8);
            b.n_quads = nq;
            if (one_shot && ngroups == 1) { d->hist_nq = nq ? nq : 1; d->hist_nq_n = n; d->hist_nq_w = w; d->hist_nq_h = h; }
            const OutLayout lay = out_layout(plan, nq, gn);
            A3_CUDA(b.h_out.reserve(lay.bytes));
            b.set_views(b.h_out.p, lay);
            if (nq == 0) {
                if (want_board) {  // no candidates: every frame of the group has the empty board pose
                    a3_board_pose e{};
                    a3_pose_default(&e.best); a3_pose_default(&e.alt);
                    for (uint32_t i = 0; i < gn; i++) reinterpret_cast<a3_board_pose *>(b.h_out.p + lay.board)[i] = e;
                }
                return A3_OK;
            }
            A3_CUDA(b.h_quads.reserve((size_t)nq * 8)); A3_CUDA(b.h_qframe.reserve(nq));
            A3_CUDA(b.d_quads.reserve((size_t)nq * 8)); A3_CUDA(b.d_qframe.reserve(nq)); A3_CUDA(b.d_out.reserve(lay.bytes));
            if (want_patches) A3_CUDA(b.d_patches.reserve(nq * np));
            uint32_t k = 0;
            // Device contour stage: K3's quads of these frames are still in device memory, so they are gathered there (the same two
            // kernels as on the one-shot route) — a small host-to-device copy would queue behind the frame chunks in flight on
            // the copy engine and hold the decode back by whole chunks.  Groups with a frame the host stage redid take the copy.
            bool on_device = gpu_contours;
            for (uint32_t i = f0; i < f1 && on_device; i++) on_device = hs.flags[i] == 0 && frame_quads[i].size() / 8 == (hs.counts[i] < quad_cap ? hs.counts[i] : quad_cap);
            if (on_device) {
                const uint32_t n_chunks = (nq + 1023) / 1024;
                A3_CUDA(b.d_info.reserve(4)); A3_CUDA(b.d_qoff.reserve((size_t)gn + 1 + n_chunks));
                pack_offsets_kernel<<<1, 1024, 0, d->s_decode>>>(ds.counts + f0, ds.flags + f0, gn, quad_cap, nq, nullptr, b.d_qoff.p, b.d_info.p,
                                                                b.d_qoff.p + gn + 1, n_chunks);
                A3_CUDA(cudaGetLastError());
                pack_quads_kernel<<<gn, 128, 0, d->s_decode>>>(d->d_k3quads.p + (size_t)f0 * quad_cap * 8, b.d_qoff.p, quad_cap, nq, b.d_info.p,
                                                              b.d_quads.p, b.d_qframe.p, f0);
                A3_CUDA(cudaGetLastError());
            } else {
                for (uint32_t i = f0; i < f1; i++) {
                    const uint32_t m = (uint32_t)(frame_quads[i].size() / 8);
                    if (m) memcpy(b.h_quads.p + (size_t)k * 8, frame_quads[i].data(), (size_t)m * 32);
                    for (uint32_t q = 0; q < m; q++) b.h_qframe.p[k + q] = i;
                    k += m;
                }
                A3_CUDA(cudaMemcpyAsync(b.d_quads.p, b.h_quads.p, (size_t)nq * 32, cudaMemcpyHostToDevice, d->s_decode));
                A3_CUDA(cudaMemcpyAsync(b.d_qframe.p, b.h_qframe.p, (size_t)nq * 4, cudaMemcpyHostToDevice, d->s_decode));
                if (want_board) {  // K6's per-frame offsets travel with the quads
                    A3_CUDA(b.h_qoff.reserve((size_t)gn + 1)); A3_CUDA(b.d_qoff.reserve((size_t)gn + 1));
                    uint32_t o = 0;
                    for (uint32_t i = f0; i < f1; i++) { b.h_qoff.p[i - f0] = o; o += (uint32_t)(frame_quads[i].size() / 8); }
                    b.h_qoff.p[gn] = o;
                    A3_CUDA(cudaMemcpyAsync(b.d_qoff.p, b.h_qoff.p, (size_t)(gn + 1) * 4, cudaMemcpyHostToDevice, d->s_decode));
                }
            }
            ChainIn in;
            in.grey = d->d_grey.p; in.w = w; in.h = h; in.quads = b.d_quads.p; in.qframe = b.d_qframe.p; in.n = nq;
            in.n_dev = on_device ? b.d_info.p : nullptr;
            A3_CUDA(k2_queue(d, nq, on_device ? b.d_info.p + 2 : nullptr, d->s_decode, &in.queue));  // d_info[2]: zeroed by pack_offsets_kernel
            in.patches = want_patches ? b.d_patches.p : nullptr; in.offsets = b.d_qoff.p; in.n_frames = gn;
            A3_CUDA(enqueue_chain(d, plan, in, b.d_out.p, lay, b, d->s_decode));
            plan.count(st);
            A3_CUDA(cudaMemcpyAsync(b.h_out.p, b.d_out.p, lay.host_end, cudaMemcpyDeviceToHost, d->s_decode));
            return A3_OK;
        };
        auto drain = [&](a3_status s) {  // an error: let the pool and the streams finish before the buffers go away
            if (!gpu_contours) {
                d->pool.publish(sn);
                d->pool.finish();
            }
            cudaStreamSynchronize(d->s_copy); cudaStreamSynchronize(d->s_pixel); cudaStreamSynchronize(d->s_decode);
            if (stage_in || stage_out) d->copy_pool.drain();
            return s;
        };

        // ---- drive: front end `kStaging` chunks ahead, feed the pool, launch decode groups as they complete ----
        const double t_host0 = now_ms();
        static const bool trace = getenv("A3_TRACE") != nullptr;  // debug aid: host timestamps of the phases of a call, on stderr
        double t_first_sync = 0, t_loop_end = 0, t_synced = 0, t_events = 0;
        a3_status err = A3_OK;
        uint32_t next_group = 0;
        for (uint32_t j = 0; j < nfe && !err; j++) {
            while (issued < nfe && issued < j + lookahead && !err) err = issue(issued++);
            if (err) break;
            const cudaError_t e = cudaEventSynchronize(ev_fe[j]);
            if (e != cudaSuccess) { err = cuda_fail(e, "cudaEventSynchronize(front end)"); break; }
            if (trace && j == 0) t_first_sync = now_ms();
            if (trace && j + 1 == nfe) t_loop_end = now_ms();
            const uint32_t upto = (j + 1) * (uint32_t)fe < sn ? (j + 1) * (uint32_t)fe : sn;
            if (gpu_contours) {
                if (k3_spec_inflight && (err = settle_one_shot())) break;
                if ((mem == A3_MEM_HOST || j == 0) && !one_shot_done)  // resident input: K3 ran once over everything
                    for (uint32_t i = (mem == A3_MEM_HOST ? j * (uint32_t)fe : 0); i < (mem == A3_MEM_HOST ? upto : sn) && !err; i++) err = take_k3_frame(i);
            } else {
                d->pool.publish(upto);
            }
            while (next_group < ngroups && !err && group_done[next_group].load() == group_size(next_group)) err = launch_group(next_group++);
        }
        if (err) return drain(err);
        for (; next_group < ngroups; next_group++) {
            const uint32_t g = next_group;
            if (!gpu_contours) d->pool.wait_caller([&] { return group_done[g].load() == group_size(g); });
            if ((err = launch_group(g))) return drain(err);
        }
        if (!gpu_contours) d->pool.finish();
        st.ms_host_quads += now_ms() - t_host0;

        // ---- gather: stage timings, then markers in frame / candidate order (src/aruco.rs:75-113) ----
        A3_CUDA(cudaStreamSynchronize(d->s_decode));
        A3_CUDA(cudaStreamSynchronize(d->s_pixel));
        if (stage_in || stage_out) d->copy_pool.drain();  // the last grey sub-chunks reach the caller's buffer
        if (trace) t_synced = now_ms();
        float ms = 0;
        for (uint32_t j = 0; j < nfe && stats; j++) {  // stage times only when the caller asked for statistics (about 2 us per query)
            if (mem == A3_MEM_HOST) { cudaEventElapsedTime(&ms, ev_h2da[j], ev_h2db[j]); st.ms_h2d += ms; }
            if (mem == A3_MEM_HOST || j == 0) { cudaEventElapsedTime(&ms, ev_k1a[j], ev_k1b[j]); st.ms_pixel_kernel += ms; }
            if (gpu_contours) {
                if (mem == A3_MEM_HOST || j == 0) {
                    cudaEventElapsedTime(&ms, ev_k1b[j], ev_k3[j]); st.ms_contour_kernels += ms;
                    cudaEventElapsedTime(&ms, ev_k3[j], ev_fe[j]); st.ms_mask_d2h += ms;
                    if (one_shot_done) st.ms_mask_d2h -= stage_ms(*d->blocks[0], nullptr);  // the decode chain sits between those two events here
                }
            } else {
                cudaEventElapsedTime(&ms, (mem == A3_MEM_HOST || j == 0) ? ev_k1b[j] : ev_fe[j - 1], ev_fe[j]);
                st.ms_mask_d2h += ms;
            }
        }
        for (uint32_t i = 0; i < sn; i++) {
            st.n_contours += frame_stats[i].n_contours;
            st.n_contour_points += frame_stats[i].n_contour_points;
            st.n_candidates_before_discard += frame_stats[i].n_before_discard;
            st.ms_host_cpu += frame_ms[i];
        }
        if (trace) {
            t_events = now_ms();
            float h2d_span = 0, gpu_tail = 0;
            if (mem == A3_MEM_HOST) {
                cudaEventElapsedTime(&h2d_span, ev_h2da[0], ev_h2db[nfe - 1]);
                cudaEventElapsedTime(&gpu_tail, ev_h2db[nfe - 1], ev_fe[nfe - 1]);
            }
            fprintf(stderr, "a3 trace: entry->loop %.3f | first front-end sync +%.3f, last +%.3f, loop end +%.3f, streams idle +%.3f, event queries +%.3f ms"
                            " | H2D first byte -> last byte %.3f, last byte -> last front end %.3f ms\n",
                    t_host0 - t_begin, t_first_sync - t_host0, t_loop_end - t_host0, st.ms_host_quads, t_synced - t_host0, t_events - t_host0,
                    h2d_span, gpu_tail);
        }
        if (lean_done) {  // the markers were assembled on the device: one block copy (lean implies a single super-batch and group)
            DecodeBlock &b = *d->blocks[0];
            if (stats) stage_ms(b, &st);
            if (want_board) memcpy(outs->board_poses, b.board_view, (size_t)sn * sizeof(a3_board_pose));
            const uint32_t nm = h_info[3], take = nm < marker_capacity ? nm : marker_capacity;
            memcpy(markers, d->h_shot.p + off_markers, (size_t)take * sizeof(a3_marker));
            if (want_poses) memcpy(outs->marker_poses, d->h_shot.p + off_mposes, (size_t)take * 2 * sizeof(a3_pose));
            if (out_corners) memcpy(out_corners, d->h_shot.p + off_mcorners, (size_t)take * 32);
            if (nm > marker_capacity) overflow = true;
            if (outs && outs->frame_marker_offsets) {
                uint32_t i = 0;
                for (uint32_t f = 0; f <= sn; f++) {
                    while (i < take && markers[i].frame < f) i++;
                    outs->frame_marker_offsets[f] = f < sn ? i : nm;
                }
            }
            total_markers = nm;
            total_cands = b.n_quads;
            continue;
        }
        for (uint32_t g = 0; g < ngroups; g++) {
            DecodeBlock &b = *d->blocks[g];
            if (stats) stage_ms(b, &st);
            const uint32_t f0 = g * group, f1 = f0 + group_size(g);
            if (want_board) memcpy(outs->board_poses + s0 + f0, b.board_view, (size_t)(f1 - f0) * sizeof(a3_board_pose));
            if (want_patches && b.n_quads && total_cands < outs->cand_capacity) {
                const uint32_t room = outs->cand_capacity - total_cands, m = b.n_quads < room ? b.n_quads : room;
                A3_CUDA(cudaMemcpy(outs->homographies + (size_t)total_cands * np, b.d_patches.p, (size_t)m * np, cudaMemcpyDeviceToHost));
            }
            uint32_t k = 0;
            for (uint32_t i = f0; i < f1; i++) {
                if (outs && outs->frame_marker_offsets) outs->frame_marker_offsets[s0 + i] = total_markers;
                const uint32_t m = (uint32_t)(frame_quads[i].size() / 8);
                for (uint32_t j = 0; j < m; j++, k++) {
                    const a3_decode &dc = b.dec_view[k];
                    const uint32_t *q = &frame_quads[i][(size_t)j * 8];
                    if (outs && total_cands < outs->cand_capacity) {
                        if (outs->candidates) memcpy(outs->candidates + (size_t)total_cands * 8, q, 32);
                        if (outs->candidate_frame) outs->candidate_frame[total_cands] = s0 + i;
                        if (outs->decodes) outs->decodes[total_cands] = dc;
                    } else if (outs && (outs->candidates || outs->decodes || outs->homographies)) {
                        overflow = true;
                    }
                    total_cands++;
                    if (!dc.accepted) continue;
                    if (markers && total_markers < marker_capacity) {
                        a3_marker &mk = markers[total_markers];
                        memset(&mk, 0, sizeof(mk));
                        mk.id = dc.id;
                        mk.code = dc.codes[dc.rotation & 3];
                        mk.frame = s0 + i;
                        mk.candidate = j;
                        mk.hamming_distance = dc.hamming_distance;
                        mk.rotation = dc.rotation;
                        for (uint32_t cidx = 0; cidx < 4; cidx++) {  // corners.rotate_left(min_rotation)
                            const uint32_t sidx = (cidx + dc.rotation) & 3;
                            mk.corners[2 * cidx] = q[2 * sidx];
                            mk.corners[2 * cidx + 1] = q[2 * sidx + 1];
                        }
                        if (want_poses) memcpy(outs->marker_poses + (size_t)total_markers * 2, b.pose_view + (size_t)k * 2, 2 * sizeof(a3_pose));
                        if (want_refine) {
                            mk.corners_refined = b.refok_view[k];
                            if (out_corners) memcpy(out_corners + (size_t)total_markers * 8, b.ref_view + (size_t)k * 8, 32);
                        }
                    } else {
                        overflow = true;
                    }
                    total_markers++;
                }
            }
        }
    }
    if (outs && outs->frame_marker_offsets) outs->frame_marker_offsets[n] = total_markers;
    if (outs) outs->n_candidates = total_cands;
    *n_markers = total_markers;
    st.n_candidates = total_cands;
    st.n_markers = total_markers;
    st.ms_total = now_ms() - t_begin;
    if (stats) *stats = st;
    if (overflow) return fail(A3_ERR_CAPACITY, "a3_detect_batch: output capacity too small (counts are valid)");
    return A3_OK;
}

// ---- pose step (src/pose.rs, src/pinhole.rs) ----------------------------------------------------------------------

a3_status a3_detector_set_pose(a3_detector *d, uint32_t mode, float marker_size_mm, const a3_camera_intrinsics *k) {
    if (!d) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_pose: null detector");
    if (mode != A3_POSE_OFF && mode != A3_POSE_UNDISTORTED && mode != A3_POSE_INTRINSICS)
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_pose: mode must be OFF, UNDISTORTED or INTRINSICS");
    if (mode == A3_POSE_INTRINSICS && !k) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_pose: intrinsics required");
    if (d->opt.dist_on && mode == A3_POSE_UNDISTORTED)
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_pose: the detector has a lens distortion, which needs INTRINSICS (or OFF)");
    d->opt.pose_mode = mode;
    d->opt.pose_marker_size = marker_size_mm;
    if (k) d->opt.pose_k = *k;
    return A3_OK;
}

// ---- board pose (K6) ------------------------------------------------------------------------------------------------

a3_status a3_detector_set_board(a3_detector *d, const a3_board *board, uint32_t mode, const a3_camera_intrinsics *k) {
    if (!d) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: null detector");
    if (!board) {
        d->opt.board_n = 0;
        d->opt.board_mode = A3_POSE_OFF;
        return A3_OK;
    }
    if (mode != A3_POSE_UNDISTORTED && mode != A3_POSE_INTRINSICS)
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: mode must be UNDISTORTED or INTRINSICS");
    if (mode == A3_POSE_INTRINSICS && !k) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: intrinsics required");
    if (d->opt.dist_on && mode != A3_POSE_INTRINSICS)
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: the detector has a lens distortion, which needs INTRINSICS");
    const uint32_t m = board->n_markers;
    if (m == 0 || m > A3_K6_MAX_MARKERS) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: a board has 1 to 1024 markers");
    if (!board->ids || !board->corners) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: null ids or corners");
    if (d->dict.n_codes > A3_K6_MAX_CODES) return fail(A3_ERR_UNSUPPORTED, "a3_detector_set_board: dictionaries of more than 8192 codes");
    std::vector<uint16_t> slots(d->dict.n_codes ? d->dict.n_codes : 1, (uint16_t)A3_K6_NO_SLOT);
    for (uint32_t i = 0; i < m; i++) {
        const uint64_t id = board->ids[i];
        if (id >= d->dict.n_codes) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: id not below the dictionary's code count");
        if (slots[id] != A3_K6_NO_SLOT) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: duplicate id");
        slots[id] = (uint16_t)i;
    }
    for (size_t i = 0; i < (size_t)m * 8; i++)
        if (!isfinite(board->corners[i])) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_board: non-finite coordinate");
    A3_CUDA(cudaSetDevice(d->device));
    A3_CUDA(d->d_board_slots.reserve(slots.size()));
    A3_CUDA(d->d_board_pts.reserve((size_t)m * 8));
    // the decode stream reads the previous board until its work is done; these copies are ordered behind it
    A3_CUDA(cudaStreamSynchronize(d->s_decode));
    A3_CUDA(cudaStreamSynchronize(d->s_pixel));
    A3_CUDA(cudaMemcpy(d->d_board_slots.p, slots.data(), slots.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    A3_CUDA(cudaMemcpy(d->d_board_pts.p, board->corners, (size_t)m * 32, cudaMemcpyHostToDevice));
    d->opt.board_n = m;
    d->opt.board_mode = mode;
    if (k) d->opt.board_k = *k;
    return A3_OK;
}

a3_status a3_solve_board(a3_detector *d, const uint64_t *ids, const float *corners, const uint32_t *frame, uint32_t n, uint32_t n_frames,
                         uint32_t image_w, uint32_t image_h, a3_board_pose *out) {
    if (!d || (n && (!ids || !corners)) || (n_frames && !out)) return fail(A3_ERR_INVALID_ARGUMENT, "a3_solve_board: null argument");
    if (d->opt.board_n == 0) return fail(A3_ERR_INVALID_ARGUMENT, "a3_solve_board: the detector has no board (a3_detector_set_board)");
    if (n_frames == 0) {
        if (n) return fail(A3_ERR_INVALID_ARGUMENT, "a3_solve_board: markers but no frames");
        return A3_OK;
    }
    if (d->opt.board_mode == A3_POSE_UNDISTORTED && (image_w == 0 || image_h == 0))
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_solve_board: undistorted mode needs the frame size");
    std::vector<uint32_t> off((size_t)n_frames + 1, 0);
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t f = frame ? frame[i] : 0;
        if (f >= n_frames || (i && frame && f < frame[i - 1])) return fail(A3_ERR_INVALID_ARGUMENT, "a3_solve_board: frame out of range or decreasing");
        off[f + 1]++;
    }
    for (uint32_t f = 0; f < n_frames; f++) off[f + 1] += off[f];
    A3_CUDA(cudaSetDevice(d->device));
    cudaStream_t s = d->s_decode;
    A3_CUDA(d->d_probe_ids.reserve(n ? n : 1));
    A3_CUDA(d->d_refined.reserve(n ? (size_t)n * 8 : 1));
    A3_CUDA(d->d_probe_off.reserve(off.size()));
    A3_CUDA(d->d_probe_out.reserve(n_frames));
    if (n) {
        A3_CUDA(cudaMemcpyAsync(d->d_probe_ids.p, ids, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        A3_CUDA(cudaMemcpyAsync(d->d_refined.p, corners, (size_t)n * 32, cudaMemcpyHostToDevice, s));
    }
    A3_CUDA(cudaMemcpyAsync(d->d_probe_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice, s));
    K6Params kp;
    kp.ids = d->d_probe_ids.p; kp.corners_f32 = d->d_refined.p; kp.offsets = d->d_probe_off.p; kp.n_frames = n_frames;
    kp.slots = d->d_board_slots.p; kp.n_codes = d->dict.n_codes; kp.board = d->d_board_pts.p; kp.n_board = d->opt.board_n;
    kp.mode = d->opt.board_mode; kp.image_w = image_w; kp.image_h = image_h; kp.k = d->opt.board_k; kp.out = d->d_probe_out.p;
    if (d->opt.dist_on && n) {  // K7 first, as a3_detect_batch runs it
        A3_CUDA(d->d_und_out.reserve((size_t)n * 8)); A3_CUDA(d->d_und_ok.reserve(n));
        K7Params up;
        up.corners_f32 = d->d_refined.p; up.n = n; up.k = d->opt.board_k; up.dist = d->opt.dist; up.out = d->d_und_out.p; up.ok = d->d_und_ok.p;
        A3_CUDA(k7_undistort(up, s));
        kp.norm = d->d_und_out.p; kp.norm_ok = d->d_und_ok.p;
    }
    A3_CUDA(k6_board(kp, s));
    A3_CUDA(cudaMemcpyAsync(out, d->d_probe_out.p, (size_t)n_frames * sizeof(a3_board_pose), cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaStreamSynchronize(s));
    return A3_OK;
}

// ---- lens distortion (K7) ------------------------------------------------------------------------------------------

a3_status a3_detector_set_distortion(a3_detector *d, const a3_camera_distortion *dist) {
    if (!d) return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_distortion: null detector");
    if (!dist || (dist->k1 == 0.0f && dist->k2 == 0.0f && dist->p1 == 0.0f && dist->p2 == 0.0f && dist->k3 == 0.0f)) {
        d->opt.dist_on = false;
        d->opt.dist = a3_camera_distortion{};
        return A3_OK;
    }
    if (!isfinite(dist->k1) || !isfinite(dist->k2) || !isfinite(dist->p1) || !isfinite(dist->p2) || !isfinite(dist->k3))
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_distortion: non-finite coefficient");
    if (d->opt.pose_mode == A3_POSE_UNDISTORTED || d->opt.pose_mode == A3_POSE_NORMALIZED)
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_distortion: the pose mode does not use the intrinsics (set INTRINSICS or OFF first)");
    if (d->opt.board_n && d->opt.board_mode != A3_POSE_INTRINSICS)
        return fail(A3_ERR_INVALID_ARGUMENT, "a3_detector_set_distortion: the board mode does not use the intrinsics (set INTRINSICS first)");
    d->opt.dist_on = true;
    d->opt.dist = *dist;
    return A3_OK;
}

a3_status a3_undistort_points(a3_detector *d, const float *points, uint32_t n, const a3_camera_intrinsics *k, const a3_camera_distortion *dist,
                              float *out, uint8_t *ok) {
    if (!d || !k || !dist || (n && (!points || !out || !ok))) return fail(A3_ERR_INVALID_ARGUMENT, "a3_undistort_points: null argument");
    if (n == 0) return A3_OK;
    A3_CUDA(cudaSetDevice(d->device));
    cudaStream_t s = d->s_decode;
    A3_CUDA(d->d_und_in.reserve((size_t)n * 2)); A3_CUDA(d->d_und_out.reserve((size_t)n * 2)); A3_CUDA(d->d_und_ok.reserve(n));
    A3_CUDA(cudaMemcpyAsync(d->d_und_in.p, points, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    A3_CUDA(k7_undistort_points(d->d_und_in.p, n, *k, *dist, d->d_und_out.p, d->d_und_ok.p, s));
    A3_CUDA(cudaMemcpyAsync(out, d->d_und_out.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaMemcpyAsync(ok, d->d_und_ok.p, n, cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaStreamSynchronize(s));
    return A3_OK;
}

static a3_status solve_poses(a3_detector *d, uint32_t mode, const void *in, uint32_t n, float marker_size_mm, uint32_t iw, uint32_t ih,
                             const a3_camera_intrinsics *k, a3_pose *best, a3_pose *alt) {
    if (!d || (n && (!in || !best || !alt))) return fail(A3_ERR_INVALID_ARGUMENT, "a3_solve_*: null argument");
    if (mode == A3_POSE_INTRINSICS && !k) return fail(A3_ERR_INVALID_ARGUMENT, "a3_solve_with_intrinsics: null intrinsics");
    if (n == 0) return A3_OK;
    A3_CUDA(cudaSetDevice(d->device));
    cudaStream_t s = d->s_decode;
    A3_CUDA(d->d_pose_in.reserve((size_t)n * 8)); A3_CUDA(d->d_pose_out.reserve((size_t)n * 2)); A3_CUDA(d->h_pose_out.reserve((size_t)n * 2));
    A3_CUDA(cudaMemcpyAsync(d->d_pose_in.p, in, (size_t)n * 32, cudaMemcpyHostToDevice, s));
    K4Params kp{};
    kp.mode = mode; kp.n = n; kp.marker_size = marker_size_mm; kp.image_w = iw; kp.image_h = ih; kp.poses = d->d_pose_out.p;
    if (mode == A3_POSE_NORMALIZED) kp.points = d->d_pose_in.p;
    else kp.corners = reinterpret_cast<const uint32_t *>(d->d_pose_in.p);
    if (k) kp.k = *k;
    A3_CUDA(k4_pose(kp, s));
    A3_CUDA(cudaMemcpyAsync(d->h_pose_out.p, d->d_pose_out.p, (size_t)n * 2 * sizeof(a3_pose), cudaMemcpyDeviceToHost, s));
    A3_CUDA(cudaStreamSynchronize(s));
    for (uint32_t i = 0; i < n; i++) { best[i] = d->h_pose_out.p[2 * (size_t)i]; alt[i] = d->h_pose_out.p[2 * (size_t)i + 1]; }
    return A3_OK;
}

a3_status a3_solve_with_intrinsics(a3_detector *d, const uint32_t *corners, uint32_t n, float marker_size_mm, const a3_camera_intrinsics *k,
                                   a3_pose *best, a3_pose *alt) {
    return solve_poses(d, A3_POSE_INTRINSICS, corners, n, marker_size_mm, 0, 0, k, best, alt);
}
a3_status a3_solve_with_undistorted_points(a3_detector *d, const uint32_t *corners, uint32_t n, float marker_size_mm, uint32_t image_width,
                                           uint32_t image_height, a3_pose *best, a3_pose *alt) {
    return solve_poses(d, A3_POSE_UNDISTORTED, corners, n, marker_size_mm, image_width, image_height, nullptr, best, alt);
}
a3_status a3_solve_with_normalized_points(a3_detector *d, const float *points, uint32_t n, float marker_size_mm, a3_pose *best, a3_pose *alt) {
    return solve_poses(d, A3_POSE_NORMALIZED, points, n, marker_size_mm, 0, 0, nullptr, best, alt);
}

void a3_pose_default(a3_pose *p) {
    if (!p) return;
    p->error = 1e31f;
    for (int i = 0; i < 9; i++) p->rotation[i] = (i % 4 == 0) ? 1.0f : 0.0f;
    p->translation[0] = p->translation[1] = p->translation[2] = 0.0f;
}

// R*p + t, or R^T*(p - t); products accumulate column by column as nalgebra's gemv does
void a3_pose_apply_transform(const a3_pose *p, const float *pts, uint32_t n, int32_t inverse, float *out) {
    if (!p || !pts || !out) return;
    const float *R = p->rotation, *t = p->translation;
    for (uint32_t i = 0; i < n; i++) {
        const float *v = pts + 3 * (size_t)i;
        float *o = out + 3 * (size_t)i;
        if (!inverse) {
            for (int r = 0; r < 3; r++) o[r] = (R[r * 3 + 2] * v[2] + (R[r * 3 + 1] * v[1] + R[r * 3] * v[0])) + t[r];
        } else {
            const float dv[3] = {v[0] - t[0], v[1] - t[1], v[2] - t[2]};
            for (int r = 0; r < 3; r++) o[r] = R[6 + r] * dv[2] + (R[3 + r] * dv[1] + R[r] * dv[0]);
        }
    }
}

void a3_camera_intrinsics_new(uint32_t iw, uint32_t ih, float fx, float fy, const float *px, const float *py, a3_camera_intrinsics *out) {
    if (!out) return;
    *out = a3_camera_intrinsics{iw, ih, fx, fy, px ? *px : (float)iw / 2.0f, py ? *py : (float)ih / 2.0f};
}

void a3_camera_intrinsics_from_fov_horizontal(float hfov, float sensor_w, uint32_t rx, uint32_t ry, a3_camera_intrinsics *out) {
    if (!out) return;
    const float aspect = (float)rx / (float)ry;
    const float vfov = hfov / aspect, sensor_h = sensor_w / aspect;
    *out = a3_camera_intrinsics{rx, ry, (sensor_w * 0.5f) / tanf(hfov * 0.5f), (sensor_h * 0.5f) / tanf(vfov * 0.5f), (float)rx * 0.5f,
                                (float)ry * 0.5f};
}

void a3_camera_project(const a3_camera_intrinsics *k, float x, float y, float z, float out[3]) {
    out[0] = (x * k->focal_x) + (z * k->principal_x);
    out[1] = (y * k->focal_y) + (z * k->principal_y);
    out[2] = z;
}

int32_t a3_camera_project_culled(const a3_camera_intrinsics *k, float x, float y, float z, float out[2]) {
    if (z <= 0.0f) return 0;
    out[0] = (x * k->focal_x) / z + k->principal_x;
    out[1] = (y * k->focal_y) / z + k->principal_y;
    return 1;
}

void a3_camera_unproject(const a3_camera_intrinsics *k, float x, float y, float out[2]) {
    out[0] = (x - k->principal_x) / k->focal_x;
    out[1] = (y - k->principal_y) / k->focal_y;
}

}  // extern "C"
