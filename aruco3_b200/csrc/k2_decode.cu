// K2 — per-candidate decode (sm_100a). Compile this file with -fmad=false: the reference is Rust, which never
// contracts a*b+c, and every float below is written in the reference's operation order.
//
// Parity status: bit-exact against the in-repo oracle (oracle/a3ref.c); parity with the upstream crates is UNPINNED — the
// reference holds no vector for this stage and imageproc solves the 8x8 system below through nalgebra's SVD, not by
// elimination.  tests/test_oracle_risk.py measures what that can change: an independent f64 SVD moves an f32 coefficient
// in about 2 % of quads, a patch byte (by one) in a tenth of those, and no code, id, rotation or distance in any.
// For each candidate quad this replaces:
//   extract_homographies            /root/reference/src/aruco.rs:234-261  (imageproc Projection::from_control_points,
//                                                                          warp_into Bilinear, default 0)
//   homography_to_code_permutations /root/reference/src/aruco.rs:263-313  (otsu_level, threshold Binary,
//                                                                          imageops::resize Triangle, >127, border test,
//                                                                          4 rotations, rotate_bit_matrix :315-326)
//   the match loop                  /root/reference/src/aruco.rs:75-96    (ARDictionary::find_nearest
//                                                                          src/dictionaries.rs:160-196, hamming lib.rs:11-21)
//
// One WARP per candidate (8 warps per CTA, no block-wide barrier after the dictionary is staged): lane 0 solves the
// homography, the warp samples the 49x49 patch and histograms it in its own shared-memory slice, Otsu by warp scans,
// the separable triangle resize, the border test by a warp vote, the four rotations on four lanes, and the dictionary
// (staged into shared memory once per CTA) matched with __popcll over all four rotations; the winner is a packed-key
// warp min so that both strict-< tie rules of the reference hold (lowest rotation, then lowest index).
// Latency-bound and tiny next to K1: what matters is how many candidates are in flight, hence a warp each.
#include <math.h>
#include <stdlib.h>

#include "a3_internal.h"

namespace a3 {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

struct Proj {
    float inv[9];  // maps patch pixels back into the image (projection.invert())
    int cls;       // 0 translation, 1 affine, 2 projection
    int ok;
};

// f64 Gaussian elimination with partial pivoting on an 8x9 system held in shared memory, by one warp.  Every element
// goes through the very sequence of operations of oracle/a3ref.c:solve8 (pivot = first row with the largest |a[r][col]|,
// f = a[r][col] / a[col][col], a[r][k] = a[r][k] - f * a[col][k] for k = col..8, back substitution top-down in k); the
// warp only spreads independent elements over lanes, which cannot change any rounding.
__device__ bool solve8_warp(double (*a)[9], int lane) {
    for (int col = 0; col < 8; col++) {
        int piv = col;
        double best = fabs(a[col][col]);
        for (int r = col + 1; r < 8; r++) {  // 8 shared-memory reads, every lane the same: no divergence, no reduction to get wrong
            const double v = fabs(a[r][col]);
            if (v > best) { best = v; piv = r; }
        }
        if (best == 0.0) return false;
        __syncwarp();
        if (piv != col && lane < 9) { const double t = a[col][lane]; a[col][lane] = a[piv][lane]; a[piv][lane] = t; }
        __syncwarp();
        // rows col+1..7, columns col..8: element e -> (row, k); the factor is read before any element of the row changes
        const int ncols = 9 - col, nelem = (7 - col) * ncols;
        double f[2], arow[2], acol[2];
        int rr[2], kk[2];
#pragma unroll
        for (int it = 0; it < 2; it++) {
            const int e = lane + 32 * it;
            rr[it] = -1;
            if (e < nelem) {
                rr[it] = col + 1 + e / ncols;
                kk[it] = col + e % ncols;
                f[it] = a[rr[it]][col] / a[col][col];
                arow[it] = a[rr[it]][kk[it]];
                acol[it] = a[col][kk[it]];
            }
        }
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 2; it++)
            if (rr[it] >= 0) a[rr[it]][kk[it]] = arow[it] - f[it] * acol[it];
        __syncwarp();
    }
    if (lane == 0) {
        for (int r = 7; r >= 0; r--) {
            double s = a[r][8];
            for (int k = r + 1; k < 8; k++) s = s - a[r][k] * a[k][8];
            a[r][8] = s / a[r][r];
        }
    }
    __syncwarp();
    return true;
}

// Projection::from_control_points(quad, [(0,0),(h,0),(h,h),(0,h)]) followed by invert() (SURVEY A.6), by one warp.
__device__ void make_projection(const uint32_t *quad, float hs, double (*a)[9], Proj *out, int lane) {
    if (lane < 8) {
        const int k = lane >> 1;
        // to = {(0,0), (hs,0), (hs,hs), (0,hs)}, chosen by select: a table indexed by lane would live in local memory
        const double xf = (double)(float)quad[2 * k], yf = (double)(float)quad[2 * k + 1];
        const double x = (double)(k == 1 || k == 2 ? hs : 0.0f), y = (double)(k >= 2 ? hs : 0.0f);
        if (lane & 1) {
            const double r1[9] = {xf, yf, 1.0, 0.0, 0.0, 0.0, -x * xf, -x * yf, x};
            for (int i = 0; i < 9; i++) a[lane][i] = r1[i];
        } else {
            const double r0[9] = {0.0, 0.0, 0.0, -xf, -yf, -1.0, y * xf, y * yf, -y};
            for (int i = 0; i < 9; i++) a[lane][i] = r0[i];
        }
    }
    if (lane == 0) out->ok = 0;
    __syncwarp();
    const bool solved = solve8_warp(a, lane);
    if (!solved || lane != 0) return;
    float t[9];
    for (int i = 0; i < 8; i++) t[i] = (float)a[i][8];
    t[8] = 1.0f;
    for (int i = 0; i < 8; i++)
        if (!isfinite(t[i])) return;
    int c = 2;
    if (fabsf(t[6]) < 1e-10f && fabsf(t[7]) < 1e-10f && fabsf(t[8] - 1.0f) < 1e-10f) {
        if (fabsf(t[0] - 1.0f) < 1e-10f && fabsf(t[1]) < 1e-10f && fabsf(t[3]) < 1e-10f && fabsf(t[4] - 1.0f) < 1e-10f) c = 0;
        else c = 1;
    }
    out->cls = c;
    // try_inverse (f32 adjugate) + normalize
    float t00 = t[0], t01 = t[1], t02 = t[2], t10 = t[3], t11 = t[4], t12 = t[5], t20 = t[6], t21 = t[7], t22 = t[8];
    float m00 = t11 * t22 - t12 * t21;
    float m01 = t10 * t22 - t12 * t20;
    float m02 = t10 * t21 - t11 * t20;
    float det = t00 * m00 - t01 * m01 + t02 * m02;
    if (fabsf(det) < 1e-10f) return;
    float m10 = t01 * t22 - t02 * t21;
    float m11 = t00 * t22 - t02 * t20;
    float m12 = t00 * t21 - t01 * t20;
    float m20 = t01 * t12 - t02 * t11;
    float m21 = t00 * t12 - t02 * t10;
    float m22 = t00 * t11 - t01 * t10;
    float rr[9] = {m00 / det, -m10 / det, m20 / det, -m01 / det, m11 / det, -m21 / det, m02 / det, -m12 / det, m22 / det};
    float s = rr[8];
    for (int i = 0; i < 8; i++) out->inv[i] = rr[i] / s;
    out->inv[8] = 1.0f;
    out->ok = 1;
}

// An integer 0 <= v < 2^23 as f32 without the conversion pipe: 2^23 + v is exact, so is the subtraction.
__device__ __forceinline__ float small_to_f32(uint32_t v) { return __uint_as_float(0x4B000000u | v) - 8388608.0f; }

// <u8 as Clamp<f32>>::clamp followed by `as u8` (x < 255 ? (x > 0 ? trunc(x) : 0) : 255, so NaN gives 255) for a blend of
// interpolate_bilinear, which is +-0, positive or NaN; returns 2^23 + the byte.  x + 2^23 rounded toward zero is 2^23 + trunc(x)
// exactly for 0 <= x < 2^23 (floats in [2^23, 2^24) are the integers), larger x and +inf stay at or above 2^23 + 255, and fminf
// returns its other operand for NaN.
__device__ __forceinline__ float clamp_u8_trunc_biased(float x) { return fminf(__fadd_rz(x, 8388608.0f), 8388608.0f + 255.0f); }

// First half of warp_into's per-pixel body (projective map + interpolate_bilinear with default 0, SURVEY A.7) for patch pixel
// (x, y): the bilinear weights, the frame offset of the top-left texel and whether the sample is outside the frame (result 0).
// The reference's test `left < 0 || right >= w || top < 0 || bottom >= h` with left = floor(px), right = left + 1 is
// `px < 0 || px >= w - 1` (and the same in y): floor(px) < 0 iff px < 0, and floor(px) + 1 >= w iff px >= w - 1 since w - 1 is
// an integer (from 2^24 on, where left + 1 rounds, both hold).  +-inf is outside.  NaN fails every comparison, as in Rust, and is
// not outside: its blend is 255 or a function of the finite weight alone, whatever bytes it reads, so it reads offset 0.
// Inside the frame 0 <= px < 2^16, where px + 2^23 rounded down is 2^23 + floor(px) exactly: the floors and their integer values
// come without FRND or F2I.  (For px = -0 the weight becomes -0 where the reference has +0; every blend that weight enters is
// >= +0 either way and clamps to the same byte.)
struct Tap {
    float rw, bw;
    uint32_t off;
    bool out;
};
template <int CLS>
__device__ __forceinline__ Tap locate(const float *t, float x, float y, float wm1, float hm1, uint32_t w) {
    float px, py;
    if constexpr (CLS == 2) {
        float d = t[6] * x + t[7] * y + t[8];
        px = (t[0] * x + t[1] * y + t[2]) / d;
        py = (t[3] * x + t[4] * y + t[5]) / d;
    } else if constexpr (CLS == 1) {
        px = t[0] * x + t[1] * y + t[2];
        py = t[3] * x + t[4] * y + t[5];
    } else {
        px = x + t[2];
        py = y + t[5];
    }
    const float fx = __fadd_rd(px, 8388608.0f), fy = __fadd_rd(py, 8388608.0f);
    const bool in = px >= 0.0f && px < wm1 && py >= 0.0f && py < hm1;
    Tap s;
    s.rw = px - (fx - 8388608.0f);
    s.bw = py - (fy - 8388608.0f);
    s.out = px < 0.0f || px >= wm1 || py < 0.0f || py >= hm1;
    s.off = in ? (__float_as_uint(fy) - 0x4B000000u) * w + (__float_as_uint(fx) - 0x4B000000u) : 0u;
    return s;
}

// Second half: blend_bilinear on the texels at off, off + 1, off + w, off + w + 1, in the reference's operation order.
__device__ __forceinline__ uint32_t blend(const Tap &s, uint32_t tl8, uint32_t tr8, uint32_t bl8, uint32_t br8) {
    const float tl = small_to_f32(tl8), tr = small_to_f32(tr8), bl = small_to_f32(bl8), br = small_to_f32(br8);
    const float topv = clamp_u8_trunc_biased((1.0f - s.rw) * tl + s.rw * tr) - 8388608.0f;
    const float botv = clamp_u8_trunc_biased((1.0f - s.rw) * bl + s.rw * br) - 8388608.0f;
    const uint32_t v = __float_as_uint(clamp_u8_trunc_biased((1.0f - s.bw) * topv + s.bw * botv)) - 0x4B000000u;
    return s.out ? 0u : v;
}

// Samples per thread whose gathers are issued before any is consumed.  Eight spill at 80 registers and were slower (K2 on
// 256 x C3 0.215 against 0.194 ms on a B200); so was building for 4 CTAs per SM (64 registers: spills, 0.52 ms), with or
// without a warp-aggregated (__match_any_sync) histogram update, which alone also lost (0.197 ms).
constexpr int kInFlight = 4;

// Read by the discarded loads of frames under 2 x 2 pixels, which have no sample inside them.
__device__ uint8_t k2_no_frame[2];

// The ps x ps patch of one candidate into `patch` and its histogram: this thread takes samples first, first + stride, ...  Each
// group of kInFlight samples is located first, then all 4 kInFlight byte loads of the group are issued with no branch between
// them, so that their latencies overlap, then the group is blended.
template <int CLS>
__device__ __forceinline__ void sample_patch(const uint8_t *grey, uint32_t w, uint32_t h, const float *inv, uint32_t ps,
                                             uint32_t first, uint32_t stride, uint8_t *patch, uint32_t *hist) {
    const uint32_t np = ps * ps;
    const bool any_inside = w >= 2 && h >= 2;
    const uint8_t *src = any_inside ? grey : k2_no_frame;
    const uint32_t row = any_inside ? w : 0u;
    const float wm1 = (float)w - 1.0f, hm1 = (float)h - 1.0f;
    // (column, row) of sample i without a division per sample: a step of `stride` adds sq rows and sr < ps columns, which wrap
    // at most once
    const uint32_t sq = stride / ps, sr = stride % ps;
    uint32_t ox = first % ps, oy = first / ps;
    for (uint32_t base = first; base < np; base += stride * kInFlight) {
        Tap s[kInFlight];
#pragma unroll
        for (int u = 0; u < kInFlight; u++) {
            s[u] = locate<CLS>(inv, small_to_f32(ox), small_to_f32(oy), wm1, hm1, w);
            ox += sr;
            oy += sq;
            if (ox >= ps) { ox -= ps; oy++; }
        }
        uint32_t b[kInFlight][4];
#pragma unroll
        for (int u = 0; u < kInFlight; u++) {
            const uint8_t *t0 = src + s[u].off, *t1 = t0 + row;
            b[u][0] = t0[0];
            b[u][1] = t0[1];
            b[u][2] = t1[0];
            b[u][3] = t1[1];
        }
#pragma unroll
        for (int u = 0; u < kInFlight; u++) {
            const uint32_t i = base + stride * u;
            const uint32_t v = blend(s[u], b[u][0], b[u][1], b[u][2], b[u][3]);
            if (i < np) {
                patch[i] = (uint8_t)v;
                atomicAdd(&hist[v], 1u);
            }
        }
    }
}

// the loop is specialised per projection class (translation, affine, projective) so that no sample branches on it
__device__ __forceinline__ void sample_patch(const uint8_t *grey, uint32_t w, uint32_t h, const float *inv, int cls, uint32_t ps,
                                             uint32_t first, uint32_t stride, uint8_t *patch, uint32_t *hist) {
    if (cls == 2) sample_patch<2>(grey, w, h, inv, ps, first, stride, patch, hist);
    else if (cls == 1) sample_patch<1>(grey, w, h, inv, ps, first, stride, patch, hist);
    else sample_patch<0>(grey, w, h, inv, ps, first, stride, patch, hist);
}

// Per-warp scratch in shared memory.
struct WarpScratch {
    double a[8][9];      // the 8x8 system of Projection::from_control_points with its right-hand side
    Proj proj;
    uint64_t codes[4];
    uint32_t hist[256];
};
__host__ __device__ inline uint32_t k2_warp_bytes(uint32_t ps, uint32_t ms) {
    const uint32_t b = (uint32_t)sizeof(WarpScratch) + ms * ps * 4 + ((ms * ms + 3) & ~3u) + ps * ps;
    return (b + 15) & ~15u;
}

// WIDE (a launch of few candidates, e.g. one frame per call): a CTA per candidate instead of a warp — all its warps take the
// 2401 bilinear samples together (the longest stretch of a candidate's chain), warp 0 does everything else in its own slice.
template <bool WIDE>
__global__ void __launch_bounds__(kThreads, 3) k2_kernel(const K2Params p, const uint32_t max_taps) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t ps = p.patch_size, ms = p.mark_size, np = ps * ps;
    // ---- carve: per CTA the dictionary and the resize taps, then one slice per warp ----
    uint64_t *dict = reinterpret_cast<uint64_t *>(smem);                       // n_codes
    float *taps = reinterpret_cast<float *>(dict + p.n_codes);                // ms * max_taps
    int *meta = reinterpret_cast<int *>(taps + ms * max_taps);                // 2 * ms
    // the slices are addressed from `smem` itself, not through an integer, so that the compiler keeps them in the shared
    // space: the patch stores and histogram atomics of the sampling loop are then STS / ATOMS instead of generic ST / ATOM
    const size_t head = ((size_t)p.n_codes * 8 + (size_t)ms * max_taps * 4 + (size_t)2 * ms * 4 + 15) & ~(size_t)15;
    const uint32_t warp_bytes = k2_warp_bytes(ps, ms);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *mine = smem + head + (size_t)(WIDE ? 0 : warp) * warp_bytes;
    WarpScratch *ws = reinterpret_cast<WarpScratch *>(mine);
    float *tmp = reinterpret_cast<float *>(mine + sizeof(WarpScratch));       // ms * ps  (vertical pass, f32)
    uint8_t *reduced = reinterpret_cast<uint8_t *>(tmp + ms * ps);            // ms * ms (padded to x4)
    uint8_t *patch = reduced + ((ms * ms + 3) & ~3u);                         // ps * ps

    // (the block has 8 warps, fewer when homography_sample_size is so large that 8 patches do not fit shared memory)
    for (uint32_t i = threadIdx.x; i < p.n_codes; i += blockDim.x) dict[i] = p.codes[i];
    for (uint32_t i = threadIdx.x; i < ms * max_taps; i += blockDim.x) taps[i] = p.resize_w[i];
    for (uint32_t i = threadIdx.x; i < 2 * ms; i += blockDim.x) meta[i] = p.resize_meta[i];
    __syncthreads();

    // one warp per candidate; warps never wait for each other
    const uint32_t n_quads = p.n_quads_dev ? min(*p.n_quads_dev, p.n_quads) : p.n_quads;
    const uint32_t nwarps = WIDE ? 1u : blockDim.x >> 5;
    const uint32_t first_q = WIDE ? blockIdx.x : blockIdx.x * nwarps + warp, stride_q = gridDim.x * nwarps;
    auto next_quad = [&](uint32_t q) -> uint32_t {  // the warp's next quad: fixed stride, or the shared counter behind the first round
        if (WIDE || !p.queue) return q + stride_q;
        uint32_t t = 0;
        if (lane == 0) t = stride_q + atomicAdd(p.queue, 1u);
        return __shfl_sync(0xffffffffu, t, 0);
    };
    for (uint32_t q = first_q; q < n_quads; q = next_quad(q)) {
        const uint32_t frame = p.quad_frame ? p.quad_frame[q] : 0;
        const uint8_t *grey = p.grey + (size_t)frame * p.w * p.h;
        if (!WIDE || warp == 0) {
            make_projection(p.quads + (size_t)q * 8, (float)ps, ws->a, &ws->proj, lane);
            for (int i = lane; i < 256; i += 32) ws->hist[i] = 0;
        }
        if constexpr (WIDE) __syncthreads(); else __syncwarp();
        const int ok = ws->proj.ok;
        uint32_t otsu_level = 0;
        if constexpr (WIDE) {
            if (ok) {  // every thread of the CTA: samples threadIdx.x, + blockDim.x, ...
                float inv[9];
#pragma unroll
                for (int k = 0; k < 9; k++) inv[k] = ws->proj.inv[k];
                sample_patch(grey, p.w, p.h, inv, ws->proj.cls, ps, threadIdx.x, blockDim.x, patch, ws->hist);
            }
            __syncthreads();   // the patch and its histogram are complete
            if (warp != 0) {   // the other warps wait for warp 0 at the end of the round
                __syncthreads();
                continue;
            }
        }
        if (ok) {
            if constexpr (!WIDE) {
                // ---- warp: ps*ps bilinear samples, histogram on the fly ----
                // The inverse map goes into registers first: it lives in shared memory next to the histogram the loop updates
                // with atomics, so the compiler would otherwise reload all nine coefficients for every sample.
                float inv[9];
#pragma unroll
                for (int k = 0; k < 9; k++) inv[k] = ws->proj.inv[k];
                sample_patch(grey, p.w, p.h, inv, ws->proj.cls, ps, lane, 32, patch, ws->hist);
            }
            __syncwarp();
            // ---- otsu_level (SURVEY A.8): integer prefix sums are exact; the f64 expression keeps the reference's order ----
            uint32_t hb[8], bw = 0, bs = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                hb[j] = ws->hist[lane * 8 + j];
                bw += hb[j];
                bs += (uint32_t)(lane * 8 + j) * hb[j];
            }
            uint32_t pw = bw, psum = bs;  // inclusive scan over lanes
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t a = __shfl_up_sync(0xffffffffu, pw, off), b = __shfl_up_sync(0xffffffffu, psum, off);
                if (lane >= off) { pw += a; psum += b; }
            }
            const double total_sum = (double)__shfl_sync(0xffffffffu, psum, 31);
            uint32_t cw = pw - bw, cs = psum - bs;  // exclusive prefix of this lane's first bin
            double best = -1.0;
            uint32_t best_t = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                cw += hb[j];
                cs += (uint32_t)(lane * 8 + j) * hb[j];
                const uint32_t fw = np - cw;
                if (cw != 0 && fw != 0) {
                    const double bsum = (double)cs;
                    const double fsum = total_sum - bsum;
                    const double bm = bsum / (double)cw;
                    const double fm = fsum / (double)fw;
                    const double diff = bm - fm;
                    const double mds = diff * diff;
                    const double v = (double)cw * (double)fw * mds;
                    if (v > best) { best = v; best_t = (uint32_t)(lane * 8 + j); }
                }
            }
            // first strict maximum over t = 0..255, starting from largest_variance = 0: larger value wins, ties go to the smaller t
#pragma unroll
            for (int off = 16; off; off >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, off);
                const uint32_t ot = __shfl_xor_sync(0xffffffffu, best_t, off);
                if (ob > best || (ob == best && ot < best_t)) { best = ob; best_t = ot; }
            }
            otsu_level = best > 0.0 ? best_t : 0u;
            // ---- threshold(Binary) + resize(Triangle): vertical pass into f32, then horizontal pass (SURVEY A.9, A.10) ----
            for (uint32_t i = lane; i < ms * ps; i += 32) {
                const uint32_t oy = i / ps, x = i % ps;
                const int left = meta[2 * oy], cnt = meta[2 * oy + 1];
                const float *wv = taps + oy * max_taps;
                float acc = 0.0f;
                for (int k = 0; k < cnt; k++) {
                    const float s = patch[(size_t)(left + k) * ps + x] > otsu_level ? 255.0f : 0.0f;
                    acc += s * wv[k];
                }
                tmp[i] = acc;
            }
            __syncwarp();
            for (uint32_t i = lane; i < ms * ms; i += 32) {
                const uint32_t y = i / ms, ox = i % ms;
                const int left = meta[2 * ox], cnt = meta[2 * ox + 1];
                const float *wv = taps + ox * max_taps;
                float acc = 0.0f;
                for (int k = 0; k < cnt; k++) acc += tmp[y * ps + left + k] * wv[k];
                const float c = acc < 0.0f ? 0.0f : (acc > 255.0f ? 255.0f : acc);
                reduced[i] = (uint8_t)roundf(c);
            }
        } else {
            // the reference decodes GrayImage::new(1,1): level 0, every cell 0 (src/aruco.rs:256; SURVEY Q5)
            for (uint32_t i = lane; i < ms * ms; i += 32) reduced[i] = 0;
        }
        if (p.patches) {
            uint8_t *dst = p.patches + (size_t)q * np;
            for (uint32_t i = lane; i < np; i += 32) dst[i] = ok ? patch[i] : 0;
        }
        __syncwarp();
        // ---- bits, border test, 4 rotations (src/aruco.rs:276-310) ----
        int good = 1;
        {
            const uint32_t end = ms ? ms - 1 : 0;
            for (uint32_t i = lane; i < ms; i += 32)
                if (reduced[i * ms] > 127 || reduced[i * ms + end] > 127 || reduced[i] > 127 || reduced[end * ms + i] > 127) good = 0;
            good = __all_sync(0xffffffffu, good);
        }
        if (lane < 4) {
            // rotation r reads the grid after r applications of rotate_bit_matrix (new[i][j] = old[j][W-1-i]):
            // r = 1: (i, j) <- (j, W-1-i);  r = 2: (W-1-i, W-1-j);  r = 3: (W-1-j, i)
            uint64_t b = 0;
            if (good) {
                const uint32_t W = ms;
                for (uint32_t y = 1; y + 1 < ms; y++)
                    for (uint32_t x = 1; x + 1 < ms; x++) {
                        uint32_t sy, sx;
                        switch (lane) {
                            case 0: sy = y; sx = x; break;
                            case 1: sy = x; sx = W - 1 - y; break;
                            case 2: sy = W - 1 - y; sx = W - 1 - x; break;
                            default: sy = W - 1 - x; sx = y; break;
                        }
                        if (reduced[sy * ms + sx] > 127) b |= 1;
                        b = (b << 1) | (b >> 63);
                    }
                b = (b >> 1) | (b << 63);
            }
            ws->codes[lane] = b;
        }
        __syncwarp();
        // ---- dictionary match: min over (dist, rotation, index) ----
        uint32_t key = 0xffffffffu;
        if (good) {
            const uint64_t c0 = ws->codes[0], c1 = ws->codes[1], c2 = ws->codes[2], c3 = ws->codes[3];
            for (uint32_t i = lane; i < p.n_codes; i += 32) {
                const uint64_t d = dict[i];
                const uint32_t k0 = ((uint32_t)__popcll(d ^ c0) << 24) | (0u << 22) | i;
                const uint32_t k1 = ((uint32_t)__popcll(d ^ c1) << 24) | (1u << 22) | i;
                const uint32_t k2 = ((uint32_t)__popcll(d ^ c2) << 24) | (2u << 22) | i;
                const uint32_t k3 = ((uint32_t)__popcll(d ^ c3) << 24) | (3u << 22) | i;
                key = min(key, min(min(k0, k1), min(k2, k3)));
            }
        }
        key = __reduce_min_sync(0xffffffffu, key);
        if (lane == 0) {
            a3_decode out;
            out.homography_ok = (uint8_t)ok;
            out.has_codes = (uint8_t)good;
            out.otsu = (uint8_t)otsu_level;
            out.reserved[0] = out.reserved[1] = 0;
            for (int r = 0; r < 4; r++) out.codes[r] = ws->codes[r];
            uint32_t dist = 255, rotation = 0, index = 0;  // find_nearest on an empty list returns (0, 255)
            if (good && p.n_codes) { dist = key >> 24; rotation = (key >> 22) & 3; index = key & 0x3fffffu; }
            out.id = index;
            out.rotation = (uint8_t)rotation;
            out.hamming_distance = (uint8_t)dist;
            out.accepted = (uint8_t)(good && (!p.filter_high_bit_errors || dist < p.tau));
            p.decodes[q] = out;
            if (p.accept_counts && out.accepted) atomicAdd(&p.accept_counts[q >> 10], 1u);
        }
        __syncwarp();
        if constexpr (WIDE) __syncthreads();  // warp 0 is done with the slice: the next candidate may overwrite it
    }
}

}  // namespace

static size_t k2_smem_for(uint32_t ps, uint32_t ms, uint32_t n_codes, uint32_t warps) {
    ResizeTaps tp = make_resize_taps(ps, ms);
    size_t b = (size_t)n_codes * 8 + (size_t)ms * tp.max_taps * 4 + (size_t)2 * ms * 4 + 16;
    return b + (size_t)warps * k2_warp_bytes(ps, ms);
}
// warps per CTA: 8, fewer when the patches of 8 candidates (homography_sample_size^2 bytes each) do not fit shared memory; 0 = not even one
static uint32_t k2_warps(uint32_t ps, uint32_t ms, uint32_t n_codes) {
    for (uint32_t w = kWarps; w >= 1; w >>= 1)
        if (k2_smem_for(ps, ms, n_codes, w) <= 220 * 1024) return w;
    return 0;
}
size_t k2_smem_bytes(uint32_t ps, uint32_t ms, uint32_t n_codes) {
    const uint32_t w = k2_warps(ps, ms, n_codes);
    return k2_smem_for(ps, ms, n_codes, w ? w : 1);
}
bool k2_supported(uint32_t ps, uint32_t ms, uint32_t n_codes) { return ps > 0 && ms >= 3 && ms <= 16 && k2_warps(ps, ms, n_codes) != 0; }

cudaError_t k2_decode(const K2Params &p, cudaStream_t stream) {
    if (p.n_quads == 0) return cudaSuccess;
    if (p.mark_size > 16 || p.mark_size < 3 || p.patch_size == 0 || p.n_codes >= (1u << 22)) return cudaErrorInvalidValue;
    ResizeTaps tp = make_resize_taps(p.patch_size, p.mark_size);
    const uint32_t warps = k2_warps(p.patch_size, p.mark_size, p.n_codes);
    if (warps == 0) return cudaErrorInvalidValue;
    const size_t smem = k2_smem_for(p.patch_size, p.mark_size, p.n_codes, warps);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // few candidates (a frame or two per call): a CTA each, one per SM and round — the time of the launch is one candidate's chain,
    // and eight warps take its samples eight times sooner than one.  A3_K2_WIDE = 0 / 1 forces the choice (tests, timing).
    static const char *wide_env = getenv("A3_K2_WIDE");
    const bool wide = wide_env ? wide_env[0] == '1' : p.n_quads <= 3u * (uint32_t)sms;  // n_quads may be a capacity (history + headroom), the real count lives on the device
    if (wide) {
        const size_t wsmem = k2_smem_for(p.patch_size, p.mark_size, p.n_codes, 1);
        cudaError_t e = cudaFuncSetAttribute(k2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem);
        if (e != cudaSuccess) return e;
        k2_kernel<true><<<p.n_quads < (uint32_t)sms * 3 ? p.n_quads : (uint32_t)sms * 3, kThreads, wsmem, stream>>>(p, tp.max_taps);
        return cudaGetLastError();
    }
    cudaError_t e = cudaFuncSetAttribute(k2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const uint32_t want = (p.n_quads + warps - 1) / warps;
    int per_sm = 0;  // CTAs that are resident together (registers allow 3, shared memory depends on the dictionary)
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k2_kernel<false>, (int)warps * 32, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    const uint32_t resident = (uint32_t)sms * (uint32_t)per_sm;
    k2_kernel<false><<<want < resident ? want : resident, warps * 32, smem, stream>>>(p, tp.max_taps);
    return cudaGetLastError();
}

// image::imageops::resize sampling taps for FilterType::Triangle (support 1.0), f32, reference expression order.
ResizeTaps make_resize_taps(uint32_t n_in, uint32_t n_out) {
    ResizeTaps t;
    t.n_in = n_in; t.n_out = n_out; t.max_taps = 0;
    std::vector<std::vector<float>> rows(n_out);
    t.meta.resize(2 * (size_t)n_out);
    const float ratio = (float)n_in / (float)n_out;
    const float sratio = ratio < 1.0f ? 1.0f : ratio;
    const float src_support = 1.0f * sratio;
    for (uint32_t o = 0; o < n_out; o++) {
        float input = ((float)o + 0.5f) * ratio;
        long long left = (long long)floorf(input - src_support);
        if (left < 0) left = 0;
        if (left > (long long)n_in - 1) left = (long long)n_in - 1;
        long long right = (long long)ceilf(input + src_support);
        if (right < left + 1) right = left + 1;
        if (right > (long long)n_in) right = (long long)n_in;
        input = input - 0.5f;
        float sum = 0.0f;
        for (long long i = left; i < right; i++) {
            float xx = ((float)i - input) / sratio;
            float wv = fabsf(xx) < 1.0f ? 1.0f - fabsf(xx) : 0.0f;
            rows[o].push_back(wv);
            sum += wv;
        }
        for (float &wv : rows[o]) wv /= sum;
        t.meta[2 * o] = (int)left;
        t.meta[2 * o + 1] = (int)(right - left);
        if (rows[o].size() > t.max_taps) t.max_taps = (uint32_t)rows[o].size();
    }
    t.weights.assign((size_t)n_out * t.max_taps, 0.0f);
    for (uint32_t o = 0; o < n_out; o++)
        for (size_t i = 0; i < rows[o].size(); i++) t.weights[(size_t)o * t.max_taps + i] = rows[o][i];
    return t;
}

}  // namespace a3
