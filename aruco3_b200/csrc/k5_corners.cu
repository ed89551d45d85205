// K5 — sub-pixel marker corners (opt-in, a3_detector_set_corner_refinement): each accepted candidate's integer corners
// become four f32 corners in the pixel-centre convention, from lines fitted to the grey image's edge profile.
//
// Specification: oracle/a3ref_refine.c, which this kernel equals bit for bit (constants in k5_refine_spec.h).  Compiled
// with -fmad=false, IEEE division and square root; every sum over an edge's 16 samples is the pairwise tree of a 16-lane
// xor-shuffle reduction, the order the oracle restates.
//
// One warp per marker: lane l takes sample (l & 15) of edges (l >> 4) and (l >> 4) + 2, i.e. each 16-lane half owns two
// edges, so every reduction stays inside a half.  Per pass and marker that is 4 x 16 x 25 bilinear reads of the grey
// (resident in L2 behind K1 and K2).  The corners are computed redundantly by every lane from the four lines, so all
// control flow that reaches a shuffle is warp-uniform.  Queued behind K2 (its `accepted` / `rotation`) and ahead of K4.
#include <math.h>

#include "a3_internal.h"
#include "k5_refine_spec.h"

namespace a3 {
namespace {

constexpr unsigned kFull = 0xffffffffu;

struct Line { float mx, my, dx, dy; };

__device__ __forceinline__ float seg_sum(float v) {  // sum over the lane's 16-lane half, tree (i, i+8), (i, i+4), ...
#pragma unroll
    for (int off = A3_K5_SAMPLES / 2; off; off >>= 1) v = v + __shfl_xor_sync(kFull, v, off);
    return v;
}
__device__ __forceinline__ float seg_min(float v) {
#pragma unroll
    for (int off = A3_K5_SAMPLES / 2; off; off >>= 1) v = fminf(v, __shfl_xor_sync(kFull, v, off));
    return v;
}

// corner k of c (k in 0..3, runtime) without indexing the register array dynamically
__device__ __forceinline__ void corner_at(const float (&c)[8], int k, float &x, float &y) {
    x = k == 0 ? c[0] : k == 1 ? c[2] : k == 2 ? c[4] : c[6];
    y = k == 0 ? c[1] : k == 1 ? c[3] : k == 2 ? c[5] : c[7];
}

__device__ __forceinline__ float bilinear(const uint8_t *__restrict__ g, uint32_t w, uint32_t h, float x, float y, bool &inside) {
    const float x0 = floorf(x), y0 = floorf(y);
    if (!(x0 >= 0.0f && x0 + 1.0f < (float)w && y0 >= 0.0f && y0 + 1.0f < (float)h)) {
        inside = false;
        return 0.0f;
    }
    const size_t ix = (size_t)x0, iy = (size_t)y0;
    const float fx = x - x0, fy = y - y0;
    const uint8_t *r0 = g + iy * w + ix, *r1 = r0 + w;
    const float a = (float)__ldg(r0), b = (float)__ldg(r0 + 1), c = (float)__ldg(r1), d = (float)__ldg(r1 + 1);
    return (a * (1.0f - fx) + b * fx) * (1.0f - fy) + (c * (1.0f - fx) + d * fx) * fy;
}

// sample i of the edge p + t * e: the edge point and its weight (0 = skipped, point (0, 0))
__device__ float edge_sample(const uint8_t *__restrict__ g, uint32_t w, uint32_t h, float px, float py, float ex, float ey, float nx, float ny,
                             int i, float &qx, float &qy) {
    const float t = A3_K5_T0 + A3_K5_TSPAN * (((float)i + 0.5f) / (float)A3_K5_SAMPLES);
    const float bx = px + t * ex, by = py + t * ey;
    float v[A3_K5_READS];
    bool inside = true;
#pragma unroll
    for (int j = 0; j < A3_K5_READS; j++) {
        const float s = -A3_K5_RANGE + A3_K5_STEP * (float)j;
        v[j] = bilinear(g, w, h, bx + s * nx, by + s * ny, inside);
    }
    qx = 0.0f;
    qy = 0.0f;
    if (!inside) return 0.0f;
    float gmax = v[2] - v[0];
#pragma unroll
    for (int j = 2; j < A3_K5_READS - 1; j++) gmax = fmaxf(gmax, v[j + 1] - v[j - 1]);
    const float floor_ = A3_K5_FLOOR * gmax;
    float sw = 0.0f, sws = 0.0f;
#pragma unroll
    for (int j = 1; j < A3_K5_READS - 1; j++) {
        const float wj = fmaxf((v[j + 1] - v[j - 1]) - floor_, 0.0f);
        sw = sw + wj;
        sws = sws + wj * (-A3_K5_RANGE + A3_K5_STEP * (float)j);
    }
    if (!(sw > 0.0f)) return 0.0f;
    const float off = sws / sw;
    qx = bx + off * nx;
    qy = by + off * ny;
    return sw;
}

// weighted total least squares line of the half's 16 points; every lane of the half returns the same line and flag
__device__ bool fit_line(float qx, float qy, float wt, Line &L) {
    const float S = seg_sum(wt), SX = seg_sum(wt * qx), SY = seg_sum(wt * qy);
    const float mx = SX / S, my = SY / S;
    const float tx = qx - mx, ty = qy - my, wx = wt * tx;
    const float a = seg_sum(wx * tx), b = seg_sum(wx * ty), c = seg_sum((wt * ty) * ty);
    const float hd = (a - c) * 0.5f;
    const float lam = (a + c) * 0.5f + sqrtf(hd * hd + b * b);
    const float v1x = b, v1y = lam - a, v2x = lam - c, v2y = b;
    const float n1 = v1x * v1x + v1y * v1y, n2 = v2x * v2x + v2y * v2y;
    const bool first = n1 >= n2;
    const float vx = first ? v1x : v2x, vy = first ? v1y : v2y, nn = first ? n1 : n2;
    const float r = sqrtf(nn);
    L.mx = mx; L.my = my; L.dx = vx / r; L.dy = vy / r;
    return S > 0.0f && nn > 0.0f;
}

// the line of edge k (this lane's half) of quad c: sample, fit, drop the far points, refit
__device__ bool fit_edge(const uint8_t *__restrict__ g, uint32_t w, uint32_t h, const float (&c)[8], int k, int i, uint32_t half_mask, Line &L) {
    float px, py, qx1, qy1;
    corner_at(c, k, px, py);
    corner_at(c, (k + 1) & 3, qx1, qy1);
    const float ex = qx1 - px, ey = qy1 - py;
    const float len = sqrtf(ex * ex + ey * ey);
    const float dx = ex / len, dy = ey / len;
    const float nx = dy, ny = -dx;  // outward for a screen-clockwise quad, y down
    float qx, qy;
    const float wt = edge_sample(g, w, h, px, py, ex, ey, nx, ny, i, qx, qy);
    Line L1;
    bool ok = fit_line(qx, qy, wt, L1);
    // lower median of the sampled points' distances to the first line: the value whose rank bracket holds (n - 1) / 2
    const bool valid = wt > 0.0f;
    const float d = fabsf((qx - L1.mx) * L1.dy - (qy - L1.my) * L1.dx);
    const float dv = valid ? d : INFINITY;
    const int base = (int)(threadIdx.x & 16);
    int less = 0, le = 0;
#pragma unroll
    for (int j = 0; j < A3_K5_SAMPLES; j++) {
        const float o = __shfl_sync(kFull, dv, base + j);
        less += o < dv;
        le += o <= dv;
    }
    const int nv = __popc(__ballot_sync(kFull, valid) & half_mask), kth = (nv - 1) / 2;
    const float med = seg_min((valid && less <= kth && kth < le) ? dv : INFINITY);
    const float lim = fmaxf(A3_K5_REJECT_MIN, A3_K5_REJECT_MEDIANS * med);
    const bool keep = valid && d <= lim;
    const int kept = __popc(__ballot_sync(kFull, keep) & half_mask);
    ok = ok && kept >= A3_K5_MIN_KEPT;
    const bool ok2 = fit_line(qx, qy, keep ? wt : 0.0f, L);
    return ok && ok2;
}

__device__ __forceinline__ bool intersect(const Line &a, const Line &b, float &x, float &y) {
    const float cr = a.dx * b.dy - a.dy * b.dx;
    const float ux = b.mx - a.mx, uy = b.my - a.my;
    const float t = (ux * b.dy - uy * b.dx) / cr;
    x = a.mx + t * a.dx;
    y = a.my + t * a.dy;
    return fabsf(cr) >= A3_K5_MIN_CROSS;
}

__device__ bool acceptable(const float (&c)[8], const float (&c0)[8], float max_move) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int k1 = (k + 1) & 3, k2 = (k + 2) & 3;
        ok = ok && isfinite(c[2 * k]) && isfinite(c[2 * k + 1]);
        const float ax = c[2 * k1] - c[2 * k], ay = c[2 * k1 + 1] - c[2 * k + 1];
        const float bx = c[2 * k2] - c[2 * k1], by = c[2 * k2 + 1] - c[2 * k1 + 1];
        ok = ok && ax * by - ay * bx > 0.0f;
        const float mx = c[2 * k] - c0[2 * k], my = c[2 * k + 1] - c0[2 * k + 1];
        ok = ok && mx * mx + my * my <= max_move * max_move;
    }
    return ok;
}

__device__ __forceinline__ Line shfl_line(const Line &l, int src) {
    return Line{__shfl_sync(kFull, l.mx, src), __shfl_sync(kFull, l.my, src), __shfl_sync(kFull, l.dx, src), __shfl_sync(kFull, l.dy, src)};
}

__global__ void __launch_bounds__(128) k5_corners_kernel(K5Params p) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t m = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (m >= p.n || (p.n_dev && m >= *p.n_dev)) return;  // warp-uniform from here on
    uint32_t rot = 0;
    if (p.decodes) {  // pipeline use: accepted candidates only; output corners.rotate_left(rotation), like a3_marker.corners
        const a3_decode &dc = p.decodes[m];
        if (!dc.accepted) return;
        rot = dc.rotation & 3u;
    }
    const uint8_t *g = p.grey + (p.quad_frame ? (size_t)p.quad_frame[m] * p.w * p.h : 0);
    float c0[8], cur[8];
#pragma unroll
    for (int k = 0; k < 8; k++) c0[k] = (float)p.quads[(size_t)m * 8 + k];
    float min_len = INFINITY;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int k1 = (k + 1) & 3;
        const float ex = c0[2 * k1] - c0[2 * k], ey = c0[2 * k1 + 1] - c0[2 * k + 1];
        min_len = fminf(min_len, sqrtf(ex * ex + ey * ey));
    }
    const float max_move = A3_K5_MAX_MOVE * min_len;
    bool good = min_len > 0.0f;
#pragma unroll
    for (int k = 0; k < 8; k++) cur[k] = c0[k];
    const int half = (int)(lane >> 4), i = (int)(lane & 15);
    const uint32_t half_mask = half ? 0xffff0000u : 0x0000ffffu;
    for (int pass = 0; pass < A3_K5_PASSES && good; pass++) {
        Line La, Lb;  // edges half and half + 2
        const bool oka = fit_edge(g, p.w, p.h, cur, half, i, half_mask, La);
        const bool okb = fit_edge(g, p.w, p.h, cur, half + 2, i, half_mask, Lb);
        const bool ok_all = __all_sync(kFull, oka && okb);
        Line L[4] = {shfl_line(La, 0), shfl_line(La, 16), shfl_line(Lb, 0), shfl_line(Lb, 16)};
        float nxt[8];
        bool ok = ok_all;
#pragma unroll
        for (int k = 0; k < 4; k++) ok = intersect(L[(k + 3) & 3], L[k], nxt[2 * k], nxt[2 * k + 1]) && ok;
        good = ok && acceptable(nxt, c0, max_move);
        if (good)
#pragma unroll
            for (int k = 0; k < 8; k++) cur[k] = nxt[k];
    }
    if (lane == 0) {
#pragma unroll
        for (int c = 0; c < 4; c++) {
            float x, y;
            corner_at(good ? cur : c0, (int)((c + rot) & 3u), x, y);
            p.corners[(size_t)m * 8 + 2 * c] = x;
            p.corners[(size_t)m * 8 + 2 * c + 1] = y;
        }
        p.ok[m] = good ? 1 : 0;
    }
}

}  // namespace

cudaError_t k5_corners(const K5Params &p, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    k5_corners_kernel<<<(p.n + 3) / 4, 128, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace a3
