/* CPU oracle of kernel K5 (see a3ref_refine.h).  Every expression is written in the order k5_corners.cu evaluates it. */
#include "a3ref_refine.h"

#include <math.h>
#include <stddef.h>

#include "../aruco3_b200/csrc/k5_refine_spec.h"

typedef struct {
    float mx, my, dx, dy;
} line_t;

/* 16 values -> one, in the order of a 16-lane xor-shuffle reduction (offsets 8, 4, 2, 1) */
static float tree16(float v[A3_K5_SAMPLES]) {
    for (int off = A3_K5_SAMPLES / 2; off; off >>= 1)
        for (int i = 0; i < off; i++) v[i] = v[i] + v[i + off];
    return v[0];
}

/* bilinear grey at (x, y); *inside = 0 when a neighbour lies outside the image */
static float bilinear(const uint8_t *g, uint32_t w, uint32_t h, float x, float y, int *inside) {
    const float x0 = floorf(x), y0 = floorf(y);
    if (!(x0 >= 0.0f && x0 + 1.0f < (float)w && y0 >= 0.0f && y0 + 1.0f < (float)h)) {
        *inside = 0;
        return 0.0f;
    }
    const size_t ix = (size_t)x0, iy = (size_t)y0;
    const float fx = x - x0, fy = y - y0;
    const uint8_t *r0 = g + iy * w + ix, *r1 = r0 + w;
    const float a = (float)r0[0], b = (float)r0[1], c = (float)r1[0], d = (float)r1[1];
    return (a * (1.0f - fx) + b * fx) * (1.0f - fy) + (c * (1.0f - fx) + d * fx) * fy;
}

/* sample i of the edge p + t * e (outward unit normal n): edge point (*qx, *qy) and its weight (0 = skipped) */
static float edge_sample(const uint8_t *g, uint32_t w, uint32_t h, float px, float py, float ex, float ey, float nx, float ny,
                         int i, float *qx, float *qy) {
    const float t = A3_K5_T0 + A3_K5_TSPAN * (((float)i + 0.5f) / (float)A3_K5_SAMPLES);
    const float bx = px + t * ex, by = py + t * ey;
    float v[A3_K5_READS];
    int inside = 1;
    for (int j = 0; j < A3_K5_READS; j++) {
        const float s = -A3_K5_RANGE + A3_K5_STEP * (float)j;
        v[j] = bilinear(g, w, h, bx + s * nx, by + s * ny, &inside);
    }
    *qx = 0.0f;
    *qy = 0.0f;
    if (!inside) return 0.0f;
    float gmax = v[2] - v[0];
    for (int j = 2; j < A3_K5_READS - 1; j++) gmax = fmaxf(gmax, v[j + 1] - v[j - 1]);
    const float floor_ = A3_K5_FLOOR * gmax;
    float sw = 0.0f, sws = 0.0f;
    for (int j = 1; j < A3_K5_READS - 1; j++) {
        const float wj = fmaxf((v[j + 1] - v[j - 1]) - floor_, 0.0f);
        sw = sw + wj;
        sws = sws + wj * (-A3_K5_RANGE + A3_K5_STEP * (float)j);
    }
    if (!(sw > 0.0f)) return 0.0f;
    const float off = sws / sw;
    *qx = bx + off * nx;
    *qy = by + off * ny;
    return sw;
}

/* weighted total least squares line through the points of weight > 0; 0 when there is no direction */
static int fit_line(const float qx[A3_K5_SAMPLES], const float qy[A3_K5_SAMPLES], const float wt[A3_K5_SAMPLES], line_t *L) {
    float s[A3_K5_SAMPLES], sx[A3_K5_SAMPLES], sy[A3_K5_SAMPLES];
    for (int i = 0; i < A3_K5_SAMPLES; i++) {
        s[i] = wt[i];
        sx[i] = wt[i] * qx[i];
        sy[i] = wt[i] * qy[i];
    }
    const float S = tree16(s), SX = tree16(sx), SY = tree16(sy);
    const float mx = SX / S, my = SY / S;
    float ca[A3_K5_SAMPLES], cb[A3_K5_SAMPLES], cc[A3_K5_SAMPLES];
    for (int i = 0; i < A3_K5_SAMPLES; i++) {
        const float tx = qx[i] - mx, ty = qy[i] - my, wx = wt[i] * tx;
        ca[i] = wx * tx;
        cb[i] = wx * ty;
        cc[i] = (wt[i] * ty) * ty;
    }
    const float a = tree16(ca), b = tree16(cb), c = tree16(cc);
    const float hd = (a - c) * 0.5f;
    const float lam = (a + c) * 0.5f + sqrtf(hd * hd + b * b);
    const float v1x = b, v1y = lam - a, v2x = lam - c, v2y = b;
    const float n1 = v1x * v1x + v1y * v1y, n2 = v2x * v2x + v2y * v2y;
    const int first = n1 >= n2;
    const float vx = first ? v1x : v2x, vy = first ? v1y : v2y, nn = first ? n1 : n2;
    const float r = sqrtf(nn);
    L->mx = mx;
    L->my = my;
    L->dx = vx / r;
    L->dy = vy / r;
    return S > 0.0f && nn > 0.0f;
}

/* edge k of the quad c: sample, fit, drop the far points, refit */
static int fit_edge(const uint8_t *g, uint32_t w, uint32_t h, const float c[8], int k, line_t *L) {
    const int k1 = (k + 1) & 3;
    const float px = c[2 * k], py = c[2 * k + 1];
    const float ex = c[2 * k1] - px, ey = c[2 * k1 + 1] - py;
    const float len = sqrtf(ex * ex + ey * ey);
    const float dx = ex / len, dy = ey / len;
    const float nx = dy, ny = -dx;  /* outward for a screen-clockwise quad, y down: the grey rises along +n */
    float qx[A3_K5_SAMPLES], qy[A3_K5_SAMPLES], wt[A3_K5_SAMPLES];
    for (int i = 0; i < A3_K5_SAMPLES; i++) wt[i] = edge_sample(g, w, h, px, py, ex, ey, nx, ny, i, &qx[i], &qy[i]);
    line_t L1;
    if (!fit_line(qx, qy, wt, &L1)) return 0;
    /* lower median of the distances of the sampled points to the first line (any sort gives the same order statistic) */
    float d[A3_K5_SAMPLES], sorted[A3_K5_SAMPLES];
    int nv = 0;
    for (int i = 0; i < A3_K5_SAMPLES; i++) {
        d[i] = fabsf((qx[i] - L1.mx) * L1.dy - (qy[i] - L1.my) * L1.dx);
        if (wt[i] > 0.0f) {
            int j = nv++;
            for (; j > 0 && sorted[j - 1] > d[i]; j--) sorted[j] = sorted[j - 1];
            sorted[j] = d[i];
        }
    }
    const float med = sorted[(nv - 1) / 2];
    const float lim = fmaxf(A3_K5_REJECT_MIN, A3_K5_REJECT_MEDIANS * med);
    float wt2[A3_K5_SAMPLES];
    int kept = 0;
    for (int i = 0; i < A3_K5_SAMPLES; i++) {
        const int keep = wt[i] > 0.0f && d[i] <= lim;
        wt2[i] = keep ? wt[i] : 0.0f;
        kept += keep;
    }
    if (kept < A3_K5_MIN_KEPT) return 0;
    return fit_line(qx, qy, wt2, L);
}

/* corner k = line of edge k-1 meets line of edge k */
static int intersect(const line_t *a, const line_t *b, float *x, float *y) {
    const float cr = a->dx * b->dy - a->dy * b->dx;
    const float ux = b->mx - a->mx, uy = b->my - a->my;
    const float t = (ux * b->dy - uy * b->dx) / cr;
    *x = a->mx + t * a->dx;
    *y = a->my + t * a->dy;
    return fabsf(cr) >= A3_K5_MIN_CROSS;
}

/* finite, convex and screen-clockwise (every turn positive), every corner within max_move of its integer corner */
static int acceptable(const float c[8], const float c0[8], float max_move) {
    for (int k = 0; k < 4; k++) {
        const int k1 = (k + 1) & 3, k2 = (k + 2) & 3;
        if (!isfinite(c[2 * k]) || !isfinite(c[2 * k + 1])) return 0;
        const float ax = c[2 * k1] - c[2 * k], ay = c[2 * k1 + 1] - c[2 * k + 1];
        const float bx = c[2 * k2] - c[2 * k1], by = c[2 * k2 + 1] - c[2 * k1 + 1];
        if (!(ax * by - ay * bx > 0.0f)) return 0;
        const float mx = c[2 * k] - c0[2 * k], my = c[2 * k + 1] - c0[2 * k + 1];
        if (!(mx * mx + my * my <= max_move * max_move)) return 0;
    }
    return 1;
}

int a3ref_refine_corners(const uint8_t *grey, uint32_t w, uint32_t h, const uint32_t corners[8], float refined[8]) {
    float c0[8], cur[8];
    for (int i = 0; i < 8; i++) c0[i] = (float)corners[i];
    float min_len = INFINITY;
    for (int k = 0; k < 4; k++) {
        const int k1 = (k + 1) & 3;
        const float ex = c0[2 * k1] - c0[2 * k], ey = c0[2 * k1 + 1] - c0[2 * k + 1];
        min_len = fminf(min_len, sqrtf(ex * ex + ey * ey));
    }
    const float max_move = A3_K5_MAX_MOVE * min_len;
    int good = min_len > 0.0f;
    for (int i = 0; i < 8; i++) cur[i] = c0[i];
    for (int pass = 0; pass < A3_K5_PASSES && good; pass++) {
        line_t L[4];
        for (int k = 0; k < 4 && good; k++) good = fit_edge(grey, w, h, cur, k, &L[k]);
        float nxt[8];
        for (int k = 0; k < 4 && good; k++) good = intersect(&L[(k + 3) & 3], &L[k], &nxt[2 * k], &nxt[2 * k + 1]);
        if (good) good = acceptable(nxt, c0, max_move);
        if (good)
            for (int i = 0; i < 8; i++) cur[i] = nxt[i];
    }
    for (int i = 0; i < 8; i++) refined[i] = good ? cur[i] : c0[i];
    return good;
}

void a3ref_solve_with_undistorted_points_f32(const float c[8], float marker_size_mm, uint32_t image_w, uint32_t image_h,
                                             a3ref_pose *best, a3ref_pose *alt) {
    float pts[8];
    for (int i = 0; i < 4; ++i) {
        pts[2 * i] = c[2 * i] / (float)image_w;
        pts[2 * i + 1] = c[2 * i + 1] / (float)image_h;
    }
    a3ref_solve_with_normalized_points(pts, marker_size_mm, best, alt);
}

void a3ref_solve_with_intrinsics_f32(const float c[8], float marker_size_mm, const a3ref_intrinsics *k, a3ref_pose *best,
                                     a3ref_pose *alt) {
    float pts[8];
    for (int i = 0; i < 4; ++i) a3ref_unproject(k, c[2 * i], c[2 * i + 1], pts + 2 * i);
    a3ref_solve_with_normalized_points(pts, marker_size_mm, best, alt);
}
