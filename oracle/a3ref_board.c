/*
 * a3ref_board.c — CPU ORACLE for the board pose (kernel K6, see a3ref_board.h).
 *
 * 1. Homography from the centred board plane to the normalised image by DLT (h22 = 1), both point sets normalised to
 *    their centroid and a mean distance of sqrt(2); f64 normal equations, Gaussian elimination with partial pivoting.
 * 2. The two rotations of the planar ambiguity from the homography's Jacobian at the centroid (a3ref_compute_rotations,
 *    pose.rs:158-235, fed as the square solve feeds it), each with its translation by linear least squares over all points.
 * 3. A3_K6_ITERS Levenberg-Marquardt steps per branch on the sum of squared reprojection distances: rotation updates by
 *    the Cayley transform (rational, so no sin / cos), 6x6 damped normal equations by Cholesky, f64 throughout.
 */
#include "a3ref_board.h"

#include <math.h>
#include <string.h>

#include "../aruco3_b200/csrc/k6_board_spec.h"

#define L A3_K6_LANES

/* the 32 lane sums -> lane 0 after the xor tree (every lane ends with the same value) */
static double tree(double v[L]) {
    double t[L];
    for (int off = L / 2; off; off >>= 1) {
        for (int l = 0; l < L; l++) t[l] = v[l] + v[l ^ off];
        memcpy(v, t, sizeof t);
    }
    return v[0];
}

/* the sums of K per-point values f(p, out) over n points, as the warp forms them */
typedef void (*point_fn)(const void *ctx, uint32_t p, double *out);
static void warp_sums(const void *ctx, point_fn f, uint32_t n, int k, double *sums) {
    double acc[L][32], val[32], col[L];
    memset(acc, 0, sizeof acc);
    for (int l = 0; l < L; l++)
        for (uint32_t p = (uint32_t)l; p < n; p += L) {
            f(ctx, p, val);
            for (int j = 0; j < k; j++) acc[l][j] = acc[l][j] + val[j];
        }
    for (int j = 0; j < k; j++) {
        for (int l = 0; l < L; l++) col[l] = acc[l][j];
        sums[j] = tree(col);
    }
}

/* Gaussian elimination with partial pivoting on a (row-major, nn x nn, destroyed), right-hand side b -> x; 0 = singular */
static int solve_ge(double *a, double *b, int nn, double *x) {
    for (int c = 0; c < nn; c++) {
        int p = c;
        for (int r = c + 1; r < nn; r++)
            if (fabs(a[r * nn + c]) > fabs(a[p * nn + c])) p = r;
        if (!(fabs(a[p * nn + c]) > 0.0) || !isfinite(a[p * nn + c])) return 0;
        if (p != c) {
            for (int k = 0; k < nn; k++) { const double t = a[c * nn + k]; a[c * nn + k] = a[p * nn + k]; a[p * nn + k] = t; }
            const double t = b[c]; b[c] = b[p]; b[p] = t;
        }
        for (int r = c + 1; r < nn; r++) {
            const double f = a[r * nn + c] / a[c * nn + c];
            for (int k = c + 1; k < nn; k++) a[r * nn + k] = a[r * nn + k] - f * a[c * nn + k];
            b[r] = b[r] - f * b[c];
        }
    }
    for (int i = nn - 1; i >= 0; i--) {
        double s = b[i];
        for (int k = i + 1; k < nn; k++) s = s - a[i * nn + k] * x[k];
        x[i] = s / a[i * nn + i];
    }
    return 1;
}

typedef struct {
    const float *uv, *xy;
    double cx, cy, mu, mv, so, si;  /* centroids, scales */
    double r[9], t[3];              /* a branch's pose (centred board frame) */
    double r2[9];                   /* translation pass: the second rotation */
} ctx_t;

static void f_centroids(const void *c_, uint32_t p, double *o) {
    const ctx_t *c = (const ctx_t *)c_;
    const double u = (double)c->uv[2 * p], v = (double)c->uv[2 * p + 1];
    o[0] = (double)c->xy[2 * p];
    o[1] = (double)c->xy[2 * p + 1];
    o[2] = u;
    o[3] = v;
    o[4] = u * u + v * v;
}
static void f_spread(const void *c_, uint32_t p, double *o) {
    const ctx_t *c = (const ctx_t *)c_;
    const double x = (double)c->xy[2 * p] - c->cx, y = (double)c->xy[2 * p + 1] - c->cy;
    const double u = (double)c->uv[2 * p] - c->mu, v = (double)c->uv[2 * p + 1] - c->mv;
    o[0] = sqrt(x * x + y * y);
    o[1] = sqrt(u * u + v * v);
}
static void f_dlt(const void *c_, uint32_t p, double *o) {
    const ctx_t *c = (const ctx_t *)c_;
    const double x = ((double)c->xy[2 * p] - c->cx) * c->so, y = ((double)c->xy[2 * p + 1] - c->cy) * c->so;
    const double a = ((double)c->uv[2 * p] - c->mu) * c->si, b = ((double)c->uv[2 * p + 1] - c->mv) * c->si;
    const double r = a * a + b * b;
    const double xx = x * x, xy = x * y, yy = y * y;
    o[0] = xx; o[1] = xy; o[2] = yy; o[3] = x; o[4] = y;
    o[5] = a * x; o[6] = a * y; o[7] = a;
    o[8] = b * x; o[9] = b * y; o[10] = b;
    o[11] = a * xx; o[12] = a * xy; o[13] = a * yy;
    o[14] = b * xx; o[15] = b * xy; o[16] = b * yy;
    o[17] = r * xx; o[18] = r * xy; o[19] = r * yy; o[20] = r * x; o[21] = r * y;
}
static void f_translation(const void *c_, uint32_t p, double *o) {
    const ctx_t *c = (const ctx_t *)c_;
    const double x = (double)c->xy[2 * p] - c->cx, y = (double)c->xy[2 * p + 1] - c->cy;
    const double u = (double)c->uv[2 * p], v = (double)c->uv[2 * p + 1];
    for (int b = 0; b < 2; b++) {
        const double *R = b ? c->r2 : c->r;
        const double rx = R[0] * x + R[1] * y, ry = R[3] * x + R[4] * y, rz = R[6] * x + R[7] * y;
        const double e0 = u * rz - rx, e1 = v * rz - ry;
        o[3 * b] = e0;
        o[3 * b + 1] = e1;
        o[3 * b + 2] = -(u * e0) - v * e1;
    }
}
/* residual of point p under (r, t), and with `o` of 28: the 21 entries of J^T J (row-major upper triangle), J^T e, e^T e */
static void residual(const ctx_t *c, uint32_t p, double *ex, double *ey, double ja[6], double jb[6]) {
    const double x = (double)c->xy[2 * p] - c->cx, y = (double)c->xy[2 * p + 1] - c->cy;
    const double u = (double)c->uv[2 * p], v = (double)c->uv[2 * p + 1];
    const double *R = c->r;
    const double qx = R[0] * x + R[1] * y, qy = R[3] * x + R[4] * y, qz = R[6] * x + R[7] * y;
    const double X = qx + c->t[0], Y = qy + c->t[1], Z = qz + c->t[2];
    const double iz = 1.0 / Z;
    const double px = X * iz, py = Y * iz;
    *ex = px - u;
    *ey = py - v;
    if (!ja) return;
    ja[0] = -px * qy * iz; ja[1] = (qz + px * qx) * iz; ja[2] = -qy * iz; ja[3] = iz; ja[4] = 0.0; ja[5] = -px * iz;
    jb[0] = (-qz - py * qy) * iz; jb[1] = py * qx * iz; jb[2] = qx * iz; jb[3] = 0.0; jb[4] = iz; jb[5] = -py * iz;
}
static void f_normal(const void *c_, uint32_t p, double *o) {
    double ex, ey, ja[6], jb[6];
    residual((const ctx_t *)c_, p, &ex, &ey, ja, jb);
    int k = 0;
    for (int i = 0; i < 6; i++)
        for (int j = i; j < 6; j++) o[k++] = ja[i] * ja[j] + jb[i] * jb[j];
    for (int i = 0; i < 6; i++) o[k++] = ja[i] * ex + jb[i] * ey;
    o[k] = ex * ex + ey * ey;
}
static void f_cost(const void *c_, uint32_t p, double *o) {
    double ex, ey;
    residual((const ctx_t *)c_, p, &ex, &ey, 0, 0);
    o[0] = ex * ex + ey * ey;
}

/* (A + lam diag(A)) d = -g by Cholesky; 0 = not positive definite */
static int solve_damped(const double s[28], double lam, double d[6]) {
    double a[6][6], l[6][6], y[6];
    int k = 0;
    for (int i = 0; i < 6; i++)
        for (int j = i; j < 6; j++) { a[i][j] = s[k]; a[j][i] = s[k]; k++; }
    for (int i = 0; i < 6; i++) a[i][i] = a[i][i] + lam * a[i][i];
    for (int i = 0; i < 6; i++)
        for (int j = 0; j <= i; j++) {
            double v = a[i][j];
            for (int m = 0; m < j; m++) v = v - l[i][m] * l[j][m];
            if (i == j) {
                if (!(v > 0.0) || !isfinite(v)) return 0;
                l[i][i] = sqrt(v);
            } else {
                l[i][j] = v / l[j][j];
            }
        }
    for (int i = 0; i < 6; i++) {
        double v = -s[21 + i];
        for (int m = 0; m < i; m++) v = v - l[i][m] * y[m];
        y[i] = v / l[i][i];
    }
    for (int i = 5; i >= 0; i--) {
        double v = y[i];
        for (int m = i + 1; m < 6; m++) v = v - l[m][i] * d[m];
        d[i] = v / l[i][i];
    }
    return 1;
}

/* Cayley transform of w / 2 applied on the left: r <- C r */
static void cayley_update(const double w[3], double r[9]) {
    const double cx = 0.5 * w[0], cy = 0.5 * w[1], cz = 0.5 * w[2];
    const double cc = cx * cx + cy * cy + cz * cz, den = 1.0 + cc, dg = 1.0 - cc;
    const double m[9] = {(dg + 2.0 * (cx * cx)) / den, 2.0 * (cx * cy - cz) / den, 2.0 * (cx * cz + cy) / den,
                         2.0 * (cx * cy + cz) / den, (dg + 2.0 * (cy * cy)) / den, 2.0 * (cy * cz - cx) / den,
                         2.0 * (cx * cz - cy) / den, 2.0 * (cy * cz + cx) / den, (dg + 2.0 * (cz * cz)) / den};
    double o[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) o[3 * i + j] = m[3 * i] * r[j] + m[3 * i + 1] * r[3 + j] + m[3 * i + 2] * r[6 + j];
    memcpy(r, o, sizeof o);
}

/* LM on one branch (c->r, c->t set); fills `out` or leaves the default; returns 1 on success */
static int refine_branch(ctx_t *c, uint32_t n, a3ref_pose *out) {
    a3ref_pose_default(out);
    double lam = A3_K6_LAMBDA0, cost = 0.0, s[28], d[6], c1;
    for (int it = 0; it < A3_K6_ITERS; it++) {
        warp_sums(c, f_normal, n, 28, s);
        cost = s[27];
        if (!solve_damped(s, lam, d)) return 0;
        const double r0[9] = {c->r[0], c->r[1], c->r[2], c->r[3], c->r[4], c->r[5], c->r[6], c->r[7], c->r[8]};
        const double t0[3] = {c->t[0], c->t[1], c->t[2]};
        cayley_update(d, c->r);
        c->t[0] = t0[0] + d[3]; c->t[1] = t0[1] + d[4]; c->t[2] = t0[2] + d[5];
        warp_sums(c, f_cost, n, 1, &c1);
        if (c1 < cost) {
            cost = c1;
            lam = lam * A3_K6_LAMBDA_DOWN;
        } else {
            memcpy(c->r, r0, sizeof r0);
            memcpy(c->t, t0, sizeof t0);
            lam = lam * A3_K6_LAMBDA_UP;
        }
    }
    double tb[3];
    for (int i = 0; i < 3; i++) tb[i] = c->t[i] - (c->r[3 * i] * c->cx + c->r[3 * i + 1] * c->cy);
    int ok = isfinite(cost) && tb[2] > 0.0 && isfinite(tb[0]) && isfinite(tb[1]) && isfinite(tb[2]);
    for (int i = 0; i < 9; i++) ok = ok && isfinite(c->r[i]);
    if (!ok) return 0;
    out->error = (float)sqrt(cost / (double)n);
    for (int i = 0; i < 9; i++) out->rotation[i] = (float)c->r[i];
    for (int i = 0; i < 3; i++) out->translation[i] = (float)tb[i];
    return 1;
}

int a3ref_board_solve(const float *uv, const float *xy, uint32_t n, a3ref_pose *best, a3ref_pose *alt) {
    a3ref_pose_default(best);
    a3ref_pose_default(alt);
    if (n == 0) return 0;
    ctx_t c;
    memset(&c, 0, sizeof c);
    c.uv = uv;
    c.xy = xy;
    const double nd = (double)n;
    double s[22];
    warp_sums(&c, f_centroids, n, 5, s);
    c.cx = s[0] / nd; c.cy = s[1] / nd; c.mu = s[2] / nd; c.mv = s[3] / nd;
    const double su = s[2], sv = s[3], sr = s[4];
    warp_sums(&c, f_spread, n, 2, s);
    if (!(s[0] > 0.0) || !(s[1] > 0.0)) return 0;
    c.so = 1.4142135623730951 * nd / s[0];
    c.si = 1.4142135623730951 * nd / s[1];
    warp_sums(&c, f_dlt, n, 22, s);
    /* rows [x y 1 0 0 0 -ax -ay] = a and [0 0 0 x y 1 -bx -by] = b */
    double m[64] = {0}, rhs[8], h[8];
    const double sxx = s[0], sxy = s[1], syy = s[2], sx = s[3], sy = s[4];
    const double blk[9] = {sxx, sxy, sx, sxy, syy, sy, sx, sy, nd};
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) { m[i * 8 + j] = blk[3 * i + j]; m[(i + 3) * 8 + j + 3] = blk[3 * i + j]; }
    const double e6[6] = {-s[11], -s[12], -s[5], -s[14], -s[15], -s[8]}, e7[6] = {-s[12], -s[13], -s[6], -s[15], -s[16], -s[9]};
    for (int i = 0; i < 6; i++) { m[i * 8 + 6] = e6[i]; m[6 * 8 + i] = e6[i]; m[i * 8 + 7] = e7[i]; m[7 * 8 + i] = e7[i]; }
    m[6 * 8 + 6] = s[17]; m[6 * 8 + 7] = s[18]; m[7 * 8 + 6] = s[18]; m[7 * 8 + 7] = s[19];
    rhs[0] = s[5]; rhs[1] = s[6]; rhs[2] = s[7]; rhs[3] = s[8]; rhs[4] = s[9]; rhs[5] = s[10]; rhs[6] = -s[20]; rhs[7] = -s[21];
    if (!solve_ge(m, rhs, 8, h)) return 0;
    /* H = Ti^-1 Hn diag(so, so, 1), Ti = [[si, 0, -si mu], [0, si, -si mv], [0, 0, 1]]; H22 = 1 */
    const double g[9] = {h[0] * c.so, h[1] * c.so, h[2], h[3] * c.so, h[4] * c.so, h[5], h[6] * c.so, h[7] * c.so, 1.0};
    double H[9];
    for (int j = 0; j < 3; j++) {
        H[j] = g[j] / c.si + c.mu * g[6 + j];
        H[3 + j] = g[3 + j] / c.si + c.mv * g[6 + j];
        H[6 + j] = g[6 + j];
    }
    /* Jacobian of the projection at the centroid, and the centroid's image */
    const float jf[4] = {(float)(H[0] - H[6] * H[2]), (float)(H[1] - H[7] * H[2]), (float)(H[3] - H[6] * H[5]),
                         (float)(H[4] - H[7] * H[5])};
    float r1[9], r2[9];
    a3ref_compute_rotations(jf, (float)H[2], (float)H[5], r1, r2);
    for (int i = 0; i < 9; i++) { c.r[i] = (double)r1[i]; c.r2[i] = (double)r2[i]; }
    warp_sums(&c, f_translation, n, 6, s);
    double t1[3], t2[3];
    int ok1, ok2;
    {
        double a[9] = {nd, 0.0, -su, 0.0, nd, -sv, -su, -sv, sr}, b[3] = {s[0], s[1], s[2]};
        ok1 = solve_ge(a, b, 3, t1);
        double a2[9] = {nd, 0.0, -su, 0.0, nd, -sv, -su, -sv, sr}, b2[3] = {s[3], s[4], s[5]};
        ok2 = solve_ge(a2, b2, 3, t2);
    }
    a3ref_pose p1, p2;
    double rr2[9];
    memcpy(rr2, c.r2, sizeof rr2);
    memcpy(c.t, t1, sizeof t1);
    ok1 = ok1 && refine_branch(&c, n, &p1);
    if (!ok1) a3ref_pose_default(&p1);
    memcpy(c.r, rr2, sizeof rr2);
    memcpy(c.t, t2, sizeof t2);
    ok2 = ok2 && refine_branch(&c, n, &p2);
    if (!ok2) a3ref_pose_default(&p2);
    if (p1.error < p2.error) {
        *best = p1;
        *alt = p2;
    } else {
        *best = p2;
        *alt = p1;
    }
    return ok1 || ok2;
}

int a3ref_board_frame(const uint64_t *board_ids, const float *board_corners, uint32_t m, uint32_t mode, uint32_t image_w,
                      uint32_t image_h, const a3ref_intrinsics *k, const uint64_t *ids, const float *corners, uint32_t n,
                      a3ref_pose *best, a3ref_pose *alt, uint32_t *n_markers) {
    static float uv[2 * 4 * A3_K6_MAX_MARKERS], xy[2 * 4 * A3_K6_MAX_MARKERS];
    uint32_t used = 0;
    for (uint32_t i = 0; i < n; i++) {
        uint32_t slot = m, seen = 0;
        for (uint32_t s = 0; s < m; s++)
            if (board_ids[s] == ids[i]) slot = s;
        if (slot == m) continue;
        for (uint32_t j = 0; j < n; j++) seen += ids[j] == ids[i];
        if (seen != 1) continue;
        for (int c = 0; c < 4; c++) {
            const float x = corners[8 * i + 2 * c], y = corners[8 * i + 2 * c + 1];
            float *o = uv + 8 * used + 2 * c;
            if (mode == 1) {
                o[0] = x / (float)image_w;
                o[1] = y / (float)image_h;
            } else {
                o[0] = (x - k->principal_x) / k->focal_x;
                o[1] = (y - k->principal_y) / k->focal_y;
            }
            xy[8 * used + 2 * c] = board_corners[8 * slot + 2 * c];
            xy[8 * used + 2 * c + 1] = board_corners[8 * slot + 2 * c + 1];
        }
        used++;
    }
    *n_markers = used;
    if (!used) {
        a3ref_pose_default(best);
        a3ref_pose_default(alt);
        return 0;
    }
    return a3ref_board_solve(uv, xy, 4 * used, best, alt);
}
