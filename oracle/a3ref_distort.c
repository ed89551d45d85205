/*
 * a3ref_distort.c — CPU ORACLE for the corner undistortion (kernel K7, see a3ref_distort.h) and the board pose on
 * undistorted corners.
 *
 * Newton's method on OpenCV's forward model from the distorted point itself, in f64, with the analytic Jacobian (symmetric:
 * dDx/dy = dDy/dx) and Cramer's rule; the expressions are written in the kernel's order.
 */
#include "a3ref_distort.h"

#include <math.h>

#include "../aruco3_b200/csrc/k6_board_spec.h"
#include "../aruco3_b200/csrc/k7_undistort_spec.h"
#include "a3ref_board.h"

int a3ref_undistort_point(const a3ref_intrinsics *k, const a3ref_distortion *d, float px, float py, float out[2]) {
    const float nu = (px - k->principal_x) / k->focal_x, nv = (py - k->principal_y) / k->focal_y;
    const double xd = (double)nu, yd = (double)nv;
    const double k1 = (double)d->k1, k2 = (double)d->k2, p1 = (double)d->p1, p2 = (double)d->p2, k3 = (double)d->k3;
    double x = xd, y = yd;
    for (int it = 0;; it++) {
        const double r2 = x * x + y * y;
        const double rad = 1.0 + r2 * (k1 + r2 * (k2 + r2 * k3));
        const double xy = x * y;
        const double fx = (x * rad + 2.0 * p1 * xy + p2 * (r2 + 2.0 * x * x)) - xd;
        const double fy = (y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * xy) - yd;
        if (!isfinite(fx) || !isfinite(fy)) return 0;
        if (fmax(fabs(fx), fabs(fy)) <= A3_UNDIST_TOL) break;
        if (it == A3_UNDIST_ITERS) return 0;
        const double dr = k1 + r2 * (2.0 * k2 + 3.0 * k3 * r2);
        const double j00 = rad + 2.0 * x * x * dr + 2.0 * p1 * y + 6.0 * p2 * x;
        const double j01 = 2.0 * xy * dr + 2.0 * p1 * x + 2.0 * p2 * y;
        const double j11 = rad + 2.0 * y * y * dr + 6.0 * p1 * y + 2.0 * p2 * x;
        const double det = j00 * j11 - j01 * j01;
        if (!(det > 0.0)) return 0;
        x = x - (fx * j11 - fy * j01) / det;
        y = y - (j00 * fy - j01 * fx) / det;
    }
    out[0] = (float)x;
    out[1] = (float)y;
    return isfinite(out[0]) && isfinite(out[1]);
}

void a3ref_undistort_points(const a3ref_intrinsics *k, const a3ref_distortion *d, const float *pts, uint32_t n, float *out, uint8_t *ok) {
    for (uint32_t i = 0; i < n; i++) {
        float o[2] = {0.0f, 0.0f};
        ok[i] = (uint8_t)a3ref_undistort_point(k, d, pts[2 * i], pts[2 * i + 1], o);
        out[2 * i] = ok[i] ? o[0] : 0.0f;
        out[2 * i + 1] = ok[i] ? o[1] : 0.0f;
    }
}

int a3ref_board_frame_distorted(const uint64_t *board_ids, const float *board_corners, uint32_t m, const a3ref_intrinsics *k,
                                const a3ref_distortion *d, const uint64_t *ids, const float *corners, uint32_t n, a3ref_pose *best,
                                a3ref_pose *alt, uint32_t *n_markers) {
    static float uv[2 * 4 * A3_K6_MAX_MARKERS], xy[2 * 4 * A3_K6_MAX_MARKERS];
    static float und[8 * 4 * A3_K6_MAX_MARKERS];
    static uint8_t good[4 * A3_K6_MAX_MARKERS];
    if (n > 4 * A3_K6_MAX_MARKERS) n = 4 * A3_K6_MAX_MARKERS;
    for (uint32_t i = 0; i < n; i++) {
        good[i] = 1;
        for (int c = 0; c < 4; c++)
            good[i] &= (uint8_t)a3ref_undistort_point(k, d, corners[8 * i + 2 * c], corners[8 * i + 2 * c + 1], und + 8 * i + 2 * c);
    }
    uint32_t used = 0;
    for (uint32_t i = 0; i < n && used < A3_K6_MAX_MARKERS; i++) {
        if (!good[i]) continue;
        uint32_t slot = m, seen = 0;
        for (uint32_t s = 0; s < m; s++)
            if (board_ids[s] == ids[i]) slot = s;
        if (slot == m) continue;
        for (uint32_t j = 0; j < n; j++) seen += good[j] && ids[j] == ids[i];
        if (seen != 1) continue;
        for (int c = 0; c < 8; c++) {
            uv[8 * used + c] = und[8 * i + c];
            xy[8 * used + c] = board_corners[8 * slot + c];
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
