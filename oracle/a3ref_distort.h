/*
 * a3ref_distort — CPU ORACLE for the corner undistortion (kernel K7) and the board pose with a lens distortion.
 * TEST INFRASTRUCTURE ONLY.
 *
 * The reference has no lens model: this file is the specification the kernel is held to, bit for bit.  Plain C, single
 * threaded, compiled with -ffp-contract=off.  Model, iteration and failure rule: aruco3_b200/csrc/k7_undistort_spec.h.
 */
#ifndef A3REF_DISTORT_H
#define A3REF_DISTORT_H

#include <stdint.h>

#include "a3ref_pose.h"

#ifdef __cplusplus
extern "C" {
#endif

/* OpenCV's k1 k2 p1 p2 k3, on the normalised coordinates of a3ref_intrinsics */
typedef struct a3ref_distortion {
    float k1, k2, p1, p2, k3;
} a3ref_distortion;

/* One pixel (pixel-centre convention) -> its normalised undistorted point out[2].  Returns 1, or 0 when the point fails
 * (out is then unspecified). */
int a3ref_undistort_point(const a3ref_intrinsics *k, const a3ref_distortion *d, float x, float y, float out[2]);

/* n points pts[2n] -> out[2n], ok[n] */
void a3ref_undistort_points(const a3ref_intrinsics *k, const a3ref_distortion *d, const float *pts, uint32_t n, float *out, uint8_t *ok);

/* a3ref_board_frame in intrinsics mode with a distortion: every corner is undistorted first, and a marker with a corner that
 * fails is skipped before the other rules (as if it had not been detected).  The board solve (a3ref_board_solve) then runs
 * on the undistorted points. */
int a3ref_board_frame_distorted(const uint64_t *board_ids, const float *board_corners, uint32_t m, const a3ref_intrinsics *k,
                                const a3ref_distortion *d, const uint64_t *ids, const float *corners, uint32_t n, a3ref_pose *best,
                                a3ref_pose *alt, uint32_t *n_markers);

#ifdef __cplusplus
}
#endif
#endif
