/*
 * a3ref_board — CPU ORACLE for the board pose (kernel K6).  TEST INFRASTRUCTURE ONLY.
 *
 * The reference has no such stage: this file is the specification the kernel is held to, bit for bit.  Plain C, single
 * threaded, compiled with -ffp-contract=off.  Every sum over a board's points is formed as the kernel forms it: point p
 * goes to lane p % 32 in increasing p, then the 32 lane sums meet in the xor tree 16, 8, 4, 2, 1.  Constants:
 * aruco3_b200/csrc/k6_board_spec.h.
 *
 * Points: image points already normalised (x / w, y / h, or (x - cx) / fx, (y - cy) / fy), f32; object points (x, y) on
 * the board plane (z = 0), x right and y up, f32.  The pose maps board points to camera coordinates, the convention of
 * a3ref_pose.  error = RMS reprojection distance over the points, in normalised units.
 */
#ifndef A3REF_BOARD_H
#define A3REF_BOARD_H

#include <stdint.h>

#include "a3ref_pose.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The solve on n >= 1 correspondences uv[2n] / xy[2n].  Returns 1 when at least one branch succeeded.  A failed branch
 * is a3ref_pose_default (error 1e31). */
int a3ref_board_solve(const float *uv, const float *xy, uint32_t n, a3ref_pose *best, a3ref_pose *alt);

/* One frame: the markers found in it (ids[n], corners[n*8] f32 in a3_marker.corners order), the board (board_ids[m],
 * board_corners[m*8]), the normalisation mode (1 undistorted: image_w / image_h, 2 intrinsics: k).  Markers whose id is not
 * on the board, and every detection of an id seen more than once in the frame, are skipped.  *n_markers = markers used.
 * Returns ok. */
int a3ref_board_frame(const uint64_t *board_ids, const float *board_corners, uint32_t m, uint32_t mode, uint32_t image_w,
                      uint32_t image_h, const a3ref_intrinsics *k, const uint64_t *ids, const float *corners, uint32_t n,
                      a3ref_pose *best, a3ref_pose *alt, uint32_t *n_markers);

#ifdef __cplusplus
}
#endif
#endif
