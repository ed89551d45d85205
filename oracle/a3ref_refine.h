/*
 * a3ref_refine — CPU ORACLE for the sub-pixel corner refinement (kernel K5).  TEST INFRASTRUCTURE ONLY.
 *
 * The reference has no such stage: this file is the specification the kernel is held to, bit for bit.  Plain C, single
 * threaded, f32, compiled with -ffp-contract=off; every sum over the 16 samples of an edge is the pairwise tree a
 * 16-lane xor-shuffle reduction produces ((v[i] + v[i+8]), then + 4, + 2, + 1).  Constants: aruco3_b200/csrc/k5_refine_spec.h.
 *
 * Input: four integer corners x0,y0..x3,y3, screen-clockwise in y-down image coordinates (a3_marker.corners, or a quad
 * before its rotation: the result is rotation-equivariant).  Output: four f32 corners in the pixel-centre convention
 * (grey pixel (x, y) is the point (x, y)).  Returns 1 when refined, 0 when it fell back to the integer corners as f32.
 */
#ifndef A3REF_REFINE_H
#define A3REF_REFINE_H

#include <stdint.h>

#include "a3ref_pose.h"

#ifdef __cplusplus
extern "C" {
#endif

int a3ref_refine_corners(const uint8_t *grey, uint32_t w, uint32_t h, const uint32_t corners[8], float refined[8]);

/* solve_with_undistorted_points / solve_with_intrinsics on f32 image corners: the same normalisation the u32 entries
 * apply after their `as f32` cast, then the same solver. */
void a3ref_solve_with_undistorted_points_f32(const float corners[8], float marker_size_mm, uint32_t image_w,
                                             uint32_t image_h, a3ref_pose *best, a3ref_pose *alt);
void a3ref_solve_with_intrinsics_f32(const float corners[8], float marker_size_mm, const a3ref_intrinsics *k,
                                     a3ref_pose *best, a3ref_pose *alt);

#ifdef __cplusplus
}
#endif
#endif
