/*
 * Constants of the sub-pixel corner refinement (kernel K5, k5_corners.cu) and of its CPU oracle (oracle/a3ref_refine.c).
 * Plain C so that both include this one file; the algorithm they share is written out in DESIGN.md §4 (K5).
 *
 * Two passes; per pass and edge, A3_K5_SAMPLES points along the edge (t = T0 + TSPAN * (i + 0.5) / SAMPLES, so the
 * corners themselves are avoided), each read bilinearly at A3_K5_READS offsets -RANGE .. +RANGE (step STEP) along the
 * outward normal; the edge point is the centroid of the positive central differences above FLOOR * their maximum.
 * Lines are weighted total least squares fits, refitted once without the points farther than
 * max(REJECT_MIN, REJECT_MEDIANS * median distance) from the first fit.
 */
#ifndef A3_K5_REFINE_SPEC_H
#define A3_K5_REFINE_SPEC_H

#define A3_K5_PASSES 2
#define A3_K5_SAMPLES 16          /* samples per edge: one 16-lane half of a warp per edge */
#define A3_K5_T0 0.12f
#define A3_K5_TSPAN 0.76f
#define A3_K5_READS 25            /* bilinear reads per sample: offsets -RANGE + STEP * j, j = 0 .. READS - 1 */
#define A3_K5_RANGE 3.0f
#define A3_K5_STEP 0.25f
#define A3_K5_FLOOR 0.3f          /* gradient weight = max(g - FLOOR * max g, 0) */
#define A3_K5_REJECT_MIN 1.0f     /* second fit keeps distance <= max(REJECT_MIN, REJECT_MEDIANS * median) */
#define A3_K5_REJECT_MEDIANS 2.5f
#define A3_K5_MIN_KEPT 4          /* fallback when an edge keeps fewer samples */
#define A3_K5_MIN_CROSS 1e-3f     /* fallback when adjacent unit directions have |cross| below this */
#define A3_K5_MAX_MOVE 0.25f      /* fallback when a corner moves more than this times the shortest integer edge */

#endif
