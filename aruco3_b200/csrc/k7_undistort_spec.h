/*
 * Specification of the corner undistortion (kernel K7, k7_undistort.cu) and of its CPU oracle (oracle/a3ref_distort.c),
 * in one place so the two cannot drift apart.  Plain C: the oracle includes it too.
 *
 * Model: OpenCV's five-coefficient Brown-Conrady distortion (k1 k2 p1 p2 k3) on the normalised coordinates of
 * a3_camera_intrinsics.  With r2 = x^2 + y^2 and rad = 1 + r2 (k1 + r2 (k2 + r2 k3)) the forward model D is
 *     Dx = x rad + 2 p1 x y + p2 (r2 + 2 x^2),    Dy = y rad + p1 (r2 + 2 y^2) + 2 p2 x y.
 * A pixel (px, py) is normalised in f32 exactly as K4 does it, xd = (px - cx) / fx, yd = (py - cy) / fy, widened to f64
 * with the coefficients, and D(x, y) = (xd, yd) is solved by Newton's method from (xd, yd): the analytic Jacobian, each
 * step by Cramer's rule, at most A3_UNDIST_ITERS steps, stopping when max(|Fx|, |Fy|) <= A3_UNDIST_TOL.  The result is
 * rounded to f32.  The point fails when the Jacobian's determinant is not > 0 at a step (the model folds there), when the
 * iteration does not converge within the step limit, or when any value is non-finite.
 */
#ifndef A3_K7_UNDISTORT_SPEC_H
#define A3_K7_UNDISTORT_SPEC_H

#define A3_UNDIST_ITERS 20     /* Newton steps at most */
#define A3_UNDIST_TOL 1e-12    /* convergence: max(|Fx|, |Fy|) in normalised units */

#endif
