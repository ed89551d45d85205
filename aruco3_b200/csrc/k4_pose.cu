// K4 — marker pose from four corners (SURVEY §8 f-3): the step that follows `detect` in both of the reference's examples
// (examples/webcam_kamera.rs:68, examples/macroquad_detect.rs:150).
//
// Restates /root/reference/src/pose.rs:52-348 (closed-form planar pose of a centred square: homography -> Jacobian at the
// centre -> the two rotations consistent with it -> translation from the normal equations -> reprojection error, best
// first) and the unproject step of src/pinhole.rs:88-93.  All f32, evaluated in the reference's operation order; this file
// is compiled with -fmad=false because Rust never contracts a*b+c.  IEEE division and square root (nvcc defaults).
//
// One thread per marker: the whole solve is ~450 dependent flops on 8 inputs, so there is nothing to share between
// threads; the kernel is launch-latency bound (5.6 k candidates of a 256-frame batch = one partial wave) and is queued
// on the decode stream right behind K2, reading K2's records (accepted, rotation) and the quads where they already lie.
#include "a3_internal.h"
#include "planar_rotations.cuh"

namespace a3 {
namespace {

using planar::M3;
using planar::V3;
using planar::two_rotations;

// nalgebra's Matrix3 * Vector3: y = col0*v0; y = col1*v1 + y; y = col2*v2 + y
__device__ __forceinline__ V3 mul(const M3 &m, const V3 &v) {
    V3 r;
    r.x = m.a[0][2] * v.z + (m.a[0][1] * v.y + m.a[0][0] * v.x);
    r.y = m.a[1][2] * v.z + (m.a[1][1] * v.y + m.a[1][0] * v.x);
    r.z = m.a[2][2] * v.z + (m.a[2][1] * v.y + m.a[2][0] * v.x);
    return r;
}

// pose.rs:96-123.  Signs of all image points are flipped first; s = half the marker side.
__device__ void square_homography(float s, const float (&px)[4], const float (&py)[4], M3 &h) {
    const float x1 = -px[0], x2 = -px[1], x3 = -px[2], x4 = -px[3];
    const float y1 = -py[0], y2 = -py[1], y3 = -py[2], y4 = -py[3];
    const float k = -1.0f / (s * (x1 * y2 - x2 * y1 - x1 * y4 + x2 * y3 - x3 * y2 + x4 * y1 + x3 * y4 - x4 * y3));
    h.a[0][0] = k * (x1 * x3 * y2 - x2 * x3 * y1 - x1 * x4 * y2 + x2 * x4 * y1 - x1 * x3 * y4 + x1 * x4 * y3 + x2 * x3 * y4 - x2 * x4 * y3);
    h.a[0][1] = k * (x1 * x2 * y3 - x1 * x3 * y2 - x1 * x2 * y4 + x2 * x4 * y1 + x1 * x3 * y4 - x3 * x4 * y1 - x2 * x4 * y3 + x3 * x4 * y2);
    h.a[0][2] = k * s * (x1 * x2 * y3 - x2 * x3 * y1 - x1 * x2 * y4 + x1 * x4 * y2 - x1 * x4 * y3 + x3 * x4 * y1 + x2 * x3 * y4 - x3 * x4 * y2);
    h.a[1][0] = k * (x1 * y2 * y3 - x2 * y1 * y3 - x1 * y2 * y4 + x2 * y1 * y4 - x3 * y1 * y4 + x4 * y1 * y3 + x3 * y2 * y4 - x4 * y2 * y3);
    h.a[1][1] = k * (x2 * y1 * y3 - x3 * y1 * y2 - x1 * y2 * y4 + x4 * y1 * y2 + x1 * y3 * y4 - x4 * y1 * y3 - x2 * y3 * y4 + x3 * y2 * y4);
    h.a[1][2] = k * s * (x1 * y2 * y3 - x3 * y1 * y2 - x2 * y1 * y4 + x4 * y1 * y2 - x1 * y3 * y4 + x3 * y1 * y4 + x2 * y3 * y4 - x4 * y2 * y3);
    h.a[2][0] = -k * (x1 * y3 - x3 * y1 - x1 * y4 - x2 * y3 + x3 * y2 + x4 * y1 + x2 * y4 - x4 * y2);
    h.a[2][1] = k * (x1 * y2 - x2 * y1 - x1 * y3 + x3 * y1 + x2 * y4 - x4 * y2 - x3 * y4 + x4 * y3);
    h.a[2][2] = 1.0f;
}

// pose.rs:269-335: t = (A^T A)^-1 A^T b with only the non-trivial coefficients kept
__device__ V3 translation_for(const M3 &rot, float s, const float (&px)[4], const float (&py)[4]) {
    const float ox[4] = {-s, s, s, -s}, oy[4] = {s, s, -s, -s};  // make_marker_square, pose.rs:85-93
    float sa = 0.0f, sb = 0.0f, sq = 0.0f, u0 = 0.0f, u1 = 0.0f, u2 = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const float rx = rot.a[0][0] * ox[i] + rot.a[0][1] * oy[i];
        const float ry = rot.a[1][0] * ox[i] + rot.a[1][1] * oy[i];
        const float rz = rot.a[2][0] * ox[i] + rot.a[2][1] * oy[i];
        const float a2 = -px[i], b2 = -py[i];
        sa += a2;
        sb += b2;
        sq += a2 * a2 + b2 * b2;
        const float bx = -a2 * rz - rx, by = -b2 * rz - ry;
        u0 += bx;
        u1 += by;
        u2 += a2 * bx + b2 * by;
    }
    // ata = [[4, 0, sa], [0, 4, sb], [sa, sb, sq]]
    const float m11 = 4.0f, m22 = 4.0f;
    const float idet = 1.0f / (m11 * m22 * sq - m11 * sb * sb - sa * m22 * sa);
    V3 t;
    t.x = idet * ((m22 * sq - sb * sb) * u0 + (sa * sb) * u1 + (-sa * m22) * u2);
    t.y = idet * ((sb * sa) * u0 + (m11 * sq - sa * sa) * u1 + (-m11 * sb) * u2);
    t.z = idet * ((-m22 * sa) * u0 + (-m11 * sb) * u1 + (m11 * m22) * u2);
    return t;
}

// pose.rs:337-348
__device__ float reprojection_error(const M3 &rot, const V3 &t, float s, const float (&px)[4], const float (&py)[4]) {
    const float ox[4] = {-s, s, s, -s}, oy[4] = {s, s, -s, -s};
    float err = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        V3 p = mul(rot, V3{ox[i], oy[i], 0.0f});
        p.x += t.x; p.y += t.y; p.z += t.z;
        const float z = fmaxf(p.z, 1e-5f);
        const float dx = p.x / z - px[i], dy = p.y / z - py[i];
        err += sqrtf(dx * dx + dy * dy);
    }
    return err;
}

__device__ void store_pose(a3_pose *out, float err, const M3 &r, const V3 &t) {
    out->error = err;
#pragma unroll
    for (int i = 0; i < 9; i++) out->rotation[i] = r.a[i / 3][i % 3];
    out->translation[0] = t.x; out->translation[1] = t.y; out->translation[2] = t.z;
}

// pose.rs:64-81 (solve_with_normalized_points) + 130-156 (solve_canonical_form)
__device__ void solve_square(const float (&px)[4], const float (&py)[4], float marker_size, a3_pose *best, a3_pose *alt) {
    const float s = 0.5f * marker_size;  // == marker_size / 2.0 exactly
    M3 h, r1, r2;
    square_homography(s, px, py, h);
    const float j[4] = {h.a[0][0] - h.a[2][0] * h.a[0][2], h.a[0][1] - h.a[2][1] * h.a[0][2],
                        h.a[1][0] - h.a[2][0] * h.a[1][2], h.a[1][1] - h.a[2][1] * h.a[1][2]};
    two_rotations(j, h.a[0][2], h.a[1][2], r1, r2);
    const V3 t1 = translation_for(r1, s, px, py), t2 = translation_for(r2, s, px, py);
    const float e1 = reprojection_error(r1, t1, s, px, py), e2 = reprojection_error(r2, t2, s, px, py);
    if (e1 < e2) {
        store_pose(best, e1, r1, t1);
        store_pose(alt, e2, r2, t2);
    } else {
        store_pose(best, e2, r2, t2);
        store_pose(alt, e1, r1, t1);
    }
}

__global__ void __launch_bounds__(128) k4_pose_kernel(K4Params p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n || (p.n_dev && i >= *p.n_dev)) return;
    uint32_t rot = 0;
    if (p.decodes) {  // pipeline use: only accepted candidates become markers; corners.rotate_left(rotation), aruco.rs:97-103
        const a3_decode &dc = p.decodes[i];
        if (!dc.accepted) return;
        rot = dc.rotation & 3;
    }
    if (p.points_ok && !p.points_ok[i]) {  // a corner K7 could not undistort: the default pair (pose.rs:42-50)
        for (int b = 0; b < 2; b++) {
            a3_pose *o = p.poses + (size_t)i * 2 + b;
            o->error = 1e31f;
#pragma unroll
            for (int j = 0; j < 9; j++) o->rotation[j] = (j % 4 == 0) ? 1.0f : 0.0f;
            o->translation[0] = o->translation[1] = o->translation[2] = 0.0f;
        }
        return;
    }
    float px[4], py[4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
        const uint32_t sidx = (c + rot) & 3;
        if (p.mode == A3_POSE_NORMALIZED) {
            px[c] = p.points[(size_t)i * 8 + 2 * sidx];
            py[c] = p.points[(size_t)i * 8 + 2 * sidx + 1];
        } else {
            float x, y;
            if (p.corners_f32) {  // K5's corners: already in marker order
                x = p.corners_f32[(size_t)i * 8 + 2 * c];
                y = p.corners_f32[(size_t)i * 8 + 2 * c + 1];
            } else {
                x = (float)p.corners[(size_t)i * 8 + 2 * sidx];
                y = (float)p.corners[(size_t)i * 8 + 2 * sidx + 1];
            }
            if (p.mode == A3_POSE_UNDISTORTED) {  // pose.rs:59-62
                px[c] = x / (float)p.image_w;
                py[c] = y / (float)p.image_h;
            } else {                              // pose.rs:52-55 + pinhole.rs:88-93
                px[c] = (x - p.k.principal_x) / p.k.focal_x;
                py[c] = (y - p.k.principal_y) / p.k.focal_y;
            }
        }
    }
    solve_square(px, py, p.marker_size, p.poses + (size_t)i * 2, p.poses + (size_t)i * 2 + 1);
}

}  // namespace

cudaError_t k4_pose(const K4Params &p, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    k4_pose_kernel<<<(p.n + 127) / 128, 128, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace a3
