// The two rotations of the planar pose ambiguity (pose.rs:158-267), shared by K4 (one marker's square) and K6 (a board's
// homography at its centroid).  Both files are compiled with -fmad=false, so the two use the same f32 arithmetic; K4's
// bit equality with oracle/a3ref_pose.c (a3ref_compute_rotations) covers this code.
#pragma once

namespace a3 {
namespace planar {

struct V3 { float x, y, z; };
struct M3 { float a[3][3]; };  // a[row][col]

// pose.rs:238-267, already transposed (pose.rs:166): returns rv = find_rotation_to_z((tx, ty, 1))^T
__device__ inline void rotation_from_z(float tx, float ty, M3 &rv) {
    const float n = sqrtf(tx * tx + ty * ty + 1.0f * 1.0f);
    const float ax = tx / n, ay = ty / n, az = 1.0f / n;
    if (fabsf(1.0f + az) < 1e-6f) {  // unreachable for z = 1, kept for fidelity
        rv = M3{{{1.0f, 0.0f, 0.0f}, {0.0f, 1.0f, 0.0f}, {0.0f, 0.0f, -1.0f}}};
        return;
    }
    const float d = 1.0f / (1.0f + az);
    const float ax2 = ax * ax, ay2 = ay * ay, axay = ax * ay;
    rv.a[0][0] = -ax2 * d + 1.0f;  rv.a[1][0] = -axay * d;        rv.a[2][0] = -ax;
    rv.a[0][1] = -axay * d;        rv.a[1][1] = -ay2 * d + 1.0f;  rv.a[2][1] = -ay;
    rv.a[0][2] = ax;               rv.a[1][2] = ay;               rv.a[2][2] = 1.0f - (ax2 + ay2) * d;
}

// pose.rs:158-235: the two rotations whose in-plane 2x2 block matches the Jacobian j (row-major) up to scale
__device__ inline void two_rotations(const float (&j)[4], float tx, float ty, M3 &r1, M3 &r2) {
    M3 rv;
    rotation_from_z(tx, ty, rv);
    const float b00 = rv.a[0][0] - tx * rv.a[2][0], b01 = rv.a[0][1] - tx * rv.a[2][1];
    const float b10 = rv.a[1][0] - ty * rv.a[2][0], b11 = rv.a[1][1] - ty * rv.a[2][1];
    const float idet = 1.0f / (b00 * b11 - b01 * b10);
    const float i00 = idet * b11, i01 = -idet * b01, i10 = -idet * b10, i11 = idet * b00;
    const float a00 = i00 * j[0] + i01 * j[2], a01 = i00 * j[1] + i01 * j[3];
    const float a10 = i10 * j[0] + i11 * j[2], a11 = i10 * j[1] + i11 * j[3];
    const float g00 = a00 * a00 + a01 * a01, g01 = a00 * a10 + a01 * a11, g11 = a10 * a10 + a11 * a11;
    const float gamma = sqrtf(0.5f * (g00 + g11 + sqrtf((g00 - g11) * (g00 - g11) + 4.0f * g01 * g01)));
    const float q00 = a00 / gamma, q01 = a01 / gamma, q10 = a10 / gamma, q11 = a11 / gamma;
    const float c0 = sqrtf(-(q00 * q00) - q10 * q10 + 1.0f);
    float c1 = sqrtf(-(q01 * q01) - q11 * q11 + 1.0f);
    if (-q00 * q01 - q10 * q11 < 0.0f) c1 = -c1;
    const float w1a = c1 * q10 - c0 * q11, w2a = c0 * q01 - c1 * q00;
    const float w1b = c0 * q11 - c1 * q10, w2b = c1 * q00 - c0 * q01;
    const float w3 = q00 * q11 - q01 * q10;
#pragma unroll
    for (int r = 0; r < 3; r++) {
        const float v1 = rv.a[r][0], v2 = rv.a[r][1], v3 = rv.a[r][2];
        r1.a[r][0] = q00 * v1 + q10 * v2 + c0 * v3;
        r1.a[r][1] = q01 * v1 + q11 * v2 + c1 * v3;
        r1.a[r][2] = w1a * v1 + w2a * v2 + w3 * v3;
        r2.a[r][0] = q00 * v1 + q10 * v2 + (-c0) * v3;
        r2.a[r][1] = q01 * v1 + q11 * v2 + (-c1) * v3;
        r2.a[r][2] = w1b * v1 + w2b * v2 + w3 * v3;
    }
}

}  // namespace planar
}  // namespace a3
