// K6 — board pose (opt-in, a3_detector_set_board): one pose per frame of a rigid planar board from the corners of every
// accepted marker whose id is on it.
//
// Specification: oracle/a3ref_board.c, which this kernel equals bit for bit (constants in k6_board_spec.h).  Compiled with
// -fmad=false, IEEE division and square root.  DLT homography at the board's centroid (f64 normal equations, Gaussian
// elimination with partial pivoting) -> the two rotations of the planar ambiguity (planar_rotations.cuh, K4's code) ->
// translations by linear least squares -> A3_K6_ITERS Levenberg-Marquardt steps per branch (Cayley rotation updates, 6x6
// Cholesky), f64.
//
// One warp per frame (a block of 32 threads).  The board's id -> slot table sits in shared memory; the frame's items are
// filtered in candidate order (accepted, on the board, id seen once in the frame) into a shared list.  Every sum over the
// points is lane-strided (point p on lane p % 32, in increasing p) and closed by an xor-shuffle tree, which leaves the same
// value on every lane, so every lane runs the small solves redundantly and all control flow stays warp-uniform; lane 0
// writes the result.  Queued behind K2 (and K5) on the decode groups and on the one-shot route.
#include <math.h>

#include "a3_internal.h"
#include "k6_board_spec.h"
#include "planar_rotations.cuh"

namespace a3 {
namespace {

constexpr unsigned kFull = 0xffffffffu;

struct Frame {
    const K6Params *p;
    const uint32_t *used;    // shared: item index of used marker i
    const uint16_t *slot;    // shared: its board slot
    double cx, cy, mu, mv, so, si;
    double r[9], t[3], r2[9];
};

// point q of the frame: normalised image point (u, v) and board point (x, y): K7's point, or the corner normalised in f32
// the way K4 normalises corners
__device__ __forceinline__ void point(const Frame &f, uint32_t q, double &u, double &v, double &x, double &y) {
    const K6Params &p = *f.p;
    const uint32_t k = f.used[q >> 2], c = q & 3u, s = f.slot[q >> 2];
    x = (double)p.board[(size_t)s * 8 + 2 * c];
    y = (double)p.board[(size_t)s * 8 + 2 * c + 1];
    if (p.norm) {  // K7's points, already normalised and undistorted, where K4 reads them
        const uint32_t sidx = (c + (p.decodes ? p.decodes[k].rotation & 3u : 0u)) & 3u;
        u = (double)p.norm[(size_t)k * 8 + 2 * sidx];
        v = (double)p.norm[(size_t)k * 8 + 2 * sidx + 1];
        return;
    }
    float px, py;
    if (p.corners_f32) {
        px = p.corners_f32[(size_t)k * 8 + 2 * c];
        py = p.corners_f32[(size_t)k * 8 + 2 * c + 1];
    } else {
        const uint32_t sidx = (c + (p.decodes ? p.decodes[k].rotation & 3u : 0u)) & 3u;
        px = (float)p.quads[(size_t)k * 8 + 2 * sidx];
        py = (float)p.quads[(size_t)k * 8 + 2 * sidx + 1];
    }
    float nu, nv;
    if (p.mode == A3_POSE_UNDISTORTED) {
        nu = px / (float)p.image_w;
        nv = py / (float)p.image_h;
    } else {
        nu = (px - p.k.principal_x) / p.k.focal_x;
        nv = (py - p.k.principal_y) / p.k.focal_y;
    }
    u = (double)nu;
    v = (double)nv;
}

// sums of K per-point values over n points: lane-strided, then the xor tree (the oracle's warp_sums)
template <int K, typename F>
__device__ __forceinline__ void warp_sums(uint32_t n, F fn, double (&s)[K]) {
    const uint32_t lane = threadIdx.x & 31u;
#pragma unroll
    for (int j = 0; j < K; j++) s[j] = 0.0;
    for (uint32_t q = lane; q < n; q += A3_K6_LANES) {
        double v[K];
        fn(q, v);
#pragma unroll
        for (int j = 0; j < K; j++) s[j] = s[j] + v[j];
    }
#pragma unroll
    for (int j = 0; j < K; j++)
#pragma unroll
        for (int off = A3_K6_LANES / 2; off; off >>= 1) s[j] = s[j] + __shfl_xor_sync(kFull, s[j], off);
}

template <int N>
__device__ bool solve_ge(double (&a)[N * N], double (&b)[N], double (&x)[N]) {
    for (int c = 0; c < N; c++) {
        int p = c;
        for (int r = c + 1; r < N; r++)
            if (fabs(a[r * N + c]) > fabs(a[p * N + c])) p = r;
        if (!(fabs(a[p * N + c]) > 0.0) || !isfinite(a[p * N + c])) return false;
        if (p != c) {
            for (int k = 0; k < N; k++) { const double t = a[c * N + k]; a[c * N + k] = a[p * N + k]; a[p * N + k] = t; }
            const double t = b[c]; b[c] = b[p]; b[p] = t;
        }
        for (int r = c + 1; r < N; r++) {
            const double f = a[r * N + c] / a[c * N + c];
            for (int k = c + 1; k < N; k++) a[r * N + k] = a[r * N + k] - f * a[c * N + k];
            b[r] = b[r] - f * b[c];
        }
    }
    for (int i = N - 1; i >= 0; i--) {
        double s = b[i];
        for (int k = i + 1; k < N; k++) s = s - a[i * N + k] * x[k];
        x[i] = s / a[i * N + i];
    }
    return true;
}

__device__ __forceinline__ void residual(const Frame &f, uint32_t q, double &ex, double &ey, double *ja, double *jb) {
    double u, v, x, y;
    point(f, q, u, v, x, y);
    x = x - f.cx;
    y = y - f.cy;
    const double qx = f.r[0] * x + f.r[1] * y, qy = f.r[3] * x + f.r[4] * y, qz = f.r[6] * x + f.r[7] * y;
    const double X = qx + f.t[0], Y = qy + f.t[1], Z = qz + f.t[2];
    const double iz = 1.0 / Z;
    const double px = X * iz, py = Y * iz;
    ex = px - u;
    ey = py - v;
    if (!ja) return;
    ja[0] = -px * qy * iz; ja[1] = (qz + px * qx) * iz; ja[2] = -qy * iz; ja[3] = iz; ja[4] = 0.0; ja[5] = -px * iz;
    jb[0] = (-qz - py * qy) * iz; jb[1] = py * qx * iz; jb[2] = qx * iz; jb[3] = 0.0; jb[4] = iz; jb[5] = -py * iz;
}

__device__ bool solve_damped(const double (&s)[28], double lam, double (&d)[6]) {
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
                if (!(v > 0.0) || !isfinite(v)) return false;
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
    return true;
}

__device__ void cayley_update(const double (&w)[6], double (&r)[9]) {
    const double cx = 0.5 * w[0], cy = 0.5 * w[1], cz = 0.5 * w[2];
    const double cc = cx * cx + cy * cy + cz * cz, den = 1.0 + cc, dg = 1.0 - cc;
    const double m[9] = {(dg + 2.0 * (cx * cx)) / den, 2.0 * (cx * cy - cz) / den, 2.0 * (cx * cz + cy) / den,
                         2.0 * (cx * cy + cz) / den, (dg + 2.0 * (cy * cy)) / den, 2.0 * (cy * cz - cx) / den,
                         2.0 * (cx * cz - cy) / den, 2.0 * (cy * cz + cx) / den, (dg + 2.0 * (cz * cz)) / den};
    double o[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) o[3 * i + j] = m[3 * i] * r[j] + m[3 * i + 1] * r[3 + j] + m[3 * i + 2] * r[6 + j];
    for (int i = 0; i < 9; i++) r[i] = o[i];
}

__device__ __forceinline__ void pose_default(a3_pose &p) {
    p.error = 1e31f;
    for (int i = 0; i < 9; i++) p.rotation[i] = (i % 4 == 0) ? 1.0f : 0.0f;
    p.translation[0] = p.translation[1] = p.translation[2] = 0.0f;
}

// Levenberg-Marquardt on the branch in f.r / f.t (the oracle's refine_branch)
__device__ bool refine_branch(Frame &f, uint32_t n, a3_pose &out) {
    pose_default(out);
    double lam = A3_K6_LAMBDA0, cost = 0.0;
    for (int it = 0; it < A3_K6_ITERS; it++) {
        double s[28], d[6], c1[1];
        warp_sums<28>(n, [&](uint32_t q, double (&o)[28]) {
            double ex, ey, ja[6], jb[6];
            residual(f, q, ex, ey, ja, jb);
            int k = 0;
#pragma unroll
            for (int i = 0; i < 6; i++)
#pragma unroll
                for (int j = i; j < 6; j++) o[k++] = ja[i] * ja[j] + jb[i] * jb[j];
#pragma unroll
            for (int i = 0; i < 6; i++) o[k++] = ja[i] * ex + jb[i] * ey;
            o[k] = ex * ex + ey * ey;
        }, s);
        cost = s[27];
        if (!solve_damped(s, lam, d)) return false;
        double r0[9], t0[3];
        for (int i = 0; i < 9; i++) r0[i] = f.r[i];
        for (int i = 0; i < 3; i++) t0[i] = f.t[i];
        cayley_update(d, f.r);
        f.t[0] = t0[0] + d[3]; f.t[1] = t0[1] + d[4]; f.t[2] = t0[2] + d[5];
        warp_sums<1>(n, [&](uint32_t q, double (&o)[1]) {
            double ex, ey;
            residual(f, q, ex, ey, nullptr, nullptr);
            o[0] = ex * ex + ey * ey;
        }, c1);
        if (c1[0] < cost) {
            cost = c1[0];
            lam = lam * A3_K6_LAMBDA_DOWN;
        } else {
            for (int i = 0; i < 9; i++) f.r[i] = r0[i];
            for (int i = 0; i < 3; i++) f.t[i] = t0[i];
            lam = lam * A3_K6_LAMBDA_UP;
        }
    }
    double tb[3];
    for (int i = 0; i < 3; i++) tb[i] = f.t[i] - (f.r[3 * i] * f.cx + f.r[3 * i + 1] * f.cy);
    bool ok = isfinite(cost) && tb[2] > 0.0 && isfinite(tb[0]) && isfinite(tb[1]) && isfinite(tb[2]);
    for (int i = 0; i < 9; i++) ok = ok && isfinite(f.r[i]);
    if (!ok) return false;
    out.error = (float)sqrt(cost / (double)n);
    for (int i = 0; i < 9; i++) out.rotation[i] = (float)f.r[i];
    for (int i = 0; i < 3; i++) out.translation[i] = (float)tb[i];
    return true;
}

// the oracle's a3ref_board_solve on the frame's n points; every lane returns the same result
__device__ bool board_solve(Frame &f, uint32_t n, a3_pose &best, a3_pose &alt) {
    pose_default(best);
    pose_default(alt);
    const double nd = (double)n;
    double s5[5], s2[2], s[22];
    warp_sums<5>(n, [&](uint32_t q, double (&o)[5]) {
        double u, v, x, y;
        point(f, q, u, v, x, y);
        o[0] = x; o[1] = y; o[2] = u; o[3] = v; o[4] = u * u + v * v;
    }, s5);
    f.cx = s5[0] / nd; f.cy = s5[1] / nd; f.mu = s5[2] / nd; f.mv = s5[3] / nd;
    const double su = s5[2], sv = s5[3], sr = s5[4];
    warp_sums<2>(n, [&](uint32_t q, double (&o)[2]) {
        double u, v, x, y;
        point(f, q, u, v, x, y);
        x = x - f.cx; y = y - f.cy; u = u - f.mu; v = v - f.mv;
        o[0] = sqrt(x * x + y * y);
        o[1] = sqrt(u * u + v * v);
    }, s2);
    if (!(s2[0] > 0.0) || !(s2[1] > 0.0)) return false;
    f.so = 1.4142135623730951 * nd / s2[0];
    f.si = 1.4142135623730951 * nd / s2[1];
    warp_sums<22>(n, [&](uint32_t q, double (&o)[22]) {
        double u, v, x, y;
        point(f, q, u, v, x, y);
        x = (x - f.cx) * f.so; y = (y - f.cy) * f.so;
        const double a = (u - f.mu) * f.si, b = (v - f.mv) * f.si;
        const double r = a * a + b * b;
        const double xx = x * x, xy = x * y, yy = y * y;
        o[0] = xx; o[1] = xy; o[2] = yy; o[3] = x; o[4] = y;
        o[5] = a * x; o[6] = a * y; o[7] = a;
        o[8] = b * x; o[9] = b * y; o[10] = b;
        o[11] = a * xx; o[12] = a * xy; o[13] = a * yy;
        o[14] = b * xx; o[15] = b * xy; o[16] = b * yy;
        o[17] = r * xx; o[18] = r * xy; o[19] = r * yy; o[20] = r * x; o[21] = r * y;
    }, s);
    double m[64], rhs[8], h[8];
    for (int i = 0; i < 64; i++) m[i] = 0.0;
    const double blk[9] = {s[0], s[1], s[3], s[1], s[2], s[4], s[3], s[4], nd};
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) { m[i * 8 + j] = blk[3 * i + j]; m[(i + 3) * 8 + j + 3] = blk[3 * i + j]; }
    const double e6[6] = {-s[11], -s[12], -s[5], -s[14], -s[15], -s[8]}, e7[6] = {-s[12], -s[13], -s[6], -s[15], -s[16], -s[9]};
    for (int i = 0; i < 6; i++) { m[i * 8 + 6] = e6[i]; m[6 * 8 + i] = e6[i]; m[i * 8 + 7] = e7[i]; m[7 * 8 + i] = e7[i]; }
    m[6 * 8 + 6] = s[17]; m[6 * 8 + 7] = s[18]; m[7 * 8 + 6] = s[18]; m[7 * 8 + 7] = s[19];
    rhs[0] = s[5]; rhs[1] = s[6]; rhs[2] = s[7]; rhs[3] = s[8]; rhs[4] = s[9]; rhs[5] = s[10]; rhs[6] = -s[20]; rhs[7] = -s[21];
    if (!solve_ge<8>(m, rhs, h)) return false;
    const double g[9] = {h[0] * f.so, h[1] * f.so, h[2], h[3] * f.so, h[4] * f.so, h[5], h[6] * f.so, h[7] * f.so, 1.0};
    double H[9];
    for (int j = 0; j < 3; j++) {
        H[j] = g[j] / f.si + f.mu * g[6 + j];
        H[3 + j] = g[3 + j] / f.si + f.mv * g[6 + j];
        H[6 + j] = g[6 + j];
    }
    const float jf[4] = {(float)(H[0] - H[6] * H[2]), (float)(H[1] - H[7] * H[2]), (float)(H[3] - H[6] * H[5]), (float)(H[4] - H[7] * H[5])};
    planar::M3 r1, r2;
    planar::two_rotations(jf, (float)H[2], (float)H[5], r1, r2);
    for (int i = 0; i < 9; i++) { f.r[i] = (double)r1.a[i / 3][i % 3]; f.r2[i] = (double)r2.a[i / 3][i % 3]; }
    double st[6];
    warp_sums<6>(n, [&](uint32_t q, double (&o)[6]) {
        double u, v, x, y;
        point(f, q, u, v, x, y);
        x = x - f.cx; y = y - f.cy;
#pragma unroll
        for (int b = 0; b < 2; b++) {
            const double *R = b ? f.r2 : f.r;
            const double rx = R[0] * x + R[1] * y, ry = R[3] * x + R[4] * y, rz = R[6] * x + R[7] * y;
            const double e0 = u * rz - rx, e1 = v * rz - ry;
            o[3 * b] = e0;
            o[3 * b + 1] = e1;
            o[3 * b + 2] = -(u * e0) - v * e1;
        }
    }, st);
    double t1[3], t2[3];
    bool ok1, ok2;
    {
        double a[9] = {nd, 0.0, -su, 0.0, nd, -sv, -su, -sv, sr}, b[3] = {st[0], st[1], st[2]};
        ok1 = solve_ge<3>(a, b, t1);
        double a2[9] = {nd, 0.0, -su, 0.0, nd, -sv, -su, -sv, sr}, b2[3] = {st[3], st[4], st[5]};
        ok2 = solve_ge<3>(a2, b2, t2);
    }
    a3_pose p1, p2;
    double rr2[9];
    for (int i = 0; i < 9; i++) rr2[i] = f.r2[i];
    for (int i = 0; i < 3; i++) f.t[i] = t1[i];
    ok1 = ok1 && refine_branch(f, n, p1);
    if (!ok1) pose_default(p1);
    for (int i = 0; i < 9; i++) f.r[i] = rr2[i];
    for (int i = 0; i < 3; i++) f.t[i] = t2[i];
    ok2 = ok2 && refine_branch(f, n, p2);
    if (!ok2) pose_default(p2);
    if (p1.error < p2.error) {
        best = p1;
        alt = p2;
    } else {
        best = p2;
        alt = p1;
    }
    return ok1 || ok2;
}

__global__ void __launch_bounds__(32) k6_board_kernel(K6Params p) {
    extern __shared__ uint16_t s_slots[];  // n_codes
    __shared__ uint32_t s_count[A3_K6_MAX_MARKERS], s_used[A3_K6_MAX_MARKERS];
    __shared__ uint16_t s_uslot[A3_K6_MAX_MARKERS];
    if (p.skip && *p.skip) return;
    const uint32_t lane = threadIdx.x, fr = blockIdx.x;
    for (uint32_t i = lane; i < p.n_codes; i += 32) s_slots[i] = p.slots[i];
    for (uint32_t i = lane; i < p.n_board; i += 32) s_count[i] = 0;
    __syncwarp();
    const uint32_t o0 = p.offsets[fr], o1 = p.offsets[fr + 1];
    auto slot_of = [&](uint32_t i) -> uint32_t {  // board slot of item i, or A3_K6_NO_SLOT
        uint64_t id;
        if (p.decodes) {
            const a3_decode &dc = p.decodes[i];
            if (!dc.accepted) return A3_K6_NO_SLOT;
            id = dc.id;
        } else {
            id = p.ids[i];
        }
        if (p.norm_ok && !p.norm_ok[i]) return A3_K6_NO_SLOT;  // a corner K7 could not undistort: as if not detected
        return id < p.n_codes ? s_slots[id] : A3_K6_NO_SLOT;
    };
    for (uint32_t i = o0 + lane; i < o1; i += 32) {
        const uint32_t s = slot_of(i);
        if (s != A3_K6_NO_SLOT) atomicAdd(&s_count[s], 1u);
    }
    __syncwarp();
    uint32_t nu = 0;
    for (uint32_t b0 = o0; b0 < o1; b0 += 32) {  // the markers used, in candidate order
        const uint32_t i = b0 + lane;
        const uint32_t s = i < o1 ? slot_of(i) : A3_K6_NO_SLOT;
        const bool use = s != A3_K6_NO_SLOT && s_count[s] == 1;
        const uint32_t bal = __ballot_sync(kFull, use);
        if (use) {
            const uint32_t pos = nu + __popc(bal & ((1u << lane) - 1u));
            s_used[pos] = i;
            s_uslot[pos] = (uint16_t)s;
        }
        nu += __popc(bal);
    }
    __syncwarp();
    a3_board_pose r;
    r.n_markers = nu;
    r.reserved[0] = r.reserved[1] = r.reserved[2] = 0;
    if (nu == 0) {
        pose_default(r.best);
        pose_default(r.alt);
        r.ok = 0;
    } else {
        Frame f;
        f.p = &p; f.used = s_used; f.slot = s_uslot;
        r.ok = board_solve(f, 4 * nu, r.best, r.alt) ? 1 : 0;
    }
    if (lane == 0) p.out[fr] = r;
}

}  // namespace

cudaError_t k6_board(const K6Params &p, cudaStream_t stream) {
    if (p.n_frames == 0) return cudaSuccess;
    k6_board_kernel<<<p.n_frames, 32, (size_t)p.n_codes * sizeof(uint16_t), stream>>>(p);
    return cudaGetLastError();
}

}  // namespace a3
