// K7 — lens undistortion of marker corners (opt-in, a3_detector_set_distortion): every corner the pose kernels read
// becomes a normalised, undistorted point once, and K4 / K6 solve from those points.
//
// Specification: k7_undistort_spec.h and oracle/a3ref_distort.c, which this kernel equals bit for bit.  Compiled with
// -fmad=false, IEEE division.  One thread per (item, corner): four consecutive lanes hold one marker, and a ballot over
// them gives the marker's flag.  Output layout: the corner K4's normalised read takes as marker corner c, i.e. screen
// corner (c + rotation) & 3 of the quad, sits at out[8 i + 2 ((c + rotation) & 3)], so K4 and K6 read these points where
// they would read the quad's integer corners.  Queued behind K2 and K5 on the decode groups and on the one-shot route.
#include <math.h>

#include "a3_internal.h"
#include "k7_undistort_spec.h"

namespace a3 {
namespace {

constexpr unsigned kFull = 0xffffffffu;

// the spec's Newton solve of D(x, y) = ((px - cx) / fx, (py - cy) / fy); false = the point fails
__device__ __forceinline__ bool undistort(float px, float py, const a3_camera_intrinsics &k, const a3_camera_distortion &dist, float &ou,
                                          float &ov) {
    const float nu = (px - k.principal_x) / k.focal_x, nv = (py - k.principal_y) / k.focal_y;
    const double xd = (double)nu, yd = (double)nv;
    const double k1 = (double)dist.k1, k2 = (double)dist.k2, p1 = (double)dist.p1, p2 = (double)dist.p2, k3 = (double)dist.k3;
    double x = xd, y = yd;
    for (int it = 0;; it++) {
        const double r2 = x * x + y * y;
        const double rad = 1.0 + r2 * (k1 + r2 * (k2 + r2 * k3));
        const double xy = x * y;
        const double fx = (x * rad + 2.0 * p1 * xy + p2 * (r2 + 2.0 * x * x)) - xd;
        const double fy = (y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * xy) - yd;
        if (!isfinite(fx) || !isfinite(fy)) return false;
        if (fmax(fabs(fx), fabs(fy)) <= A3_UNDIST_TOL) break;
        if (it == A3_UNDIST_ITERS) return false;
        const double dr = k1 + r2 * (2.0 * k2 + 3.0 * k3 * r2);  // d rad / d r2
        const double j00 = rad + 2.0 * x * x * dr + 2.0 * p1 * y + 6.0 * p2 * x;
        const double j01 = 2.0 * xy * dr + 2.0 * p1 * x + 2.0 * p2 * y;  // = j10
        const double j11 = rad + 2.0 * y * y * dr + 6.0 * p1 * y + 2.0 * p2 * x;
        const double det = j00 * j11 - j01 * j01;
        if (!(det > 0.0)) return false;
        x = x - (fx * j11 - fy * j01) / det;
        y = y - (j00 * fy - j01 * fx) / det;
    }
    ou = (float)x;
    ov = (float)y;
    return isfinite(ou) && isfinite(ov);
}

__global__ void __launch_bounds__(128) k7_markers_kernel(K7Params p) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, i = t >> 2, s = t & 3u, lane = threadIdx.x & 31u;
    bool live = i < p.n && !(p.n_dev && i >= *p.n_dev);
    uint32_t rot = 0;
    if (live && p.decodes) {
        const a3_decode &dc = p.decodes[i];
        live = dc.accepted != 0;
        rot = dc.rotation & 3u;
    }
    bool good = false;
    float u = 0.0f, v = 0.0f;
    if (live) {
        float px, py;
        if (p.corners_f32) {  // marker order: screen corner s is marker corner (s - rotation) & 3
            const uint32_t c = (s + 4u - rot) & 3u;
            px = p.corners_f32[(size_t)i * 8 + 2 * c];
            py = p.corners_f32[(size_t)i * 8 + 2 * c + 1];
        } else {
            px = (float)p.quads[(size_t)i * 8 + 2 * s];
            py = (float)p.quads[(size_t)i * 8 + 2 * s + 1];
        }
        good = undistort(px, py, p.k, p.dist, u, v);
    }
    const uint32_t grp = (__ballot_sync(kFull, good) >> (lane & ~3u)) & 0xfu;
    if (!live) return;
    p.out[(size_t)i * 8 + 2 * s] = u;
    p.out[(size_t)i * 8 + 2 * s + 1] = v;
    if (s == 0) p.ok[i] = grp == 0xfu ? 1 : 0;
}

__global__ void __launch_bounds__(128) k7_points_kernel(const float *pts, uint32_t n, a3_camera_intrinsics k, a3_camera_distortion dist,
                                                        float *out, uint8_t *ok) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float u = 0.0f, v = 0.0f;
    const bool good = undistort(pts[2 * (size_t)i], pts[2 * (size_t)i + 1], k, dist, u, v);
    out[2 * (size_t)i] = good ? u : 0.0f;  // a failed point reads (0, 0)
    out[2 * (size_t)i + 1] = good ? v : 0.0f;
    ok[i] = good ? 1 : 0;
}

}  // namespace

cudaError_t k7_undistort(const K7Params &p, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    const size_t threads = (size_t)p.n * 4;
    k7_markers_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t k7_undistort_points(const float *pts, uint32_t n, const a3_camera_intrinsics &k, const a3_camera_distortion &dist, float *out,
                                uint8_t *ok, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    k7_points_kernel<<<(n + 127) / 128, 128, 0, stream>>>(pts, n, k, dist, out, ok);
    return cudaGetLastError();
}

}  // namespace a3
