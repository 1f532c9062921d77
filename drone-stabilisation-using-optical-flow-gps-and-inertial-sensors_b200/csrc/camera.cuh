// camera.cuh -- OpenCV's inverse lens model (cv2.undistortPoints), the one implementation every device path uses:
// the standalone ofb_undistort_points kernel, the frame-pair solve and the tracker's filter (r_tilde gate + solve).
#pragma once
#include <math.h>
#include "common.cuh"

// Rejects what OpenCV would not model: a camera matrix that is not positive, an unsupported coefficient count, a
// non-finite entry, an iteration count outside 1..1000, a rate <= 0. `who` prefixes the error message.
static inline int ofb_camera_check(const ofb_camera* c, const char* who)
{
    OFB_REQUIRE(c, "%s: null camera", who);
    OFB_REQUIRE(c->n_dist == 0 || c->n_dist == 4 || c->n_dist == 5 || c->n_dist == 8,
                "%s: n_dist must be 0, 4, 5 or 8 (got %d)", who, c->n_dist);
    OFB_REQUIRE(c->iterations >= 1 && c->iterations <= 1000, "%s: iterations must be in 1..1000 (got %d)", who, c->iterations);
    bool finite = isfinite(c->fx) && isfinite(c->fy) && isfinite(c->cx) && isfinite(c->cy) && isfinite(c->rate);
    for (int k = 0; k < c->n_dist; ++k) finite = finite && isfinite(c->dist[k]);
    OFB_REQUIRE(finite, "%s: non-finite camera parameter", who);
    OFB_REQUIRE(c->fx > 0 && c->fy > 0, "%s: fx and fy must be positive", who);
    OFB_REQUIRE(c->rate > 0, "%s: rate must be positive", who);
    return OFB_OK;
}

// Pixel -> normalised image coordinates, cvUndistortPointsInternal's arithmetic in its operation order (the identity
// rectification is left to the caller). The explicitly rounded operations keep nvcc from contracting them into FMAs,
// so the result is OpenCV's to the last bit.
__device__ __forceinline__ double ofb_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ofb_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double ofb_sub(double a, double b) { return __dsub_rn(a, b); }

__device__ __forceinline__ void ofb_undistort(const ofb_camera& c, double px, double py, double& x, double& y)
{
    const double x0 = ofb_mul(ofb_sub(px, c.cx), 1.0 / c.fx), y0 = ofb_mul(ofb_sub(py, c.cy), 1.0 / c.fy);
    x = x0; y = y0;
    if (c.n_dist == 0) return;
    const double k1 = c.dist[0], k2 = c.dist[1], p1 = c.dist[2], p2 = c.dist[3];
    const double k3 = c.n_dist > 4 ? c.dist[4] : 0.0;
    const double k4 = c.n_dist > 5 ? c.dist[5] : 0.0, k5 = c.n_dist > 5 ? c.dist[6] : 0.0, k6 = c.n_dist > 5 ? c.dist[7] : 0.0;
    for (int j = 0; j < c.iterations; ++j) {
        const double r2 = ofb_add(ofb_mul(x, x), ofb_mul(y, y));
        // (1 + ((k6 r2 + k5) r2 + k4) r2) / (1 + ((k3 r2 + k2) r2 + k1) r2)
        const double icdist = ofb_add(1.0, ofb_mul(ofb_add(ofb_mul(ofb_add(ofb_mul(k6, r2), k5), r2), k4), r2)) /
                              ofb_add(1.0, ofb_mul(ofb_add(ofb_mul(ofb_add(ofb_mul(k3, r2), k2), r2), k1), r2));
        if (icdist < 0) { x = x0; y = y0; return; }
        // 2 p1 x y + p2 (r2 + 2 x x),  p1 (r2 + 2 y y) + 2 p2 x y
        const double dx = ofb_add(ofb_mul(ofb_mul(2.0 * p1, x), y), ofb_mul(p2, ofb_add(r2, ofb_mul(2.0 * x, x))));
        const double dy = ofb_add(ofb_mul(p1, ofb_add(r2, ofb_mul(2.0 * y, y))), ofb_mul(ofb_mul(2.0 * p2, x), y));
        x = ofb_mul(ofb_sub(x0, dx), icdist);
        y = ofb_mul(ofb_sub(y0, dy), icdist);
    }
}

// Normalised image coordinates -> pixel, OpenCV's forward lens model: cv2.projectPoints of the object point (x, y, 1)
// with zero rvec / tvec, in cvProjectPoints2Internal's operation order (the zero rotation, translation and tilt terms
// are exact identities there and are left out). The inverse of ofb_undistort where that converges.
__device__ __forceinline__ void ofb_project(const ofb_camera& c, double x, double y, double& px, double& py)
{
    const int nd = c.n_dist;
    const double k1 = nd ? c.dist[0] : 0.0, k2 = nd ? c.dist[1] : 0.0, p1 = nd ? c.dist[2] : 0.0, p2 = nd ? c.dist[3] : 0.0;
    const double k3 = nd > 4 ? c.dist[4] : 0.0;
    const double k4 = nd > 5 ? c.dist[5] : 0.0, k5 = nd > 5 ? c.dist[6] : 0.0, k6 = nd > 5 ? c.dist[7] : 0.0;
    const double r2 = ofb_add(ofb_mul(x, x), ofb_mul(y, y));
    const double r4 = ofb_mul(r2, r2), r6 = ofb_mul(r4, r2);
    const double a1 = ofb_mul(2.0 * x, y);
    const double a2 = ofb_add(r2, ofb_mul(2.0 * x, x)), a3 = ofb_add(r2, ofb_mul(2.0 * y, y));
    // cdist = 1 + k1 r2 + k2 r4 + k3 r6,  icdist2 = 1 / (1 + k4 r2 + k5 r4 + k6 r6)
    const double cdist = ofb_add(ofb_add(ofb_add(1.0, ofb_mul(k1, r2)), ofb_mul(k2, r4)), ofb_mul(k3, r6));
    const double icdist2 = 1.0 / ofb_add(ofb_add(ofb_add(1.0, ofb_mul(k4, r2)), ofb_mul(k5, r4)), ofb_mul(k6, r6));
    const double xd = ofb_add(ofb_add(ofb_mul(ofb_mul(x, cdist), icdist2), ofb_mul(p1, a1)), ofb_mul(p2, a2));
    const double yd = ofb_add(ofb_add(ofb_mul(ofb_mul(y, cdist), icdist2), ofb_mul(p1, a3)), ofb_mul(p2, a1));
    px = ofb_add(ofb_mul(xd, c.fx), c.cx);
    py = ofb_add(ofb_mul(yd, c.fy), c.cy);
}

// Calibrated position and flow of one track: x = undistort(p_new), u = (x - undistort(p_old)) * rate.
__device__ __forceinline__ double4 ofb_calibrate(const ofb_camera& c, float nx, float ny, float ox, float oy)
{
    double xn, yn, xo, yo;
    ofb_undistort(c, (double)nx, (double)ny, xn, yn);
    ofb_undistort(c, (double)ox, (double)oy, xo, yo);
    return make_double4(xn, yn, (xn - xo) * c.rate, (yn - yo) * c.rate);
}
