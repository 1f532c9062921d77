// gyro.cuh -- gyro-predicted initial flow for LK: where a point of the previous frame lands in the next one when the
// camera only rotates by the gyro increment omega * dt. Rotational image motion does not depend on depth, and on a drone
// it is the large part of the motion between two frames; LK starts from the prediction (OFB_LK_USE_INITIAL_FLOW).
#pragma once
#include <math.h>
#include "camera.cuh"

// Pixel <-> normalised model of a prediction: the calibrated camera when cam != NULL (ofb_undistort / ofb_project, dt =
// 1 / rate), else the pair configuration's pinhole x = (p - c) * ps with dt = ps / fs (u = dp * fs, so that omega is
// per unit of the flow's time, as the solve reads it).
struct GyroPinhole { double cx, cy, ps, dt; };

// Guess for the pixel (px, py) under the rotation R = exp([omega * dt]x), fp64: X = (x, y, 1), X' = R X, x' = X'_xy / X'_z,
// back to pixels. To first order X' - X = dt (omega x X), the rotational flow the solve subtracts. Falls back to the
// point itself when X'_z <= 0 or anything is not finite (the IMU sample is device data, not validated on the host), and
// when omega = 0 (project(undistort(p)) is p only to the convergence of the inverse lens model).
__device__ __forceinline__ float2 ofb_gyro_predict_point(const GyroPinhole& ph, const ofb_camera* cam, double wx, double wy,
                                                         double wz, float px, float py)
{
    if (wx == 0.0 && wy == 0.0 && wz == 0.0) return make_float2(px, py);
    double x, y, dt;
    if (cam) { ofb_undistort(*cam, (double)px, (double)py, x, y); dt = 1.0 / cam->rate; }
    else { x = ((double)px - ph.cx) * ph.ps; y = ((double)py - ph.cy) * ph.ps; dt = ph.dt; }
    const double rx = wx * dt, ry = wy * dt, rz = wz * dt;
    const double t2 = rx * rx + ry * ry + rz * rz;
    // Rodrigues: R X = X + a (r x X) + b r x (r x X), a = sin(t) / t, b = (1 - cos(t)) / t^2 = 2 sin^2(t/2) / t^2; the
    // series below t^2 = 1e-4 are exact to the last bit of fp64 there (first omitted terms t^6 / 5040, t^6 / 40320)
    double a, b;
    if (t2 < 1e-4) {
        a = 1.0 - t2 * (1.0 / 6.0 - t2 * (1.0 / 120.0));
        b = 0.5 - t2 * (1.0 / 24.0 - t2 * (1.0 / 720.0));
    } else {
        const double t = sqrt(t2), s = sin(0.5 * t);
        a = sin(t) / t;
        b = 2.0 * s * s / t2;
    }
    const double c0 = ry - rz * y, c1 = rz * x - rx, c2 = rx * y - ry * x;            // r x X
    const double d0 = ry * c2 - rz * c1, d1 = rz * c0 - rx * c2, d2 = rx * c1 - ry * c0; // r x (r x X)
    const double X = x + a * c0 + b * d0, Y = y + a * c1 + b * d1, Z = 1.0 + a * c2 + b * d2;
    if (!(Z > 0.0)) return make_float2(px, py);
    const double xn = X / Z, yn = Y / Z;
    double gx, gy;
    if (cam) ofb_project(*cam, xn, yn, gx, gy);
    else { gx = ph.cx + xn / ph.ps; gy = ph.cy + yn / ph.ps; }
    const float fx = (float)gx, fy = (float)gy;
    if (!(isfinite(fx) && isfinite(fy))) return make_float2(px, py);
    return make_float2(fx, fy);
}

// Launches the prediction kernel: one thread per point, guess[pair][i] for i < counts[pair * counts_stride] (counts NULL:
// n_uniform points per pair), omega of pair p at w[p * w_stride] (three doubles). cam: device pointer or NULL (pinhole).
int ofb_gyro_predict_device(ofb_ctx* ctx, const GyroPinhole& ph, const ofb_camera* cam, const double* w, int w_stride,
                            int n_pairs, const float* pts, const int* counts, int counts_stride, int n_uniform,
                            size_t pts_stride, float* guess);

// The pinhole model of a pair configuration, or OFB_E_INVALID when its dt = pos_scale / flow_scale is not a finite number
static inline int ofb_gyro_pinhole(const ofb_pair_cfg* cfg, const char* who, GyroPinhole* ph)
{
    OFB_REQUIRE(cfg->flow_scale != 0.0, "%s: gyro prediction with the pinhole needs flow_scale != 0", who);
    const double dt = cfg->pos_scale / cfg->flow_scale;
    OFB_REQUIRE(isfinite(dt) && isfinite(cfg->cx) && isfinite(cfg->cy) && cfg->pos_scale != 0.0,
                "%s: gyro prediction needs finite cx, cy and a finite, non-zero pos_scale / flow_scale", who);
    *ph = GyroPinhole{cfg->cx, cfg->cy, cfg->pos_scale, dt};
    return OFB_OK;
}
