// camera.cu -- cv2.undistortPoints / cv2.undistortPointsIter (COUNT criterion) on the device: one thread per point,
// the lens model of camera.cuh, then OpenCV's rectification / projection H = P[:, :3] @ R.
#include "camera.cuh"

namespace {

struct Homography { double h[9]; int identity; };

__global__ void __launch_bounds__(256)
undistort_points_kernel(ofb_camera cam, Homography H, const double2* pts, int n, double2* out)   // out may alias pts
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2 p = pts[i];
    double x, y;
    ofb_undistort(cam, p.x, p.y, x, y);
    if (!H.identity) {
        const double xx = ofb_add(ofb_add(ofb_mul(H.h[0], x), ofb_mul(H.h[1], y)), H.h[2]);
        const double yy = ofb_add(ofb_add(ofb_mul(H.h[3], x), ofb_mul(H.h[4], y)), H.h[5]);
        const double ww = 1. / ofb_add(ofb_add(ofb_mul(H.h[6], x), ofb_mul(H.h[7], y)), H.h[8]);
        x = ofb_mul(xx, ww); y = ofb_mul(yy, ww);
    }
    out[i] = make_double2(x, y);
}

}  // namespace

extern "C" int ofb_undistort_points(ofb_ctx* ctx, const ofb_camera* cam, const double* pts, int n, const double* H, double* out)
{
    OFB_REQUIRE(ctx, "undistort_points: null context");
    OFB_TRY(ofb_camera_check(cam, "undistort_points"));
    OFB_REQUIRE(n >= 0, "undistort_points: n must be >= 0");
    OFB_REQUIRE(n == 0 || (pts && out), "undistort_points: null point array");
    Homography hm;
    hm.identity = H ? 0 : 1;
    for (int k = 0; k < 9; ++k) {
        hm.h[k] = H ? H[k] : (k % 4 == 0 ? 1.0 : 0.0);
        OFB_REQUIRE(isfinite(hm.h[k]), "undistort_points: non-finite entry in H");
    }
    if (n == 0) return OFB_OK;
    OFB_CUDA(cudaSetDevice(ctx->device));
    const size_t bytes = sizeof(double) * 2 * (size_t)n;
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, out, bytes, &o));
    const void* dpts;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, pts, bytes, &dpts));
    undistort_points_kernel<<<ofb_div_up(n, 256), 256, 0, ctx->stream>>>(*cam, hm, (const double2*)dpts, n, (double2*)o.dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, &o, 1);
}
