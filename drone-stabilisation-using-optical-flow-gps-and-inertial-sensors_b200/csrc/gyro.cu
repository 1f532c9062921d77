// gyro.cu -- the gyro prediction of gyro.cuh as a kernel of its own (one thread per point, fp64, fp32 guesses into the
// next-points buffer LK then reads with OFB_LK_USE_INITIAL_FLOW), and the standalone ofb_gyro_predict.
#include "gyro.cuh"

namespace {

__global__ void __launch_bounds__(256)
gyro_predict_kernel(GyroPinhole ph, const ofb_camera* __restrict__ cam, const double* __restrict__ w, int w_stride,
                    const float* __restrict__ pts, const int* __restrict__ counts, int counts_stride, int n_uniform,
                    size_t pts_stride, float* __restrict__ guess)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x, pair = blockIdx.y;
    const int n = counts ? counts[(size_t)pair * counts_stride] : n_uniform;
    if (i >= n) return;
    OFB_DEV_ASSERT(i < n_uniform);
    const size_t o = (size_t)pair * pts_stride + i;
    const double* wp = w + (size_t)pair * w_stride;
    const float2 g = ofb_gyro_predict_point(ph, cam, wp[0], wp[1], wp[2], pts[2 * o], pts[2 * o + 1]);
    guess[2 * o] = g.x; guess[2 * o + 1] = g.y;
}

}  // namespace

int ofb_gyro_predict_device(ofb_ctx* ctx, const GyroPinhole& ph, const ofb_camera* cam, const double* w, int w_stride,
                            int n_pairs, const float* pts, const int* counts, int counts_stride, int n_uniform,
                            size_t pts_stride, float* guess)
{
    if (n_uniform <= 0 || n_pairs <= 0) return OFB_OK;
    dim3 grid(ofb_div_up(n_uniform, 256), n_pairs);
    gyro_predict_kernel<<<grid, 256, 0, ctx->stream>>>(ph, cam, w, w_stride, pts, counts, counts_stride, n_uniform, pts_stride,
                                                       guess);
    OFB_LAUNCH_CHECK(ctx);
    return OFB_OK;
}

extern "C" int ofb_gyro_predict(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, const float* pts, int n,
                                const double* w3, float* guess_out)
{
    OFB_REQUIRE(ctx && (cfg || cam), "gyro_predict: null context, or neither cfg nor camera");
    OFB_REQUIRE(w3, "gyro_predict: null w3");
    OFB_REQUIRE(n >= 0, "gyro_predict: n must be >= 0");
    OFB_REQUIRE(n == 0 || (pts && guess_out), "gyro_predict: null point array");
    GyroPinhole ph{0.0, 0.0, 0.0, 0.0};
    if (cam) OFB_TRY(ofb_camera_check(cam, "gyro_predict"));
    else OFB_TRY(ofb_gyro_pinhole(cfg, "gyro_predict", &ph));
    if (n == 0) return OFB_OK;
    OFB_CUDA(cudaSetDevice(ctx->device));
    const size_t bytes = sizeof(float) * 2 * (size_t)n;
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, guess_out, bytes, &o));
    const void *dpts, *dw;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, pts, bytes, &dpts));
    OFB_TRY(ofb_stage_in(ctx, SC_IN1, w3, sizeof(double) * 3, &dw));
    const ofb_camera* dcam = nullptr;
    if (cam) {
        const void* dc;
        OFB_TRY(ofb_stage_in(ctx, SC_IN2, cam, sizeof(ofb_camera), &dc));
        dcam = (const ofb_camera*)dc;
    }
    OFB_TRY(ofb_gyro_predict_device(ctx, ph, dcam, (const double*)dw, 0, 1, (const float*)dpts, nullptr, 0, n, 0,
                                    (float*)o.dev));
    return ofb_finish_out(ctx, &o, 1);
}
