// pairs.cu -- fused frame-pair path: pyramid -> Shi-Tomasi -> pyramidal LK -> velocity solve for a
// batch of independent frame pairs (or of consecutive frames of one stream), with no host round-trip
// between stages (feature counts stay on the device). Work is ordered on the context's stream; inside a
// call it fans out to helper streams and joins back before the call's results are read:
//   * aux streams: the pyramid kernels run beside the one-CTA-per-image selection kernel;
//   * twin context (own stream + scratch): every other chunk of a batch, so the selection/pyramid phase of
//     one chunk hides behind the lambda_min kernel of the next;
//   * copy stream: host frames are uploaded in sub-batches while the previous sub-batch computes.
//
// Replaces the per-frame dataflow of velocity_measurment_node:224-267 (centre with of.pix_trans,
// scale by `scaling`, solve_lgs) and flight_experiments/evaluate_exp.py:77-120
// (calcOpticalFlowPyrLK -> status filter -> solve_lgs(new_pos, new_pos-old_pos, ...)).
#include "common.cuh"
#include "features.cuh"
#include "pyrlk.cuh"
#include "velocity_device.cuh"
#include "camera.cuh"
#include "gyro.cuh"
#include <stddef.h>
#include <type_traits>

namespace {

// One CTA per pair: the velocity solve; with EGO the ego-motion solve and with ROBUST the robust velocity solve of the pair
// follow on the same points (ego[f], rob[f]). CALIB: every tracked point is undistorted once into ld.xu first.
template <bool EGO, bool ROBUST, bool CALIB>
__global__ void __launch_bounds__(OFB_SOLVE_THREADS)
pair_solve_kernel(TrackLoader<CALIB> ld, ofb_camera cam, int variant, const ofb_imu_sample* __restrict__ imu,
                  ofb_pair_result* __restrict__ out, const FeatImageState* __restrict__ det, ofb_ego_result* __restrict__ ego,
                  ofb_robust_cfg rcfg, ofb_robust_result* __restrict__ rob)
{
    const int f = blockIdx.x;
    if (CALIB) {
        const int n = ld.end(f);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const size_t o = (size_t)f * ld.stride + i;
            if (ld.status[o]) ld.xu[o] = ofb_calibrate(cam, ld.next[2 * o], ld.next[2 * o + 1], ld.prev[2 * o], ld.prev[2 * o + 1]);
        }
        __syncthreads();
    }
    const ofb_imu_sample& s = imu[f];
    const OfbSolveOut o = ofb_block_solve(ld, f, variant, s.d, s.n, s.w, s.t);
    if (threadIdx.x == 0) {
        ofb_pair_result r;
        for (int k = 0; k < 3; ++k) { r.v[k] = o.v[k]; r.s[k] = o.s[k]; }
        r.res = o.res; r.rank = o.rank;
        r.n_features = ld.end(f);
        r.n_tracked = o.count;
        r.flags = (det && det[f].overflow) ? OFB_PAIR_OVERFLOW : 0;     // detector ran out of candidate slots
        out[f] = r;
    }
    if (EGO) {
        const OfbEgoOut e = ofb_block_solve_ego(ld, f, variant, s.d, s.n, s.t);
        if (threadIdx.x == 0) ego[f] = ofb_ego_record(e, OFB_EGO_SOLVED);
    }
    if (ROBUST) {
        const OfbRobustOut r = ofb_block_solve_robust(ld, f, variant, s.d, s.n, s.w, s.t, rcfg.c, rcfg.iterations);
        if (threadIdx.x == 0) rob[f] = ofb_robust_record(r, OFB_ROBUST_SOLVED);
    }
}

}  // namespace

// Stages 1b-4 for pairs [c0, c0+n) whose level-0 frames already sit in pp/pn (images 0..n-1 of each).
// gyro (NULL: off): the pinhole model of the gyro prediction, with dcam the device copy of the camera (NULL: pinhole).
// d_ego (NULL: off): the pairs' ego-motion records, solved in the velocity solve's kernel; d_rob (NULL: off) likewise
// the robust records under rcfg.
// Sequence layout (pn == pp): pp holds n+1 consecutive frames of one stream, pair i = (image i, image i+1), so every
// interior frame's pyramid is built once and serves as "next" of one pair and "prev" of the following one.
static int run_pairs_chunk(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, double fb_max_err,
                           const GyroPinhole* gyro, const ofb_camera* dcam, ofb_pyr* pp, ofb_pyr* pn, int n, int c0,
                           const ofb_imu_sample* dimu, const int* counts_in, float* d_prev, float* d_next, uint8_t* d_stat,
                           ofb_pair_result* d_res, ofb_ego_result* d_ego, const ofb_robust_cfg& rcfg, ofb_robust_result* d_rob,
                           bool mark)
{
    const bool seq = pn == pp;
    const int w = cfg->width, h = cfg->height, K = cfg->max_corners;
#define STAGE_MARK(i) do { if (mark) OFB_CUDA(cudaEventRecord(ctx->stage_ev[i], ctx->stream)); } while (0)
    // Detection only needs level 0, and the selection kernel keeps just one SM per image busy: unless stage
    // timing is on, the pyramids are built on aux_stream while the selection runs (fork after lambda_min).
    const bool overlap = cfg->detect && !mark;
    if (overlap && !ctx->aux_stream) {
        OFB_CUDA(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
        OFB_CUDA(cudaStreamCreateWithFlags(&ctx->aux2_stream, cudaStreamNonBlocking));
        OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
        OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_join2, cudaEventDisableTiming));
    }
    STAGE_MARK(0);
    if (!overlap) {
        OFB_TRY(ofb_pyr_build_device(ctx, pp));
        if (!seq) OFB_TRY(ofb_pyr_build_device(ctx, pn));
    }
    STAGE_MARK(1);
    float* cp = d_prev + (size_t)c0 * 2 * K;
    float* cn = d_next + (size_t)c0 * 2 * K;
    uint8_t* cs = d_stat + (size_t)c0 * K;
    const int* counts; int counts_stride;
    FeatImageState* st = nullptr;
    if (cfg->detect) {
        unsigned int cand_cap = (unsigned int)(((size_t)w * h) / 4 + 1024);
        ctx->fork_after_eig = overlap;
        int fr = ofb_features_device(ctx, pp->level0, w, h, pp->level0_pitch, pp->level0_stride, n, nullptr, 0, 0, K,
                                     cfg->quality, cfg->min_distance, cfg->block_size, cand_cap, cp, (size_t)2 * K, K, &st);
        ctx->fork_after_eig = false;
        OFB_TRY(fr);
        counts = &st->n_out; counts_stride = (int)(sizeof(FeatImageState) / sizeof(int));
        if (overlap) {
            // aux streams: wait for the lambda_min kernel, build the two pyramids beside the selection kernel (one
            // stream each: the small upper levels are latency-bound launches and overlap)
            OFB_CUDA(cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_fork, 0));
            OFB_CUDA(cudaStreamWaitEvent(ctx->aux2_stream, ctx->ev_fork, 0));
            cudaStream_t main_stream = ctx->stream;
            ctx->stream = ctx->aux_stream;
            int pr = ofb_pyr_build_device(ctx, pp);
            ctx->stream = ctx->aux2_stream;
            if (pr == OFB_OK && !seq) pr = ofb_pyr_build_device(ctx, pn);
            ctx->stream = main_stream;
            OFB_TRY(pr);
            OFB_CUDA(cudaEventRecord(ctx->ev_join, ctx->aux_stream));
            OFB_CUDA(cudaEventRecord(ctx->ev_join2, ctx->aux2_stream));
            OFB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
            OFB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join2, 0));
        }
    } else {
        if (mark) OFB_CUDA(cudaEventRecord(ctx->stage_ev[2], ctx->stream));
        counts = counts_in + c0; counts_stride = 1;
    }
    STAGE_MARK(3);
    OFB_TRY(ctx->scratch[SC_ERR].reserve(sizeof(float) * (size_t)n * K));
    int lk_flags = 0;
    if (gyro) {
        // LK starts from the rotation the gyro measured: the guesses go where LK writes its result
        OFB_TRY(ofb_gyro_predict_device(ctx, *gyro, dcam, (const double*)((const char*)(dimu + c0) + offsetof(ofb_imu_sample, w)),
                                        (int)(sizeof(ofb_imu_sample) / sizeof(double)), n, cp, counts, counts_stride, K,
                                        (size_t)K, cn));
        lk_flags = OFB_LK_USE_INITIAL_FLOW | OFB_LK_FB_INITIAL_FLOW;
    }
    OFB_TRY(ofb_lk_device(ctx, pp, 0, 1, pn, seq ? 1 : 0, 1, n, cp, counts, counts_stride, K, (size_t)K, cfg->win_w, cfg->win_h,
                          cfg->max_level, cfg->max_count, cfg->eps, lk_flags, cfg->min_eig_thr, cn, cs,
                          ctx->scratch[SC_ERR].as<float>(), fb_max_err));
    STAGE_MARK(4);
    double4* xu = nullptr;
    if (cam) {
        OFB_TRY(ctx->scratch[SC_CALIB].reserve(sizeof(double4) * (size_t)n * K));
        xu = ctx->scratch[SC_CALIB].as<double4>();
    }
    auto launch = [&](auto calib) {
        constexpr bool C = decltype(calib)::value;
        const TrackLoader<C> ld{cp, cn, cs, counts, counts_stride, 0, (size_t)K, cfg->cx, cfg->cy, cfg->pos_scale, cfg->flow_scale, xu};
        auto kern = d_ego ? (d_rob ? pair_solve_kernel<true, true, C> : pair_solve_kernel<true, false, C>)
                          : (d_rob ? pair_solve_kernel<false, true, C> : pair_solve_kernel<false, false, C>);
        kern<<<n, OFB_SOLVE_THREADS, 0, ctx->stream>>>(ld, cam ? *cam : ofb_camera{}, cfg->variant, dimu + c0, d_res + c0, st,
                                                       d_ego ? d_ego + c0 : nullptr, rcfg, d_rob ? d_rob + c0 : nullptr);
    };
    if (cam) launch(std::true_type{});
    else launch(std::false_type{});
    OFB_LAUNCH_CHECK(ctx);
    STAGE_MARK(5);
#undef STAGE_MARK
    return OFB_OK;
}

extern "C" int ofb_frame_pairs(ofb_ctx* ctx, const ofb_pair_cfg* cfg, int n_pairs,
                               const uint8_t* prev, const uint8_t* next, int pitch, size_t image_stride,
                               const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                               ofb_pair_result* results, float* prev_pts, float* next_pts, uint8_t* status)
{
    return ofb_frame_pairs_cam(ctx, cfg, nullptr, n_pairs, prev, next, pitch, image_stride, imu, pts_in, n_in, results, prev_pts,
                               next_pts, status);
}

extern "C" int ofb_frame_pairs_cam(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, int n_pairs,
                                   const uint8_t* prev, const uint8_t* next, int pitch, size_t image_stride,
                                   const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                                   ofb_pair_result* results, float* prev_pts, float* next_pts, uint8_t* status)
{
    return ofb_frame_pairs_fb(ctx, cfg, cam, 0.0, n_pairs, prev, next, pitch, image_stride, imu, pts_in, n_in, results, prev_pts,
                              next_pts, status);
}

extern "C" int ofb_frame_pairs_fb(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, double fb_max_err, int n_pairs,
                                  const uint8_t* prev, const uint8_t* next, int pitch, size_t image_stride,
                                  const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                                  ofb_pair_result* results, float* prev_pts, float* next_pts, uint8_t* status)
{
    return ofb_frame_pairs_gyro(ctx, cfg, cam, fb_max_err, 0, n_pairs, prev, next, pitch, image_stride, imu, pts_in, n_in, results,
                                prev_pts, next_pts, status);
}

extern "C" int ofb_frame_pairs_gyro(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, double fb_max_err,
                                    int gyro_predict, int n_pairs, const uint8_t* prev, const uint8_t* next, int pitch,
                                    size_t image_stride, const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                                    ofb_pair_result* results, float* prev_pts, float* next_pts, uint8_t* status)
{
    return ofb_frame_pairs_ego(ctx, cfg, cam, fb_max_err, gyro_predict, n_pairs, prev, next, pitch, image_stride, imu, pts_in, n_in,
                               results, nullptr, prev_pts, next_pts, status);
}

extern "C" int ofb_frame_pairs_ego(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, double fb_max_err,
                                   int gyro_predict, int n_pairs, const uint8_t* prev, const uint8_t* next, int pitch,
                                   size_t image_stride, const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                                   ofb_pair_result* results, ofb_ego_result* ego, float* prev_pts, float* next_pts,
                                   uint8_t* status)
{
    return ofb_frame_pairs_robust(ctx, cfg, cam, fb_max_err, gyro_predict, n_pairs, prev, next, pitch, image_stride, imu, pts_in,
                                  n_in, results, ego, nullptr, nullptr, prev_pts, next_pts, status);
}

extern "C" int ofb_frame_pairs_robust(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, double fb_max_err,
                                      int gyro_predict, int n_pairs, const uint8_t* prev, const uint8_t* next, int pitch,
                                      size_t image_stride, const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                                      ofb_pair_result* results, ofb_ego_result* ego, const ofb_robust_cfg* robust,
                                      ofb_robust_result* rob, float* prev_pts, float* next_pts, uint8_t* status)
{
    OFB_REQUIRE(ctx && cfg && prev && next && imu && results, "frame_pairs: null argument");
    ofb_robust_cfg rcfg{0.0, 0};
    if (rob) {
        OFB_REQUIRE(cfg->variant >= 0 && cfg->variant <= 2, "frame_pairs: unknown variant");
        OFB_TRY(ofb_robust_check(robust, "frame_pairs"));
        rcfg = *robust;
    }
    if (cam) OFB_TRY(ofb_camera_check(cam, "frame_pairs"));
    OFB_REQUIRE(ofb_fb_thr_ok(fb_max_err), "frame_pairs: fb_max_err must be >= 0 (0 = no forward-backward check)");
    GyroPinhole gph{0.0, 0.0, 0.0, 0.0};
    if (gyro_predict && !cam) OFB_TRY(ofb_gyro_pinhole(cfg, "frame_pairs", &gph));
    OFB_REQUIRE(n_pairs > 0 && n_pairs <= 65535, "frame_pairs: n_pairs must be in 1..65535");
    const int w = cfg->width, h = cfg->height, K = cfg->max_corners;
    OFB_REQUIRE(w > 0 && h > 0 && pitch >= w, "frame_pairs: bad image geometry");
    OFB_REQUIRE(K > 0, "frame_pairs: max_corners must be positive");
    OFB_REQUIRE(cfg->max_level >= 0, "frame_pairs: max_level must be >= 0");
    OFB_REQUIRE(cfg->variant >= 0 && cfg->variant <= 2, "frame_pairs: unknown variant");
    OFB_REQUIRE(cfg->detect || (pts_in && n_in), "frame_pairs: detect==0 needs pts_in and n_in");
    OFB_REQUIRE(n_pairs == 1 || image_stride >= (size_t)pitch * (h - 1) + w, "frame_pairs: image_stride too small");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const size_t npts = (size_t)n_pairs * K;
    OutStage o[6];
    OFB_TRY(ofb_stage_out(ctx, SC_PTS0, prev_pts, sizeof(float) * 2 * npts, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_PTS1, next_pts, sizeof(float) * 2 * npts, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_STAT, status, npts, &o[2]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT3, results, sizeof(ofb_pair_result) * n_pairs, &o[3]));
    OFB_TRY(ofb_stage_out(ctx, SC_EGO, ego, sizeof(ofb_ego_result) * n_pairs, &o[4]));
    OFB_TRY(ofb_stage_out(ctx, SC_ROBUST, rob, sizeof(ofb_robust_result) * n_pairs, &o[5]));
    // optional outputs still need device storage when the caller passes NULL
    float* d_prev = (float*)o[0].dev; float* d_next = (float*)o[1].dev; uint8_t* d_stat = (uint8_t*)o[2].dev;
    if (!d_prev) { OFB_TRY(ctx->scratch[SC_PTS0].reserve(sizeof(float) * 2 * npts)); d_prev = ctx->scratch[SC_PTS0].as<float>(); }
    if (!d_next) { OFB_TRY(ctx->scratch[SC_PTS1].reserve(sizeof(float) * 2 * npts)); d_next = ctx->scratch[SC_PTS1].as<float>(); }
    if (!d_stat) { OFB_TRY(ctx->scratch[SC_STAT].reserve(npts)); d_stat = ctx->scratch[SC_STAT].as<uint8_t>(); }
    const void* dimu;
    OFB_TRY(ofb_stage_in(ctx, SC_IN3, imu, sizeof(ofb_imu_sample) * n_pairs, &dimu));
    const void* dcam = nullptr;                     // the prediction kernel reads the camera from device memory
    if (gyro_predict && cam) OFB_TRY(ofb_stage_in(ctx, SC_IN5, cam, sizeof(ofb_camera), &dcam));
    const int* counts_in = nullptr;
    if (!cfg->detect) {
        const void* dn;
        OFB_TRY(ofb_stage_in(ctx, SC_IN4, n_in, sizeof(int) * n_pairs, &dn));
        counts_in = (const int*)dn;
        if ((const float*)pts_in != d_prev)
            OFB_CUDA(cudaMemcpyAsync(d_prev, pts_in, sizeof(float) * 2 * npts, cudaMemcpyDefault, ctx->stream));
    }
    const bool dev_prev = ofb_is_device_ptr(prev), dev_next = ofb_is_device_ptr(next);
    // consecutive frames of one stream in one buffer: each frame is uploaded and its pyramid built once per chunk
    const bool seq = next == prev + image_stride && n_pairs > 1;
    const int extra = seq ? 1 : 0;                  // a chunk of n pairs holds n + extra prev frames
    // Chunk schedule. Chunks of at most `cap` pairs (the capacity of their pyramids) alternate between this context and a
    // twin context with its own stream and scratch, so the lambda_min kernel (shared-memory heavy, issue bound) of one
    // chunk and the selection and LK kernels of the other are co-resident on the SMs instead of running back to back.
    //   * host frames (staged): the frames of the whole call are staged in one device buffer by back-to-back H2D copies on
    //     a copy stream (the PCIe copy is the bound: nothing else is ever queued between two copies); a chunk of 8 pairs
    //     starts as soon as its frames have landed, with level 0 aliasing the staging buffer (in the sequence layout a
    //     frame shared by two chunks is simply read by both). The last chunks are smaller (8, ..., 8, 4, 2, 2): what
    //     remains after the last copy is one short chain.
    //   * device frames: two halves of the batch, level 0 is the caller's buffer.
    //   * otherwise (a small batch, mixed host / device frames, stage timing): one pass over the whole batch.
    const bool staged = !dev_prev && !dev_next && n_pairs > 8 && !ctx->profile;
    int cap = n_pairs;
    if (staged) cap = 8;
    else if (dev_prev && dev_next && n_pairs >= 2 && !ctx->profile) cap = (n_pairs + 1) / 2;
    const bool use_twin = n_pairs > cap;
    if (use_twin && !ctx->twin) {
        OFB_TRY(ofb_ctx_create(ctx->device, &ctx->twin));
        OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_twin_fork, cudaEventDisableTiming));
        OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_twin_join, cudaEventDisableTiming));
    }
    // level 0 of the chunk pyramids: prev frame i at fprev + i * fstride, next frame i at fnext + i * fstride
    const uint8_t* fprev = prev; const uint8_t* fnext = next;
    int fpitch = pitch; size_t fstride = image_stride;
    uint8_t* frames = nullptr;                      // staging buffer: the prev frames, then (unless seq) the next frames
    if (staged) {
        if (!ctx->copy_stream) OFB_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        if (!ctx->ev_free[0]) OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_free[0], cudaEventDisableTiming));
        fpitch = (w + 15) & ~15;
        fstride = (((size_t)fpitch * h) + 255) & ~(size_t)255;
        OFB_TRY(ctx->scratch[SC_FRAMES].reserve(fstride * (seq ? (size_t)n_pairs + 1 : 2 * (size_t)n_pairs) + 256));
        frames = ctx->scratch[SC_FRAMES].as<uint8_t>();
        fprev = frames;
        fnext = frames + fstride * (seq ? 1 : (size_t)n_pairs);
        // the staging buffer may still be read by work enqueued earlier (a previous call with device-side outputs)
        OFB_CUDA(cudaEventRecord(ctx->ev_free[0], ctx->stream));
        OFB_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_free[0], 0));
    }
    auto upload = [&](uint8_t* dst, const uint8_t* src, int count) -> int {
        if (count <= 0) return OFB_OK;
        if (pitch == fpitch && image_stride == fstride) {            // same layout on both sides: one copy
            OFB_CUDA(cudaMemcpyAsync(dst, src, fstride * (size_t)(count - 1) + (size_t)pitch * (h - 1) + w,
                                     cudaMemcpyHostToDevice, ctx->copy_stream));
            return OFB_OK;
        }
        for (int i = 0; i < count; ++i)
            OFB_CUDA(cudaMemcpy2DAsync(dst + (size_t)i * fstride, fpitch, src + (size_t)i * image_stride, pitch, w, h,
                                       cudaMemcpyHostToDevice, ctx->copy_stream));
        return OFB_OK;
    };
    ofb_ctx* tw = ctx->twin;
    uint64_t tw0 = 0;
    if (use_twin) {
        // staged inputs (IMU samples, seed points) were enqueued on this context's stream
        OFB_CUDA(cudaEventRecord(ctx->ev_twin_fork, ctx->stream));
        OFB_CUDA(cudaStreamWaitEvent(tw->stream, ctx->ev_twin_fork, 0));
        tw0 = tw->launches;
    }
    for (int c0 = 0, ci = 0, n = 0; c0 < n_pairs; c0 += n, ++ci) {
        const int left = n_pairs - c0;
        n = !staged ? (left < cap ? left : cap) : left > 12 ? 8 : left > 4 ? 4 : left > 2 ? 2 : left;
        ofb_ctx* c = (ci & 1) ? tw : ctx;
        const int slot = (ci >> 1) & 1;
        if (staged) {
            if (seq) {
                // frames c0 .. c0+n; frame c0 came with the previous chunk
                const int f0 = ci == 0 ? 0 : c0 + 1;
                OFB_TRY(upload(frames + (size_t)f0 * fstride, prev + (size_t)f0 * image_stride, c0 + n + 1 - f0));
            } else {
                OFB_TRY(upload(frames + (size_t)c0 * fstride, prev + (size_t)c0 * image_stride, n));
                OFB_TRY(upload(frames + ((size_t)n_pairs + c0) * fstride, next + (size_t)c0 * image_stride, n));
            }
            if ((int)ctx->ev_piece.size() <= ci) {
                cudaEvent_t e;
                OFB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                ctx->ev_piece.push_back(e);
            }
            OFB_CUDA(cudaEventRecord(ctx->ev_piece[ci], ctx->copy_stream));
            OFB_CUDA(cudaStreamWaitEvent(c->stream, ctx->ev_piece[ci], 0));
        }
        // (c, slot) is reused every fourth chunk, on the same stream: stream order protects its upper levels
        OFB_TRY(ofb_pyr_prepare(c, &c->pair_pyr[slot][0], fprev + (size_t)c0 * fstride, w, h, fpitch, fstride, n + extra,
                                cap + extra, cfg->max_level, false));
        if (!seq)
            OFB_TRY(ofb_pyr_prepare(c, &c->pair_pyr[slot][1], fnext + (size_t)c0 * fstride, w, h, fpitch, fstride, n, cap,
                                    cfg->max_level, false));
        OFB_TRY(run_pairs_chunk(c, cfg, cam, fb_max_err, gyro_predict ? &gph : nullptr, (const ofb_camera*)dcam,
                                c->pair_pyr[slot][0], seq ? c->pair_pyr[slot][0] : c->pair_pyr[slot][1], n, c0,
                                (const ofb_imu_sample*)dimu, counts_in, d_prev, d_next, d_stat, (ofb_pair_result*)o[3].dev,
                                (ofb_ego_result*)o[4].dev, rcfg, (ofb_robust_result*)o[5].dev, ctx->profile));
    }
    if (use_twin) {
        ctx->launches += tw->launches - tw0;
        OFB_CUDA(cudaEventRecord(ctx->ev_twin_join, tw->stream));
        OFB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_twin_join, 0));
    }
    int rc = ofb_finish_out(ctx, o, 6);
    if (rc == OFB_OK && ctx->profile) {
        // stage order: 0 pyramids, 1 lambda_min+NMS, 2 ordered selection, 3 LK, 4 solve
        OFB_CUDA(cudaEventSynchronize(ctx->stage_ev[5]));
        for (int i = 0; i < OFB_NSTAGES; ++i) {
            float ms = 0.f;
            OFB_CUDA(cudaEventElapsedTime(&ms, ctx->stage_ev[i], ctx->stage_ev[i + 1]));
            ctx->stage_ms[i] += ms;
        }
        ctx->stage_calls++;
    }
    return rc;
}
