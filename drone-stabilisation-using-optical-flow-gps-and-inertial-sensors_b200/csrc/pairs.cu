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

namespace {

struct TrackLoader {
    const float* prev; const float* next; const uint8_t* status;
    const int* counts; int counts_stride; size_t stride;
    double cx, cy, ps, fs;
    __device__ int begin(int) const { return 0; }
    __device__ int end(int f) const { return counts[(size_t)f * counts_stride]; }
    __device__ bool load(int f, int i, double& px, double& py, double& ux, double& uy) const {
        size_t o = (size_t)f * stride + i;
        if (!status[o]) return false;                       // new_pos[status==1]  (node:134, evaluate_exp.py:99)
        float nx = next[2 * o], ny = next[2 * o + 1];
        float dx = nx - prev[2 * o], dy = ny - prev[2 * o + 1];   // flow formed in fp32 as cv2 arrays are (node:136)
        px = ((double)nx - cx) * ps; py = ((double)ny - cy) * ps;  // node:232-233
        ux = (double)dx * fs; uy = (double)dy * fs;                // node:235
        return true;
    }
    __device__ bool dist(int, int, double&) const { return false; }
};

template <class Loader>
__device__ __forceinline__ void pair_solve(const Loader& ld, int variant, const ofb_imu_sample* __restrict__ imu,
                                           ofb_pair_result* __restrict__ out, const FeatImageState* __restrict__ det)
{
    int f = blockIdx.x;
    const ofb_imu_sample& s = imu[f];
    OfbSolveOut o = ofb_block_solve(ld, f, variant, s.d, s.n, s.w, s.t);
    if (threadIdx.x == 0) {
        ofb_pair_result r;
        for (int k = 0; k < 3; ++k) { r.v[k] = o.v[k]; r.s[k] = o.s[k]; }
        r.res = o.res; r.rank = o.rank;
        r.n_features = ld.end(f);
        r.n_tracked = o.count;
        r.flags = (det && det[f].overflow) ? OFB_PAIR_OVERFLOW : 0;     // detector ran out of candidate slots
        out[f] = r;
    }
}

__global__ void __launch_bounds__(OFB_SOLVE_THREADS)
pair_solve_kernel(TrackLoader ld, int variant, const ofb_imu_sample* __restrict__ imu, ofb_pair_result* __restrict__ out,
                  const FeatImageState* __restrict__ det)
{
    pair_solve(ld, variant, imu, out, det);
}

// With a calibrated camera: every tracked point is undistorted once into xu (the solve reads each point twice), then
// solved from there.
__global__ void __launch_bounds__(OFB_SOLVE_THREADS)
pair_solve_cam_kernel(TrackLoader tl, ofb_camera cam, double4* __restrict__ xu, int variant,
                      const ofb_imu_sample* __restrict__ imu, ofb_pair_result* __restrict__ out,
                      const FeatImageState* __restrict__ det)
{
    const int f = blockIdx.x, n = tl.end(f);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const size_t o = (size_t)f * tl.stride + i;
        if (tl.status[o]) xu[o] = ofb_calibrate(cam, tl.next[2 * o], tl.next[2 * o + 1], tl.prev[2 * o], tl.prev[2 * o + 1]);
    }
    __syncthreads();
    pair_solve(CalibLoader{xu, tl.stride, tl.status, tl.counts, tl.counts_stride, 0}, variant, imu, out, det);
}

}  // namespace

// Stages 1b-4 for pairs [c0, c0+n) whose level-0 frames already sit in pp/pn (images 0..n-1 of each).
// Sequence layout (pn == pp): pp holds n+1 consecutive frames of one stream, pair i = (image i, image i+1), so every
// interior frame's pyramid is built once and serves as "next" of one pair and "prev" of the following one.
static int run_pairs_chunk(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, double fb_max_err, ofb_pyr* pp, ofb_pyr* pn,
                           int n, int c0,
                           const ofb_imu_sample* dimu, const int* counts_in, float* d_prev, float* d_next, uint8_t* d_stat,
                           ofb_pair_result* d_res, bool mark)
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
    OFB_TRY(ofb_lk_device(ctx, pp, 0, 1, pn, seq ? 1 : 0, 1, n, cp, counts, counts_stride, K, (size_t)K, cfg->win_w, cfg->win_h,
                          cfg->max_level, cfg->max_count, cfg->eps, 0, cfg->min_eig_thr, cn, cs, ctx->scratch[SC_ERR].as<float>(),
                          fb_max_err));
    STAGE_MARK(4);
    TrackLoader ld{cp, cn, cs, counts, counts_stride, (size_t)K, cfg->cx, cfg->cy, cfg->pos_scale, cfg->flow_scale};
    if (cam) {
        OFB_TRY(ctx->scratch[SC_CALIB].reserve(sizeof(double4) * (size_t)n * K));
        pair_solve_cam_kernel<<<n, OFB_SOLVE_THREADS, 0, ctx->stream>>>(ld, *cam, ctx->scratch[SC_CALIB].as<double4>(), cfg->variant,
                                                                       dimu + c0, d_res + c0, st);
    } else {
        pair_solve_kernel<<<n, OFB_SOLVE_THREADS, 0, ctx->stream>>>(ld, cfg->variant, dimu + c0, d_res + c0, st);
    }
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
    OFB_REQUIRE(ctx && cfg && prev && next && imu && results, "frame_pairs: null argument");
    if (cam) OFB_TRY(ofb_camera_check(cam, "frame_pairs"));
    OFB_REQUIRE(ofb_fb_thr_ok(fb_max_err), "frame_pairs: fb_max_err must be >= 0 (0 = no forward-backward check)");
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
    OutStage o[4];
    OFB_TRY(ofb_stage_out(ctx, SC_PTS0, prev_pts, sizeof(float) * 2 * npts, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_PTS1, next_pts, sizeof(float) * 2 * npts, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_STAT, status, npts, &o[2]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT3, results, sizeof(ofb_pair_result) * n_pairs, &o[3]));
    // optional outputs still need device storage when the caller passes NULL
    float* d_prev = (float*)o[0].dev; float* d_next = (float*)o[1].dev; uint8_t* d_stat = (uint8_t*)o[2].dev;
    if (!d_prev) { OFB_TRY(ctx->scratch[SC_PTS0].reserve(sizeof(float) * 2 * npts)); d_prev = ctx->scratch[SC_PTS0].as<float>(); }
    if (!d_next) { OFB_TRY(ctx->scratch[SC_PTS1].reserve(sizeof(float) * 2 * npts)); d_next = ctx->scratch[SC_PTS1].as<float>(); }
    if (!d_stat) { OFB_TRY(ctx->scratch[SC_STAT].reserve(npts)); d_stat = ctx->scratch[SC_STAT].as<uint8_t>(); }
    const void* dimu;
    OFB_TRY(ofb_stage_in(ctx, SC_IN3, imu, sizeof(ofb_imu_sample) * n_pairs, &dimu));
    const int* counts_in = nullptr;
    if (!cfg->detect) {
        const void* dn;
        OFB_TRY(ofb_stage_in(ctx, SC_IN4, n_in, sizeof(int) * n_pairs, &dn));
        counts_in = (const int*)dn;
        if ((const float*)pts_in != d_prev)
            OFB_CUDA(cudaMemcpyAsync(d_prev, pts_in, sizeof(float) * 2 * npts, cudaMemcpyDefault, ctx->stream));
    }
    const bool host_frames = !ofb_is_device_ptr(prev) && !ofb_is_device_ptr(next);
    // consecutive frames of one stream in one buffer: each frame is uploaded and its pyramid built once per sub-batch
    const bool seq = next == prev + image_stride && n_pairs > 1;
    const int chunk = 8;
    if (host_frames && n_pairs > chunk && !ctx->profile) {
        // Host frames: pipeline sub-batches. The frames of the whole call are staged in one device buffer by
        // back-to-back H2D copies on a copy stream (the PCIe copy is the bound: nothing else is ever queued between
        // two copies); a sub-batch starts as soon as its frames have landed and then runs exactly the resident path
        // (level 0 aliases the staging buffer; in the sequence layout a frame shared by two sub-batches is simply
        // read by both). Sub-batches compute alternately on this context and on its twin (own stream and scratch),
        // so the one-CTA-per-image selection of sub-batch i runs beside the lambda_min kernel of sub-batch i+1. The
        // last sub-batches are smaller: what remains after the last copy is one short chain.
        if (!ctx->twin) {
            OFB_TRY(ofb_ctx_create(ctx->device, &ctx->twin));
            OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_twin_fork, cudaEventDisableTiming));
            OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_twin_join, cudaEventDisableTiming));
        }
        ofb_ctx* tw = ctx->twin;
        if (!ctx->copy_stream) OFB_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        if (!ctx->ev_free[0]) OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_free[0], cudaEventDisableTiming));
        const int pitch_d = (w + 15) & ~15;
        const size_t stride_d = (((size_t)pitch_d * h) + 255) & ~(size_t)255;
        const size_t n_frames = seq ? (size_t)n_pairs + 1 : 2 * (size_t)n_pairs;
        OFB_TRY(ctx->scratch[SC_FRAMES].reserve(stride_d * n_frames + 256));
        uint8_t* d_frames = ctx->scratch[SC_FRAMES].as<uint8_t>();
        uint8_t* d_prevf = d_frames;
        uint8_t* d_nextf = seq ? d_frames + stride_d : d_frames + stride_d * (size_t)n_pairs;
        auto upload = [&](uint8_t* dst, const uint8_t* src, int count) -> int {
            if (count <= 0) return OFB_OK;
            if (pitch == pitch_d && image_stride == stride_d) {            // same layout on both sides: one copy
                OFB_CUDA(cudaMemcpyAsync(dst, src, stride_d * (size_t)(count - 1) + (size_t)pitch * (h - 1) + w,
                                         cudaMemcpyHostToDevice, ctx->copy_stream));
                return OFB_OK;
            }
            for (int i = 0; i < count; ++i)
                OFB_CUDA(cudaMemcpy2DAsync(dst + (size_t)i * stride_d, pitch_d, src + (size_t)i * image_stride, pitch, w, h,
                                           cudaMemcpyHostToDevice, ctx->copy_stream));
            return OFB_OK;
        };
        // the staging buffer may still be read by work enqueued earlier (a previous call with device-side outputs)
        OFB_CUDA(cudaEventRecord(ctx->ev_free[0], ctx->stream));
        OFB_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_free[0], 0));
        // staged inputs (IMU samples, seed points) were enqueued on this context's stream
        OFB_CUDA(cudaEventRecord(ctx->ev_twin_fork, ctx->stream));
        OFB_CUDA(cudaStreamWaitEvent(tw->stream, ctx->ev_twin_fork, 0));
        const uint64_t tw0 = tw->launches;
        int ci = 0;
        for (int c0 = 0; c0 < n_pairs; ++ci) {
            const int left = n_pairs - c0;
            const int n = left > 12 ? chunk : left > 4 ? 4 : left > 2 ? 2 : left;
            ofb_ctx* c = (ci & 1) ? tw : ctx;
            const int slot = (ci >> 1) & 1;
            if (seq) {
                // frames c0 .. c0+n; frame c0 came with the previous sub-batch
                const int f0 = ci == 0 ? 0 : c0 + 1;
                OFB_TRY(upload(d_frames + (size_t)f0 * stride_d, prev + (size_t)f0 * image_stride, c0 + n + 1 - f0));
            } else {
                OFB_TRY(upload(d_prevf + (size_t)c0 * stride_d, prev + (size_t)c0 * image_stride, n));
                OFB_TRY(upload(d_nextf + (size_t)c0 * stride_d, next + (size_t)c0 * image_stride, n));
            }
            if ((int)ctx->ev_piece.size() <= ci) {
                cudaEvent_t e;
                OFB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                ctx->ev_piece.push_back(e);
            }
            OFB_CUDA(cudaEventRecord(ctx->ev_piece[ci], ctx->copy_stream));
            OFB_CUDA(cudaStreamWaitEvent(c->stream, ctx->ev_piece[ci], 0));
            // (c, slot) is reused every fourth sub-batch, on the same stream: stream order protects its upper levels
            OFB_TRY(ofb_pyr_prepare(c, &c->pair_pyr[slot][0], d_prevf + (size_t)c0 * stride_d, w, h, pitch_d, stride_d,
                                    seq ? n + 1 : n, seq ? chunk + 1 : chunk, cfg->max_level, false));
            if (!seq)
                OFB_TRY(ofb_pyr_prepare(c, &c->pair_pyr[slot][1], d_nextf + (size_t)c0 * stride_d, w, h, pitch_d, stride_d, n,
                                        chunk, cfg->max_level, false));
            OFB_TRY(run_pairs_chunk(c, cfg, cam, fb_max_err, c->pair_pyr[slot][0], seq ? c->pair_pyr[slot][0] : c->pair_pyr[slot][1], n, c0,
                                    (const ofb_imu_sample*)dimu, counts_in, d_prev, d_next, d_stat, (ofb_pair_result*)o[3].dev, false));
            c0 += n;
        }
        ctx->launches += tw->launches - tw0;
        OFB_CUDA(cudaEventRecord(ctx->ev_twin_join, tw->stream));
        OFB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_twin_join, 0));
        return ofb_finish_out(ctx, o, 4);
    }
    // Resident frames: the batch is cut into chunks that alternate between this context and a twin context with its own
    // stream and scratch. The lambda_min kernel (shared-memory heavy, issue bound) of one chunk and the LK kernel
    // (register heavy, latency bound) of the other are then co-resident on the SMs instead of running back to back.
    static const int twin_chunks = [] { const char* e = getenv("OFB_TWIN_CHUNKS"); return e ? atoi(e) : 2; }();
    if (!host_frames && ofb_is_device_ptr(prev) && ofb_is_device_ptr(next) && !ctx->profile && twin_chunks >= 2 &&
        n_pairs >= twin_chunks) {
        if (!ctx->twin) {
            OFB_TRY(ofb_ctx_create(ctx->device, &ctx->twin));
            OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_twin_fork, cudaEventDisableTiming));
            OFB_CUDA(cudaEventCreateWithFlags(&ctx->ev_twin_join, cudaEventDisableTiming));
        }
        ofb_ctx* tw = ctx->twin;
        // staged inputs (IMU samples, seed points) were enqueued on this context's stream
        OFB_CUDA(cudaEventRecord(ctx->ev_twin_fork, ctx->stream));
        OFB_CUDA(cudaStreamWaitEvent(tw->stream, ctx->ev_twin_fork, 0));
        const int per = (n_pairs + twin_chunks - 1) / twin_chunks;
        const uint64_t tw0 = tw->launches;
        int ci = 0;
        for (int c0 = 0; c0 < n_pairs; c0 += per, ++ci) {
            const int n = n_pairs - c0 < per ? n_pairs - c0 : per;
            ofb_ctx* c = (ci & 1) ? tw : ctx;
            const int slot = (ci >> 1) & 1;
            OFB_TRY(ofb_pyr_prepare(c, &c->pair_pyr[slot][0], prev + (size_t)c0 * image_stride, w, h, pitch, image_stride,
                                    seq ? n + 1 : n, seq ? per + 1 : per, cfg->max_level, false));
            if (!seq)
                OFB_TRY(ofb_pyr_prepare(c, &c->pair_pyr[slot][1], next + (size_t)c0 * image_stride, w, h, pitch, image_stride, n, per,
                                        cfg->max_level, false));
            OFB_TRY(run_pairs_chunk(c, cfg, cam, fb_max_err, c->pair_pyr[slot][0], seq ? c->pair_pyr[slot][0] : c->pair_pyr[slot][1], n, c0,
                                    (const ofb_imu_sample*)dimu, counts_in, d_prev, d_next, d_stat, (ofb_pair_result*)o[3].dev, false));
        }
        ctx->launches += tw->launches - tw0;
        OFB_CUDA(cudaEventRecord(ctx->ev_twin_join, tw->stream));
        OFB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_twin_join, 0));
        return ofb_finish_out(ctx, o, 4);
    }
    // resident frames (or a small batch): one pass over the whole batch
    OFB_TRY(ofb_pyr_prepare(ctx, &ctx->pair_pyr[0][0], prev, w, h, pitch, image_stride, seq ? n_pairs + 1 : n_pairs,
                            seq ? n_pairs + 1 : n_pairs, cfg->max_level, false));
    if (!seq)
        OFB_TRY(ofb_pyr_prepare(ctx, &ctx->pair_pyr[0][1], next, w, h, pitch, image_stride, n_pairs, n_pairs, cfg->max_level, false));
    OFB_TRY(run_pairs_chunk(ctx, cfg, cam, fb_max_err, ctx->pair_pyr[0][0], seq ? ctx->pair_pyr[0][0] : ctx->pair_pyr[0][1], n_pairs, 0,
                            (const ofb_imu_sample*)dimu, counts_in, d_prev, d_next, d_stat, (ofb_pair_result*)o[3].dev, ctx->profile));
    int rc = ofb_finish_out(ctx, o, 4);
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
