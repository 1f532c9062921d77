// tracker.cu -- feature lifecycle around the tracker (SURVEY 8f-2): the point sets of n_streams camera streams
// live on the device between frames; one step = ingest -> pyramid -> LK -> status filter + gates -> solve ->
// top-up detection, with no host round trip between the stages (counts and "needs top-up" flags stay on the device).
//
// Replaces the per-frame loops around cv2.calcOpticalFlowPyrLK in the reference:
//   flight_experiments/evaluate_exp.py:97-120   track, new_pos[status==1], top-up when <= min_feat, solve_lgs
//   velocity_measurment_node:129-172, 224-260   track + status filter, r_tilde gate, solve, masked top-up
//   optical_flow_experiments/of_module.py:83-131 re-detect when <= 10 remain, r_tilde gate with `status`
//   of_library.py:88-92                          static_immobile speed gate
//
// Kernels (all tiny next to the pyramid / LK / lambda_min kernels they sit between):
//   ingest_bgr_kernel        BGR8 -> grey straight into the tracker's level-0 buffer (cv2.cvtColor arithmetic)
//   track_filter_solve_kernel one CTA per stream: ordered compaction of the surviving points (ballot + block
//                            scan), the two gates, then the fp64 normal-equation solve on the kept points
//   mask_render_kernel       exclusion mask of the masked top-up (ones + filled circles), only for streams that need it
//   topup_append_kernel      appends the first (max_features - count) detected corners (greedy selection has the
//                            prefix property: the first m corners of a longer run are the run with maxCorners = m)
#include "common.cuh"
#include "features.cuh"
#include "pyrlk.cuh"
#include "velocity_device.cuh"
#include "camera.cuh"
#include "gyro.cuh"
#include <stddef.h>
#include <type_traits>

struct ofb_tracker {
    ofb_ctx* ctx = nullptr;
    ofb_tracker_cfg cfg;
    int cap = 0;                       // points per stream
    int pitch_d = 0;                   // level-0 pitch of the tracker's own frame buffers
    size_t stride_d = 0;
    DevBuf frames[2];                  // grey level 0 of the previous / current frame (ping-pong)
    ofb_pyr* pyr[2] = {nullptr, nullptr};
    int cur = 0;                       // slot the NEXT frame goes to
    bool have_prev = false;
    DevBuf pts[2];                     // float2 [S][cap]; pts[pcur] = current point sets
    int pcur = 0;
    DevBuf counts;                     // int [3][S]: count, need (top-up flag), kept (count after the gates)
    DevBuf nxt, status, err, kept_prev, det, vlast, mask, hw, bgr;
    // CUDA-graph replay of the steady-state step for small fleets fed from host memory (the launch-bound case: a
    // step is ~15 tiny launches/copies). Inputs are staged in pinned buffers at fixed addresses, so one captured
    // graph per ping-pong parity (x with/without v_prior) serves every later step.
    PinBuf pin_in, pin_out;
    DevBuf dev_io;                     // imu | v_prior | results
    cudaGraphExec_t gexec[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
    uint64_t glaunches[2][2] = {{0, 0}, {0, 0}};
    uint64_t gsig[2][2] = {{0, 0}, {0, 0}};   // signature of the context's scratch arenas the graph's pointers refer to
    bool graph_ok = true;
    bool capturing = false;
    // the new frame's ingest + pyramid run on their own stream: they only have to wait for the LK of the previous step (it
    // read the pyramid slot that is overwritten), so they overlap the previous step's filter / solve / top-up kernels
    cudaStream_t pyr_stream = nullptr;
    cudaEvent_t ev_lk = nullptr, ev_pyr = nullptr;
    bool lk_recorded = false;          // ev_lk marks the LK launch of the previous step
    uint64_t launches_end = ~0ull, async_end = 0;   // the context's counters when the previous step returned
    // split solve: with device-resident inputs and result records the fp64 solve of a step runs on its own stream beside
    // the next frame's LK (track_filter_solve_kernel<1> / <2>); the next filter and the context's sync points wait for it
    cudaStream_t sol_stream = nullptr;
    cudaEvent_t ev_filt = nullptr, ev_sol = nullptr, ev_sol_join = nullptr;
    bool sol_pending = false;
    int plain_steps = 0;               // steps run launch by launch since creation (scratch arenas are sized by them)
    // calibrated camera (ofb_tracker_set_camera): the filter kernel reads it from cam_dev, which is written in stream order,
    // so a graph captured with a camera replays whatever camera is current; calib holds the kept points' (x, y, ux, uy)
    bool has_cam = false;
    ofb_camera cam_host;
    DevBuf cam_dev, calib;
    // forward-backward check of the LK tracks (ofb_tracker_set_fb_check), 0 = off: a kernel argument, so captured graphs
    // hold the value they were captured with
    double fb_max_err = 0.0;
    // gyro-predicted initial flow of the LK tracks (ofb_tracker_set_gyro_prediction): whether the prediction kernel is
    // launched is decided when a step is enqueued, so a change drops the captured graphs
    bool gyro = false;
    // ego-motion solve after the velocity solve (ofb_tracker_set_ego_motion): which kernel is launched is decided when a
    // step is enqueued, so a change drops the captured graphs; records the caller did not ask for go to ego_buf
    bool ego = false;
    DevBuf ego_buf;
    // robust velocity solve after them (ofb_tracker_set_robust), as ego: the setting is a kernel argument, so any change
    // drops the captured graphs; records the caller did not ask for go to rob_buf
    bool robust = false;
    ofb_robust_cfg rcfg = {0.0, 0};
    DevBuf rob_buf;
    uint64_t graph_steps = 0;
};

static cudaError_t tracker_join_solve(ofb_tracker* t);

namespace {

struct TrackerDev {
    const float* prev; const float* next; const uint8_t* status;   // [S][cap] LK input / output
    float* kept_prev; float* kept_next;                             // [S][cap] compacted
    int* count; int* need; int* kept;
    double* vlast;                                                  // [S][3]
    int cap;
    int variant; double cx, cy, ps, fs;
    const ofb_camera* cam; double4* calib;                          // calibrated camera (NULL: the pinhole cx, cy, ps, fs)
    double max_speed, dummy; int gate_mode; double gate_T;
    int min_solve, min_features, topup_mode, max_features;
    int have_prev;
    FeatImageState* feat_state; int* cell_grid; size_t cell_stride; // detector scratch, reset here instead of by memsets
};

// of.r_tilde (of_library.py:365-386, 5-argument form), feasibility value only
__device__ __forceinline__ double r_tilde_point(double px, double py, double ux, double uy, const double n3[3],
                                                const double v[3])
{
    // a = -(X x v), b = X x u3 with X = (px, py, 1), u3 = (ux, uy, 0)
    double a0 = -(py * v[2] - v[1]), a1 = -(v[0] - px * v[2]), a2 = -(px * v[1] - py * v[0]);
    double b0 = -uy, b1 = ux, b2 = px * uy - py * ux;
    double na = sqrt(a0 * a0 + a1 * a1 + a2 * a2), nb = sqrt(b0 * b0 + b1 * b1 + b2 * b2);
    if (nb * na == 0.0) return 1.0;                                   // of_library.py:377-379
    double r = (a0 * b0 + a1 * b1 + a2 * b2) * (1.0 / nb) / na;
    if (n3[0] * px + n3[1] * py + n3[2] < 0) r = -r;
    return r;
}

// EGO: the ego-motion solve of the stream follows the velocity solve on the same kept points (ego[s], zero with flags 0
// when the stream did not solve); ROBUST: then the robust velocity solve under rcfg (rob[s], likewise). Both false is
// the velocity solve alone. CALIB (a camera is attached): the solves read the kept points' calibrated values (T.calib).
// PART 0: filter + solve in one launch. PART 1: the filter alone (compaction, gates, counts, top-up decision -- all the next
// step's LK needs); PART 2: the solve of a stream an earlier PART 1 launch compacted. The split lets the solve run beside
// the next frame's LK on a stream of its own: nothing but the NEXT filter (its r_tilde gate uses the solved velocity) and
// the reader of the result record depend on it.
template <int PART, bool EGO = false, bool ROBUST = false, bool CALIB = false>
__global__ void __launch_bounds__(OFB_SOLVE_THREADS)
track_filter_solve_kernel(TrackerDev T, const ofb_imu_sample* __restrict__ imu, const double* __restrict__ v_prior,
                          ofb_track_result* __restrict__ out, ofb_ego_result* __restrict__ ego, ofb_robust_cfg rcfg,
                          ofb_robust_result* __restrict__ rob)
{
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ int wtot[OFB_SOLVE_THREADS / 32];
    const ofb_imu_sample& im = imu[s];
    const int n = min(max(T.count[s], 0), T.cap);                     // first frame: seeded points (or none) carry over
                                                                      // (clamped: device-side counts are not validated)
    const size_t base = (size_t)s * T.cap;
    double vp[3];
    {
        const double* src = v_prior ? v_prior + 3 * s : T.vlast + 3 * s;
        vp[0] = src[0]; vp[1] = src[1]; vp[2] = src[2];
    }
    // r_tilde is 1 for every point when the prior velocity is zero (of_library.py:377-379): a "keep r <= T" gate
    // would then drop every point and the stream could never solve its first velocity -- no prior, no gate
    const bool have_prior = vp[0] != 0.0 || vp[1] != 0.0 || vp[2] != 0.0;
    const double n3[3] = {im.n[0], im.n[1], im.n[2]};
    // static_immobile compares float32 arrays with a Python scalar: the threshold takes the arrays' type
    const float speed_thr = T.max_speed > 0 ? (float)(T.max_speed / im.d) : 0.f;
    const float dummy = (float)T.dummy;
    int kept = 0, tracked = 0;
    if (PART == 2) kept = T.kept[s];
    for (int i0 = 0; PART != 2 && i0 < n; i0 += OFB_SOLVE_THREADS) {
        const int i = i0 + tid;
        bool st = false, keep = false;
        float px = 0, py = 0, qx = 0, qy = 0;
        if (i < n) {
            px = T.prev[2 * (base + i)]; py = T.prev[2 * (base + i) + 1];
            if (T.have_prev) {
                st = T.status[base + i] != 0;                        // new_pos[status==1]  evaluate_exp.py:99
                qx = T.next[2 * (base + i)]; qy = T.next[2 * (base + i) + 1];
            } else { st = true; qx = px; qy = py; }
            keep = st;
            if (keep && T.have_prev && T.max_speed > 0) {                           // of_library.py:88-92
                const bool speed_ok = fabsf(qx - px) < speed_thr && fabsf(qy - py) < speed_thr;
                const bool not_dummy = px != dummy && py != dummy;
                keep = speed_ok && not_dummy;
            }
            if (keep && T.have_prev && T.gate_mode != OFB_GATE_NONE && have_prior) { // node:238-245, of_module.py:125-131
                const float dx = qx - px, dy = qy - py;
                double r;
                if (T.cam) {
                    const double4 xu = ofb_calibrate(*T.cam, qx, qy, px, py);
                    r = r_tilde_point(xu.x, xu.y, xu.z, xu.w, n3, vp);
                } else {
                    r = r_tilde_point(((double)qx - T.cx) * T.ps, ((double)qy - T.cy) * T.ps, (double)dx * T.fs, (double)dy * T.fs,
                                      n3, vp);
                }
                keep = T.gate_mode == OFB_GATE_R_GE ? r >= T.gate_T : r <= T.gate_T;
            }
        }
        const unsigned int bal = __ballot_sync(0xffffffffu, keep);
        const unsigned int bst = __ballot_sync(0xffffffffu, st);
        if (lane == 0) wtot[warp] = __popc(bal);
        tracked += __popc(bst);                                       // per-warp partial, summed below
        __syncthreads();
        int off = kept, tot = 0;
#pragma unroll
        for (int k = 0; k < OFB_SOLVE_THREADS / 32; ++k) { if (k < warp) off += wtot[k]; tot += wtot[k]; }
        if (keep) {
            const size_t o = base + off + __popc(bal & ((1u << lane) - 1u));
            OFB_DEV_ASSERT(o >= (size_t)s * T.cap && o < (size_t)(s + 1) * T.cap);
            T.kept_prev[2 * o] = px; T.kept_prev[2 * o + 1] = py;
            T.kept_next[2 * o] = qx; T.kept_next[2 * o + 1] = qy;
        }
        kept += tot;
        __syncthreads();
    }
    // calibrated camera: the kept points are undistorted once more, in their compacted order, for the solve (it reads
    // every point twice); keeping the gate's values instead would hold them across the compaction and spill
    if (PART != 2 && T.cam && T.have_prev)
        for (int i = tid; i < kept; i += OFB_SOLVE_THREADS) {
            const size_t o = base + i;
            T.calib[o] = ofb_calibrate(*T.cam, T.kept_next[2 * o], T.kept_next[2 * o + 1], T.kept_prev[2 * o], T.kept_prev[2 * o + 1]);
        }
    if (PART != 2) {
        // tracked: every lane of a warp holds its warp's total; the record takes the sum over warps
        if (lane == 0) wtot[warp] = tracked;
        __syncthreads();                                              // wtot and kept_* visible to the whole CTA
    }
    const bool solve = T.have_prev && kept >= T.min_solve && kept > 0;
    const TrackLoader<CALIB> ld{T.kept_prev, T.kept_next, nullptr, nullptr, 0, kept, (size_t)T.cap, T.cx, T.cy, T.ps, T.fs, T.calib};
    OfbSolveOut o;                                                    // vp: MODULE's per-point distances (of_module.py:125)
    if (PART != 1 && solve) o = ofb_block_solve(ld, s, T.variant, im.d, im.n, im.w, im.t, vp);
    OfbEgoOut e;
    if (EGO && PART != 1 && solve) e = ofb_block_solve_ego(ld, s, T.variant, im.d, im.n, im.t);
    OfbRobustOut rb;
    if (ROBUST && PART != 1 && solve) rb = ofb_block_solve_robust(ld, s, T.variant, im.d, im.n, im.w, im.t, rcfg.c, rcfg.iterations);
    // the detector's per-image state and (for streams that will top up) its min-distance cell grid start clean
    if (PART != 2 && kept <= T.min_features)
        for (size_t i = tid; i < T.cell_stride; i += OFB_SOLVE_THREADS) T.cell_grid[(size_t)s * T.cell_stride + i] = -1;
    if (tid == 0) {
        ofb_track_result& r = out[s];                                 // (the two parts own disjoint fields of the record)
        if (PART != 1) {
            for (int k = 0; k < 3; ++k) { r.v[k] = solve ? o.v[k] : 0.0; r.s[k] = solve ? o.s[k] : 0.0; }
            r.res = solve ? o.res : 0.0; r.rank = solve ? o.rank : 0;
            r.flags = solve ? OFB_TRACK_SOLVED : 0;
            if (solve) { T.vlast[3 * s] = o.v[0]; T.vlast[3 * s + 1] = o.v[1]; T.vlast[3 * s + 2] = o.v[2]; }
            if (EGO) {
                if (solve) ego[s] = ofb_ego_record(e, OFB_EGO_SOLVED);
                else { ofb_ego_result z = {}; ego[s] = z; }
            }
            if (ROBUST) {
                if (solve) rob[s] = ofb_robust_record(rb, OFB_ROBUST_SOLVED);
                else { ofb_robust_result z = {}; rob[s] = z; }
            }
        }
        if (PART != 2) {
            FeatImageState z; z.max_key = 0; z.n_cand = 0; z.n_out = 0; z.overflow = 0;
            T.feat_state[s] = z;
            tracked = 0;
#pragma unroll
            for (int k = 0; k < OFB_SOLVE_THREADS / 32; ++k) tracked += wtot[k];
            r.n_prev = n; r.n_tracked = tracked; r.n_kept = kept; r.n_added = 0; r.n_points = kept;
            const int need = kept <= T.min_features;
            T.kept[s] = kept;
            T.need[s] = need;
            T.count[s] = (need && T.topup_mode == OFB_TOPUP_REPLACE) ? 0 : kept;    // of_module.py:86 replaces the set
        }
    }
}

// (3735 B + 19235 G + 9798 R + 2^14) >> 15, four pixels per thread
__global__ void ingest_bgr_kernel(const uint8_t* __restrict__ bgr, int w, int h, int pitch, size_t istride,
                                  uint8_t* __restrict__ gray, int gpitch, size_t gstride, int vec)
{
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x4 >= w) return;
    const uint8_t* p = bgr + (size_t)blockIdx.z * istride + (size_t)y * pitch + 3 * (size_t)x4;
    uint8_t* g = gray + (size_t)blockIdx.z * gstride + (size_t)y * gpitch + x4;
    uint8_t b[12];
    const int npx = min(4, w - x4);
    if (vec && npx == 4) {
        const uint32_t* q = (const uint32_t*)p;
        uint32_t a0 = __ldg(q), a1 = __ldg(q + 1), a2 = __ldg(q + 2);
#pragma unroll
        for (int k = 0; k < 4; ++k) { b[k] = (a0 >> (8 * k)) & 255; b[4 + k] = (a1 >> (8 * k)) & 255; b[8 + k] = (a2 >> (8 * k)) & 255; }
    } else {
        for (int k = 0; k < 3 * npx; ++k) b[k] = p[k];
    }
    uint32_t o = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < npx) {
            const uint32_t v = (3735u * b[3 * k] + 19235u * b[3 * k + 1] + 9798u * b[3 * k + 2] + 16384u) >> 15;
            o |= v << (8 * k);
        }
    if (npx == 4) *(uint32_t*)g = o;                                  // gpitch and gstride are multiples of 16
    else for (int k = 0; k < npx; ++k) g[k] = (o >> (8 * k)) & 255;
}

// Exclusion mask of the masked top-up: ones, with cv2.circle(mask, (int(x), int(y)), radius, 0, FILLED) at every
// surviving point = the clipped union of the midpoint-circle spans; hw[|dy|] is the half width of row cy+dy (computed
// once on the host from OpenCV's loop). MASK_CTAS CTAs per stream, each owning a band of rows: it fills its band
// with ones, then draws the part of every circle that falls into the band (warps over points, lanes over the bytes
// of a row) -- no ordering between CTAs is needed. Streams that need no top-up cost one exiting CTA row.
#define MASK_CTAS 16
__global__ void __launch_bounds__(256)
mask_render_kernel(uint8_t* __restrict__ mask, int w, int h, int mpitch, size_t mstride, const float* __restrict__ pts,
                   size_t pts_stride, const int* __restrict__ count, const int* __restrict__ need,
                   const int* __restrict__ hw, int radius)
{
    const int s = blockIdx.y;
    if (need && !need[s]) return;
    const int r0 = (int)((long long)blockIdx.x * h / gridDim.x), r1 = (int)((long long)(blockIdx.x + 1) * h / gridDim.x);
    uint8_t* m = mask + (size_t)s * mstride;
    {
        uint4* band = (uint4*)(m + (size_t)r0 * mpitch);              // mpitch is a multiple of 16, mstride of 256
        const size_t n16 = (size_t)(r1 - r0) * mpitch / 16;
        for (size_t i = threadIdx.x; i < n16; i += blockDim.x) band[i] = make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
    }
    __syncthreads();
    const int n = count ? count[s] : 0, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int i = warp; i < n; i += nwarps) {
        const float fx = pts[2 * ((size_t)s * pts_stride + i)], fy = pts[2 * ((size_t)s * pts_stride + i) + 1];
        const int cx = (int)fx, cy = (int)fy;                         // Python-2 cv2 truncates float coordinates
        const int ya = max(cy - radius, r0), yb = min(cy + radius, r1 - 1);
        for (int y = ya; y <= yb; ++y) {
            const int dy = y - cy, half = hw[dy < 0 ? -dy : dy];
            const int x0 = max(cx - half, 0), x1 = min(cx + half, w - 1);
            for (int x = x0 + lane; x <= x1; x += 32) m[(size_t)y * mpitch + x] = 0;
        }
    }
}

__global__ void topup_append_kernel(TrackerDev T, const FeatImageState* __restrict__ st, const float* __restrict__ det,
                                    float* __restrict__ pts, ofb_track_result* __restrict__ out)
{
    const int s = blockIdx.x;
    if (!T.need[s]) return;
    const int ndet = st[s].n_out, cnt = T.count[s];
    int take = T.topup_mode == OFB_TOPUP_APPEND ? T.max_features : T.max_features - T.kept[s];
    take = min(take, ndet);
    take = min(take, T.cap - cnt);
    if (take < 0) take = 0;
    const float2* src = (const float2*)det + (size_t)s * T.max_features;
    float2* dst = (float2*)pts + (size_t)s * T.cap + cnt;
    for (int i = threadIdx.x; i < take; i += blockDim.x) dst[i] = src[i];
    if (threadIdx.x == 0) {
        T.count[s] = cnt + take;
        out[s].n_added = take;
        out[s].n_points = cnt + take;
        if (st[s].overflow) out[s].flags |= OFB_TRACK_OVERFLOW;
    }
}

// OpenCV's Circle() (imgproc/drawing.cpp) walks (dx, dy) from (radius, 0) while dx >= dy, filling rows cy+-dy over
// cx+-dx and rows cy+-dx over cx+-dy; the half width of a row is the widest span that touched it.
void circle_half_widths(int radius, std::vector<int>& hw)
{
    hw.assign((size_t)radius + 1, -1);
    int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
    while (dx >= dy) {
        if (hw[dy] < dx) hw[dy] = dx;
        if (hw[dx] < dy) hw[dx] = dy;
        dy++;
        err += plus;
        plus += 2;
        const int m = (err <= 0) - 1;
        err -= minus & m;
        dx += m;
        minus -= m & 2;
    }
    for (int r = 0; r <= radius; ++r) if (hw[r] < 0) hw[r] = 0;
}

int render_mask_device(ofb_ctx* ctx, uint8_t* mask, int w, int h, int mpitch, size_t mstride, int n_streams,
                       const float* pts, size_t pts_stride, int max_pts, const int* count, const int* need, const int* hw,
                       int radius)
{
    (void)max_pts;
    dim3 grid(h < MASK_CTAS ? h : MASK_CTAS, n_streams);
    mask_render_kernel<<<grid, 256, 0, ctx->stream>>>(mask, w, h, mpitch, mstride, pts, pts_stride, count, need, hw, radius);
    OFB_LAUNCH_CHECK(ctx);
    return OFB_OK;
}

}  // namespace

// every stream's prior velocity (the r_tilde gate's `self.vel`) starts from cfg.v_init
static cudaError_t tracker_seed_prior(ofb_tracker* t)
{
    const int S = t->cfg.n_streams;
    std::vector<double> v((size_t)3 * S);
    for (int s = 0; s < S; ++s) for (int k = 0; k < 3; ++k) v[3 * s + k] = t->cfg.v_init[k];
    cudaError_t e = cudaMemcpyAsync(t->vlast.p, v.data(), sizeof(double) * 3 * S, cudaMemcpyHostToDevice, t->ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(t->ctx->stream);          // v is a local
    return e;
}

extern "C" int ofb_tracker_create(ofb_ctx* ctx, const ofb_tracker_cfg* cfg, ofb_tracker** out)
{
    OFB_REQUIRE(ctx && cfg && out, "tracker_create: null argument");
    const ofb_pair_cfg& p = cfg->pair;
    OFB_REQUIRE(p.width >= 2 && p.height >= 2, "tracker_create: bad image geometry");
    OFB_REQUIRE(p.max_corners > 0, "tracker_create: max_features (pair.max_corners) must be positive");
    OFB_REQUIRE(p.max_level >= 0, "tracker_create: max_level must be >= 0");
    OFB_REQUIRE(p.variant >= 0 && p.variant <= OFB_VARIANT_MODULE, "tracker_create: unknown variant");
    OFB_REQUIRE(cfg->n_streams >= 1 && cfg->n_streams <= 65535, "tracker_create: n_streams must be in 1..65535");
    OFB_REQUIRE(cfg->min_features >= 0 && cfg->min_features < p.max_corners,
                "tracker_create: min_features must be in 0..max_features-1");
    OFB_REQUIRE(cfg->topup_mode >= 0 && cfg->topup_mode <= 2, "tracker_create: unknown topup_mode");
    OFB_REQUIRE(cfg->gate_mode >= 0 && cfg->gate_mode <= 2, "tracker_create: unknown gate_mode");
    OFB_REQUIRE(cfg->mask_radius >= 0 && cfg->mask_radius <= 4096, "tracker_create: mask_radius must be in 0..4096");
    OFB_REQUIRE(cfg->min_solve >= 0, "tracker_create: min_solve must be >= 0");
    OFB_CUDA(cudaSetDevice(ctx->device));
    ofb_tracker* t = new ofb_tracker();
    t->ctx = ctx; t->cfg = *cfg;
    const int S = cfg->n_streams, K = p.max_corners;
    t->cap = K + (cfg->topup_mode == OFB_TOPUP_APPEND ? cfg->min_features : 0);
    t->pitch_d = (p.width + 15) & ~15;
    t->stride_d = (((size_t)t->pitch_d * p.height) + 255) & ~(size_t)255;
    int rc = OFB_OK;
    auto R = [&](DevBuf& b, size_t bytes) { if (rc == OFB_OK) rc = b.reserve(bytes); };
    R(t->frames[0], t->stride_d * S + 256); R(t->frames[1], t->stride_d * S + 256);
    const size_t np = (size_t)S * t->cap;
    R(t->pts[0], sizeof(float) * 2 * np); R(t->pts[1], sizeof(float) * 2 * np);
    R(t->nxt, sizeof(float) * 2 * np); R(t->kept_prev, sizeof(float) * 2 * np);
    R(t->status, np); R(t->err, sizeof(float) * np);
    R(t->counts, sizeof(int) * 3 * S); R(t->det, sizeof(float) * 2 * (size_t)S * K);
    R(t->vlast, sizeof(double) * 3 * S);
    if (cfg->topup_mode == OFB_TOPUP_APPEND_MASKED && cfg->mask_radius > 0) {
        R(t->mask, t->stride_d * S);
        R(t->hw, sizeof(int) * ((size_t)cfg->mask_radius + 1));
    }
    if (rc != OFB_OK) { ofb_tracker_destroy(t); return rc; }
    cudaError_t ce = cudaSuccess;
    if (t->hw.p) {
        std::vector<int> hw;
        circle_half_widths(cfg->mask_radius, hw);
        ce = cudaMemcpyAsync(t->hw.p, hw.data(), sizeof(int) * hw.size(), cudaMemcpyHostToDevice, ctx->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);      // hw is a local
    }
    if (ce == cudaSuccess) ce = cudaMemsetAsync(t->counts.p, 0, sizeof(int) * 3 * S, ctx->stream);
    if (ce == cudaSuccess) ce = tracker_seed_prior(t);
    if (ce != cudaSuccess) {
        ofb_set_error("tracker_create: %s", cudaGetErrorString(ce));
        ofb_tracker_destroy(t);
        return OFB_E_CUDA;
    }
    *out = t;
    return OFB_OK;
}

extern "C" int ofb_tracker_destroy(ofb_tracker* t)
{
    OFB_REQUIRE(t, "tracker_destroy: null tracker");
    if (t->ctx) { cudaSetDevice(t->ctx->device); cudaStreamSynchronize(t->ctx->stream); }
    for (int i = 0; i < 2; ++i) {
        if (t->pyr[i]) { cudaFree(t->pyr[i]->base); delete t->pyr[i]; }
        t->frames[i].release(); t->pts[i].release();
    }
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j) if (t->gexec[i][j]) cudaGraphExecDestroy(t->gexec[i][j]);
    t->pin_in.release(); t->pin_out.release();
    if (t->pyr_stream) { cudaStreamSynchronize(t->pyr_stream); cudaStreamDestroy(t->pyr_stream); }
    if (t->sol_stream) {
        cudaStreamSynchronize(t->sol_stream);
        if (t->ctx)
            for (size_t i = 0; i < t->ctx->aux_join.size(); ++i)
                if (t->ctx->aux_join[i].first == t->sol_stream) { t->ctx->aux_join.erase(t->ctx->aux_join.begin() + i); break; }
        cudaStreamDestroy(t->sol_stream);
    }
    if (t->ev_filt) cudaEventDestroy(t->ev_filt);
    if (t->ev_sol) cudaEventDestroy(t->ev_sol);
    if (t->ev_sol_join) cudaEventDestroy(t->ev_sol_join);
    if (t->ev_lk) cudaEventDestroy(t->ev_lk);
    if (t->ev_pyr) cudaEventDestroy(t->ev_pyr);
    DevBuf* bufs[] = {&t->counts, &t->nxt, &t->status, &t->err, &t->kept_prev, &t->det, &t->vlast, &t->mask, &t->hw, &t->bgr, &t->dev_io,
                      &t->cam_dev, &t->calib, &t->ego_buf, &t->rob_buf};
    for (DevBuf* b : bufs) b->release();
    delete t;
    return OFB_OK;
}

extern "C" int ofb_tracker_reset(ofb_tracker* t)
{
    OFB_REQUIRE(t, "tracker_reset: null tracker");
    OFB_CUDA(cudaSetDevice(t->ctx->device));
    t->have_prev = false;
    t->lk_recorded = false;
    OFB_CUDA(tracker_join_solve(t));
    OFB_CUDA(cudaMemsetAsync(t->counts.p, 0, sizeof(int) * 3 * t->cfg.n_streams, t->ctx->stream));
    OFB_CUDA(tracker_seed_prior(t));
    return OFB_OK;
}

extern "C" int ofb_tracker_capacity(const ofb_tracker* t, int* capacity_out)
{
    OFB_REQUIRE(t && capacity_out, "tracker_capacity: null argument");
    *capacity_out = t->cap;
    return OFB_OK;
}

extern "C" int ofb_tracker_set_points(ofb_tracker* t, const float* pts, const int* counts)
{
    OFB_REQUIRE(t && pts && counts, "tracker_set_points: null argument");
    ofb_ctx* ctx = t->ctx;
    OFB_CUDA(cudaSetDevice(ctx->device));
    OFB_CUDA(tracker_join_solve(t));
    const int S = t->cfg.n_streams;
    if (!ofb_is_device_ptr(counts))
        for (int s = 0; s < S; ++s)
            OFB_REQUIRE(counts[s] >= 0 && counts[s] <= t->cap, "tracker_set_points: counts[%d] = %d outside 0..%d", s, counts[s], t->cap);
    OFB_CUDA(cudaMemcpyAsync(t->pts[t->pcur].p, pts, sizeof(float) * 2 * (size_t)S * t->cap, cudaMemcpyDefault, ctx->stream));
    OFB_CUDA(cudaMemcpyAsync(t->counts.p, counts, sizeof(int) * S, cudaMemcpyDefault, ctx->stream));
    OFB_CUDA(cudaStreamSynchronize(ctx->stream));                     // the caller's buffers are free on return
    return OFB_OK;
}

// order the context's stream behind a split solve that is still pending (see ofb_tracker::sol_stream)
static cudaError_t tracker_join_solve(ofb_tracker* t)
{
    if (!t->sol_pending) return cudaSuccess;
    t->sol_pending = false;
    return cudaStreamWaitEvent(t->ctx->stream, t->ev_sol, 0);
}

// One step, launch by launch, on ctx->stream (also the body that is captured into a graph).
static int tracker_step_launches(ofb_tracker* t, const uint8_t* frames, int pitch, size_t image_stride,
                                 const ofb_imu_sample* imu, const double* v_prior, ofb_track_result* results,
                                 float* pts_out, int* n_out, float* kept_prev, float* kept_next, ofb_ego_result* ego,
                                 ofb_robust_result* rob)
{
    ofb_ctx* ctx = t->ctx;
    const ofb_tracker_cfg& cfg = t->cfg;
    const ofb_pair_cfg& pc = cfg.pair;
    const int S = cfg.n_streams, w = pc.width, h = pc.height, K = pc.max_corners, cap = t->cap;
    const size_t np = (size_t)S * cap;
    OutStage o[4];
    OFB_TRY(ofb_stage_out(ctx, SC_OUT3, results, sizeof(ofb_track_result) * S, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT2, n_out, sizeof(int) * S, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_EGO, ego, sizeof(ofb_ego_result) * S, &o[2]));
    OFB_TRY(ofb_stage_out(ctx, SC_ROBUST, rob, sizeof(ofb_robust_result) * S, &o[3]));
    ofb_ego_result* d_ego = (ofb_ego_result*)o[2].dev;
    if (t->ego && !d_ego) {
        OFB_TRY(t->ego_buf.reserve(sizeof(ofb_ego_result) * S));
        d_ego = t->ego_buf.as<ofb_ego_result>();
    }
    ofb_robust_result* d_rob = (ofb_robust_result*)o[3].dev;
    if (t->robust && !d_rob) {
        OFB_TRY(t->rob_buf.reserve(sizeof(ofb_robust_result) * S));
        d_rob = t->rob_buf.as<ofb_robust_result>();
    }
    const void *dimu, *dvp = nullptr;
    OFB_TRY(ofb_stage_in(ctx, SC_IN3, imu, sizeof(ofb_imu_sample) * S, &dimu));
    if (v_prior) OFB_TRY(ofb_stage_in(ctx, SC_IN4, v_prior, sizeof(double) * 3 * S, &dvp));
    // 1. ingest: the tracker keeps its own copy of the frame (it is "old_image" of the next step) unless the caller
    //    lends device-resident frames (borrow_frames)
    const uint8_t* f = t->frames[t->cur].as<uint8_t>();
    uint8_t* fown = t->frames[t->cur].as<uint8_t>();
    int fpitch = t->pitch_d; size_t fstride = t->stride_d;
    bool fused_bgr = false; const uint8_t* bgr_src = nullptr; int bgr_pitch = 0; size_t bgr_stride = 0;
    // Ingest + pyramid go to their own stream (OFB_TRACKER_EARLY_PYR=0: everything on the context's stream): the slot they
    // write was last read by the previous step's LK, nothing else of that step touches it, so they overlap the previous
    // step's filter / solve / top-up. Not while a graph is captured (the graph is for the launch-bound host-fed case),
    // not in profile mode (stage events live on one stream), and never on a stream the caller owns or has been handed
    // (work enqueued there must stay ordered in front of this step). On the context's own stream other API calls may
    // have produced this frame since the previous step (a kernel launch, an asynchronous copy into device memory): the
    // ingest is then ordered behind everything enqueued so far, which costs the overlap for this step only.
    cudaStream_t const main_stream0 = ctx->stream;
    bool early = false;
    {
        const char* ee = getenv("OFB_TRACKER_EARLY_PYR");
        early = !t->capturing && !ctx->profile && ctx->own_stream && !ctx->stream_exported && !(ee && ee[0] == '0');
        // a large grey fleet saturates the GPU by itself: there is no latency to hide and the second stream only costs
        // (256 x 720p: 283 k -> 280 k pairs/s; the heavier BGR ingest still gains 2 %)
        if (early && !cfg.bgr_input && (size_t)S * w * h > ((size_t)32 << 20) && !(ee && ee[0] == '1')) early = false;
    }
    if (ctx->launches != t->launches_end || ctx->async_writes != t->async_end) t->lk_recorded = false;
    if (early) {
        if (!t->pyr_stream) {
            OFB_CUDA(cudaStreamCreateWithFlags(&t->pyr_stream, cudaStreamNonBlocking));
            OFB_CUDA(cudaEventCreateWithFlags(&t->ev_lk, cudaEventDisableTiming));
            OFB_CUDA(cudaEventCreateWithFlags(&t->ev_pyr, cudaEventDisableTiming));
        }
        if (!t->lk_recorded) OFB_CUDA(cudaEventRecord(t->ev_lk, main_stream0));   // no LK to wait for: behind all earlier work
        OFB_CUDA(cudaStreamWaitEvent(t->pyr_stream, t->ev_lk, 0));
        ctx->stream = t->pyr_stream;
    }
    const int ingest_rc = [&]() -> int {
    if (cfg.bgr_input) {
        const uint8_t* src = frames; int spitch = pitch; size_t sstride = image_stride;
        if (!ofb_is_device_ptr(frames)) {
            spitch = (3 * w + 3) & ~3; sstride = ((size_t)spitch * h + 15) & ~(size_t)15;
            OFB_TRY(t->bgr.reserve(sstride * S));
            for (int s = 0; s < S; ++s)
                OFB_CUDA(cudaMemcpy2DAsync(t->bgr.as<uint8_t>() + (size_t)s * sstride, spitch, frames + (size_t)s * image_stride,
                                           pitch, (size_t)3 * w, h, cudaMemcpyHostToDevice, ctx->stream));
            src = t->bgr.as<uint8_t>();
        }
        // the conversion is fused into the first pyramid step (grey level 0 and level 1 from one read of the BGR frame)
        // whenever there is a level 1; OFB_BGR_FUSED=0 keeps the separate conversion kernel (cross-check)
        const char* fe = getenv("OFB_BGR_FUSED");
        fused_bgr = pc.max_level >= 1 && w >= 4 && h >= 4 && !(fe && fe[0] == '0');
        if (fused_bgr) { bgr_src = src; bgr_pitch = spitch; bgr_stride = sstride; }
        else {
            const int vec = ((uintptr_t)src % 4 == 0 && spitch % 4 == 0 && sstride % 4 == 0) ? 1 : 0;
            dim3 grid(ofb_div_up(ofb_div_up(w, 4), 128), h, S);
            ingest_bgr_kernel<<<grid, 128, 0, ctx->stream>>>(src, w, h, spitch, sstride, fown, t->pitch_d, t->stride_d, vec);
            OFB_LAUNCH_CHECK(ctx);
        }
    } else if (cfg.borrow_frames && ofb_is_device_ptr(frames)) {
        f = frames; fpitch = pitch; fstride = image_stride;
    } else if (pitch == t->pitch_d && (S == 1 || image_stride == t->stride_d)) {
        OFB_CUDA(cudaMemcpyAsync(fown, frames, t->stride_d * (size_t)(S - 1) + (size_t)pitch * (h - 1) + w, cudaMemcpyDefault, ctx->stream));
    } else {
        for (int s = 0; s < S; ++s)
            OFB_CUDA(cudaMemcpy2DAsync(fown + (size_t)s * t->stride_d, t->pitch_d, frames + (size_t)s * image_stride, pitch, w, h,
                                       cudaMemcpyDefault, ctx->stream));
    }
    OFB_TRY(ofb_pyr_prepare(ctx, &t->pyr[t->cur], f, w, h, fpitch, fstride, S, S, pc.max_level, !fused_bgr));
    if (fused_bgr) OFB_TRY(ofb_pyr_ingest_bgr(ctx, t->pyr[t->cur], bgr_src, bgr_pitch, bgr_stride));
    return OFB_OK;
    }();
    ctx->stream = main_stream0;
    if (ingest_rc != OFB_OK) return ingest_rc;
    if (early) {
        OFB_CUDA(cudaEventRecord(t->ev_pyr, t->pyr_stream));
        OFB_CUDA(cudaStreamWaitEvent(main_stream0, t->ev_pyr, 0));
    }
    int* count = t->counts.as<int>();
    int* need = count + S;
    int* keptn = count + 2 * S;
    float* P = t->pts[t->pcur].as<float>();
    float* Pn = t->pts[t->pcur ^ 1].as<float>();
    TrackerDev T;
    T.prev = P; T.next = t->nxt.as<float>(); T.status = t->status.as<uint8_t>();
    T.kept_prev = t->kept_prev.as<float>(); T.kept_next = Pn;
    T.count = count; T.need = need; T.kept = keptn; T.vlast = t->vlast.as<double>();
    T.cap = cap; T.variant = pc.variant; T.cx = pc.cx; T.cy = pc.cy; T.ps = pc.pos_scale; T.fs = pc.flow_scale;
    T.cam = t->has_cam ? t->cam_dev.as<ofb_camera>() : nullptr; T.calib = t->calib.as<double4>();
    T.max_speed = cfg.max_speed; T.dummy = cfg.dummy_value; T.gate_mode = cfg.gate_mode; T.gate_T = cfg.gate_T;
    T.min_solve = cfg.min_solve; T.min_features = cfg.min_features; T.topup_mode = cfg.topup_mode; T.max_features = K;
    T.have_prev = t->have_prev ? 1 : 0;
    OFB_TRY(ofb_features_scratch(ctx, w, h, pc.min_distance, S, &T.feat_state, &T.cell_grid, &T.cell_stride));
    // 2. track the stream's points from the kept frame into the new one (with the gyro prediction: starting from where
    //    this step's rotation moves them, predicted on the context's stream from this step's staged IMU samples)
    if (t->have_prev) {
        int lk_flags = 0;
        if (t->gyro) {
            GyroPinhole gph{0.0, 0.0, 0.0, 0.0};
            if (!t->has_cam) OFB_TRY(ofb_gyro_pinhole(&pc, "tracker_step", &gph));
            OFB_TRY(ofb_gyro_predict_device(ctx, gph, T.cam, (const double*)((const char*)dimu + offsetof(ofb_imu_sample, w)),
                                            (int)(sizeof(ofb_imu_sample) / sizeof(double)), S, P, count, 1, cap, (size_t)cap,
                                            t->nxt.as<float>()));
            lk_flags = OFB_LK_USE_INITIAL_FLOW | OFB_LK_FB_INITIAL_FLOW;
        }
        OFB_TRY(ofb_lk_device(ctx, t->pyr[t->cur ^ 1], 0, 1, t->pyr[t->cur], 0, 1, S, P, count, 1, cap, (size_t)cap, pc.win_w,
                              pc.win_h, pc.max_level, pc.max_count, pc.eps, lk_flags, pc.min_eig_thr, t->nxt.as<float>(),
                              t->status.as<uint8_t>(), t->err.as<float>(), t->fb_max_err));
    }
    t->lk_recorded = false;
    if (early && t->have_prev) { OFB_CUDA(cudaEventRecord(t->ev_lk, ctx->stream)); t->lk_recorded = true; }
    // 3.+4. status filter, gates, solve; the compacted new positions become the point set (Pn)
    // (the previous step's solve wrote the prior velocity of this step's gate and read the buffers this filter overwrites)
    OFB_CUDA(tracker_join_solve(t));
    bool split = false;
    {
        const char* se = getenv("OFB_TRACKER_SPLIT_SOLVE");
        split = early && t->have_prev && ofb_is_device_ptr(results) && ofb_is_device_ptr(imu) && (!v_prior || ofb_is_device_ptr(v_prior)) &&
                (!ego || ofb_is_device_ptr(ego)) && (!rob || ofb_is_device_ptr(rob)) && !(se && se[0] == '0');
    }
    if (split) {
        if (!t->sol_stream) {
            OFB_CUDA(cudaStreamCreateWithFlags(&t->sol_stream, cudaStreamNonBlocking));
            OFB_CUDA(cudaEventCreateWithFlags(&t->ev_filt, cudaEventDisableTiming));
            OFB_CUDA(cudaEventCreateWithFlags(&t->ev_sol, cudaEventDisableTiming));
            OFB_CUDA(cudaEventCreateWithFlags(&t->ev_sol_join, cudaEventDisableTiming));
            ctx->aux_join.push_back(std::make_pair(t->sol_stream, t->ev_sol_join));
        }
        track_filter_solve_kernel<1><<<S, OFB_SOLVE_THREADS, 0, ctx->stream>>>(T, (const ofb_imu_sample*)dimu, (const double*)dvp,
                                                                               (ofb_track_result*)o[0].dev, nullptr, t->rcfg, nullptr);
        OFB_LAUNCH_CHECK(ctx);
        OFB_CUDA(cudaEventRecord(t->ev_filt, ctx->stream));
        OFB_CUDA(cudaStreamWaitEvent(t->sol_stream, t->ev_filt, 0));
    }
    // the solve: in one launch with the filter, or (split) on the solve stream behind the filter launched above; CALIB when
    // a camera is attached (attaching or detaching one drops the captured graphs)
    auto launch = [&](auto calib) {
        constexpr bool C = decltype(calib)::value;
        auto kern = split ? (t->ego ? (t->robust ? track_filter_solve_kernel<2, true, true, C> : track_filter_solve_kernel<2, true, false, C>)
                                    : (t->robust ? track_filter_solve_kernel<2, false, true, C> : track_filter_solve_kernel<2, false, false, C>))
                          : (t->ego ? (t->robust ? track_filter_solve_kernel<0, true, true, C> : track_filter_solve_kernel<0, true, false, C>)
                                    : (t->robust ? track_filter_solve_kernel<0, false, true, C> : track_filter_solve_kernel<0, false, false, C>));
        kern<<<S, OFB_SOLVE_THREADS, 0, split ? t->sol_stream : ctx->stream>>>(T, (const ofb_imu_sample*)dimu, (const double*)dvp,
                                                                               (ofb_track_result*)o[0].dev, d_ego, t->rcfg, d_rob);
    };
    if (t->has_cam) launch(std::true_type{});
    else launch(std::false_type{});
    OFB_LAUNCH_CHECK(ctx);
    if (split) {
        OFB_CUDA(cudaEventRecord(t->ev_sol, t->sol_stream));
        t->sol_pending = true;
    }
    bool host_out = false;
    auto copy_out = [&](float* dst, const float* src) -> int {
        if (!dst) return OFB_OK;
        OFB_CUDA(cudaMemcpyAsync(dst, src, sizeof(float) * 2 * np, cudaMemcpyDefault, ctx->stream));
        if (!ofb_is_device_ptr(dst)) host_out = true;
        return OFB_OK;
    };
    OFB_TRY(copy_out(kept_prev, t->kept_prev.as<float>()));
    OFB_TRY(copy_out(kept_next, Pn));                                 // the head of the new point set, before any top-up
    // 5. top-up on the current frame; streams that do not need it are skipped inside the kernels (no host sync)
    const uint8_t* mask = nullptr;
    if (cfg.topup_mode == OFB_TOPUP_APPEND_MASKED && cfg.mask_radius > 0) {
        OFB_TRY(render_mask_device(ctx, t->mask.as<uint8_t>(), w, h, t->pitch_d, t->stride_d, S, Pn, (size_t)cap, cap, count,
                                   need, t->hw.as<int>(), cfg.mask_radius));
        mask = t->mask.as<uint8_t>();
    }
    FeatImageState* st = nullptr;
    const unsigned int cand_cap = (unsigned int)(((size_t)w * h) / 4 + 1024);
    ctx->feat_active = need;
    ctx->feat_prezeroed = true;                                       // done by track_filter_solve_kernel
    int fr = ofb_features_device(ctx, f, w, h, fpitch, (S == 1 ? 0 : fstride), S, mask, t->pitch_d, t->stride_d, K, pc.quality,
                                 pc.min_distance, pc.block_size, cand_cap, t->det.as<float>(), (size_t)2 * K, K, &st);
    ctx->feat_active = nullptr;
    ctx->feat_prezeroed = false;
    if (fr != OFB_OK) return fr;
    topup_append_kernel<<<S, 128, 0, ctx->stream>>>(T, st, t->det.as<float>(), Pn, (ofb_track_result*)o[0].dev);
    ctx->launches++;
    {
        const cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess) { ofb_set_error("tracker_step: topup_append launch -> %s", cudaGetErrorString(le)); return OFB_E_CUDA; }
    }
    if (o[1].dev) OFB_CUDA(cudaMemcpyAsync(o[1].dev, count, sizeof(int) * S, cudaMemcpyDeviceToDevice, ctx->stream));
    OFB_TRY(copy_out(pts_out, Pn));
    t->pcur ^= 1;
    t->cur ^= 1;
    t->have_prev = true;
    t->launches_end = ctx->launches; t->async_end = ctx->async_writes;
    int rc = ofb_finish_out(ctx, o, 4);
    if (rc == OFB_OK && host_out) OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    return rc;
}

// The context's scratch arenas are shared with every other call on the context and grow on demand: a graph holds their
// addresses, so it is rebuilt when any of them moved (another call needed a larger arena in between).
static uint64_t scratch_signature(const ofb_ctx* ctx)
{
    uint64_t h = 1469598103934665603ull;
    for (int i = 0; i < OFB_NSCRATCH; ++i) { h ^= (uint64_t)(uintptr_t)ctx->scratch[i].p; h *= 1099511628211ull; }
    return h;
}

// Steady-state step replayed from a captured CUDA graph. Returns OFB_E_UNSUPPORTED when the graph could not be
// built (the caller then runs the step launch by launch; nothing has executed and the tracker state is unchanged).
static int tracker_step_graph(ofb_tracker* t, const uint8_t* frames, int pitch, size_t image_stride,
                              const ofb_imu_sample* imu, const double* v_prior, ofb_track_result* results, ofb_ego_result* ego,
                              ofb_robust_result* rob)
{
    ofb_ctx* ctx = t->ctx;
    const int S = t->cfg.n_streams, w = t->cfg.pair.width, h = t->cfg.pair.height;
    const size_t row = (size_t)(t->cfg.bgr_input ? 3 : 1) * w, fbytes = row * h;
    const size_t off_imu = (fbytes * S + 255) & ~(size_t)255, off_vp = off_imu + sizeof(ofb_imu_sample) * S;
    const size_t in_bytes = off_vp + sizeof(double) * 3 * S;
    const size_t d_vp = sizeof(ofb_imu_sample) * S, d_res = d_vp + sizeof(double) * 3 * S;
    const size_t d_ego = d_res + sizeof(ofb_track_result) * S, out_bytes = sizeof(ofb_track_result) * S;
    const size_t ego_bytes = sizeof(ofb_ego_result) * S, d_rob = d_ego + ego_bytes, rob_bytes = sizeof(ofb_robust_result) * S;
    if (!t->pin_in.p) {                 // fixed sizes: allocated once, the addresses are baked into the graphs
        OFB_TRY(t->pin_in.reserve(in_bytes));
        OFB_TRY(t->pin_out.reserve(out_bytes + ego_bytes + rob_bytes));    // results | ego records | robust records
        OFB_TRY(t->dev_io.reserve(d_rob + rob_bytes));
    }
    uint8_t* pin = (uint8_t*)t->pin_in.p;
    uint8_t* dio = t->dev_io.as<uint8_t>();
    for (int s = 0; s < S; ++s) {
        const uint8_t* src = frames + (size_t)s * image_stride;
        if ((size_t)pitch == row) memcpy(pin + (size_t)s * fbytes, src, fbytes);
        else for (int y = 0; y < h; ++y) memcpy(pin + (size_t)s * fbytes + (size_t)y * row, src + (size_t)y * pitch, row);
    }
    memcpy(pin + off_imu, imu, sizeof(ofb_imu_sample) * S);
    if (v_prior) memcpy(pin + off_vp, v_prior, sizeof(double) * 3 * S);
    const int par = t->cur, hp = v_prior ? 1 : 0;
    if (t->gexec[par][hp] && t->gsig[par][hp] != scratch_signature(ctx)) {
        cudaGraphExecDestroy(t->gexec[par][hp]);
        t->gexec[par][hp] = nullptr;
    }
    if (!t->gexec[par][hp]) {
        // capture = a dry run of the launch-by-launch body: it advances the host-side ping-pong state, which is
        // restored afterwards (the graph launch below is what executes the step)
        const int cur0 = t->cur, pcur0 = t->pcur; const bool hp0 = t->have_prev; const uint64_t l0 = ctx->launches;
        cudaGraph_t g = nullptr;
        if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) { cudaGetLastError(); return OFB_E_UNSUPPORTED; }
        int rc = OFB_OK;
        t->capturing = true;
        if (cudaMemcpyAsync(dio, pin + off_imu, sizeof(ofb_imu_sample) * S, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) rc = OFB_E_CUDA;
        if (rc == OFB_OK && v_prior &&
            cudaMemcpyAsync(dio + d_vp, pin + off_vp, sizeof(double) * 3 * S, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) rc = OFB_E_CUDA;
        if (rc == OFB_OK)
            rc = tracker_step_launches(t, pin, (int)row, fbytes, (const ofb_imu_sample*)dio, v_prior ? (const double*)(dio + d_vp) : nullptr,
                                       (ofb_track_result*)(dio + d_res), nullptr, nullptr, nullptr, nullptr,
                                       t->ego ? (ofb_ego_result*)(dio + d_ego) : nullptr,
                                       t->robust ? (ofb_robust_result*)(dio + d_rob) : nullptr);
        // the ego and robust records follow the results in dev_io and pin_out: one copy brings them all back
        const size_t copy_bytes = out_bytes + (t->robust ? ego_bytes + rob_bytes : t->ego ? ego_bytes : 0);
        if (rc == OFB_OK && cudaMemcpyAsync(t->pin_out.p, dio + d_res, copy_bytes, cudaMemcpyDeviceToHost,
                                            ctx->stream) != cudaSuccess) rc = OFB_E_CUDA;
        const cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
        const uint64_t captured = ctx->launches - l0;
        t->capturing = false;
        t->cur = cur0; t->pcur = pcur0; t->have_prev = hp0; ctx->launches = l0;
        cudaGraphExec_t ex = nullptr;
        bool ok = rc == OFB_OK && e == cudaSuccess && g;
        if (ok) ok = cudaGraphInstantiate(&ex, g, 0) == cudaSuccess && ex;
        if (g) cudaGraphDestroy(g);
        if (!ok) {
            cudaGetLastError();
            return OFB_E_UNSUPPORTED;
        }
        t->gexec[par][hp] = ex; t->glaunches[par][hp] = captured;
        t->gsig[par][hp] = scratch_signature(ctx);                    // (the dry run cannot grow an arena: three plain steps sized them)
    }
    OFB_CUDA(tracker_join_solve(t));
    OFB_CUDA(cudaGraphLaunch(t->gexec[par][hp], ctx->stream));
    t->lk_recorded = false;             // (a later launch-by-launch step orders its ingest behind this graph)
    ctx->launches += t->glaunches[par][hp];
    t->pcur ^= 1; t->cur ^= 1; t->graph_steps++;
    OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    memcpy(results, t->pin_out.p, out_bytes);
    if (ego) memcpy(ego, (const uint8_t*)t->pin_out.p + out_bytes, ego_bytes);
    if (rob) memcpy(rob, (const uint8_t*)t->pin_out.p + out_bytes + ego_bytes, rob_bytes);
    return OFB_OK;
}

extern "C" int ofb_tracker_step(ofb_tracker* t, const uint8_t* frames, int pitch, size_t image_stride,
                                const ofb_imu_sample* imu, const double* v_prior, ofb_track_result* results,
                                float* pts_out, int* n_out, float* kept_prev, float* kept_next)
{
    return ofb_tracker_step_ego(t, frames, pitch, image_stride, imu, v_prior, results, pts_out, n_out, kept_prev, kept_next, nullptr);
}

extern "C" int ofb_tracker_step_ego(ofb_tracker* t, const uint8_t* frames, int pitch, size_t image_stride,
                                    const ofb_imu_sample* imu, const double* v_prior, ofb_track_result* results,
                                    float* pts_out, int* n_out, float* kept_prev, float* kept_next, ofb_ego_result* ego)
{
    return ofb_tracker_step_robust(t, frames, pitch, image_stride, imu, v_prior, results, pts_out, n_out, kept_prev, kept_next, ego,
                                   nullptr);
}

extern "C" int ofb_tracker_step_robust(ofb_tracker* t, const uint8_t* frames, int pitch, size_t image_stride,
                                       const ofb_imu_sample* imu, const double* v_prior, ofb_track_result* results,
                                       float* pts_out, int* n_out, float* kept_prev, float* kept_next, ofb_ego_result* ego,
                                       ofb_robust_result* rob)
{
    OFB_REQUIRE(t && frames && imu && results, "tracker_step: null argument");
    OFB_REQUIRE(!ego || t->ego, "tracker_step: ego records need ofb_tracker_set_ego_motion(trk, 1)");
    OFB_REQUIRE(!rob || t->robust, "tracker_step: robust records need ofb_tracker_set_robust");
    ofb_ctx* ctx = t->ctx;
    const int S = t->cfg.n_streams, w = t->cfg.pair.width, h = t->cfg.pair.height, bpp = t->cfg.bgr_input ? 3 : 1;
    OFB_REQUIRE(pitch >= bpp * w, "tracker_step: pitch smaller than a row");
    OFB_REQUIRE(S == 1 || image_stride >= (size_t)pitch * (h - 1) + (size_t)bpp * w, "tracker_step: image_stride too small");
    if (t->gyro && !t->has_cam) {
        GyroPinhole gph;
        OFB_TRY(ofb_gyro_pinhole(&t->cfg.pair, "tracker_step", &gph));
    }
    OFB_CUDA(cudaSetDevice(ctx->device));
    // launch-bound case (a few small frames from host memory, only the result records wanted): replay a graph
    const char* genv = getenv("OFB_TRACKER_GRAPH");
    const bool graphs_on = !(genv && genv[0] == '0');
    if (graphs_on && t->graph_ok && t->have_prev && t->plain_steps >= 3 && !pts_out && !n_out && !kept_prev && !kept_next &&
        (size_t)S * bpp * w * h <= ((size_t)16 << 20) && !ofb_is_device_ptr(frames) && !ofb_is_device_ptr(imu) &&
        !ofb_is_device_ptr(results) && !(v_prior && ofb_is_device_ptr(v_prior)) && !(ego && ofb_is_device_ptr(ego)) &&
        !(rob && ofb_is_device_ptr(rob))) {
        const int rc = tracker_step_graph(t, frames, pitch, image_stride, imu, v_prior, results, ego, rob);
        if (rc != OFB_E_UNSUPPORTED) return rc;
        t->graph_ok = false;            // this build / driver cannot capture the step: stay on plain launches
    }
    t->plain_steps++;
    return tracker_step_launches(t, frames, pitch, image_stride, imu, v_prior, results, pts_out, n_out, kept_prev, kept_next, ego,
                                 rob);
}

// A setting that changes what a step launches, or a launch argument, makes the graphs captured before it stale: they are
// rebuilt on the next eligible step (no graph is in flight: a replayed step synchronises before it returns).
static void tracker_drop_graphs(ofb_tracker* t)
{
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j)
            if (t->gexec[i][j]) { cudaGraphExecDestroy(t->gexec[i][j]); t->gexec[i][j] = nullptr; }
}

extern "C" int ofb_tracker_set_camera(ofb_tracker* t, const ofb_camera* cam)
{
    OFB_REQUIRE(t, "tracker_set_camera: null tracker");
    if (cam) OFB_TRY(ofb_camera_check(cam, "tracker_set_camera"));
    ofb_ctx* ctx = t->ctx;
    OFB_CUDA(cudaSetDevice(ctx->device));
    if (cam) {
        OFB_TRY(t->cam_dev.reserve(sizeof(ofb_camera)));
        OFB_TRY(t->calib.reserve(sizeof(double4) * (size_t)t->cfg.n_streams * t->cap));
        // Stream order on the context's stream places the update behind the filter kernels of every step enqueued so far
        // (the only readers of the camera; a split solve reads the calibrated points its filter wrote) and in front of
        // the next step's, whether that step is launched or replayed from a graph. A pageable source is staged before
        // cudaMemcpyAsync returns.
        t->cam_host = *cam;
        OFB_CUDA(cudaMemcpyAsync(t->cam_dev.p, &t->cam_host, sizeof(ofb_camera), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (t->has_cam != (cam != nullptr)) {
        // attaching or detaching changes the solve kernel and the filter kernel's arguments
        tracker_drop_graphs(t);
        t->has_cam = cam != nullptr;
    }
    return OFB_OK;
}

extern "C" int ofb_tracker_set_fb_check(ofb_tracker* t, double fb_max_err)
{
    OFB_REQUIRE(t, "tracker_set_fb_check: null tracker");
    OFB_REQUIRE(ofb_fb_thr_ok(fb_max_err), "tracker_set_fb_check: fb_max_err must be >= 0 (0 = off)");
    if (fb_max_err != t->fb_max_err) {
        // the threshold is an argument of the LK launch
        tracker_drop_graphs(t);
        t->fb_max_err = fb_max_err;
    }
    return OFB_OK;
}

extern "C" int ofb_tracker_set_gyro_prediction(ofb_tracker* t, int enable)
{
    OFB_REQUIRE(t, "tracker_set_gyro_prediction: null tracker");
    if (enable && !t->has_cam) {
        GyroPinhole gph;
        OFB_TRY(ofb_gyro_pinhole(&t->cfg.pair, "tracker_set_gyro_prediction", &gph));
    }
    if ((enable != 0) != t->gyro) {
        // the prediction is a launch of the step and the LK flags are a launch argument
        tracker_drop_graphs(t);
        t->gyro = enable != 0;
    }
    return OFB_OK;
}

extern "C" int ofb_tracker_set_ego_motion(ofb_tracker* t, int enable)
{
    OFB_REQUIRE(t, "tracker_set_ego_motion: null tracker");
    OFB_REQUIRE(!enable || t->cfg.pair.variant != OFB_VARIANT_MODULE,
                "tracker_set_ego_motion: the MODULE variant has no gyro term to estimate");
    if ((enable != 0) != t->ego) {
        // the solve kernel is chosen when a step is enqueued
        tracker_drop_graphs(t);
        t->ego = enable != 0;
    }
    return OFB_OK;
}

extern "C" int ofb_tracker_set_robust(ofb_tracker* t, const ofb_robust_cfg* cfg)
{
    OFB_REQUIRE(t, "tracker_set_robust: null tracker");
    if (cfg) {
        OFB_REQUIRE(t->cfg.pair.variant != OFB_VARIANT_MODULE, "tracker_set_robust: the MODULE variant is not supported");
        OFB_TRY(ofb_robust_check(cfg, "tracker_set_robust"));
    }
    const bool on = cfg != nullptr;
    if (on != t->robust || (on && (cfg->c != t->rcfg.c || cfg->iterations != t->rcfg.iterations))) {
        // the kernel and its setting are chosen when a step is enqueued
        tracker_drop_graphs(t);
        t->robust = on;
        t->rcfg = on ? *cfg : ofb_robust_cfg{0.0, 0};
    }
    return OFB_OK;
}

/* steps replayed from a CUDA graph so far (0 when graphs are off or were never eligible); *conditional_out is always 0
 * (the captured graphs hold no conditional node) */
extern "C" int ofb_tracker_graph_info(const ofb_tracker* t, uint64_t* steps_out, int* conditional_out)
{
    OFB_REQUIRE(t && steps_out, "tracker_graph_info: null argument");
    *steps_out = t->graph_steps;
    if (conditional_out) *conditional_out = 0;
    return OFB_OK;
}

extern "C" int ofb_tracker_render_mask(ofb_ctx* ctx, const float* pts, int n, int radius, int w, int h, uint8_t* mask_out)
{
    OFB_REQUIRE(ctx && mask_out && (pts || n == 0), "tracker_render_mask: null argument");
    OFB_REQUIRE(w > 0 && h > 0 && n >= 0 && radius >= 0 && radius <= 4096, "tracker_render_mask: bad arguments");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const int mpitch = (w + 15) & ~15;
    const size_t mstride = ((size_t)mpitch * h + 255) & ~(size_t)255;
    OFB_TRY(ctx->scratch[SC_TMP0].reserve(mstride));
    OFB_TRY(ctx->scratch[SC_TMP1].reserve(sizeof(int) * ((size_t)radius + 2)));
    std::vector<int> hw;
    circle_half_widths(radius, hw);
    hw.push_back(n);                                                  // the count rides behind the table
    OFB_CUDA(cudaMemcpyAsync(ctx->scratch[SC_TMP1].p, hw.data(), sizeof(int) * hw.size(), cudaMemcpyHostToDevice, ctx->stream));
    OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    const void* dpts = nullptr;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, pts, sizeof(float) * 2 * (size_t)n, &dpts));
    const int* dhw = ctx->scratch[SC_TMP1].as<int>();
    OFB_TRY(render_mask_device(ctx, ctx->scratch[SC_TMP0].as<uint8_t>(), w, h, mpitch, mstride, 1, (const float*)dpts, (size_t)n, n,
                               dhw + radius + 1, nullptr, dhw, radius));
    OFB_CUDA(cudaMemcpy2DAsync(mask_out, w, ctx->scratch[SC_TMP0].p, mpitch, w, h, cudaMemcpyDefault, ctx->stream));
    OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    return OFB_OK;
}
