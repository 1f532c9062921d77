/*
 * ofb200.h -- C ABI of libofb200.so: the B200 (sm_100a) velocity-measurement hot path.
 *
 * The reference (liquidcronos/Drone-stabilisation-using-Optical-Flow-Gps-and-Inertial-Sensors)
 * is pure Python and has no FFI layer; the boundary it offers is the set of Python call shapes
 * its drivers use (SURVEY.md 8b). Each entry point below names the reference call it replaces
 * (paths relative to the reference checkout). The Python mirror of those call shapes lives in
 * drone-stabilisation-using-optical-flow-gps-and-inertial-sensors_b200/ and binds these symbols
 * with ctypes; INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *  - every function returns 0 on success, <0 on error (OFB_E_*); ofb_last_error() returns the
 *    message of the calling thread's last failure. No exception crosses the boundary.
 *  - pointer arguments may be HOST or DEVICE memory; the library classifies each pointer with
 *    cudaPointerGetAttributes. Host inputs are copied in, host outputs copied out, on the
 *    context's stream; a call with any host OUTPUT returns after that output is complete.
 *    Calls whose outputs are all device-resident return after enqueueing (use ofb_ctx_sync).
 *  - a context = one CUDA device + one stream + grow-only scratch arenas. Not thread-safe per
 *    context; contexts are independent (one per camera stream / callback thread).
 *  - images are 8-bit single channel, row pitch in bytes.
 */
#ifndef OFB200_H
#define OFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFB_OK            0
#define OFB_E_INVALID    -1   /* bad argument (Python layer raises ValueError) */
#define OFB_E_CUDA       -2   /* CUDA runtime failure */
#define OFB_E_NOMEM      -3
#define OFB_E_UNSUPPORTED -4

#define OFB_MAX_LEVELS   16

typedef struct ofb_ctx ofb_ctx;
typedef struct ofb_pyr ofb_pyr;

const char* ofb_last_error(void);
int  ofb_version(void);

/* ---- context ----------------------------------------------------------------------------- */
int ofb_ctx_create(int device, ofb_ctx** out);
/* same, but all work is enqueued on an existing cudaStream_t (e.g. torch's current stream) */
int ofb_ctx_create_on_stream(int device, void* cuda_stream, ofb_ctx** out);
int ofb_ctx_destroy(ofb_ctx* ctx);
int ofb_ctx_sync(ofb_ctx* ctx);
int ofb_ctx_stream(ofb_ctx* ctx, void** cuda_stream_out);
/* number of kernels this context has launched since creation (bench.py's gpu_launches) */
int ofb_ctx_launch_count(ofb_ctx* ctx, uint64_t* out);
/* per-stage CUDA-event timing of ofb_frame_pairs on the context's stream. ms_out[5] accumulates, in
 * order: pyramids (+H2D of host frames), lambda_min+NMS kernel, ordered-selection kernel, LK kernel,
 * velocity-solve kernel; *calls_out = number of ofb_frame_pairs calls accumulated. */
int ofb_ctx_set_profile(ofb_ctx* ctx, int enable);
int ofb_ctx_stage_times(ofb_ctx* ctx, float* ms_out, uint64_t* calls_out);
/* CUDA-event bracket on the context's stream: ofb_timer_start, ..., ofb_timer_stop -> ms */
int ofb_timer_start(ofb_ctx* ctx);
int ofb_timer_stop(ofb_ctx* ctx, float* ms_out);
/* device scratch for callers that want resident inputs without torch: plain cudaMalloc/cudaFree,
 * host<->device copies on the context's stream */
int ofb_dev_alloc(ofb_ctx* ctx, size_t bytes, void** out);
int ofb_dev_free(ofb_ctx* ctx, void* p);
int ofb_host_alloc_pinned(ofb_ctx* ctx, size_t bytes, void** out);
int ofb_host_free_pinned(ofb_ctx* ctx, void* p);
int ofb_memcpy(ofb_ctx* ctx, void* dst, const void* src, size_t bytes);   /* direction inferred; synchronous */
int ofb_memcpy_async(ofb_ctx* ctx, void* dst, const void* src, size_t bytes);

/* ---- stage 0: BGR -> grey. Replaces cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
 *      velocity_measurment_node:113, flight_experiments/evaluate_exp.py:65,85,
 *      optical_flow_experiments/of_module.py:40,80.  (3735 B + 19235 G + 9798 R + 2^14) >> 15 */
int ofb_bgr2gray(ofb_ctx* ctx, const uint8_t* bgr, int w, int h, int pitch, uint8_t* gray, int gray_pitch);

/* ---- stage 1: Gaussian pyramid. Replaces the pyramid built inside cv2.calcOpticalFlowPyrLK
 *      (velocity_measurment_node:133, evaluate_exp.py:98, of_module.py:88, of_library.py:249);
 *      same arithmetic as cv2.pyrDown: [1 4 6 4 1]^2, reflect-101, (sum+128)>>8.
 *      n_images images of identical size, image i at img + i*image_stride. Level l of image i is
 *      ((w+1)/2^l...) as in OpenCV. The pyramid is owned by the context until ofb_pyr_free. */
int ofb_pyramid(ofb_ctx* ctx, const uint8_t* img, int w, int h, int pitch, size_t image_stride,
                int n_images, int max_level, ofb_pyr** out);
/* The same from BGR8 frames (3 bytes per pixel, pitch >= 3*w): cv2.cvtColor(BGR2GRAY) fused into the first pyramid step --
 * one kernel reads the BGR frame, writes the grey level 0 and level 1 (velocity_measurment_node:113 + :133). */
int ofb_pyramid_bgr(ofb_ctx* ctx, const uint8_t* bgr, int w, int h, int pitch, size_t image_stride,
                    int n_images, int max_level, ofb_pyr** out);
int ofb_pyr_free(ofb_ctx* ctx, ofb_pyr* pyr);
int ofb_pyr_info(const ofb_pyr* pyr, int* n_images, int* n_levels, int* widths, int* heights, int* pitches);
/* copy level `level` of image `image` to dst (host or device), dst_pitch bytes per row */
int ofb_pyr_download(ofb_ctx* ctx, const ofb_pyr* pyr, int image, int level, uint8_t* dst, int dst_pitch);

/* ---- stage 2: Shi-Tomasi. Replaces cv2.goodFeaturesToTrack(gray, mask=..., maxCorners,
 *      qualityLevel, minDistance, blockSize)  velocity_measurment_node:120,163,
 *      evaluate_exp.py:66,106, of_module.py:44,86, of_library.py:238.
 *      xy_out: capacity `capacity` points (x,y float32, integer valued); *n_out = number found
 *      (cv2 returns None when 0). max_corners <= 0 means "all" (as in cv2). */
int ofb_good_features(ofb_ctx* ctx, const uint8_t* img, int w, int h, int pitch,
                      const uint8_t* mask, int mask_pitch,
                      int max_corners, double quality, double min_distance, int block_size,
                      float* xy_out, int capacity, int* n_out);
/* the lambda_min map itself (cv2.cornerMinEigenVal(gray, blockSize)); eig_out is w*h float32 */
int ofb_min_eig_map(ofb_ctx* ctx, const uint8_t* img, int w, int h, int pitch, int block_size, float* eig_out);

/* ---- stage 3: pyramidal Lucas-Kanade. Replaces cv2.calcOpticalFlowPyrLK(prev, next, prevPts,
 *      None, winSize, maxLevel, criteria)  (same call sites as stage 1).
 *      prev/next: pyramids from ofb_pyramid; image index selects the image inside each pyramid.
 *      max_level < 0 uses every level of the pyramid; levels whose size is <= the window are cut
 *      as in OpenCV. criteria: max_count (clamped to [0,100]) and eps (clamped to [0,10]).
 *      flags: OFB_LK_USE_INITIAL_FLOW (next_pts holds the initial guess). */
#define OFB_LK_USE_INITIAL_FLOW 4
int ofb_pyrlk(ofb_ctx* ctx, const ofb_pyr* prev, int prev_image, const ofb_pyr* next, int next_image,
              const float* prev_pts, int n, int win_w, int win_h, int max_level,
              int max_count, double eps, int flags, double min_eig_thr,
              float* next_pts, uint8_t* status, float* err);

/* ---- stage 4: planar-flow velocity least squares. Replaces solve_lgs
 *      variant OFB_VARIANT_NODE  velocity_measurment_node:30-42   (x,u,d,n,omega)
 *      variant OFB_VARIANT_EXP   flight_experiments/evaluate_exp.py:18-31 (x,u,d,n,omega,t)
 *      variant OFB_VARIANT_SIM   numerical_simulation/simulation.py:15-30 (x,u,d,n,omega,t)
 *      x,u: n x 2 float64 (metric). Outputs: v[3]; res[1] (sum of squared residuals; valid only
 *      when *rank==3 and 3n>3, as np.linalg.lstsq); rank; s[3] singular values (descending).
 *      Batched form: n_frames problems, problem f uses points [offsets[f], offsets[f+1]). */
#define OFB_VARIANT_NODE 0
#define OFB_VARIANT_EXP  1
#define OFB_VARIANT_SIM  2
#define OFB_VARIANT_MODULE 3   /* the inline system of optical_flow_experiments/of_module.py:136-146: rows [X]x / dist_i,
                                  rhs [X]x u3 / (dist_i (n.X)) with a per-point distance dist_i from the older 4-argument
                                  of.r_tilde (of_module.py:125); no gyro term, no common height, no lever arm. Accepted by
                                  ofb_solve_velocity_module and by the tracker (ofb_tracker_cfg.pair.variant), where dist_i
                                  comes from the step's prior velocity. */
int ofb_solve_velocity(ofb_ctx* ctx, int variant, const double* x, const double* u, int n, double d,
                       const double n3[3], const double w3[3], const double t3[3],
                       double v_out[3], double* res, int* rank, double s_out[3]);
int ofb_solve_velocity_batched(ofb_ctx* ctx, int variant, const double* x, const double* u,
                               const int* offsets, int n_frames,
                               const double* d, const double* n3, const double* w3, const double* t3,
                               double* v_out, double* res, int* rank, double* s_out);
/* Variant MODULE (of_module.py:136-146): np.linalg.lstsq(A, B) with A_i = [X_i]x / dist_i and
 * B_i = A_i u_i / (n . X_i). x,u: n x ld doubles (ld = 2, or 3 for the homogeneous rows (x, y, 1) / (ux, uy, 0) the
 * reference builds at of_module.py:96-108). dist: n per-point distances (the `distance` output of the 4-argument
 * of.r_tilde); when NULL they are derived from v_prior[3] exactly as that r_tilde does (an all-zero prior, for which
 * the reference would divide by zero, gives unit distances). Outputs as ofb_solve_velocity. */
int ofb_solve_velocity_module(ofb_ctx* ctx, const double* x, const double* u, int n, int ld, const double* dist,
                              const double n3[3], const double* v_prior,
                              double v_out[3], double* res, int* rank, double s_out[3]);
/* generate_test_data: simulation.py:7-12 (t3 != NULL) / velocity_measurment_node:25-29 (t3 NULL) */
int ofb_generate_flow(ofb_ctx* ctx, const double* x, int n, const double v3[3], const double w3[3],
                      double d, const double n3[3], const double* t3, double* u_out);
/* Time-evolution sweep driver (simulation.py:472-501): k steps of `data += generate_test_data(data, v, 0, h, n, t);
 * h += v.n`. pos_out[k][n][2] = the points of every step, flow_out[k][n][2] (may be NULL) = the step's true flow
 * generate_test_data(data_s, v, w, h_s, n, t), d_out[k] (may be NULL) = the heights h_s. One launch for all k steps. */
int ofb_advect_points(ofb_ctx* ctx, const double* x0, int n, const double v3[3], const double w3[3], double d0,
                      const double n3[3], const double t3[3], int k, double* pos_out, double* flow_out, double* d_out);
/* r_tilde: of_library.py:365-386. x,u are n x ld doubles (ld = 2, or 3 for the homogeneous 4-arg
 * copy in sensor_precision_experiments/pixhawk_pure_IMU/of_library.py:365-384, then dist is ignored
 * when <= 0). Outputs r[n], d_out[n]. */
int ofb_r_tilde(ofb_ctx* ctx, const double* x, const double* u, int n, int ld, const double n3[3],
                const double v3[3], double dist, double* r_out, double* d_out);
/* feasibility: simulation.py:108-120 -> out[2*n] = parallelity[n] then length[n] */
int ofb_feasibility(ofb_ctx* ctx, const double* x, const double* v3, const double* u, int n,
                    const double w3[3], const double t3[3], const double n3[3], double* out);

/* ---- fused frame pairs (stages 1-4): what velocity_measurment_node:224-267 and
 *      evaluate_exp.py:77-120 do per frame: detect on prev, track into next, convert pixel
 *      positions/flows to metric, solve. n_pairs independent pairs, images of identical size. */
typedef struct {
    int    width, height;
    int    max_level;                 /* LK maxLevel (levels = max_level+1 before the cut) */
    int    max_corners;               /* > 0 */
    double quality, min_distance;
    int    block_size;
    int    win_w, win_h, max_count;
    double eps, min_eig_thr;
    int    variant;                   /* OFB_VARIANT_* */
    double cx, cy;                    /* principal point (of.pix_trans) */
    double pos_scale;                 /* x = (p_new - c) * pos_scale     node:229-233 */
    double flow_scale;                /* u = (p_new - p_old) * flow_scale  node:235 */
    int    detect;                    /* 1: detect on prev (detect+track+solve); 0: use pts_in */
} ofb_pair_cfg;

typedef struct {   /* per pair IMU/sonar sample */
    double d;        /* height above ground */
    double n[3];     /* plane normal (third column of R) */
    double w[3];     /* gyro rate */
    double t[3];     /* lever arm (EXP/SIM variants) */
} ofb_imu_sample;

#define OFB_PAIR_OVERFLOW 2        /* ofb_pair_result.flags: the detector's candidate buffer (w*h/4 + 1024 local maxima
                                      per image) overflowed -- plateau images; the feature list of this pair is
                                      truncated and must not be trusted (same bit as OFB_TRACK_OVERFLOW) */
typedef struct {
    double v[3];
    double s[3];
    double res;
    int    rank;
    int    n_features;   /* detected (or given) */
    int    n_tracked;    /* status==1 (ofb_frame_pairs_fb: and passed the forward-backward check) */
    int    flags;        /* OFB_PAIR_* (occupies what used to be tail padding: the record is still 72 bytes) */
} ofb_pair_result;

/* prev/next: n_pairs images each, image i at base + i*image_stride (host or device).
 * pts_in (detect==0): n_pairs x max_corners x 2 float32 with counts n_in[n_pairs].
 * Optional outputs (may be NULL): prev_pts/next_pts (n_pairs x max_corners x 2 f32),
 * status (n_pairs x max_corners u8).
 * Sequence layout: when next == prev + image_stride the n_pairs+1 images are consecutive frames of one
 * camera stream (pair i = frames i, i+1 -- what the node sees, it keeps the previous callback's image,
 * velocity_measurment_node:224-267 `old_gray`); every frame is then uploaded and its pyramid built once.
 * Results are identical to passing the same pairs in two separate buffers. */
int ofb_frame_pairs(ofb_ctx* ctx, const ofb_pair_cfg* cfg, int n_pairs,
                    const uint8_t* prev, const uint8_t* next, int pitch, size_t image_stride,
                    const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                    ofb_pair_result* results, float* prev_pts, float* next_pts, uint8_t* status);

/* ---- calibrated camera: OpenCV's pinhole + lens model (plumb_bob / rational_polynomial), no skew.
 *      Replaces the ideal pinhole of velocity_measurment_node:229-235 (one focal length, no distortion) with what a
 *      caller of the reference's style does with cv2.undistortPoints before the solve. Per point, in fp64 and in
 *      OpenCV's operation order (cvUndistortPointsInternal):
 *        x0 = (px - cx) * (1/fx), y0 = (py - cy) * (1/fy); x = x0, y = y0;
 *        `iterations` times (none when n_dist == 0): r2 = x^2 + y^2,
 *          icdist = (1 + ((k6 r2 + k5) r2 + k4) r2) / (1 + ((k3 r2 + k2) r2 + k1) r2)  (icdist < 0: x = x0, y = y0, stop)
 *          x = (x0 - (2 p1 x y + p2 (r2 + 2 x^2))) icdist,  y = (y0 - (p1 (r2 + 2 y^2) + 2 p2 x y)) icdist
 *      A ROS camera_info maps as fx = K[0], fy = K[4], cx = K[2], cy = K[5], dist = D (plumb_bob: 5 coefficients,
 *      rational_polynomial: 8). cv2.undistortPoints iterates 5 times; wide-angle lenses need more to converge (a
 *      k1 = -0.3 lens: 0.48 px left after 5, 1e-8 px after 20), so the struct carries the count explicitly. */
typedef struct {
    double fx, fy, cx, cy;   /* camera matrix K (no skew); fx, fy > 0 */
    double dist[8];          /* k1 k2 p1 p2 k3 k4 k5 k6 (OpenCV order); entries past n_dist are ignored */
    int    n_dist;           /* 0, 4, 5 or 8 */
    int    iterations;       /* fixed-point iterations of the inverse lens model, 1..1000 */
    double rate;             /* > 0: u = (x_new - x_old) * rate, e.g. the frame rate 1/dt */
} ofb_camera;

/* cv2.undistortPointsIter(src, K, D, R, P, (TERM_CRITERIA_COUNT, iterations, 0)): pts and out are n x 2 float64 (host
 * or device; out may equal pts). H = P[:, :3] @ R as 9 row-major doubles, applied as OpenCV does
 * (x, y) <- ((H0 x + H1 y + H2) w, (H3 x + H4 y + H5) w), w = 1 / (H6 x + H7 y + H8); NULL = identity.
 * cam->rate is not used here. */
int ofb_undistort_points(ofb_ctx* ctx, const ofb_camera* cam, const double* pts, int n, const double* H, double* out);

/* ofb_frame_pairs with a calibrated camera: x = undistort(p_new), u = (undistort(p_new) - undistort(p_old)) * rate
 * (cfg->cx / cy / pos_scale / flow_scale are not used). cam == NULL is exactly ofb_frame_pairs. */
int ofb_frame_pairs_cam(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, int n_pairs,
                        const uint8_t* prev, const uint8_t* next, int pitch, size_t image_stride,
                        const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                        ofb_pair_result* results, float* prev_pts, float* next_pts, uint8_t* status);

/* ---- forward-backward check of the LK tracks (OpenCV's samples/python/lk_track.py): every point with forward status 1
 *      is tracked back from next to prev, starting at its forward result, with the same window, levels, criteria and
 *      min_eig_thr and no initial flow. fb_err = max(|x0 - x0r|, |y0 - y0r|) in fp32; the point keeps status 1 iff the
 *      forward and the backward status are 1 and (double)fb_err < fb_max_err. LK's status only says that the window
 *      was well conditioned and stayed inside the image: a point that is covered or uncovered between the frames, a
 *      patch that changes appearance or a window that slides along an edge is tracked with status 1 to a wrong place,
 *      and rarely returns to where it started. Both passes run in one launch, in the warp that owns the feature.
 *      fb_max_err > 0 (+inf allowed) enables the check, 0 disables it; negative values and NaN return OFB_E_INVALID. */
/* calcOpticalFlowPyrLK + the check, without initial flow: next_pts and err are exactly ofb_pyrlk's, status is the
 * combined decision, fb_err (n floats, may be NULL) the distance where both passes had status 1 and +inf elsewhere
 * (everywhere when fb_max_err == 0). */
int ofb_pyrlk_fb(ofb_ctx* ctx, const ofb_pyr* prev, int prev_image, const ofb_pyr* next, int next_image,
                 const float* prev_pts, int n, int win_w, int win_h, int max_level, int max_count, double eps,
                 double min_eig_thr, double fb_max_err, float* next_pts, uint8_t* status, float* err, float* fb_err);
/* ofb_frame_pairs_cam with the check folded into the track status: the solve, ofb_pair_result.n_tracked and the
 * optional status output see only the points that passed it. The check runs on pixel positions, before any camera
 * model. fb_max_err == 0 is exactly ofb_frame_pairs_cam. */
int ofb_frame_pairs_fb(ofb_ctx* ctx, const ofb_pair_cfg* cfg, const ofb_camera* cam, double fb_max_err, int n_pairs,
                       const uint8_t* prev, const uint8_t* next, int pitch, size_t image_stride,
                       const ofb_imu_sample* imu, const float* pts_in, const int* n_in,
                       ofb_pair_result* results, float* prev_pts, float* next_pts, uint8_t* status);

/* ---- feature lifecycle around the tracker (SURVEY 8f-2): the point set of every camera stream stays on the
 *      device between frames. One step does what the reference's per-frame loops do around the tracker
 *      (flight_experiments/evaluate_exp.py:97-120, velocity_measurment_node:129-172 and 224-260,
 *      optical_flow_experiments/of_module.py:83-131):
 *        1. (optional) BGR -> grey of the new frame (node:113), Gaussian pyramid of the new frame only;
 *        2. calcOpticalFlowPyrLK from the kept previous frame at the stream's points (evaluate_exp.py:98);
 *        3. new_pos[status==1], order preserved (evaluate_exp.py:99, node:134-136), then the optional gates:
 *           of.static_immobile (of_library.py:88-92: |new-old| < maxspeed/distance per component and
 *           old != dummy_value) and the r_tilde threshold (node:238-245 keeps r <= T, of_module.py:125-131
 *           keeps r >= T); points that fail are dropped from the set (node:245);
 *        4. px -> metric and solve_lgs on the kept points when at least min_solve remain (node:247-250);
 *        5. top-up when count <= min_features (node:157, evaluate_exp.py:105, of_module.py:83):
 *           goodFeaturesToTrack on the CURRENT frame, see OFB_TOPUP_*.
 *      The first step (no previous frame) only detects (evaluate_exp.py:66, of_module.py:44).
 *      n_streams streams advance in lockstep, one frame each per step (the fleet configuration). */
#define OFB_TOPUP_APPEND_MASKED 0  /* node:157-172: mask = ones with cv2.circle(mask,(int)p,mask_radius,0,FILLED) at every
                                      surviving point, maxCorners = max_features - count, appended */
#define OFB_TOPUP_APPEND        1  /* evaluate_exp.py:105-107: no mask, maxCorners = max_features, appended
                                      (capacity max_features + min_features) */
#define OFB_TOPUP_REPLACE       2  /* of_module.py:83-86: the set is replaced by maxCorners = max_features - count */
#define OFB_GATE_NONE 0
#define OFB_GATE_R_GE 1            /* keep r_tilde >= gate_T   (of_module.py:129) */
#define OFB_GATE_R_LE 2            /* keep r_tilde <= gate_T   (node:240-245) */
#define OFB_TRACK_SOLVED   1       /* ofb_track_result.flags: a velocity was solved this step */
#define OFB_TRACK_OVERFLOW 2       /* detector candidate buffer overflowed during the top-up */
typedef struct ofb_tracker ofb_tracker;

typedef struct {
    ofb_pair_cfg pair;       /* geometry, detector, LK and solve parameters; max_corners = max_features
                                (node:95 max_feat); `detect` is ignored */
    int    n_streams;        /* >= 1 */
    int    min_features;     /* top up when count <= min_features; must be < max_features */
    int    topup_mode;       /* OFB_TOPUP_* */
    int    mask_radius;      /* OFB_TOPUP_APPEND_MASKED: circle radius in px (30 at node:161); 0 = no mask */
    int    bgr_input;        /* 1: frames are BGR8, 3 bytes per pixel (pitch >= 3*width) */
    double max_speed;        /* > 0 enables of.static_immobile(new, old, max_speed, d, dummy_value) */
    double dummy_value;
    int    gate_mode;        /* OFB_GATE_* on of.r_tilde(x, u, n, v_prior, d) */
    double gate_T;
    int    min_solve;        /* solve only when at least this many points are kept (3 at node:247) */
    int    borrow_frames;    /* 1: device-resident grey frames are used in place instead of being copied into the
                                tracker; the caller keeps frame k unchanged until step k+1 has completed (a ring of
                                two buffers per stream is enough). Ignored for host or BGR frames. */
    double v_init[3];        /* prior velocity of the r_tilde gate before the first solve (velocity_measurment_node:183
                                starts from self.vel = [0.1, 0.1, 0.1]). While the prior is exactly zero (no v_init, no
                                v_prior, nothing solved yet) the gate is skipped: r_tilde is 1 for every point then. */
} ofb_tracker_cfg;

typedef struct {
    double v[3];             /* solve_lgs velocity (zeros unless flags & OFB_TRACK_SOLVED) */
    double s[3];
    double res;
    int    rank;
    int    flags;
    int    n_prev;           /* points tracked from (count before the step) */
    int    n_tracked;        /* status == 1 (with ofb_tracker_set_fb_check: and passed the forward-backward check) */
    int    n_kept;           /* after the gates = points the solve used */
    int    n_added;          /* appended by the top-up */
    int    n_points;         /* count after the step */
} ofb_track_result;

/* The tracker works on ctx's stream and scratch arenas: use it from the thread that uses ctx, and destroy it before
 * the context. */
int ofb_tracker_create(ofb_ctx* ctx, const ofb_tracker_cfg* cfg, ofb_tracker** out);
int ofb_tracker_destroy(ofb_tracker* trk);
/* forget the previous frame and all points: the next step detects */
int ofb_tracker_reset(ofb_tracker* trk);
/* points per stream the tracker can hold (pts arrays are n_streams x capacity x 2 float32) */
int ofb_tracker_capacity(const ofb_tracker* trk, int* capacity_out);
/* replace the point sets (host or device): pts n_streams x capacity x 2, counts[n_streams] */
int ofb_tracker_set_points(ofb_tracker* trk, const float* pts, const int* counts);
/* frames: n_streams images (grey u8, or BGR8 when bgr_input), image i at frames + i*image_stride, host or
 * device; imu: one sample per stream; v_prior: n_streams x 3 prior velocity for the r_tilde gate (NULL = the
 * stream's last solved velocity, cfg.v_init before the first solve; an all-zero prior skips the gate). Outputs (host or device; optional ones may be
 * NULL): results[n_streams]; pts_out n_streams x capacity x 2 and n_out[n_streams] = point sets after the step;
 * kept_prev / kept_next n_streams x capacity x 2 = the (old, new) positions the solve used (first n_kept).
 * Streams: on a context that owns its stream (ofb_ctx_create) the ingest + pyramid of the new frame run on a stream of
 * the tracker, ordered behind the previous step's LK kernel only, so that they overlap that step's filter / solve /
 * top-up; they are ordered behind everything on the context's stream whenever another call of this library enqueued
 * work there since the previous step (a kernel launch, ofb_memcpy_async into device memory). Device-resident frames
 * produced by other means must be complete when the call is made. Contexts on a caller's stream
 * (ofb_ctx_create_on_stream) and contexts whose stream was handed out (ofb_ctx_stream) keep every operation on that
 * stream. OFB_TRACKER_EARLY_PYR=0 in the environment disables the second stream. With device-resident frames, IMU samples and
 * result records the fp64 solve of a step also runs on a stream of its own, beside the next frame's LK: the records are
 * complete after ofb_ctx_sync / ofb_timer_stop / ofb_memcpy* on the context (they join that stream), or after the next step
 * of the tracker has been synchronised; OFB_TRACKER_SPLIT_SOLVE=0 disables it. */
int ofb_tracker_step(ofb_tracker* trk, const uint8_t* frames, int pitch, size_t image_stride,
                     const ofb_imu_sample* imu, const double* v_prior, ofb_track_result* results,
                     float* pts_out, int* n_out, float* kept_prev, float* kept_next);
/* Small fleets fed from host memory (<= 16 MB of frames per step, host imu/results, no optional outputs) are
 * launch bound: from the fourth step on such a step is replayed from a captured CUDA graph (inputs staged in
 * pinned buffers at fixed addresses; one graph per ping-pong parity). Results are identical to the launch-by-launch
 * path; OFB_TRACKER_GRAPH=0 in the environment disables the graph. *steps_out = steps replayed from a graph so far;
 * *conditional_out (may be NULL) is always 0: the graphs hold no conditional node. */
int ofb_tracker_graph_info(const ofb_tracker* trk, uint64_t* steps_out, int* conditional_out);
/* Attach a calibrated camera to every stream of the tracker (cam == NULL detaches it: back to cfg.pair's pinhole).
 * From the next ofb_tracker_step on, the r_tilde gate, the MODULE variant's per-point distances and the solve see
 * x = undistort(p_new), u = (undistort(p_new) - undistort(p_old)) * rate; static_immobile stays in pixels. A step
 * already enqueued (split solve, graph replay) keeps the camera it was enqueued with. */
int ofb_tracker_set_camera(ofb_tracker* trk, const ofb_camera* cam);
/* Forward-backward check of every stream's LK tracks (see ofb_pyrlk_fb) from the next ofb_tracker_step on; 0 turns it
 * off (the default). A point that fails it counts as lost (status 0): it leaves the set before the gates, the solve
 * and the top-up. A change of the value rebuilds the captured CUDA graphs. */
int ofb_tracker_set_fb_check(ofb_tracker* trk, double fb_max_err);
/* the exclusion mask OFB_TOPUP_APPEND_MASKED would use for `n` points (n x 2 float32): mask_out h x w u8
 * (1 = allowed, 0 = inside a circle). Exposed for parity tests against cv2.circle. */
int ofb_tracker_render_mask(ofb_ctx* ctx, const float* pts, int n, int radius, int w, int h, uint8_t* mask_out);

/* ---- stage 5: Monte-Carlo error propagation. Replaces of_simulation (simulation.py:36-66),
 *      feas_simulation (simulation.py:70-104) and the per-step np.mean/np.std of the sweep
 *      drivers (e.g. simulation.py:183-202). One ofb_mc_step = one call of of_simulation. */
#define OFB_MC_MAX_POINTS 256
typedef struct {
    double v[3], w[3], n[3], t[3];       /* truth: linear/angular velocity, normal, lever arm */
    double height;
    double ang_vel_sig, translation_sig, height_sig, flow_sig, position_sig, normal_sig;
    double velocity_sig;                 /* feas_simulation only (global at simulation.py:172) */
    double true_vel[3];                  /* feas_simulation only */
    int    n_points;
    int    pos_offset;                   /* index (in points) of this step's first point in pos/flow */
} ofb_mc_step;

typedef struct {                         /* per step, sums over trials (mergeable across shards) */
    double n;                            /* trials accumulated */
    double sum_dv[3];                    /* sum (v_obs - v_true) */
    double sum_dv2[3];                   /* sum (v_obs - v_true)^2 */
    double sum_R;                        /* sum of the analytic bound R */
} ofb_mc_sums;

/* pos / true_flow: all steps' points, (total_points x 2) float64. Trials [trial_begin,
 * trial_begin+trials) of every step are run; RNG = Philox4x32-10 keyed by seed with counter
 * (trial id, draw block, step id + step_id_base) so any sharding of the trial range reproduces
 * the same union. sums_out: n_steps entries (host or device), OVERWRITTEN. Optional dumps (may
 * be NULL; device or host): v_dump (n_steps x trials x 3), R_dump (n_steps x trials).
 * precision: 0 = fp32 per-point arithmetic with fp64 solve/statistics, 1 = fp64 throughout; +2 skips the
 * analytic bound R (sum_R = 0) for callers that only consume v_obs. */
int ofb_mc_sweep(ofb_ctx* ctx, const ofb_mc_step* steps, int n_steps, int step_id_base,
                 const double* pos, const double* true_flow, int total_points,
                 uint64_t trial_begin, uint64_t trials, uint64_t seed, int precision,
                 ofb_mc_sums* sums_out, double* v_dump, double* R_dump);

/* The same sweep over SEVERAL contexts of this process (any mix of devices): contiguous trial shards, all enqueued
 * before the first is waited for, sums merged on the host in context order. pos, true_flow and sums_out are host
 * memory. The union of trials equals the one-context run (counter RNG); no torch, no NCCL. */
int ofb_mc_sweep_multi(ofb_ctx** ctxs, int n_ctx, const ofb_mc_step* steps, int n_steps, int step_id_base,
                       const double* pos, const double* true_flow, int total_points,
                       uint64_t trial_begin, uint64_t trials, uint64_t seed, int precision,
                       ofb_mc_sums* sums_out);

/* feas_simulation: per-point sums over trials of the six quantities returned at
 * simulation.py:104 (backward par, backward dist, forward par, forward dist, backward res,
 * forward res): sums_out[6*n_points] (+ n in *n_out); means = sums / n. */
int ofb_mc_feas(ofb_ctx* ctx, const ofb_mc_step* step, int step_id,
                const double* pos, const double* true_flow,
                uint64_t trial_begin, uint64_t trials, uint64_t seed,
                double* sums_out);

/* overlap (simulation.py:124-136) split so shards can merge: range, then 100-bin counts over
 * [lo,hi] with numpy's histogram binning (last bin closed). */
int ofb_minmax(ofb_ctx* ctx, const double* data, size_t n, double* lo_out, double* hi_out);
int ofb_histogram(ofb_ctx* ctx, const double* data, size_t n, double lo, double hi, int bins,
                  unsigned long long* counts_out);

#ifdef __cplusplus
}
#endif
#endif /* OFB200_H */
