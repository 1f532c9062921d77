// velocity.cu -- stage 4: IMU-derotated planar-flow velocity least squares and the per-point
// helpers around it (generate_test_data, r_tilde, feasibility).
//
// Replaces (reference paths): solve_lgs velocity_measurment_node:30-42 (NODE),
// flight_experiments/evaluate_exp.py:18-31 (EXP), numerical_simulation/simulation.py:15-30 (SIM);
// generate_test_data simulation.py:7-12 / node:25-29; r_tilde of_library.py:365-386;
// feasibility simulation.py:108-120; px->metric node:229-235; body->world is done on the host.
//
// The reference stacks a (3N x 3) matrix row by row and calls np.linalg.lstsq. Here each frame is
// one CTA: per-point contributions to the 3x3 normal equations are accumulated in fp64 registers,
// reduced with warp shuffles + one shared-memory hop, and solved by a Jacobi eigen-decomposition
// (which also yields the singular values and the rank lstsq returns). A second pass over the
// points gives the residual sum without the cancellation of the one-pass formula.
#include "common.cuh"
#include "math3.cuh"
#include "velocity_device.cuh"

namespace {

struct PointsF64 {          // x,u as n x ld doubles, frame f covers [offsets[f], offsets[f+1])
    const double* x; const double* u; const int* offsets; int single_n;
    int ld = 2; const double* dists = nullptr;        // MODULE variant: optional per-point distances
    __device__ int begin(int f) const { return offsets ? offsets[f] : 0; }
    __device__ int end(int f) const { return offsets ? offsets[f + 1] : single_n; }
    __device__ bool load(int, int i, double& px, double& py, double& ux, double& uy) const {
        px = x[ld * i]; py = x[ld * i + 1]; ux = u[ld * i]; uy = u[ld * i + 1];
        return true;
    }
    __device__ bool dist(int, int i, double& d) const { if (!dists) return false; d = dists[i]; return true; }
};

__global__ void __launch_bounds__(OFB_SOLVE_THREADS)
solve_velocity_kernel(PointsF64 ld, int variant, const double* __restrict__ d_arr, const double* __restrict__ n_arr,
                      const double* __restrict__ w_arr, const double* __restrict__ t_arr, int d_stride, int imu_stride,
                      double* __restrict__ v_out, double* __restrict__ res_out, int* __restrict__ rank_out,
                      double* __restrict__ s_out, int* __restrict__ count_out, const double* __restrict__ vprior_arr)
{
    int f = blockIdx.x;
    const double* n3 = n_arr + (size_t)f * imu_stride;
    const double* w3 = w_arr + (size_t)f * imu_stride;
    const double* t3 = t_arr ? t_arr + (size_t)f * imu_stride : nullptr;
    double d = d_arr ? d_arr[(size_t)f * d_stride] : 1.0;
    OfbSolveOut o = ofb_block_solve(ld, f, variant, d, n3, w3, t3, vprior_arr ? vprior_arr + (size_t)f * imu_stride : nullptr);
    if (threadIdx.x == 0) {
        v_out[3 * f] = o.v[0]; v_out[3 * f + 1] = o.v[1]; v_out[3 * f + 2] = o.v[2];
        if (res_out) res_out[f] = o.res;
        if (rank_out) rank_out[f] = o.rank;
        if (s_out) { s_out[3 * f] = o.s[0]; s_out[3 * f + 1] = o.s[1]; s_out[3 * f + 2] = o.s[2]; }
        if (count_out) count_out[f] = o.count;
    }
}

__global__ void __launch_bounds__(OFB_SOLVE_THREADS)
solve_ego_kernel(PointsF64 ld, int variant, const double* __restrict__ d_arr, const double* __restrict__ n_arr,
                 const double* __restrict__ t_arr, ofb_ego_result* __restrict__ out)
{
    const int f = blockIdx.x;
    const OfbEgoOut o = ofb_block_solve_ego(ld, f, variant, d_arr[f], n_arr + 3 * (size_t)f, t_arr ? t_arr + 3 * (size_t)f : nullptr);
    if (threadIdx.x == 0) out[f] = ofb_ego_record(o, OFB_EGO_SOLVED);
}

__global__ void __launch_bounds__(OFB_SOLVE_THREADS)
solve_robust_kernel(PointsF64 ld, int variant, const double* __restrict__ d_arr, const double* __restrict__ n_arr,
                    const double* __restrict__ w_arr, const double* __restrict__ t_arr, ofb_robust_cfg cfg,
                    ofb_robust_result* __restrict__ out, double* __restrict__ wout)
{
    const int f = blockIdx.x;
    const OfbRobustOut o = ofb_block_solve_robust(ld, f, variant, d_arr[f], n_arr + 3 * (size_t)f, w_arr + 3 * (size_t)f,
                                                  t_arr ? t_arr + 3 * (size_t)f : nullptr, cfg.c, cfg.iterations, wout);
    if (threadIdx.x == 0) out[f] = ofb_robust_record(o, OFB_ROBUST_SOLVED);
}

__global__ void generate_flow_kernel(const double* __restrict__ x, int n, double3 v, double3 w, double d,
                                     double3 nrm, double* __restrict__ u)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double px = x[2 * i], py = x[2 * i + 1];
    double nx = nrm.x * px + nrm.y * py + nrm.z;
    // omega x X
    double cx = w.y - w.z * py, cy = w.z * px - w.x, cz = w.x * py - w.y * px;
    double s = nx / d;
    u[2 * i]     = s * (v.x - v.z * px) + (cx - cz * px);
    u[2 * i + 1] = s * (v.y - v.z * py) + (cy - cz * py);
}

// Time-evolution sweep (simulation.py:472-501): between two steps every point moves by its own translational flow,
// data += generate_test_data(data, v, 0, h, n, t), and the height grows by v.n. A point's trajectory depends on no other
// point, so one thread walks all k steps of its point (one launch instead of k dependent host round trips) and
// writes, per step, the position and the true flow of the step (generate_test_data with the real gyro rate).
__global__ void advect_points_kernel(const double* __restrict__ x0, int n, double3 v, double3 vlev, double3 w, double d0,
                                     double dstep, double3 nrm, int k, double* __restrict__ pos_out,
                                     double* __restrict__ flow_out, double* __restrict__ d_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double px = x0[2 * i], py = x0[2 * i + 1], d = d0;
    for (int s = 0; s < k; ++s) {
        const size_t o = 2 * ((size_t)s * n + i);
        pos_out[o] = px; pos_out[o + 1] = py;
        const double nx = nrm.x * px + nrm.y * py + nrm.z, sc = nx / d;
        if (flow_out) {     // simulation.py:7-12 with v' = v + w x t
            const double cx = w.y - w.z * py, cy = w.z * px - w.x, cz = w.x * py - w.y * px;
            flow_out[o] = sc * (vlev.x - vlev.z * px) + (cx - cz * px);
            flow_out[o + 1] = sc * (vlev.y - vlev.z * py) + (cy - cz * py);
        }
        if (d_out && i == 0) d_out[s] = d;
        const double ax = sc * (v.x - v.z * px), ay = sc * (v.y - v.z * py);     // gyro rate 0: v' = v (simulation.py:497)
        px += ax; py += ay;
        d += dstep;                                                              // simulation.py:499
    }
}

__global__ void r_tilde_kernel(const double* __restrict__ x, const double* __restrict__ u, int n, int ld,
                               double3 nrm, double3 v, double dist, double* __restrict__ r_out,
                               double* __restrict__ d_out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double X0 = x[ld * i], X1 = x[ld * i + 1], X2 = ld == 3 ? x[ld * i + 2] : 1.0;
    double U0 = u[ld * i], U1 = u[ld * i + 1], U2 = ld == 3 ? u[ld * i + 2] : 0.0;
    // v_cross = -(X x v), u_cross = X x U
    double vc0 = -(X1 * v.z - X2 * v.y), vc1 = -(X2 * v.x - X0 * v.z), vc2 = -(X0 * v.y - X1 * v.x);
    double uc0 = X1 * U2 - X2 * U1, uc1 = X2 * U0 - X0 * U2, uc2 = X0 * U1 - X1 * U0;
    double nv = sqrt(vc0 * vc0 + vc1 * vc1 + vc2 * vc2);
    double nu = sqrt(uc0 * uc0 + uc1 * uc1 + uc2 * uc2);
    double inv_u = 1.0 / nu;
    bool five_arg = (ld == 2);
    if (five_arg && nu * nv == 0.0) { r_out[i] = 1.0; d_out[i] = 1.0; return; }   // of_library.py:377-379
    double r = (vc0 * uc0 + vc1 * uc1 + vc2 * uc2) * inv_u / nv;
    double nx = X0 * nrm.x + X1 * nrm.y + X2 * nrm.z;
    if (nx < 0) r = -r;
    r_out[i] = r;
    double dd = nx * nv * inv_u;
    if (five_arg || dist > 0) dd /= dist;
    d_out[i] = dd;
}

__global__ void feasibility_kernel(const double* __restrict__ x, double3 v, const double* __restrict__ u, int n,
                                   double3 w, double3 t, double3 nrm, double* __restrict__ out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double px = x[2 * i], py = x[2 * i + 1];
    // a = v - w x t
    double a0 = v.x - (w.y * t.z - w.z * t.y), a1 = v.y - (w.z * t.x - w.x * t.z), a2 = v.z - (w.x * t.y - w.y * t.x);
    // f1 = X x a
    double f10 = py * a2 - a1, f11 = a0 - px * a2, f12 = px * a1 - py * a0;
    // b = u3 - w x X
    double b0 = u[2 * i] - (w.y - w.z * py), b1 = u[2 * i + 1] - (w.z * px - w.x), b2 = -(w.x * py - w.y * px);
    double f20 = py * b2 - b1, f21 = b0 - px * b2, f22 = px * b1 - py * b0;
    double n1 = sqrt(f10 * f10 + f11 * f11 + f12 * f12);
    double n2 = sqrt(f20 * f20 + f21 * f21 + f22 * f22);
    out[i] = (f10 * f20 + f11 * f21 + f12 * f22) / (n1 * n2);
    out[n + i] = n1 / n2 * (nrm.x * px + nrm.y * py + nrm.z);
}

inline double3 d3(const double* p) { return make_double3(p[0], p[1], p[2]); }

// The device inputs of a batched solve. x and u hold offsets[n_frames] rows.
struct BatchIn { const void *x, *u, *offsets, *d, *n3, *w3, *t3; int total; };

// Copies the offsets to the host (they size the point copies), checks them and stages x, u, offsets, d, n3 and the
// optional w3 and t3 (NULL: not staged). `who` prefixes the error messages.
int stage_batch(ofb_ctx* ctx, const char* who, const double* x, const double* u, const int* offsets, int n_frames,
                const double* d, const double* n3, const double* w3, const double* t3, BatchIn* in)
{
    std::vector<int> hoff(n_frames + 1);
    if (ofb_is_device_ptr(offsets)) {
        OFB_CUDA(cudaMemcpyAsync(hoff.data(), offsets, sizeof(int) * (n_frames + 1), cudaMemcpyDeviceToHost, ctx->stream));
        OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    } else memcpy(hoff.data(), offsets, sizeof(int) * (n_frames + 1));
    OFB_REQUIRE(hoff[0] >= 0, "%s: offsets[0] = %d is negative", who, hoff[0]);
    for (int f = 0; f < n_frames; ++f)
        OFB_REQUIRE(hoff[f + 1] >= hoff[f], "%s: offsets must be non-decreasing (offsets[%d] = %d > offsets[%d] = %d)", who, f, hoff[f],
                    f + 1, hoff[f + 1]);
    *in = BatchIn{};
    in->total = hoff[n_frames];
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, x, sizeof(double) * 2 * (size_t)in->total, &in->x));
    OFB_TRY(ofb_stage_in(ctx, SC_IN1, u, sizeof(double) * 2 * (size_t)in->total, &in->u));
    OFB_TRY(ofb_stage_in(ctx, SC_IN2, offsets, sizeof(int) * (n_frames + 1), &in->offsets));
    OFB_TRY(ofb_stage_in(ctx, SC_IN3, d, sizeof(double) * n_frames, &in->d));
    OFB_TRY(ofb_stage_in(ctx, SC_IN4, n3, sizeof(double) * 3 * n_frames, &in->n3));
    if (w3) OFB_TRY(ofb_stage_in(ctx, SC_IN5, w3, sizeof(double) * 3 * n_frames, &in->w3));
    if (t3) OFB_TRY(ofb_stage_in(ctx, SC_TMP0, t3, sizeof(double) * 3 * n_frames, &in->t3));
    return OFB_OK;
}

}  // namespace

extern "C" int ofb_solve_velocity_batched(ofb_ctx* ctx, int variant, const double* x, const double* u,
                                          const int* offsets, int n_frames,
                                          const double* d, const double* n3, const double* w3, const double* t3,
                                          double* v_out, double* res, int* rank, double* s_out)
{
    OFB_REQUIRE(ctx && x && u && offsets && d && n3 && w3 && v_out, "solve_velocity_batched: null argument");
    OFB_REQUIRE(variant >= 0 && variant <= 2, "solve_velocity: unknown variant %d", variant);
    OFB_REQUIRE(n_frames > 0, "solve_velocity_batched: n_frames must be positive");
    OFB_CUDA(cudaSetDevice(ctx->device));
    BatchIn in;
    OFB_TRY(stage_batch(ctx, "solve_velocity_batched", x, u, offsets, n_frames, d, n3, w3, t3, &in));
    OutStage o[4];
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, v_out, sizeof(double) * 3 * n_frames, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT1, res, sizeof(double) * n_frames, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT2, rank, sizeof(int) * n_frames, &o[2]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT3, s_out, sizeof(double) * 3 * n_frames, &o[3]));
    const PointsF64 ld{(const double*)in.x, (const double*)in.u, (const int*)in.offsets, 0};
    solve_velocity_kernel<<<n_frames, OFB_SOLVE_THREADS, 0, ctx->stream>>>(
        ld, variant, (const double*)in.d, (const double*)in.n3, (const double*)in.w3, (const double*)in.t3, 1, 3,
        (double*)o[0].dev, (double*)o[1].dev, (int*)o[2].dev, (double*)o[3].dev, nullptr, nullptr);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, o, 4);
}

extern "C" int ofb_solve_velocity_module(ofb_ctx* ctx, const double* x, const double* u, int n, int ld, const double* dist,
                                         const double n3[3], const double* v_prior,
                                         double v_out[3], double* res, int* rank, double s_out[3])
{
    OFB_REQUIRE(ctx && n3 && v_out, "solve_velocity_module: null argument");
    OFB_REQUIRE(ld == 2 || ld == 3, "solve_velocity_module: leading dimension must be 2 or 3");
    OFB_REQUIRE(n >= 0, "solve_velocity_module: negative point count");
    OFB_REQUIRE(n == 0 || (x && u), "solve_velocity_module: null points");
    OFB_REQUIRE(dist || v_prior, "solve_velocity_module: needs per-point distances or the prior velocity they derive from");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const double zero3[3] = {0.0, 0.0, 0.0};
    const void *dx = nullptr, *du = nullptr, *dd = nullptr, *dn, *dw, *dvp = nullptr;
    if (n) {
        OFB_TRY(ofb_stage_in(ctx, SC_IN0, x, sizeof(double) * ld * (size_t)n, &dx));
        OFB_TRY(ofb_stage_in(ctx, SC_IN1, u, sizeof(double) * ld * (size_t)n, &du));
        if (dist) OFB_TRY(ofb_stage_in(ctx, SC_IN2, dist, sizeof(double) * (size_t)n, &dd));
    }
    OFB_TRY(ofb_stage_in(ctx, SC_IN4, n3, sizeof(double) * 3, &dn));
    OFB_TRY(ofb_stage_in(ctx, SC_IN5, zero3, sizeof(double) * 3, &dw));       // (pageable source: the copy is staged at once)
    if (v_prior) OFB_TRY(ofb_stage_in(ctx, SC_TMP0, v_prior, sizeof(double) * 3, &dvp));
    OutStage o[4];
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, v_out, sizeof(double) * 3, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT1, res, sizeof(double), &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT2, rank, sizeof(int), &o[2]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT3, s_out, sizeof(double) * 3, &o[3]));
    PointsF64 ldr{(const double*)dx, (const double*)du, nullptr, n};
    ldr.ld = ld; ldr.dists = (const double*)dd;
    solve_velocity_kernel<<<1, OFB_SOLVE_THREADS, 0, ctx->stream>>>(
        ldr, OFB_VARIANT_MODULE, nullptr, (const double*)dn, (const double*)dw, nullptr, 1, 3,
        (double*)o[0].dev, (double*)o[1].dev, (int*)o[2].dev, (double*)o[3].dev, nullptr, (const double*)dvp);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, o, 4);
}

extern "C" int ofb_solve_velocity(ofb_ctx* ctx, int variant, const double* x, const double* u, int n, double d,
                                  const double n3[3], const double w3[3], const double t3[3],
                                  double v_out[3], double* res, int* rank, double s_out[3])
{
    OFB_REQUIRE(ctx && n3 && w3 && v_out, "solve_velocity: null argument");
    OFB_REQUIRE(n >= 0, "solve_velocity: negative point count");
    OFB_REQUIRE(n == 0 || (x && u), "solve_velocity: null points");
    int offsets[2] = {0, n};
    double dummy[2] = {0, 0};
    return ofb_solve_velocity_batched(ctx, variant, n ? x : dummy, n ? u : dummy, offsets, 1, &d, n3, w3, t3,
                                      v_out, res, rank, s_out);
}

extern "C" int ofb_solve_ego_motion_batched(ofb_ctx* ctx, int variant, const double* x, const double* u, const int* offsets,
                                            int n_frames, const double* d, const double* n3, const double* t3, ofb_ego_result* out)
{
    OFB_REQUIRE(ctx && x && u && offsets && d && n3 && out, "solve_ego_motion_batched: null argument");
    OFB_REQUIRE(variant >= 0 && variant <= 2, "solve_ego_motion: unknown variant %d (MODULE has no gyro term to estimate)", variant);
    OFB_REQUIRE(n_frames > 0, "solve_ego_motion_batched: n_frames must be positive");
    OFB_CUDA(cudaSetDevice(ctx->device));
    BatchIn in;
    OFB_TRY(stage_batch(ctx, "solve_ego_motion_batched", x, u, offsets, n_frames, d, n3, nullptr, t3, &in));
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, out, sizeof(ofb_ego_result) * n_frames, &o));
    const PointsF64 ld{(const double*)in.x, (const double*)in.u, (const int*)in.offsets, 0};
    solve_ego_kernel<<<n_frames, OFB_SOLVE_THREADS, 0, ctx->stream>>>(ld, variant, (const double*)in.d, (const double*)in.n3,
                                                                       (const double*)in.t3, (ofb_ego_result*)o.dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, &o, 1);
}

extern "C" int ofb_solve_ego_motion(ofb_ctx* ctx, int variant, const double* x, const double* u, int n, double d,
                                    const double n3[3], const double t3[3], ofb_ego_result* out)
{
    OFB_REQUIRE(ctx && n3 && out, "solve_ego_motion: null argument");
    OFB_REQUIRE(n >= 0, "solve_ego_motion: negative point count");
    OFB_REQUIRE(n == 0 || (x && u), "solve_ego_motion: null points");
    int offsets[2] = {0, n};
    double dummy[2] = {0, 0};
    return ofb_solve_ego_motion_batched(ctx, variant, n ? x : dummy, n ? u : dummy, offsets, 1, &d, n3, t3, out);
}

extern "C" int ofb_solve_velocity_robust_batched(ofb_ctx* ctx, int variant, const double* x, const double* u, const int* offsets,
                                                 int n_frames, const double* d, const double* n3, const double* w3, const double* t3,
                                                 const ofb_robust_cfg* cfg, ofb_robust_result* out, double* weights_out)
{
    OFB_REQUIRE(ctx && x && u && offsets && d && n3 && w3 && out, "solve_velocity_robust_batched: null argument");
    OFB_REQUIRE(variant >= 0 && variant <= 2, "solve_velocity_robust: unknown variant %d (MODULE is not supported)", variant);
    OFB_TRY(ofb_robust_check(cfg, "solve_velocity_robust"));
    OFB_REQUIRE(n_frames > 0, "solve_velocity_robust_batched: n_frames must be positive");
    OFB_CUDA(cudaSetDevice(ctx->device));
    BatchIn in;
    OFB_TRY(stage_batch(ctx, "solve_velocity_robust_batched", x, u, offsets, n_frames, d, n3, w3, t3, &in));
    OutStage o[2];
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, out, sizeof(ofb_robust_result) * n_frames, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT1, weights_out, sizeof(double) * (size_t)in.total, &o[1]));
    if (o[1].dev) OFB_CUDA(cudaMemsetAsync(o[1].dev, 0, sizeof(double) * (size_t)in.total, ctx->stream));   // rows in no frame
    const PointsF64 ld{(const double*)in.x, (const double*)in.u, (const int*)in.offsets, 0};
    solve_robust_kernel<<<n_frames, OFB_SOLVE_THREADS, 0, ctx->stream>>>(ld, variant, (const double*)in.d, (const double*)in.n3,
                                                                          (const double*)in.w3, (const double*)in.t3, *cfg,
                                                                          (ofb_robust_result*)o[0].dev, (double*)o[1].dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, o, 2);
}

extern "C" int ofb_solve_velocity_robust(ofb_ctx* ctx, int variant, const double* x, const double* u, int n, double d,
                                         const double n3[3], const double w3[3], const double t3[3], const ofb_robust_cfg* cfg,
                                         ofb_robust_result* out, double* weights_out)
{
    OFB_REQUIRE(ctx && n3 && w3 && out, "solve_velocity_robust: null argument");
    OFB_REQUIRE(n >= 0, "solve_velocity_robust: negative point count");
    OFB_REQUIRE(n == 0 || (x && u), "solve_velocity_robust: null points");
    int offsets[2] = {0, n};
    double dummy[2] = {0, 0};
    return ofb_solve_velocity_robust_batched(ctx, variant, n ? x : dummy, n ? u : dummy, offsets, 1, &d, n3, w3, t3, cfg, out,
                                             n ? weights_out : nullptr);
}

extern "C" int ofb_generate_flow(ofb_ctx* ctx, const double* x, int n, const double v3[3], const double w3[3],
                                 double d, const double n3[3], const double* t3, double* u_out)
{
    OFB_REQUIRE(ctx && v3 && w3 && n3 && u_out, "generate_flow: null argument");
    OFB_REQUIRE(n >= 0, "generate_flow: negative point count");
    if (n == 0) return OFB_OK;
    OFB_REQUIRE(x, "generate_flow: null points");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void* dx;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, x, sizeof(double) * 2 * (size_t)n, &dx));
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, u_out, sizeof(double) * 2 * (size_t)n, &o));
    double3 v = d3(v3), w = d3(w3);
    if (t3) {   // v' = v + w x t   (simulation.py:9)
        v.x += w.y * t3[2] - w.z * t3[1];
        v.y += w.z * t3[0] - w.x * t3[2];
        v.z += w.x * t3[1] - w.y * t3[0];
    }
    generate_flow_kernel<<<ofb_div_up(n, 256), 256, 0, ctx->stream>>>((const double*)dx, n, v, w, d, d3(n3), (double*)o.dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, &o, 1);
}

extern "C" int ofb_advect_points(ofb_ctx* ctx, const double* x0, int n, const double v3[3], const double w3[3], double d0,
                                 const double n3[3], const double t3[3], int k, double* pos_out, double* flow_out,
                                 double* d_out)
{
    OFB_REQUIRE(ctx && v3 && w3 && n3 && pos_out, "advect_points: null argument");
    OFB_REQUIRE(n >= 0 && k >= 1, "advect_points: bad point or step count");
    if (n == 0) return OFB_OK;
    OFB_REQUIRE(x0, "advect_points: null points");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void* dx;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, x0, sizeof(double) * 2 * (size_t)n, &dx));
    OutStage o[3];
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, pos_out, sizeof(double) * 2 * (size_t)n * k, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT1, flow_out, sizeof(double) * 2 * (size_t)n * k, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT2, d_out, sizeof(double) * (size_t)k, &o[2]));
    double3 v = d3(v3), w = d3(w3), vl = v;
    if (t3) { vl.x += w.y * t3[2] - w.z * t3[1]; vl.y += w.z * t3[0] - w.x * t3[2]; vl.z += w.x * t3[1] - w.y * t3[0]; }
    const double dstep = v3[0] * n3[0] + v3[1] * n3[1] + v3[2] * n3[2];
    advect_points_kernel<<<ofb_div_up(n, 128), 128, 0, ctx->stream>>>((const double*)dx, n, v, vl, w, d0, dstep, d3(n3), k,
                                                                      (double*)o[0].dev, (double*)o[1].dev, (double*)o[2].dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, o, 3);
}

extern "C" int ofb_r_tilde(ofb_ctx* ctx, const double* x, const double* u, int n, int ld, const double n3[3],
                           const double v3[3], double dist, double* r_out, double* d_out)
{
    OFB_REQUIRE(ctx && n3 && v3 && r_out && d_out, "r_tilde: null argument");
    OFB_REQUIRE(ld == 2 || ld == 3, "r_tilde: leading dimension must be 2 or 3");
    OFB_REQUIRE(n >= 0, "r_tilde: negative point count");
    if (n == 0) return OFB_OK;
    OFB_REQUIRE(x && u, "r_tilde: null points");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void *dx, *du;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, x, sizeof(double) * ld * (size_t)n, &dx));
    OFB_TRY(ofb_stage_in(ctx, SC_IN1, u, sizeof(double) * ld * (size_t)n, &du));
    OutStage o[2];
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, r_out, sizeof(double) * (size_t)n, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT1, d_out, sizeof(double) * (size_t)n, &o[1]));
    r_tilde_kernel<<<ofb_div_up(n, 256), 256, 0, ctx->stream>>>((const double*)dx, (const double*)du, n, ld, d3(n3),
                                                                d3(v3), dist, (double*)o[0].dev, (double*)o[1].dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, o, 2);
}

extern "C" int ofb_feasibility(ofb_ctx* ctx, const double* x, const double* v3, const double* u, int n,
                               const double w3[3], const double t3[3], const double n3[3], double* out)
{
    OFB_REQUIRE(ctx && v3 && w3 && t3 && n3 && out, "feasibility: null argument");
    OFB_REQUIRE(n >= 0, "feasibility: negative point count");
    if (n == 0) return OFB_OK;
    OFB_REQUIRE(x && u, "feasibility: null points");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void *dx, *du;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, x, sizeof(double) * 2 * (size_t)n, &dx));
    OFB_TRY(ofb_stage_in(ctx, SC_IN1, u, sizeof(double) * 2 * (size_t)n, &du));
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, out, sizeof(double) * 2 * (size_t)n, &o));
    feasibility_kernel<<<ofb_div_up(n, 256), 256, 0, ctx->stream>>>((const double*)dx, d3(v3), (const double*)du, n,
                                                                    d3(w3), d3(t3), d3(n3), (double*)o.dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, &o, 1);
}
