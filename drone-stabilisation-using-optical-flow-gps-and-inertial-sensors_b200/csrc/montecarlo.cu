// montecarlo.cu -- stage 5: Monte-Carlo error propagation of the velocity solve.
//
// Replaces of_simulation (numerical_simulation/simulation.py:36-66), feas_simulation
// (simulation.py:70-104), the per-step np.mean/np.std of the sweep drivers (e.g. simulation.py:183-202)
// and the pieces of overlap (simulation.py:124-136) that touch bulk data.
//
// Mapping: one thread = one trial (all points of the trial stay in registers as running sums of the
// 3x3 normal equations), blockIdx.y = sweep step, trials strided over blockIdx.x. Noise comes from
// Philox4x32-10 keyed by the seed with counter (trial id, draw block, step id): block 0 = gyro(3)+height,
// block 1 = lever arm(3) [+ angle 1 for feas], block 2 = forward velocity(3)+angle 2 (feas only; the
// normal-vector noise of of_simulation is drawn-and-discarded by the reference, simulation.py:45-46, so
// it is never generated), block 3+j = point j: flow(2)+position(2). Any sharding of the trial range
// therefore reproduces the same union of trials. Statistics are fp64 sums of (v - v_true), their
// squares and R; per-block partials are reduced in a fixed order so a given launch shape is
// bit-reproducible.
#include "common.cuh"
#include "math3.cuh"

namespace {

constexpr int MC_THREADS = 128;
constexpr int MC_NSTAT = 8;     // n, dv(3), dv2(3), R

template <class T> struct McParams {
    T v[3], w[3], n[3], nh[3], t[3];
    T h, sw, st, sh, sf, sp;
    double baseR;
    double vtrue[3];
    int N, pos_offset;
};

template <class T>
OFB_HD void mc_normals4(uint32_t tlo, uint32_t thi, uint32_t blk, uint32_t step, uint2 key,
                                            T& z0, T& z1, T& z2, T& z3)
{
    uint4 r = ofb_philox4x32_10(make_uint4(tlo, thi, blk, step), key);
    ofb_box_muller(r.x, r.y, z0, z1);
    ofb_box_muller(r.z, r.w, z2, z3);
}

template <class T>
__host__ __device__ void mc_load_params(const ofb_mc_step& s, McParams<T>& p)
{
    double nn = sqrt(s.n[0] * s.n[0] + s.n[1] * s.n[1] + s.n[2] * s.n[2]);
    for (int k = 0; k < 3; ++k) {
        p.v[k] = (T)s.v[k]; p.w[k] = (T)s.w[k]; p.n[k] = (T)s.n[k]; p.nh[k] = (T)(s.n[k] / nn); p.t[k] = (T)s.t[k];
        p.vtrue[k] = s.v[k];
    }
    p.h = (T)s.height; p.sw = (T)s.ang_vel_sig; p.st = (T)s.translation_sig; p.sh = (T)s.height_sig;
    p.sf = (T)s.flow_sig; p.sp = (T)s.position_sig;
    double nw = sqrt(s.w[0] * s.w[0] + s.w[1] * s.w[1] + s.w[2] * s.w[2]);
    double nt = sqrt(s.t[0] * s.t[0] + s.t[1] * s.t[1] + s.t[2] * s.t[2]);
    // simulation.py:64: |w| sigma_t + sigma_w |t| + sigma_w sigma_t
    p.baseR = nw * s.translation_sig + s.ang_vel_sig * nt + s.ang_vel_sig * s.translation_sig;
    p.N = s.n_points; p.pos_offset = s.pos_offset;
}

// Per-point constants of the analytic error bound (simulation.py:57-58 evaluated at the TRUE position, which does not
// depend on the trial): sconst[2j] = n . x_j, sconst[2j+1] = (n/|n| - n) . x_j. Filled once per step.
template <class T>
OFB_HD void mc_point_consts(const McParams<T>& P, const T* __restrict__ spos, int j, T* __restrict__ sconst)
{
    const T dn0 = P.nh[0] - P.n[0], dn1 = P.nh[1] - P.n[1], dn2 = P.nh[2] - P.n[2];
    const T px0 = spos[2 * j], py0 = spos[2 * j + 1];
    sconst[2 * j] = P.n[0] * px0 + P.n[1] * py0 + P.n[2];
    sconst[2 * j + 1] = dn0 * px0 + dn1 * py0 + dn2;
}

// One trial of of_simulation (simulation.py:39-64).
// WANT_R = false skips the analytic error bound R (simulation.py:56-64) for callers that only consume v_obs
// (every saved sweep except sim_err_vs_num); R_out is then 0.
template <class T, bool WANT_R = true>
OFB_HD void mc_trial(const McParams<T>& P, const T* __restrict__ spos, const T* __restrict__ sflow,
                                         const T* __restrict__ sconst, uint64_t trial, uint2 key, uint32_t step,
                                         double v_out[3], double& R_out)
{
    uint32_t tlo = (uint32_t)trial, thi = (uint32_t)(trial >> 32);
    T z0, z1, z2, z3;
    mc_normals4<T>(tlo, thi, 0u, step, key, z0, z1, z2, z3);
    T dw0 = P.sw * z0, dw1 = P.sw * z1, dw2 = P.sw * z2;
    T w0 = P.w[0] + dw0, w1 = P.w[1] + dw1, w2 = P.w[2] + dw2;
    T dh = P.sh * z3;
    mc_normals4<T>(tlo, thi, 1u, step, key, z0, z1, z2, z3);
    T t0 = P.t[0] + P.st * z0, t1 = P.t[1] + P.st * z1, t2 = P.t[2] + P.st * z2;
    T dh_rel = dh / P.h;

    T m0 = 0, m1 = 0, m2 = 0, m3 = 0, m4 = 0, m5 = 0, g0 = 0, g1 = 0, g2 = 0, accR = 0;
#pragma unroll 2
    for (int j = 0; j < P.N; ++j) {
        mc_normals4<T>(tlo, thi, 3u + (uint32_t)j, step, key, z0, z1, z2, z3);
        T dfx = P.sf * z0, dfy = P.sf * z1, dpx = P.sp * z2, dpy = P.sp * z3;
        T px0 = spos[2 * j], py0 = spos[2 * j + 1];
        T px = px0 + dpx, py = py0 + dpy;
        T ux = sflow[2 * j] + dfx, uy = sflow[2 * j + 1] + dfy;
        // solve_lgs variant SIM (simulation.py:19-23)
        T nx = P.nh[0] * px + P.nh[1] * py + P.nh[2];
        T ax = py * w2 - w1, ay = w0 - px * w2, az = px * w1 - py * w0;
        T cx = ux + ax, cy = uy + ay, cz = az;
        T bx = py * cz - cy, by = cx - px * cz, bz = px * cy - py * cx;
        T q2 = nx * nx, xx = px * px, yy = py * py;
        m0 += q2 * (yy + (T)1); m1 -= q2 * (px * py); m2 -= q2 * px;
        m3 += q2 * (xx + (T)1); m4 -= q2 * py;        m5 += q2 * (xx + yy);
        g0 -= nx * (py * bz - by); g1 -= nx * (bx - px * bz); g2 -= nx * (px * by - py * bx);
        if (WANT_R) {
            // analytic error bound, simulation.py:57-63 (xp = true position)
            // (n . x and dn . x of the TRUE position do not depend on the trial: sconst, filled once per step)
            T v_e = dh_rel * sconst[2 * j] + sconst[2 * j + 1] + (P.n[0] * dpx + P.n[1] * dpy);
            T e0 = dfx + (dpy * P.w[2]) + (py0 * dw2 - dw1) + dpx;
            T e1 = dfy + (-dpx * P.w[2]) + (dw0 - px0 * dw2) + dpy;
            T e2 = (dpx * P.w[1] - dpy * P.w[0]) + (px0 * dw1 - py0 * dw0);
            T r0 = v_e * P.v[0] + P.h * e0, r1 = v_e * P.v[1] + P.h * e1, r2 = v_e * P.v[2] + P.h * e2;
            T qx = py0 * r2 - r1, qy = r0 - px0 * r2, qz = px0 * r1 - py0 * r0;
            accR += qx * qx + qy * qy + qz * qz;
        }
    }
    double M[6] = {(double)m0, (double)m1, (double)m2, (double)m3, (double)m4, (double)m5};
    double g[3] = {(double)g0, (double)g1, (double)g2};
    double v[3];
    ofb_solve_sym3(M, g, v);
    double he = (double)P.h + (double)dh;
    double W0 = (double)w0, W1 = (double)w1, W2 = (double)w2, T0 = (double)t0, T1 = (double)t1, T2 = (double)t2;
    v_out[0] = v[0] * he - (W1 * T2 - W2 * T1);
    v_out[1] = v[1] * he - (W2 * T0 - W0 * T2);
    v_out[2] = v[2] * he - (W0 * T1 - W1 * T0);
    if (WANT_R) {
        double lmin = ofb_min_eig_sym3(M);
        R_out = sqrt((double)accR / lmin) + P.baseR;
    } else R_out = 0.0;
}

// Register budget left to the compiler (128 for fp32): forcing 5 CTAs/SM (96 registers) was measured slower
// (2.19e9 vs 2.40e9 trials/s) -- the spills cost more than the extra warps gain.
template <class T, bool WANT_R>
__global__ void __launch_bounds__(MC_THREADS)
mc_sweep_kernel(const ofb_mc_step* __restrict__ steps, int step_id_base, const double* __restrict__ pos,
                const double* __restrict__ flow, uint64_t trial_begin, uint64_t trials, uint2 key,
                double* __restrict__ partials, double* __restrict__ v_dump, double* __restrict__ R_dump)
{
    __shared__ McParams<T> P;
    __shared__ T spos[2 * OFB_MC_MAX_POINTS];
    __shared__ T sflow[2 * OFB_MC_MAX_POINTS];
    __shared__ T sconst[2 * OFB_MC_MAX_POINTS];     // per point: n . x, (n/|n| - n) . x of the true position (error bound R)
    __shared__ double red[MC_NSTAT][MC_THREADS / 32];
    int step = blockIdx.y;
    if (threadIdx.x == 0) mc_load_params<T>(steps[step], P);
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * P.N; i += blockDim.x) {
        spos[i] = (T)pos[2 * (size_t)P.pos_offset + i];
        sflow[i] = (T)flow[2 * (size_t)P.pos_offset + i];
    }
    __syncthreads();
    if (WANT_R) {
        for (int j = threadIdx.x; j < P.N; j += blockDim.x) mc_point_consts<T>(P, spos, j, sconst);
        __syncthreads();
    }
    double acc[MC_NSTAT] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < trials; k += stride) {
        double v[3], R;
        mc_trial<T, WANT_R>(P, spos, sflow, sconst, trial_begin + k, key, (uint32_t)(step_id_base + step), v, R);
        if (v_dump) {
            double* o = v_dump + ((size_t)step * trials + k) * 3;
            o[0] = v[0]; o[1] = v[1]; o[2] = v[2];
        }
        if (R_dump) R_dump[(size_t)step * trials + k] = R;
        double d0 = v[0] - P.vtrue[0], d1 = v[1] - P.vtrue[1], d2 = v[2] - P.vtrue[2];
        acc[0] += 1.0;
        acc[1] += d0; acc[2] += d1; acc[3] += d2;
        acc[4] += d0 * d0; acc[5] += d1 * d1; acc[6] += d2 * d2;
        acc[7] += R;
    }
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int s = 0; s < MC_NSTAT; ++s) {
        double x = acc[s];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) red[s][warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < MC_NSTAT) {
        double x = 0;
        for (int w = 0; w < MC_THREADS / 32; ++w) x += red[threadIdx.x][w];
        partials[((size_t)step * gridDim.x + blockIdx.x) * MC_NSTAT + threadIdx.x] = x;
    }
}

// fixed-order reduction of the per-block partials of one step (one warp per step)
__global__ void mc_finalize_kernel(const double* __restrict__ partials, int blocks_per_step, ofb_mc_sums* __restrict__ out)
{
    int step = blockIdx.x, lane = threadIdx.x;
    double acc[MC_NSTAT] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int b = lane; b < blocks_per_step; b += 32)
#pragma unroll
        for (int s = 0; s < MC_NSTAT; ++s) acc[s] += partials[((size_t)step * blocks_per_step + b) * MC_NSTAT + s];
#pragma unroll
    for (int s = 0; s < MC_NSTAT; ++s)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[s] += __shfl_xor_sync(0xffffffffu, acc[s], o);
    if (lane == 0) {
        ofb_mc_sums r;
        r.n = acc[0];
        r.sum_dv[0] = acc[1]; r.sum_dv[1] = acc[2]; r.sum_dv[2] = acc[3];
        r.sum_dv2[0] = acc[4]; r.sum_dv2[1] = acc[5]; r.sum_dv2[2] = acc[6];
        r.sum_R = acc[7];
        out[step] = r;
    }
}

// ---- feas_simulation (simulation.py:70-104), fp64 -------------------------------------------
struct FeasParams {
    double w[3], n[3], t[3], tv[3];
    double h, sw, st, sh, sf, sp, sn, sv;
    int N, pos_offset;
};

struct FeasNoise { double w[3], t[3], he, ve[3], ne[3]; };

__device__ __forceinline__ void feas_point(const FeasParams& P, const double* spos, const double* sflow, uint32_t tlo,
                                           uint32_t thi, int j, uint32_t step, uint2 key, double& px, double& py,
                                           double& ux, double& uy)
{
    double z0, z1, z2, z3;
    mc_normals4<double>(tlo, thi, 3u + (uint32_t)j, step, key, z0, z1, z2, z3);
    px = spos[2 * j] + P.sp * z2; py = spos[2 * j + 1] + P.sp * z3;
    ux = sflow[2 * j] + P.sf * z0; uy = sflow[2 * j + 1] + P.sf * z1;
}

__device__ __forceinline__ void feas_pair(double px, double py, double ux, double uy, const double v[3],
                                          const double w[3], const double t[3], const double ne[3], double& par,
                                          double& len)
{   // simulation.py:111-118
    double a0 = v[0] - (w[1] * t[2] - w[2] * t[1]), a1 = v[1] - (w[2] * t[0] - w[0] * t[2]),
           a2 = v[2] - (w[0] * t[1] - w[1] * t[0]);
    double f10 = py * a2 - a1, f11 = a0 - px * a2, f12 = px * a1 - py * a0;
    double b0 = ux - (w[1] - w[2] * py), b1 = uy - (w[2] * px - w[0]), b2 = -(w[0] * py - w[1] * px);
    double f20 = py * b2 - b1, f21 = b0 - px * b2, f22 = px * b1 - py * b0;
    double n1 = sqrt(f10 * f10 + f11 * f11 + f12 * f12), n2 = sqrt(f20 * f20 + f21 * f21 + f22 * f22);
    par = (f10 * f20 + f11 * f21 + f12 * f22) / (n1 * n2);
    len = n1 / n2 * (ne[0] * px + ne[1] * py + ne[2]);
}

__global__ void __launch_bounds__(MC_THREADS)
mc_feas_kernel(const ofb_mc_step* __restrict__ stepp, int step_id, const double* __restrict__ pos,
               const double* __restrict__ flow, uint64_t trial_begin, uint64_t trials, uint2 key,
               double* __restrict__ sums /* 6*N */)
{
    __shared__ FeasParams P;
    __shared__ double spos[2 * OFB_MC_MAX_POINTS];
    __shared__ double sflow[2 * OFB_MC_MAX_POINTS];
    __shared__ double ssum[6 * OFB_MC_MAX_POINTS];
    if (threadIdx.x == 0) {
        const ofb_mc_step& s = *stepp;
        for (int k = 0; k < 3; ++k) { P.w[k] = s.w[k]; P.n[k] = s.n[k]; P.t[k] = s.t[k]; P.tv[k] = s.true_vel[k]; }
        P.h = s.height; P.sw = s.ang_vel_sig; P.st = s.translation_sig; P.sh = s.height_sig; P.sf = s.flow_sig;
        P.sp = s.position_sig; P.sn = s.normal_sig; P.sv = s.velocity_sig; P.N = s.n_points; P.pos_offset = s.pos_offset;
    }
    __syncthreads();
    int N = P.N;
    for (int i = threadIdx.x; i < 2 * N; i += blockDim.x) {
        spos[i] = pos[2 * (size_t)P.pos_offset + i];
        sflow[i] = flow[2 * (size_t)P.pos_offset + i];
    }
    for (int i = threadIdx.x; i < 6 * N; i += blockDim.x) ssum[i] = 0.0;
    __syncthreads();
    uint32_t step = (uint32_t)step_id;
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < trials; k += stride) {
        uint64_t trial = trial_begin + k;
        uint32_t tlo = (uint32_t)trial, thi = (uint32_t)(trial >> 32);
        double z0, z1, z2, z3;
        double w[3], t[3], ve[3], ne[3];
        mc_normals4<double>(tlo, thi, 0u, step, key, z0, z1, z2, z3);
        w[0] = P.w[0] + P.sw * z0; w[1] = P.w[1] + P.sw * z1; w[2] = P.w[2] + P.sw * z2;
        double he = P.h + P.sh * z3;
        mc_normals4<double>(tlo, thi, 1u, step, key, z0, z1, z2, z3);
        t[0] = P.t[0] + P.st * z0; t[1] = P.t[1] + P.st * z1; t[2] = P.t[2] + P.st * z2;
        double a1 = P.sn * (P.sn * z3);          // simulation.py:87: normal_sig*N(0,normal_sig)
        mc_normals4<double>(tlo, thi, 2u, step, key, z0, z1, z2, z3);
        ve[0] = P.tv[0] + P.sv * z0; ve[1] = P.tv[1] + P.sv * z1; ve[2] = P.tv[2] + P.sv * z2;
        double a2 = P.sn * (P.sn * z3);          // simulation.py:88
        {   // simulation.py:89: Ry(a2) Rx(a1) n
            double c1 = cos(a1), s1 = sin(a1), c2 = cos(a2), s2 = sin(a2);
            double r0 = P.n[0], r1 = c1 * P.n[1] - s1 * P.n[2], r2 = s1 * P.n[1] + c1 * P.n[2];
            ne[0] = c2 * r0 + s2 * r2; ne[1] = r1; ne[2] = -s2 * r0 + c2 * r2;
        }
        // pass 1: normal equations, variant SIM
        double M[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
        for (int j = 0; j < N; ++j) {
            double px, py, ux, uy;
            feas_point(P, spos, sflow, tlo, thi, j, step, key, px, py, ux, uy);
            double nx = ne[0] * px + ne[1] * py + ne[2];
            double ax = py * w[2] - w[1], ay = w[0] - px * w[2], az = px * w[1] - py * w[0];
            double cx = ux + ax, cy = uy + ay, cz = az;
            double bx = py * cz - cy, by = cx - px * cz, bz = px * cy - py * cx;
            double q2 = nx * nx, xx = px * px, yy = py * py;
            M[0] += q2 * (yy + 1.0); M[1] -= q2 * px * py; M[2] -= q2 * px;
            M[3] += q2 * (xx + 1.0); M[4] -= q2 * py;      M[5] += q2 * (xx + yy);
            g[0] -= nx * (py * bz - by); g[1] -= nx * (bx - px * bz); g[2] -= nx * (px * by - py * bx);
        }
        double v[3];
        ofb_solve_sym3(M, g, v);
        v[0] = v[0] * he - (w[1] * t[2] - w[2] * t[1]);
        v[1] = v[1] * he - (w[2] * t[0] - w[0] * t[2]);
        v[2] = v[2] * he - (w[0] * t[1] - w[1] * t[0]);
        // pass 2: regenerate each point's noise, emit the six per-point quantities. Lanes walk the
        // points in rotated order so the shared-memory atomics of a warp hit distinct addresses.
        int rot = threadIdx.x & 31;
        for (int jj = 0; jj < N; ++jj) {
            int j = jj + rot; if (j >= N) j -= N; if (j >= N) j %= N;
            double px, py, ux, uy;
            feas_point(P, spos, sflow, tlo, thi, j, step, key, px, py, ux, uy);
            double bpar, bdist, fpar, fdist;
            feas_pair(px, py, ux, uy, v, w, t, ne, bpar, bdist);
            feas_pair(px, py, ux, uy, ve, w, t, ne, fpar, fdist);
            double nx = ne[0] * px + ne[1] * py + ne[2];
            double ax = py * w[2] - w[1], ay = w[0] - px * w[2], az = px * w[1] - py * w[0];
            double cx = ux + ax, cy = uy + ay, cz = az;
            double bx = py * cz - cy, by = cx - px * cz, bz = px * cy - py * cx;
            // simulation.py:102-103: ||(n.X)[X]x v - b_i||
            double rb0 = nx * (py * v[2] - v[1]) - bx, rb1 = nx * (v[0] - px * v[2]) - by, rb2 = nx * (px * v[1] - py * v[0]) - bz;
            double rf0 = nx * (py * ve[2] - ve[1]) - bx, rf1 = nx * (ve[0] - px * ve[2]) - by, rf2 = nx * (px * ve[1] - py * ve[0]) - bz;
            atomicAdd(&ssum[0 * N + j], bpar);
            atomicAdd(&ssum[1 * N + j], bdist);
            atomicAdd(&ssum[2 * N + j], fpar);
            atomicAdd(&ssum[3 * N + j], fdist);
            atomicAdd(&ssum[4 * N + j], sqrt(rb0 * rb0 + rb1 * rb1 + rb2 * rb2));
            atomicAdd(&ssum[5 * N + j], sqrt(rf0 * rf0 + rf1 * rf1 + rf2 * rf2));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 6 * N; i += blockDim.x) atomicAdd(&sums[i], ssum[i]);
}

// ---- overlap helpers --------------------------------------------------------------------------
__global__ void minmax_kernel(const double* __restrict__ data, size_t n, double* __restrict__ part /* 2*gridDim.x */)
{
    double lo = INFINITY, hi = -INFINITY;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        double v = data[i]; lo = fmin(lo, v); hi = fmax(hi, v);
    }
    __shared__ double slo[8], shi[8];
    for (int o = 16; o > 0; o >>= 1) { lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o)); }
    if ((threadIdx.x & 31) == 0) { slo[threadIdx.x >> 5] = lo; shi[threadIdx.x >> 5] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { lo = fmin(lo, slo[w]); hi = fmax(hi, shi[w]); }
        part[2 * blockIdx.x] = lo; part[2 * blockIdx.x + 1] = hi;
    }
}
__global__ void minmax_final_kernel(double* part, int nblocks)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double lo = part[0], hi = part[1];
        for (int b = 1; b < nblocks; ++b) { lo = fmin(lo, part[2 * b]); hi = fmax(hi, part[2 * b + 1]); }
        part[0] = lo; part[1] = hi;
    }
}
// Edge k of numpy.linspace(lo, hi, bins + 1), bit for bit: k * ((hi - lo) / bins) + lo, rounded after the product and
// after the sum (the intrinsics keep nvcc from contracting the two into one FMA); the last edge is hi itself.
__device__ __forceinline__ double linspace_edge(double lo, double hi, double step, int k, int bins)
{
    return k == bins ? hi : __dadd_rn(__dmul_rn((double)k, step), lo);
}

// numpy.histogram semantics for uniform bins over [lo,hi]: bin = floor((x-lo)/(hi-lo)*bins), x==hi
// falls in the last bin, values outside are dropped; the computed index is then corrected against the
// actual linspace edges the way numpy does, so a sample on an edge lands where numpy puts it.
__global__ void histogram_kernel(const double* __restrict__ data, size_t n, double lo, double hi, int bins,
                                 unsigned long long* __restrict__ counts)
{
    extern __shared__ unsigned int sh[];
    for (int i = threadIdx.x; i < bins; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    double norm = (double)bins / (hi - lo);
    double step = (hi - lo) / bins;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        double v = data[i];
        if (!(v >= lo && v <= hi)) continue;
        int b = (int)((v - lo) * norm);
        if (b >= bins) b = bins - 1;
        double e0 = linspace_edge(lo, hi, step, b, bins), e1 = linspace_edge(lo, hi, step, b + 1, bins);
        if (v < e0 && b > 0) --b;
        else if (v >= e1 && b + 1 < bins) ++b;
        atomicAdd(&sh[b], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += blockDim.x)
        if (sh[i]) atomicAdd(&counts[i], (unsigned long long)sh[i]);
}

int validate_steps(const ofb_mc_step* steps, int n_steps, int total_points)
{
    for (int i = 0; i < n_steps; ++i) {
        // one point leaves the 3x3 normal matrix singular (its own ray is in the null space): at least two
        OFB_REQUIRE(steps[i].n_points >= 2 && steps[i].n_points <= OFB_MC_MAX_POINTS,
                    "mc: step %d has %d points (2..%d supported: one point does not determine the velocity)", i,
                    steps[i].n_points, OFB_MC_MAX_POINTS);
        OFB_REQUIRE(steps[i].pos_offset >= 0 && steps[i].pos_offset + steps[i].n_points <= total_points,
                    "mc: step %d point range outside pos/true_flow", i);
        OFB_REQUIRE(steps[i].height != 0.0, "mc: step %d has zero height", i);
    }
    return OFB_OK;
}

}  // namespace

extern "C" int ofb_mc_sweep(ofb_ctx* ctx, const ofb_mc_step* steps, int n_steps, int step_id_base,
                            const double* pos, const double* true_flow, int total_points,
                            uint64_t trial_begin, uint64_t trials, uint64_t seed, int precision,
                            ofb_mc_sums* sums_out, double* v_dump, double* R_dump)
{
    OFB_REQUIRE(ctx && steps && pos && true_flow && sums_out, "mc_sweep: null argument");
    OFB_REQUIRE(n_steps > 0 && n_steps <= 65535, "mc_sweep: n_steps must be in 1..65535");
    OFB_REQUIRE(trials > 0, "mc_sweep: iterations must be a positive number");
    OFB_REQUIRE(precision >= 0 && precision <= 3, "mc_sweep: precision must be 0 (fp32) or 1 (fp64), +2 to skip R");
    OFB_REQUIRE(!ofb_is_device_ptr(steps), "mc_sweep: steps must be host memory");
    OFB_TRY(validate_steps(steps, n_steps, total_points));
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void *dsteps, *dpos, *dflow;
    OFB_TRY(ofb_stage_in(ctx, SC_MC0, steps, sizeof(ofb_mc_step) * n_steps, &dsteps));
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, pos, sizeof(double) * 2 * (size_t)total_points, &dpos));
    OFB_TRY(ofb_stage_in(ctx, SC_IN1, true_flow, sizeof(double) * 2 * (size_t)total_points, &dflow));
    // launch shape: enough CTAs to fill the machine several times over, ~4 trials per thread at most
    uint64_t want = (trials + (uint64_t)MC_THREADS * 4 - 1) / ((uint64_t)MC_THREADS * 4);
    uint64_t fill = ((uint64_t)ctx->sm_count * 16 + n_steps - 1) / n_steps;   // >= 16 CTAs per SM in flight overall
    uint64_t cap = (trials + MC_THREADS - 1) / MC_THREADS;
    uint64_t bps = want > fill ? want : fill;
    if (bps > cap) bps = cap;
    if (bps < 1) bps = 1;
    if (bps > 16384) bps = 16384;
    int blocks_per_step = (int)bps;
    OFB_TRY(ctx->scratch[SC_MC1].reserve(sizeof(double) * MC_NSTAT * (size_t)blocks_per_step * n_steps));
    OutStage o[3];
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, sums_out, sizeof(ofb_mc_sums) * n_steps, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT1, v_dump, sizeof(double) * 3 * (size_t)n_steps * trials, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT2, R_dump, sizeof(double) * (size_t)n_steps * trials, &o[2]));
    uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    dim3 grid(blocks_per_step, n_steps);
#define OFB_MC_LAUNCH(T, WR)                                                                                          \
    mc_sweep_kernel<T, WR><<<grid, MC_THREADS, 0, ctx->stream>>>((const ofb_mc_step*)dsteps, step_id_base,             \
        (const double*)dpos, (const double*)dflow, trial_begin, trials, key, ctx->scratch[SC_MC1].as<double>(),        \
        (double*)o[1].dev, (double*)o[2].dev)
    switch (precision) {
        case 0: OFB_MC_LAUNCH(float, true); break;
        case 1: OFB_MC_LAUNCH(double, true); break;
        case 2: OFB_MC_LAUNCH(float, false); break;
        default: OFB_MC_LAUNCH(double, false); break;
    }
#undef OFB_MC_LAUNCH
    OFB_LAUNCH_CHECK(ctx);
    mc_finalize_kernel<<<n_steps, 32, 0, ctx->stream>>>(ctx->scratch[SC_MC1].as<double>(), blocks_per_step,
                                                        (ofb_mc_sums*)o[0].dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, o, 3);
}

// Single-process multi-GPU sweep (SURVEY 8b proposed ofb_mc_sweep(ctx_list, n_ctx, ...)): the trial range is cut into
// contiguous shards, one per context (any mix of devices), every shard is enqueued before the first one is waited for,
// and the per-step sums are merged on the host in context order -- the counter RNG makes the union identical to a
// one-context run up to fp64 summation order. A ctypes-only consumer gets all GPUs of a box without torch or NCCL;
// multi-PROCESS runs (one rank per GPU) merge the same 8 doubles per step with one all-reduce instead (simulation.py).
extern "C" int ofb_mc_sweep_multi(ofb_ctx** ctxs, int n_ctx, const ofb_mc_step* steps, int n_steps, int step_id_base,
                                  const double* pos, const double* true_flow, int total_points,
                                  uint64_t trial_begin, uint64_t trials, uint64_t seed, int precision,
                                  ofb_mc_sums* sums_out)
{
    OFB_REQUIRE(ctxs && n_ctx >= 1 && n_ctx <= 64, "mc_sweep_multi: needs 1..64 contexts");
    OFB_REQUIRE(steps && pos && true_flow && sums_out, "mc_sweep_multi: null argument");
    OFB_REQUIRE(n_steps > 0 && n_steps <= 65535, "mc_sweep_multi: n_steps must be in 1..65535");
    OFB_REQUIRE(trials > 0, "mc_sweep: iterations must be a positive number");
    OFB_REQUIRE(!ofb_is_device_ptr(sums_out) && !ofb_is_device_ptr(pos) && !ofb_is_device_ptr(true_flow),
                "mc_sweep_multi: pos, true_flow and sums_out must be host memory (they are read / merged for several devices)");
    for (int c = 0; c < n_ctx; ++c) OFB_REQUIRE(ctxs[c], "mc_sweep_multi: null context %d", c);
    const uint64_t base = trials / (uint64_t)n_ctx, rem = trials % (uint64_t)n_ctx;
    std::vector<uint64_t> cnt(n_ctx);
    uint64_t begin = trial_begin;
    for (int c = 0; c < n_ctx; ++c) {                       // enqueue every shard (device-resident sums: no wait)
        cnt[c] = base + ((uint64_t)c < rem ? 1 : 0);
        if (cnt[c] == 0) continue;
        ofb_ctx* ctx = ctxs[c];
        OFB_CUDA(cudaSetDevice(ctx->device));
        OFB_TRY(ctx->scratch[SC_MC2].reserve(sizeof(ofb_mc_sums) * n_steps));
        OFB_TRY(ofb_mc_sweep(ctx, steps, n_steps, step_id_base, pos, true_flow, total_points, begin, cnt[c], seed, precision,
                             ctx->scratch[SC_MC2].as<ofb_mc_sums>(), nullptr, nullptr));
        begin += cnt[c];
    }
    std::vector<ofb_mc_sums> part((size_t)n_steps);
    memset(sums_out, 0, sizeof(ofb_mc_sums) * n_steps);
    for (int c = 0; c < n_ctx; ++c) {                       // merge in context order: a fixed summation order
        if (cnt[c] == 0) continue;
        ofb_ctx* ctx = ctxs[c];
        OFB_CUDA(cudaSetDevice(ctx->device));
        OFB_CUDA(cudaMemcpyAsync(part.data(), ctx->scratch[SC_MC2].p, sizeof(ofb_mc_sums) * n_steps, cudaMemcpyDeviceToHost, ctx->stream));
        OFB_CUDA(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < n_steps; ++i) {
            sums_out[i].n += part[i].n; sums_out[i].sum_R += part[i].sum_R;
            for (int k = 0; k < 3; ++k) { sums_out[i].sum_dv[k] += part[i].sum_dv[k]; sums_out[i].sum_dv2[k] += part[i].sum_dv2[k]; }
        }
    }
    return OFB_OK;
}

extern "C" int ofb_mc_feas(ofb_ctx* ctx, const ofb_mc_step* step, int step_id, const double* pos,
                           const double* true_flow, uint64_t trial_begin, uint64_t trials, uint64_t seed,
                           double* sums_out)
{
    OFB_REQUIRE(ctx && step && pos && true_flow && sums_out, "mc_feas: null argument");
    OFB_REQUIRE(trials > 0, "mc_feas: iterations must be a positive number");
    OFB_REQUIRE(!ofb_is_device_ptr(step), "mc_feas: step must be host memory");
    int total_points = step->pos_offset + step->n_points;
    OFB_TRY(validate_steps(step, 1, total_points));
    OFB_CUDA(cudaSetDevice(ctx->device));
    int N = step->n_points;
    const void *dstep, *dpos, *dflow;
    OFB_TRY(ofb_stage_in(ctx, SC_MC0, step, sizeof(ofb_mc_step), &dstep));
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, pos, sizeof(double) * 2 * (size_t)total_points, &dpos));
    OFB_TRY(ofb_stage_in(ctx, SC_IN1, true_flow, sizeof(double) * 2 * (size_t)total_points, &dflow));
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, sums_out, sizeof(double) * 6 * (size_t)N, &o));
    OFB_CUDA(cudaMemsetAsync(o.dev, 0, sizeof(double) * 6 * (size_t)N, ctx->stream));
    uint64_t nb = (trials + MC_THREADS - 1) / MC_THREADS;
    uint64_t maxb = (uint64_t)ctx->sm_count * 8;
    if (nb > maxb) nb = maxb;
    uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    mc_feas_kernel<<<(int)nb, MC_THREADS, 0, ctx->stream>>>((const ofb_mc_step*)dstep, step_id, (const double*)dpos,
                                                           (const double*)dflow, trial_begin, trials, key, (double*)o.dev);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, &o, 1);
}

extern "C" int ofb_minmax(ofb_ctx* ctx, const double* data, size_t n, double* lo_out, double* hi_out)
{
    OFB_REQUIRE(ctx && data && lo_out && hi_out, "minmax: null argument");
    OFB_REQUIRE(n > 0, "minmax: empty input");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void* dd;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, data, sizeof(double) * n, &dd));
    int nb = (int)((n + 255) / 256); if (nb > ctx->sm_count * 4) nb = ctx->sm_count * 4;
    OFB_TRY(ctx->scratch[SC_TMP0].reserve(sizeof(double) * 2 * nb));
    minmax_kernel<<<nb, 256, 0, ctx->stream>>>((const double*)dd, n, ctx->scratch[SC_TMP0].as<double>());
    OFB_LAUNCH_CHECK(ctx);
    minmax_final_kernel<<<1, 32, 0, ctx->stream>>>(ctx->scratch[SC_TMP0].as<double>(), nb);
    OFB_LAUNCH_CHECK(ctx);
    double r[2];
    OFB_CUDA(cudaMemcpyAsync(r, ctx->scratch[SC_TMP0].p, sizeof(r), cudaMemcpyDeviceToHost, ctx->stream));
    OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    *lo_out = r[0]; *hi_out = r[1];
    return OFB_OK;
}

extern "C" int ofb_histogram(ofb_ctx* ctx, const double* data, size_t n, double lo, double hi, int bins,
                             unsigned long long* counts_out)
{
    OFB_REQUIRE(ctx && data && counts_out, "histogram: null argument");
    OFB_REQUIRE(bins > 0 && bins <= 4096, "histogram: bins must be in 1..4096");
    OFB_REQUIRE(isfinite(lo) && isfinite(hi), "histogram: range [%g, %g] is not finite", lo, hi);
    OFB_REQUIRE(hi >= lo, "histogram: max must be larger than min");
    OFB_CUDA(cudaSetDevice(ctx->device));
    if (hi == lo) { lo -= 0.5; hi += 0.5; }   // numpy widens a degenerate range
    const void* dd;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, data, sizeof(double) * n, &dd));
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, counts_out, sizeof(unsigned long long) * bins, &o));
    OFB_CUDA(cudaMemsetAsync(o.dev, 0, sizeof(unsigned long long) * bins, ctx->stream));
    if (n > 0) {
        int nb = (int)((n + 255) / 256); if (nb > ctx->sm_count * 4) nb = ctx->sm_count * 4;
        histogram_kernel<<<nb, 256, sizeof(unsigned int) * bins, ctx->stream>>>((const double*)dd, n, lo, hi, bins,
                                                                              (unsigned long long*)o.dev);
        OFB_LAUNCH_CHECK(ctx);
    }
    return ofb_finish_out(ctx, &o, 1);
}
