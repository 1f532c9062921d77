// velocity_device.cuh -- block-cooperative planar-flow least squares (one CTA = one frame).
// Shared by ofb_solve_velocity* (fp64 point arrays) and the fused frame-pair path (float tracks).
#pragma once
#include "math3.cuh"

constexpr int OFB_SOLVE_THREADS = 256;   // threads of a one-CTA-per-frame solve

struct OfbSolveOut { double v[3]; double s[3]; double res; int rank; int count; };

// Per-point contribution (SURVEY App. A). X=(px,py,1), beta = X x (u3 + X x w).
//   SIM  : A_i = (n.X)[X]x, b_i = beta            simulation.py:19-23
//   NODE/EXP: A_i = [X]x,   b_i = beta/(n.X)      node:34-38, evaluate_exp.py:22-26
//   MODULE: A_i = [X]x / dist_i, b_i = A_i u3 / (n.X) = [X]x u3 / (dist_i (n.X)); no gyro term (the caller passes
//           w = 0), right-hand side not scaled by a common height    optical_flow_experiments/of_module.py:141-146
struct OfbPointTerms { double wA, wb, bx, by, bz; };

__device__ __forceinline__ OfbPointTerms ofb_point_terms(int variant, double px, double py, double ux, double uy,
                                                         const double n3[3], const double w3[3], double inv_dist = 1.0)
{
    // a = X x w
    double ax = py * w3[2] - w3[1], ay = w3[0] - px * w3[2], az = px * w3[1] - py * w3[0];
    double cx = ux + ax, cy = uy + ay, cz = az;
    OfbPointTerms t;
    t.bx = py * cz - cy; t.by = cx - px * cz; t.bz = px * cy - py * cx;
    double nx = n3[0] * px + n3[1] * py + n3[2];
    if (variant == OFB_VARIANT_SIM) { t.wA = nx; t.wb = 1.0; }
    else if (variant == OFB_VARIANT_MODULE) { t.wA = inv_dist; t.wb = inv_dist / nx; }
    else { t.wA = 1.0; t.wb = 1.0 / nx; }
    return t;
}

// 1 / dist_i of the older 4-argument of.r_tilde (sensor_precision_experiments/pixhawk_pure_IMU/of_library.py:365-384,
// called at of_module.py:125): dist_i = (n.X) |X x v| / |X x u3|
__device__ __forceinline__ double ofb_module_inv_dist(double px, double py, double ux, double uy, const double n3[3],
                                                      const double v[3])
{
    const double a0 = py * v[2] - v[1], a1 = v[0] - px * v[2], a2 = px * v[1] - py * v[0];      // X x v
    const double b0 = -uy, b1 = ux, b2 = px * uy - py * ux;                                     // X x u3
    const double na = sqrt(a0 * a0 + a1 * a1 + a2 * a2), nb = sqrt(b0 * b0 + b1 * b1 + b2 * b2);
    return nb / ((n3[0] * px + n3[1] * py + n3[2]) * na);
}

__device__ __forceinline__ double ofb_warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum of K doubles per thread; result valid in every thread.
template <int K>
__device__ __forceinline__ void ofb_block_sum(double (&acc)[K], double* smem /* K*32 doubles */)
{
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = ofb_warp_sum(acc[k]);
    __syncthreads();
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < K; ++k) smem[k * 32 + warp] = acc[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double v = lane < nwarps ? smem[k * 32 + lane] : 0.0;
        acc[k] = ofb_warp_sum(v);
    }
}

// Adds one point's contribution, weighted by om, to the normal equations acc[0..5] v = d acc[6..8] and the count acc[9].
// The plain solve passes om = 1, which multiplies exactly.
__device__ __forceinline__ void ofb_normal_add(double (&acc)[10], const OfbPointTerms& t, double px, double py, double om)
{
    const double w2 = t.wA * t.wA * om;
    const double xx = px * px, yy = py * py;
    // |X|^2 I - X X^T
    acc[0] += w2 * (yy + 1.0);      // xx
    acc[1] += w2 * (-px * py);      // xy
    acc[2] += w2 * (-px);           // xz
    acc[3] += w2 * (xx + 1.0);      // yy
    acc[4] += w2 * (-py);           // yz
    acc[5] += w2 * (xx + yy);       // zz
    // A^T b = -wA wb (X x beta)
    const double s = -t.wA * t.wb * om;
    acc[6] += s * (py * t.bz - t.by);
    acc[7] += s * (t.bx - px * t.bz);
    acc[8] += s * (px * t.by - py * t.bx);
    acc[9] += 1.0;
}

// numpy lstsq (rcond=None) of the normal equations acc[0..5] v = d acc[6..8] (M packed xx, xy, xz, yy, yz, zz) of
// acc[9] points (3 rows each): sets o.count, o.s and o.rank, returns the solution in v.
__device__ __forceinline__ void ofb_lstsq3(const double (&acc)[10], double d, OfbSolveOut& o, double (&v)[3])
{
    o.count = (int)(acc[9] + 0.5);
    double M[6] = {acc[0], acc[1], acc[2], acc[3], acc[4], acc[5]};
    double ev[3], q[3][3];
    ofb_jacobi3(M, ev, q);
    // numpy lstsq (rcond=None): singular values below eps*max(M,N)*s_max are treated as zero.
    // s comes from eig(A^T A), so it cannot resolve below ~1e-8*s_max; use 1e-7 as the floor.
    double rows = 3.0 * (double)o.count;
    double rc = 2.220446049250313e-16 * (rows > 3.0 ? rows : 3.0);
    if (rc < 1e-7) rc = 1e-7;
    double smax = ev[0] > 0 ? sqrt(ev[0]) : 0.0;
    int rank = 0;
    v[0] = v[1] = v[2] = 0.0;
    for (int k = 0; k < 3; ++k) {
        double sk = ev[k] > 0 ? sqrt(ev[k]) : 0.0;
        o.s[k] = sk;
        if (sk > rc * smax && smax > 0) {
            ++rank;
            double c = (q[k][0] * acc[6] + q[k][1] * acc[7] + q[k][2] * acc[8]) * d / ev[k];
            v[0] += c * q[k][0]; v[1] += c * q[k][1]; v[2] += c * q[k][2];
        }
    }
    o.rank = rank;
}

// ||A_i v - d b_i||^2 of one point (the residual of the plain solve's second pass)
__device__ __forceinline__ double ofb_point_res2(const OfbPointTerms& t, double px, double py, double d, const double (&v)[3])
{
    double rx = t.wA * (py * v[2] - v[1]) - d * t.wb * t.bx;
    double ry = t.wA * (v[0] - px * v[2]) - d * t.wb * t.by;
    double rz = t.wA * (px * v[1] - py * v[0]) - d * t.wb * t.bz;
    return rx * rx + ry * ry + rz * rz;
}

// Loader concept: begin(f), end(f), load(f, i, px, py, ux, uy) -> bool (false = point skipped),
// dist(f, i, d) -> bool (MODULE variant: true = per-point distance supplied by the caller, false = derive it from the
// prior velocity `vprior` with the 4-argument r_tilde).

// Loader over LK tracks (frame pairs, tracker): point i of frame f sits at o = f*stride + i, and is used when status is
// NULL or status[o] != 0; points per frame from counts[f*counts_stride] (counts NULL: n). CALIB: xu[o] holds the point's
// (x, y, ux, uy) of a calibrated camera, undistorted once before the solves (they read every point several times);
// otherwise the pinhole model maps the track. CALIB is a compile-time choice: behind a runtime branch nvcc contracts the
// pinhole flow scale differently into the solves' sums, and the pinhole results would change in the last bit.
template <bool CALIB>
struct TrackLoader {
    const float* prev; const float* next;                            // (x, y) pairs
    const uint8_t* status;
    const int* counts; int counts_stride; int n; size_t stride;
    double cx, cy, ps, fs;
    double4* xu;
    __device__ int begin(int) const { return 0; }
    __device__ int end(int f) const { return counts ? counts[(size_t)f * counts_stride] : n; }
    __device__ bool load(int f, int i, double& px, double& py, double& ux, double& uy) const {
        const size_t o = (size_t)f * stride + i;
        if (status && !status[o]) return false;                      // new_pos[status==1]  (node:134, evaluate_exp.py:99)
        if constexpr (CALIB) {
            const double4 v = xu[o];
            px = v.x; py = v.y; ux = v.z; uy = v.w;
        } else {
            const float nx = next[2 * o], ny = next[2 * o + 1];
            const float dx = nx - prev[2 * o], dy = ny - prev[2 * o + 1];   // flow formed in fp32 as cv2 arrays are (node:136)
            px = ((double)nx - cx) * ps; py = ((double)ny - cy) * ps;         // node:232-233
            ux = (double)dx * fs; uy = (double)dy * fs;                       // node:235
        }
        return true;
    }
    __device__ bool dist(int, int, double&) const { return false; }  // MODULE: distances from the prior velocity
};

template <class Loader>
__device__ OfbSolveOut ofb_block_solve(const Loader& ld, int f, int variant, double d, const double* n3g,
                                       const double* w3g, const double* t3g, const double* vprior = nullptr)
{
    __shared__ double red[11 * 32];
    const bool module = variant == OFB_VARIANT_MODULE;
    double n3[3] = {n3g[0], n3g[1], n3g[2]};
    double w3[3] = {w3g[0], w3g[1], w3g[2]};
    double vp[3] = {0.0, 0.0, 0.0};
    if (module) {                                   // flow is used as given (no gyro term), rhs is not scaled by a height
        w3[0] = w3[1] = w3[2] = 0.0; d = 1.0;
        if (vprior) { vp[0] = vprior[0]; vp[1] = vprior[1]; vp[2] = vprior[2]; }
    }
    // a zero prior would make every derived distance zero (the reference then divides by zero): unit distances instead
    const bool unit_dist = module && vp[0] == 0.0 && vp[1] == 0.0 && vp[2] == 0.0;
    auto inv_dist = [&](int i, double px, double py, double ux, double uy) -> double {
        if (!module) return 1.0;
        double di;
        if (ld.dist(f, i, di)) return 1.0 / di;
        if (unit_dist) return 1.0;
        return ofb_module_inv_dist(px, py, ux, uy, n3, vp);
    };
    int i0 = ld.begin(f), i1 = ld.end(f);
    // M (6), g (3), count
    double acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double px, py, ux, uy;
        if (!ld.load(f, i, px, py, ux, uy)) continue;
        ofb_normal_add(acc, ofb_point_terms(variant, px, py, ux, uy, n3, w3, inv_dist(i, px, py, ux, uy)), px, py, 1.0);
    }
    ofb_block_sum<10>(acc, red);
    OfbSolveOut o;
    double v[3];
    ofb_lstsq3(acc, d, o, v);
    // second pass: residual sum ||A_i v - d b_i||^2
    double r[1] = {0};
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double px, py, ux, uy;
        if (!ld.load(f, i, px, py, ux, uy)) continue;
        r[0] += ofb_point_res2(ofb_point_terms(variant, px, py, ux, uy, n3, w3, inv_dist(i, px, py, ux, uy)), px, py, d, v);
    }
    ofb_block_sum<1>(r, red);
    o.res = r[0];
    // lever arm: v_obs = v' - w x t   (simulation.py:28, evaluate_exp.py:29); NODE has none
    if (variant != OFB_VARIANT_NODE && !module && t3g) {
        v[0] -= w3[1] * t3g[2] - w3[2] * t3g[1];
        v[1] -= w3[2] * t3g[0] - w3[0] * t3g[2];
        v[2] -= w3[0] * t3g[1] - w3[1] * t3g[0];
    }
    o.v[0] = v[0]; o.v[1] = v[1]; o.v[2] = v[2];
    return o;
}

// Ego-motion solve: the angular rate is estimated together with the velocity instead of being taken from the gyro.
// Moving the gyro term of ofb_point_terms to the left side makes every point's block linear in (v', w):
//   X = (x, y, 1), C = [X]x, P = |X|^2 I - X X^T = C^T C, u3 = (ux, uy, 0), v' = v + w x t
//   A_i = [ wA C , d wb P ],  b_i = d wb C u3        (wA, wb: the variant weights of ofb_point_terms; MODULE has no
//                                                      gyro term and is not accepted)
// The normal-equation blocks have closed forms (C X = 0, C P = |X|^2 C, P^2 = |X|^2 P):
//   A^T A: vv = wA^2 P, vw = -wA d wb |X|^2 C, ww = d^2 wb^2 |X|^2 P;   A^T b: v = wA d wb P u3, w = d^2 wb^2 |X|^2 C u3
// C is antisymmetric with entries (-1, y, -x) above the diagonal, so vw needs three sums: 6 + 3 + 6 + 6 + a count =
// 22 fp64 accumulators per thread. The 6x6 system is decomposed by one warp (ofb_jacobi_n<6>, the other warps wait);
// the pseudo-inverse keeps the eigenpairs of A^T A that pass ofb_block_solve's rank rule; a second pass sums the
// residual r_i = X x (wA v' - d wb (X x w) - d wb u3) = A_i (v', w) - b_i.
struct OfbEgoOut { double v[3]; double w[3]; double s[6]; double res; int rank; int count; };

template <class Loader>
__device__ OfbEgoOut ofb_block_solve_ego(const Loader& ld, int f, int variant, double d, const double* n3g, const double* t3g)
{
    __shared__ double red[22 * 32];
    __shared__ double sol[6 + 6 + 1];                // (v', w), s descending, rank
    const double n3[3] = {n3g[0], n3g[1], n3g[2]};
    const bool sim = variant == OFB_VARIANT_SIM;
    const int i0 = ld.begin(f), i1 = ld.end(f);
    double acc[22];
#pragma unroll
    for (int k = 0; k < 22; ++k) acc[k] = 0.0;
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double px, py, ux, uy;
        if (!ld.load(f, i, px, py, ux, uy)) continue;
        const double nx = n3[0] * px + n3[1] * py + n3[2];
        const double wA = sim ? nx : 1.0, e = sim ? d : d / nx;           // e = d wb
        const double xx = px * px, yy = py * py, xy = px * py, r2 = xx + yy + 1.0;
        // P packed as (xx, xy, xz, yy, yz, zz)
        const double P[6] = {yy + 1.0, -xy, -px, xx + 1.0, -py, xx + yy};
        const double a2 = wA * wA, e2r = e * e * r2;
#pragma unroll
        for (int k = 0; k < 6; ++k) { acc[k] += a2 * P[k]; acc[9 + k] += e2r * P[k]; }
        const double kc = -wA * e * r2;                                    // vw = kc C
        acc[6] += kc; acc[7] += kc * py; acc[8] += kc * px;
        const double s = px * ux + py * uy, we = wA * e;                   // P u3 = r2 u3 - X (X . u3)
        acc[15] += we * (r2 * ux - px * s);
        acc[16] += we * (r2 * uy - py * s);
        acc[17] += we * (-s);
        acc[18] += e2r * (-uy);                                            // C u3 = X x u3
        acc[19] += e2r * ux;
        acc[20] += e2r * (px * uy - py * ux);
        acc[21] += 1.0;
    }
    ofb_block_sum<22>(acc, red);
    OfbEgoOut o;
    o.count = (int)(acc[21] + 0.5);
    if (threadIdx.x < 32) {
        const double k0 = acc[6], k1 = acc[7], k2 = acc[8];
        // vw block = sum kc C, C = [[0, -1, y], [1, 0, -x], [-y, x, 0]]
        double a[6][6] = {
            {acc[0], acc[1], acc[2], 0.0, -k0, k1},
            {acc[1], acc[3], acc[4], k0, 0.0, -k2},
            {acc[2], acc[4], acc[5], -k1, k2, 0.0},
            {0.0, k0, -k1, acc[9], acc[10], acc[11]},
            {-k0, 0.0, k2, acc[10], acc[12], acc[13]},
            {k1, -k2, 0.0, acc[11], acc[13], acc[14]}};
        double q[6][6];
        ofb_jacobi_n<6>(a, q);
        double ev[6], smax = 0.0;
#pragma unroll
        for (int k = 0; k < 6; ++k) { ev[k] = a[k][k]; smax = fmax(smax, ev[k] > 0 ? sqrt(ev[k]) : 0.0); }
        // numpy lstsq's rank rule (rcond=None), floored as in ofb_block_solve
        const double rows = 3.0 * (double)o.count;
        double rc = 2.220446049250313e-16 * (rows > 6.0 ? rows : 6.0);
        if (rc < 1e-7) rc = 1e-7;
        double x[6] = {0, 0, 0, 0, 0, 0}, sk[6];
        int rank = 0;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            sk[k] = ev[k] > 0 ? sqrt(ev[k]) : 0.0;
            if (sk[k] > rc * smax && smax > 0) {
                ++rank;
                double c = 0.0;
#pragma unroll
                for (int j = 0; j < 6; ++j) c += q[j][k] * acc[15 + j];
                c /= ev[k];
#pragma unroll
                for (int j = 0; j < 6; ++j) x[j] += c * q[j][k];
            }
        }
#pragma unroll
        for (int i = 0; i < 5; ++i)                                        // descending, fixed compare-exchange order
#pragma unroll
            for (int j = 0; j < 5 - i; ++j) {
                const double hi = fmax(sk[j], sk[j + 1]), lo = fmin(sk[j], sk[j + 1]);
                sk[j] = hi; sk[j + 1] = lo;
            }
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < 6; ++k) { sol[k] = x[k]; sol[6 + k] = sk[k]; }
            sol[12] = (double)rank;
        }
    }
    __syncthreads();
    const double vp[3] = {sol[0], sol[1], sol[2]}, w[3] = {sol[3], sol[4], sol[5]};
    double r[1] = {0};
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double px, py, ux, uy;
        if (!ld.load(f, i, px, py, ux, uy)) continue;
        const double nx = n3[0] * px + n3[1] * py + n3[2];
        const double wA = sim ? nx : 1.0, e = sim ? d : d / nx;
        const double cx = py * w[2] - w[1], cy = w[0] - px * w[2], cz = px * w[1] - py * w[0];   // X x w
        const double ax = wA * vp[0] - e * (cx + ux), ay = wA * vp[1] - e * (cy + uy), az = wA * vp[2] - e * cz;
        const double rx = py * az - ay, ry = ax - px * az, rz = px * ay - py * ax;
        r[0] += rx * rx + ry * ry + rz * rz;
    }
    ofb_block_sum<1>(r, red);
    o.res = r[0];
    o.rank = (int)sol[12];
    for (int k = 0; k < 3; ++k) { o.v[k] = vp[k]; o.w[k] = w[k]; }
    for (int k = 0; k < 6; ++k) o.s[k] = sol[6 + k];
    // lever arm: v = v' - w x t with the estimated rate (EXP, SIM); NODE has none
    if (variant != OFB_VARIANT_NODE && t3g) {
        o.v[0] -= w[1] * t3g[2] - w[2] * t3g[1];
        o.v[1] -= w[2] * t3g[0] - w[0] * t3g[2];
        o.v[2] -= w[0] * t3g[1] - w[1] * t3g[0];
    }
    return o;
}

// the C ABI record of a solve
__device__ __forceinline__ ofb_ego_result ofb_ego_record(const OfbEgoOut& o, int flags)
{
    ofb_ego_result r;
    for (int k = 0; k < 3; ++k) { r.v[k] = o.v[k]; r.w[k] = o.w[k]; }
    for (int k = 0; k < 6; ++k) r.s[k] = o.s[k];
    r.res = o.res; r.rank = o.rank; r.flags = flags;
    return r;
}

// Robust velocity solve: iteratively reweighted least squares with Tukey's biweight and a median scale.
//   iteration 0: the plain solve (ofb_block_solve's v' before the lever arm, bit for bit), all weights 1;
//   iteration k = 1..K: rho_i = ||r_i(v'_{k-1})|| (fp64; r_i = wA (X x v') - d wb beta_i, the plain solve's residual),
//     sigma = the lower median of (float)rho_i (rank floor((N-1)/2), exact), tau = c sigma; tau 0 or not finite: stop,
//     keeping v'_{k-1} and its weights (an exact fit of at least half the points);
//     w_i = (1 - (rho_i / tau)^2)^2 for rho_i < tau, else 0; v'_k = lstsq of the weighted normal equations, 3 N_in rows.
// Each weight multiplies its point's terms, so a weight of 1 changes nothing. The median is a radix select over the
// fp32 keys (the bits of non-negative floats sort as unsigned integers): 4 passes of 8 bits, each recomputing rho_i from
// the loader, counting into a shared-memory histogram with integer atomics and picking the digit by a warp scan. So
// there is no cap on N and no per-point scratch, and the result does not depend on the order of the atomics.
// Per iteration that is 5 passes over the points (4 select passes and the weighted accumulation); one more pass at the
// end sums res = sum w_i rho_i(v'_K)^2 with the last solve's weights (and writes them to wout when given).
struct OfbRobustOut { double v[3]; double s[3]; double res; double scale; int rank; int n_inliers; int iterations; };

__device__ __forceinline__ double ofb_tukey_weight(double rho, double tau)
{
    if (!(rho < tau)) return 0.0;
    const double q = rho / tau, a = 1.0 - __dmul_rn(q, q);      // rounded as NumPy rounds (no fused multiply-add)
    return a * a;
}

template <class Loader>
__device__ OfbRobustOut ofb_block_solve_robust(const Loader& ld, int f, int variant, double d, const double* n3g,
                                               const double* w3g, const double* t3g, double c, int iterations,
                                               double* __restrict__ wout = nullptr)
{
    __shared__ double red[11 * 32];
    __shared__ unsigned hist[256];
    __shared__ unsigned sel[2];                      // selected key prefix, rank left inside it
    const double n3[3] = {n3g[0], n3g[1], n3g[2]};
    const double w3[3] = {w3g[0], w3g[1], w3g[2]};
    const int i0 = ld.begin(f), i1 = ld.end(f);
    // weighted normal equations with weights from (vw, tau); tau = 0: all weights 1 (the plain solve)
    auto solve = [&](const double (&vw)[3], double tau, OfbSolveOut& o, double (&v)[3]) {
        double acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
            double px, py, ux, uy;
            if (!ld.load(f, i, px, py, ux, uy)) continue;
            const OfbPointTerms t = ofb_point_terms(variant, px, py, ux, uy, n3, w3);
            double om = 1.0;
            if (tau > 0.0) {
                om = ofb_tukey_weight(sqrt(ofb_point_res2(t, px, py, d, vw)), tau);
                if (om == 0.0) continue;
            }
            ofb_normal_add(acc, t, px, py, om);
        }
        ofb_block_sum<10>(acc, red);
        ofb_lstsq3(acc, d, o, v);
    };
    // the key of rank m (0-based, ascending) of (float)rho_i(vk)
    auto select = [&](const double (&vk)[3], unsigned m) -> unsigned {
        unsigned prefix = 0u, rank = m;
        for (int shift = 24; shift >= 0; shift -= 8) {
            const unsigned hi = shift == 24 ? 0u : 0xffffffffu << (shift + 8);
            for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0u;
            __syncthreads();
            for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
                double px, py, ux, uy;
                if (!ld.load(f, i, px, py, ux, uy)) continue;
                const OfbPointTerms t = ofb_point_terms(variant, px, py, ux, uy, n3, w3);
                const unsigned key = __float_as_uint((float)sqrt(ofb_point_res2(t, px, py, d, vk)));
                if ((key & hi) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (threadIdx.x < 32) {                  // lane l holds bins 8l .. 8l+7
                const int lane = threadIdx.x;
                unsigned cnt[8], sum = 0u;
#pragma unroll
                for (int j = 0; j < 8; ++j) { cnt[j] = hist[8 * lane + j]; sum += cnt[j]; }
                unsigned incl = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned y = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += y;
                }
                unsigned cum = incl - sum;
                if (rank >= cum && rank < incl) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (rank < cum + cnt[j]) { sel[0] = prefix | ((unsigned)(8 * lane + j) << shift); sel[1] = rank - cum; break; }
                        cum += cnt[j];
                    }
                }
            }
            __syncthreads();
            prefix = sel[0]; rank = sel[1];
        }
        return prefix;
    };
    OfbRobustOut r;
    OfbSolveOut o;
    double vk[3], vprev[3] = {0.0, 0.0, 0.0};
    solve(vprev, 0.0, o, vk);
    const int n = o.count;
    double tau_last = 0.0;                           // tau of the weights of the last solve (0: all weights 1)
    r.scale = 0.0; r.iterations = 0;
    for (int k = 1; k <= iterations && n > 0; ++k) {
        const double sigma = (double)__uint_as_float(select(vk, (unsigned)(n - 1) / 2u));
        const double tau = c * sigma;
        if (!(tau > 0.0) || !isfinite(tau)) break;
        OfbSolveOut ok;
        double vn[3];
        solve(vk, tau, ok, vn);
        for (int j = 0; j < 3; ++j) { vprev[j] = vk[j]; vk[j] = vn[j]; }
        o = ok; tau_last = tau; r.scale = sigma; r.iterations = k;
    }
    // last pass: res with the last solve's weights (from vprev and tau_last)
    double acc[1] = {0.0};
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double px, py, ux, uy;
        double om = 0.0;
        if (ld.load(f, i, px, py, ux, uy)) {
            const OfbPointTerms t = ofb_point_terms(variant, px, py, ux, uy, n3, w3);
            om = tau_last > 0.0 ? ofb_tukey_weight(sqrt(ofb_point_res2(t, px, py, d, vprev)), tau_last) : 1.0;
            if (om != 0.0) acc[0] += om * ofb_point_res2(t, px, py, d, vk);
        }
        if (wout) wout[i] = om;
    }
    ofb_block_sum<1>(acc, red);
    r.res = acc[0];
    r.rank = o.rank; r.n_inliers = o.count;
    for (int k = 0; k < 3; ++k) { r.s[k] = o.s[k]; r.v[k] = vk[k]; }
    // lever arm: v = v' - w x t (EXP, SIM); NODE has none
    if (variant != OFB_VARIANT_NODE && t3g) {
        r.v[0] -= w3[1] * t3g[2] - w3[2] * t3g[1];
        r.v[1] -= w3[2] * t3g[0] - w3[0] * t3g[2];
        r.v[2] -= w3[0] * t3g[1] - w3[1] * t3g[0];
    }
    return r;
}

// the C ABI record of a robust solve
__device__ __forceinline__ ofb_robust_result ofb_robust_record(const OfbRobustOut& o, int flags)
{
    ofb_robust_result r;
    for (int k = 0; k < 3; ++k) { r.v[k] = o.v[k]; r.s[k] = o.s[k]; }
    r.res = o.res; r.scale = o.scale;
    r.rank = o.rank; r.n_inliers = o.n_inliers; r.iterations = o.iterations; r.flags = flags;
    return r;
}

// host-side check of a robust setting: c finite and >= 1.5 (so that at least half the points keep a weight), 0..64 iterations
static inline int ofb_robust_check(const ofb_robust_cfg* r, const char* who)
{
    OFB_REQUIRE(r, "%s: null robust setting", who);
    OFB_REQUIRE(r->c >= 1.5 && r->c < HUGE_VAL, "%s: robust c must be finite and >= 1.5 (got %g)", who, r->c);
    OFB_REQUIRE(r->iterations >= 0 && r->iterations <= 64, "%s: robust iterations must be in 0..64 (got %d)", who, r->iterations);
    return OFB_OK;
}
