// math3.cuh -- small fp64 linear algebra and the counter-based RNG shared by stages 4 and 5.
// Everything is __host__ __device__ so tools/host_check.cu can exercise it without a GPU.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#define OFB_HD __host__ __device__ __forceinline__

// ---- Philox4x32-10 (Salmon et al., SC'11) ------------------------------------------------------
OFB_HD void ofb_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo)
{
    uint64_t p = (uint64_t)a * b;          // one IMAD.WIDE.U32 on the device
    lo = (uint32_t)p; hi = (uint32_t)(p >> 32);
}

OFB_HD uint4 ofb_philox4x32_10(uint4 c, uint2 k)
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        ofb_mulhilo(M0, c.x, hi0, lo0);
        ofb_mulhilo(M1, c.z, hi1, lo1);
        uint4 n;
        n.x = hi1 ^ c.y ^ k.x; n.y = lo1; n.z = hi0 ^ c.w ^ k.y; n.w = lo0;
        c = n;
        k.x += W0; k.y += W1;
    }
    return c;
}

// Box-Muller on two 32-bit words: u0=(r0+0.5)2^-32 in (0,1], angle 2*pi*(u1-0.5).
// fp32 path uses the SFU intrinsics on device; the fp64 path is used for parity runs.
OFB_HD void ofb_box_muller(uint32_t r0, uint32_t r1, float& z0, float& z1)
{
#ifdef __CUDA_ARCH__
    // (float)r * 2^-32 + 2^-33 in one FMA: bit-identical to ((float)r + 0.5f) * 2^-32 (below 2^24 both are exact,
    // above it the half is below half an ulp either way)
    const float u0 = fmaf((float)r0, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
    const float u1 = fmaf((float)r1, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
    // radius: -2 ln u = (-2 ln 2) lg2 u, square root by the SFU (MUFU.LG2, FMUL, MUFU.SQRT: ~1 ulp, as accurate as
    // the fast logarithm in front of it; the IEEE sqrtf sequence with its range-check branch cost 5x as much)
    float rad;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(-1.3862943611198906f * __log2f(u0)));
    float s, c;
    __sincosf(6.2831853071795865f * (u1 - 0.5f), &s, &c);
#else
    float u0 = ((float)r0 + 0.5f) * 2.3283064365386963e-10f;
    float u1 = ((float)r1 + 0.5f) * 2.3283064365386963e-10f;
    float rad = sqrtf(-2.0f * logf(u0));
    float a = 6.2831853071795865f * (u1 - 0.5f);
    float s = sinf(a), c = cosf(a);
#endif
    z0 = rad * c; z1 = rad * s;
}
OFB_HD void ofb_box_muller(uint32_t r0, uint32_t r1, double& z0, double& z1)
{
    float u0 = ((float)r0 + 0.5f) * 2.3283064365386963e-10f;   // same uniforms as the fp32 path
    float u1 = ((float)r1 + 0.5f) * 2.3283064365386963e-10f;
    double rad = sqrt(-2.0 * log((double)u0));
    double a = 6.283185307179586476925 * ((double)u1 - 0.5);
    z0 = rad * cos(a); z1 = rad * sin(a);
}

// ---- 3x3 symmetric helpers (fp64) -------------------------------------------------------------
// M packed as (xx, xy, xz, yy, yz, zz)

// Cyclic Jacobi eigen-decomposition: M = Q diag(ev) Q^T, columns of Q in q[col][row].
// Eigenvalues sorted descending.
OFB_HD void ofb_jacobi3(const double M[6], double ev[3], double q[3][3])
{
    double a[3][3] = {{M[0], M[1], M[2]}, {M[1], M[3], M[4]}, {M[2], M[4], M[5]}};
    double v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};   // v[row][col]
    for (int sweep = 0; sweep < 16; ++sweep) {
        double off = fabs(a[0][1]) + fabs(a[0][2]) + fabs(a[1][2]);
        double diag = fabs(a[0][0]) + fabs(a[1][1]) + fabs(a[2][2]);
        if (off <= 1e-300 || off <= 1e-18 * diag) break;
        for (int p = 0; p < 2; ++p)
            for (int r = p + 1; r < 3; ++r) {
                double apq = a[p][r];
                if (apq == 0.0) continue;
                // tan of the rotation angle, t = sgn(theta) / (|theta| + sqrt(theta^2 + 1)) with theta = d / (2 apq),
                // multiplied through by |2 apq|: one square root and one division instead of two of each
                const double d = a[r][r] - a[p][p], two = 2.0 * apq;
                const double sg = (d == 0.0 || ((d > 0.0) == (apq > 0.0))) ? 1.0 : -1.0;
                double t = sg * fabs(two) / (fabs(d) + sqrt(d * d + two * two));
#ifdef __CUDA_ARCH__
                double c = rsqrt(t * t + 1.0), s = t * c;
#else
                double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#endif
                // A <- J^T A J
                for (int k = 0; k < 3; ++k) {
                    double akp = a[k][p], akq = a[k][r];
                    a[k][p] = c * akp - s * akq;
                    a[k][r] = s * akp + c * akq;
                }
                for (int k = 0; k < 3; ++k) {
                    double apk = a[p][k], aqk = a[r][k];
                    a[p][k] = c * apk - s * aqk;
                    a[r][k] = s * apk + c * aqk;
                }
                for (int k = 0; k < 3; ++k) {
                    double vkp = v[k][p], vkq = v[k][r];
                    v[k][p] = c * vkp - s * vkq;
                    v[k][r] = s * vkp + c * vkq;
                }
            }
    }
    int idx[3] = {0, 1, 2};
    double e[3] = {a[0][0], a[1][1], a[2][2]};
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2 - i; ++j)
            if (e[idx[j]] < e[idx[j + 1]]) { int tmp = idx[j]; idx[j] = idx[j + 1]; idx[j + 1] = tmp; }
    for (int i = 0; i < 3; ++i) {
        ev[i] = e[idx[i]];
        for (int k = 0; k < 3; ++k) q[i][k] = v[k][idx[i]];
    }
}

// Cyclic Jacobi eigen-decomposition of an N x N symmetric matrix a (overwritten: its diagonal holds the eigenvalues on
// return, unsorted), eigenvectors in the columns of v (v[row][col]). Same rotation and stopping rule as ofb_jacobi3.
// Every index is a compile-time constant once the loops are unrolled, so both matrices stay in registers.
template <int N>
OFB_HD void ofb_jacobi_n(double (&a)[N][N], double (&v)[N][N])
{
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) v[i][j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 16; ++sweep) {
        double off = 0.0, diag = 0.0;
#pragma unroll
        for (int p = 0; p < N; ++p) {
            diag += fabs(a[p][p]);
#pragma unroll
            for (int r = p + 1; r < N; ++r) off += fabs(a[p][r]);
        }
        if (off <= 1e-300 || off <= 1e-18 * diag) break;
#pragma unroll
        for (int p = 0; p < N - 1; ++p)
#pragma unroll
            for (int r = p + 1; r < N; ++r) {
                const double apq = a[p][r];
                if (apq == 0.0) continue;
                const double d = a[r][r] - a[p][p], two = 2.0 * apq;
                const double sg = (d == 0.0 || ((d > 0.0) == (apq > 0.0))) ? 1.0 : -1.0;
                const double t = sg * fabs(two) / (fabs(d) + sqrt(d * d + two * two));
#ifdef __CUDA_ARCH__
                const double c = rsqrt(t * t + 1.0), s = t * c;
#else
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#endif
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double akp = a[k][p], akq = a[k][r];
                    a[k][p] = c * akp - s * akq;
                    a[k][r] = s * akp + c * akq;
                }
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double apk = a[p][k], aqk = a[r][k];
                    a[p][k] = c * apk - s * aqk;
                    a[r][k] = s * apk + c * aqk;
                }
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double vkp = v[k][p], vkq = v[k][r];
                    v[k][p] = c * vkp - s * vkq;
                    v[k][r] = s * vkp + c * vkq;
                }
            }
    }
}

// Solve M v = g for SPD M by the adjugate (cofactors); returns det.
OFB_HD double ofb_solve_sym3(const double M[6], const double g[3], double v[3])
{
    double c00 = M[3] * M[5] - M[4] * M[4];
    double c01 = M[2] * M[4] - M[1] * M[5];
    double c02 = M[1] * M[4] - M[2] * M[3];
    double c11 = M[0] * M[5] - M[2] * M[2];
    double c12 = M[1] * M[2] - M[0] * M[4];
    double c22 = M[0] * M[3] - M[1] * M[1];
    double det = M[0] * c00 + M[1] * c01 + M[2] * c02;
    double inv = 1.0 / det;
    v[0] = (c00 * g[0] + c01 * g[1] + c02 * g[2]) * inv;
    v[1] = (c01 * g[0] + c11 * g[1] + c12 * g[2]) * inv;
    v[2] = (c02 * g[0] + c12 * g[1] + c22 * g[2]) * inv;
    return det;
}

// Smallest eigenvalue of an SPD 3x3 by Newton on the characteristic cubic started at 0
// (left of the smallest root the monic cubic is increasing and concave, so the iteration is
// monotone and cannot overshoot).
OFB_HD double ofb_min_eig_sym3(const double M[6])
{
    double c2 = M[0] + M[3] + M[5];
    double c1 = (M[0] * M[3] - M[1] * M[1]) + (M[0] * M[5] - M[2] * M[2]) + (M[3] * M[5] - M[4] * M[4]);
    double c0 = M[0] * (M[3] * M[5] - M[4] * M[4]) - M[1] * (M[1] * M[5] - M[4] * M[2]) +
                M[2] * (M[1] * M[4] - M[3] * M[2]);
    double lam = 0.0;
    for (int it = 0; it < 64; ++it) {
        double f = ((lam - c2) * lam + c1) * lam - c0;
        double fp = (3.0 * lam - 2.0 * c2) * lam + c1;
        if (!(fp > 0.0)) break;
        double step = f / fp;
        lam -= step;
        if (fabs(step) <= 4e-16 * c2) break;
    }
    return lam;
}

template <class T> struct ofb_vec3 { T x, y, z; };
template <class T> OFB_HD ofb_vec3<T> ofb_cross(const ofb_vec3<T>& a, const ofb_vec3<T>& b)
{
    return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
template <class T> OFB_HD T ofb_dot(const ofb_vec3<T>& a, const ofb_vec3<T>& b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
