// pyrlk.cu -- stage 3: pyramidal Lucas-Kanade tracking, one warp per feature.
//
// Replaces cv2.calcOpticalFlowPyrLK(prev, next, prevPts, None, winSize, maxLevel, criteria)
// (velocity_measurment_node:133; flight_experiments/evaluate_exp.py:98;
// optical_flow_experiments/of_module.py:88; of_library.py:249). Arithmetic follows OpenCV's
// lkpyramid.cpp as summarised in SURVEY App. B.3/B.4: Scharr gradients (int16, reflect-101 inside the
// image, ZERO outside), Q14 fixed-point bilinear patches with 5 fractional bits, fp32 2x2 system,
// <= maxCount Newton steps with the eps / oscillation exits, L1 patch error at level 0.
//
// Mapping: a warp owns one feature for all levels (coarse -> fine) so the whole track is one launch.
// Per level the (win+3)^2 u8 neighbourhood of I is staged in the warp's shared-memory slice, the
// Scharr gradients of the (win+1)^2 footprint are formed there once, and the template patch and its
// two interpolated gradients are kept in shared memory as int16 for the iterations. Each iteration
// stages the (win+1)^2 window of J (reflect-101 fix-up only for windows that touch the border,
// a warp-uniform branch), accumulates the mismatch vector in exact int32 per lane, reduces it with
// 64-bit shuffles and solves the 2x2 system redundantly in every lane's registers. OpenCV builds
// full-frame Scharr images per level; here gradients are formed only under the windows, so the
// derivative images (the largest share of OpenCV's LK time, SURVEY 6) never exist.
// The kernel is latency/issue bound (dependent iterations), not HBM bound: DESIGN.md, "LK".
#include <climits>
#include "common.cuh"
#include "pyrlk.cuh"

namespace {

constexpr int LK_WARPS = 4;

__device__ __forceinline__ int refl101(int p, int len)
{
    if (len == 1) return 0;
    while ((unsigned)p >= (unsigned)len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}

__device__ __forceinline__ long long warp_sum_ll(long long v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Stage the RW x RH block of `img` whose top-left corner is (x0,y0) into dst (row pitch dp),
// reflect-101 outside the image.
__device__ __forceinline__ void stage_block(const uint8_t* __restrict__ img, int w, int h, int pitch, int x0, int y0,
                                            int RW, int RH, uint8_t* dst, int dp, int lane)
{
    bool inside = x0 >= 0 && y0 >= 0 && x0 + RW <= w && y0 + RH <= h;
    if (inside) {
        const uint8_t* s = img + (size_t)y0 * pitch + x0;
        for (int r = 0; r < RH; ++r)
            for (int c = lane; c < RW; c += 32) dst[r * dp + c] = __ldg(s + (size_t)r * pitch + c);
    } else {
        for (int r = 0; r < RH; ++r) {
            const uint8_t* s = img + (size_t)refl101(y0 + r, h) * pitch;
            for (int c = lane; c < RW; c += 32) dst[r * dp + c] = __ldg(s + refl101(x0 + c, w));
        }
    }
}

__device__ __forceinline__ void bil_weights(float a, float b, int& w00, int& w01, int& w10, int& w11)
{
    w00 = __float2int_rn(__fmul_rn(__fmul_rn(1.f - a, 1.f - b), 16384.f));
    w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, 1.f - b), 16384.f));
    w10 = __float2int_rn(__fmul_rn(__fmul_rn(1.f - a, b), 16384.f));
    w11 = 16384 - w00 - w01 - w10;
}

// FB: the forward-backward check, as lk_track_fast2_kernel<true>.
template <bool FB>
__global__ void __launch_bounds__(LK_WARPS * 32)
lk_track_kernel(LKParams P, const float* __restrict__ prev_pts, float* __restrict__ next_pts,
                uint8_t* __restrict__ status, float* __restrict__ err, const int* __restrict__ counts,
                int counts_stride, int n_uniform, size_t pts_stride, size_t warp_smem, double fb_thr,
                float* __restrict__ fb_err)
{
    extern __shared__ __align__(16) unsigned char lk_smem[];
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int pair = blockIdx.y;
    int n = counts ? counts[(size_t)pair * counts_stride] : n_uniform;
    int feat = blockIdx.x * LK_WARPS + warp;
    if (feat >= n) return;
    const int winW = P.win_w, winH = P.win_h, npx = winW * winH;
    const int RW = winW + 3, RH = winH + 3, RP = (RW + 3) & ~3;
    const int DW = winW + 1, DH = winH + 1;
    size_t po = (size_t)pair * pts_stride + feat;
    float ptx = prev_pts[2 * po], pty = prev_pts[2 * po + 1];
    float nx = 0.f, ny = 0.f;
    if (P.flags & OFB_LK_USE_INITIAL_FLOW) { nx = next_pts[2 * po]; ny = next_pts[2 * po + 1]; }
    // (the point is loaded before the slices are set up: in this order ptxas spills 20 / 20 bytes for FB = false and
    // 16 / 32 for FB = true, the least of the orders tried)
    unsigned char* base = lk_smem + (size_t)warp * warp_smem;
    uint8_t* reg = base;                                       // RP x RH staged image bytes
    short* ders = (short*)(base + (((size_t)RP * RH + 15) & ~(size_t)15));   // Ix, Iy over DW x DH
    short* pat = ders + 2 * DW * DH;                           // Ipatch, dIx, dIy over npx
    const float hwx = P.hwx, hwy = P.hwy;
    const float FLT_SCALE = 1.f / (1 << 20);
    bool st = true;
    float errv = 0.f;
    int pimg = P.prev_image0 + pair * P.prev_image_step, nimg = P.next_image0 + pair * P.next_image_step;

#pragma unroll
    for (int pass = 0; pass < (FB ? 2 : 1); ++pass) {
        const bool bwd = FB && pass == 1;
        for (int level = P.nlev - 1; level >= 0; --level) {
            const LKLevel& L = P.lv[level];
            const uint8_t* I = bwd ? L.J + (size_t)nimg * L.jstride : L.I + (size_t)pimg * L.istride;
            const uint8_t* J = bwd ? L.I + (size_t)pimg * L.istride : L.J + (size_t)nimg * L.jstride;
            const int w = L.w, h = L.h;
            const int ipitch = bwd ? L.jpitch : L.ipitch, jpitch = bwd ? L.ipitch : L.jpitch;
            float sc = 1.f / (float)(1 << level);
            float ppx = ptx * sc, ppy = pty * sc;
            if (level == P.nlev - 1) {
                if (bwd ? (P.flags & OFB_LK_FB_INITIAL_FLOW) : (P.flags & OFB_LK_USE_INITIAL_FLOW)) { nx = nx * sc; ny = ny * sc; }
                else { nx = ppx; ny = ppy; }
            } else { nx = nx * 2.f; ny = ny * 2.f; }
            float px = ppx - hwx, py = ppy - hwy;
            int ix = __float2int_rd(px), iy = __float2int_rd(py);
            if (ix < -winW || ix >= w || iy < -winH || iy >= h) {
                if (level == 0) { st = false; errv = 0.f; }
                continue;
            }
            float a = px - (float)ix, b = py - (float)iy;
            int w00, w01, w10, w11;
            bil_weights(a, b, w00, w01, w10, w11);
            // ---- template: stage I neighbourhood, Scharr under the window, interpolated patches ----
            __syncwarp();
            stage_block(I, w, h, ipitch, ix - 1, iy - 1, RW, RH, reg, RP, lane);
            __syncwarp();
            for (int i = lane; i < DW * DH; i += 32) {
                int r = i / DW, c = i - r * DW;
                int X = ix + c, Y = iy + r;
                short gx = 0, gy = 0;
                if ((unsigned)X < (unsigned)w && (unsigned)Y < (unsigned)h) {
                    const uint8_t* r0 = reg + r * RP + c;          // (X-1, Y-1)
                    const uint8_t* r1 = r0 + RP;
                    const uint8_t* r2 = r1 + RP;
                    gx = (short)(3 * ((int)r0[2] - (int)r0[0]) + 10 * ((int)r1[2] - (int)r1[0]) + 3 * ((int)r2[2] - (int)r2[0]));
                    gy = (short)(3 * ((int)r2[0] - (int)r0[0]) + 10 * ((int)r2[1] - (int)r0[1]) + 3 * ((int)r2[2] - (int)r0[2]));
                }
                ders[i] = gx; ders[DW * DH + i] = gy;
            }
            __syncwarp();
            int iA11 = 0, iA12 = 0, iA22 = 0;
            for (int i = lane; i < npx; i += 32) {
                int y = i / winW, x = i - y * winW;
                const uint8_t* s0 = reg + (y + 1) * RP + x + 1;
                const uint8_t* s1 = s0 + RP;
                int iv = ((int)s0[0] * w00 + (int)s0[1] * w01 + (int)s1[0] * w10 + (int)s1[1] * w11 + (1 << 8)) >> 9;
                const short* d0 = ders + y * DW + x;
                const short* d1 = d0 + DW;
                int gx = ((int)d0[0] * w00 + (int)d0[1] * w01 + (int)d1[0] * w10 + (int)d1[1] * w11 + (1 << 13)) >> 14;
                const short* e0 = d0 + DW * DH;
                const short* e1 = e0 + DW;
                int gy = ((int)e0[0] * w00 + (int)e0[1] * w01 + (int)e1[0] * w10 + (int)e1[1] * w11 + (1 << 13)) >> 14;
                pat[i] = (short)iv; pat[npx + i] = (short)gx; pat[2 * npx + i] = (short)gy;
                iA11 += gx * gx; iA12 += gx * gy; iA22 += gy * gy;
            }
            float A11 = (float)warp_sum_ll(iA11) * FLT_SCALE;
            float A12 = (float)warp_sum_ll(iA12) * FLT_SCALE;
            float A22 = (float)warp_sum_ll(iA22) * FLT_SCALE;
            float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
            float dd = A11 - A22;
            float minEig = (A22 + A11 - sqrtf(__fadd_rn(__fmul_rn(dd, dd), __fmul_rn(__fmul_rn(4.f, A12), A12)))) /
                           (float)(2 * winW * winH);
            if ((double)minEig < P.min_eig_thr || D < 1.1920928955078125e-7f) {
                if (level == 0) st = false;
                continue;
            }
            D = 1.f / D;
            float qx = nx - hwx, qy = ny - hwy;
            float pdx = 0.f, pdy = 0.f;
            bool lost = false;
            for (int j = 0; j < P.max_count; ++j) {
                int jx = __float2int_rd(qx), jy = __float2int_rd(qy);
                if (jx < -winW || jx >= w || jy < -winH || jy >= h) { lost = true; break; }
                a = qx - (float)jx; b = qy - (float)jy;
                bil_weights(a, b, w00, w01, w10, w11);
                __syncwarp();
                stage_block(J, w, h, jpitch, jx, jy, DW, DH, reg, RP, lane);
                __syncwarp();
                int ib1 = 0, ib2 = 0;
                for (int i = lane; i < npx; i += 32) {
                    int y = i / winW, x = i - y * winW;
                    const uint8_t* s0 = reg + y * RP + x;
                    const uint8_t* s1 = s0 + RP;
                    int jv = ((int)s0[0] * w00 + (int)s0[1] * w01 + (int)s1[0] * w10 + (int)s1[1] * w11 + (1 << 8)) >> 9;
                    int diff = jv - (int)pat[i];
                    ib1 += diff * (int)pat[npx + i];
                    ib2 += diff * (int)pat[2 * npx + i];
                }
                float b1 = (float)warp_sum_ll(ib1) * FLT_SCALE;
                float b2 = (float)warp_sum_ll(ib2) * FLT_SCALE;
                float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), D);
                float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), D);
                qx += dx; qy += dy;
                nx = qx + hwx; ny = qy + hwy;
                if ((double)dx * (double)dx + (double)dy * (double)dy <= P.eps) break;
                if (j > 0 && fabsf(dx + pdx) < 0.01f && fabsf(dy + pdy) < 0.01f) {
                    nx -= dx * 0.5f; ny -= dy * 0.5f;
                    break;
                }
                pdx = dx; pdy = dy;
            }
            if (lost && level == 0) st = false;
            if (st && level == 0) {
                float rx = nx - hwx, ry = ny - hwy;
                int jx = __float2int_rd(rx), jy = __float2int_rd(ry);
                if (jx < -winW || jx >= w || jy < -winH || jy >= h) { st = false; }
                else if (!bwd) {                  // (the backward pass only needs the status of this bounds test)
                    a = rx - (float)jx; b = ry - (float)jy;
                    bil_weights(a, b, w00, w01, w10, w11);
                    __syncwarp();
                    stage_block(J, w, h, jpitch, jx, jy, DW, DH, reg, RP, lane);
                    __syncwarp();
                    int ie = 0;
                    for (int i = lane; i < npx; i += 32) {
                        int y = i / winW, x = i - y * winW;
                        const uint8_t* s0 = reg + y * RP + x;
                        const uint8_t* s1 = s0 + RP;
                        int jv = ((int)s0[0] * w00 + (int)s0[1] * w01 + (int)s1[0] * w10 + (int)s1[1] * w11 + (1 << 8)) >> 9;
                        ie += abs(jv - (int)pat[i]);
                    }
                    errv = (float)__reduce_add_sync(0xffffffffu, ie) * (1.f / (float)(32 * winW * winH));
                }
            }
        }
        if (FB && pass == 0) {
            // the forward result is stored now and the starting point re-read at the end, so that neither stays in
            // registers across the backward pass; likewise the initial flow g is re-read here, before the store
            // overwrites it, rather than kept from the forward pass's load
            float gx = 0.f, gy = 0.f;
            const bool seed = (P.flags & OFB_LK_FB_INITIAL_FLOW) != 0;
            if (seed) { gx = next_pts[2 * po]; gy = next_pts[2 * po + 1]; __syncwarp(); }
            if (lane == 0) {
                OFB_DEV_ASSERT(feat >= 0 && feat < n && (gridDim.y == 1 || po < (size_t)(pair + 1) * pts_stride));
                next_pts[2 * po] = nx; next_pts[2 * po + 1] = ny;
                if (err) err[po] = st ? errv : 0.f;
                if (!st) { status[po] = 0; if (fb_err) fb_err[po] = INFINITY; }
            }
            if (!st) return;
            const float p0x = ptx, p0y = pty;
            ptx = nx; pty = ny;
            if (seed) { nx = nx + (p0x - gx); ny = ny + (p0y - gy); }     // backward initial flow p1 + (p0 - g)
        }
    }
    if (FB) {
        if (lane == 0) {
            const float d = fmaxf(fabsf(prev_pts[2 * po] - nx), fabsf(prev_pts[2 * po + 1] - ny));
            status[po] = st && (double)d < fb_thr ? 1 : 0;
            if (fb_err) fb_err[po] = st ? d : INFINITY;
        }
        return;
    }
    if (lane == 0) {
        OFB_DEV_ASSERT(feat >= 0 && feat < n && (gridDim.y == 1 || po < (size_t)(pair + 1) * pts_stride));   // (one pair: the stride is unused)
        next_pts[2 * po] = nx; next_pts[2 * po + 1] = ny;
        status[po] = st ? 1 : 0;
        if (err) err[po] = st ? errv : 0.f;
    }
}

// ================= register-resident fast path: winW <= 16, winH <= 15 (the reference uses 15x15) ============
constexpr int LKF_WARPS = 1;                 // one feature per CTA: see lk_track_fast2_kernel

__device__ __forceinline__ int dp2a_lo(int w16x2, unsigned int bytes, int c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w16x2), "r"(bytes), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi(int w16x2, unsigned int bytes, int c)
{
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w16x2), "r"(bytes), "r"(c));
    return d;
}

// Column index reflected into [0, len): exact reflect-101 for p in [-len, 2*len) (two folds), which covers every
// patch position the tracker can reach (|offset| <= window + 9 columns, len > window).
__device__ __forceinline__ int refl_col(int p, int len)
{
    p = p < 0 ? -p : p;
    p = p >= len ? 2 * len - 2 - p : p;
    p = p < 0 ? -p : p;
    return min(p, len - 1);
}

// 12 bytes of image row Yr (already inside the image) starting at column X0 (bytes j=0..11 <-> columns X0+j) as
// three words. colfast (warp-uniform): the 16 bytes from the aligned-down address are inside the row -> four
// 32-bit loads and funnel shifts; else twelve independent byte loads with reflect-101 columns.
__device__ __forceinline__ void load12(const uint8_t* __restrict__ img, int w, int pitch, int X0, int Yr, bool colfast,
                                       unsigned int& o0, unsigned int& o1, unsigned int& o2)
{
    const uint8_t* row = img + (size_t)Yr * pitch;
    OFB_DEV_ASSERT(Yr >= 0 && (!colfast || (X0 >= 0 && X0 + 12 <= w)));
    if (colfast) {
        unsigned long long a = (unsigned long long)(row + X0);
        const unsigned int* q = (const unsigned int*)(a & ~3ull);
        unsigned int sh = (unsigned int)(a & 3ull) * 8u;
        unsigned int a0 = __ldg(q), a1 = __ldg(q + 1), a2 = __ldg(q + 2), a3 = __ldg(q + 3);
        o0 = __funnelshift_r(a0, a1, sh); o1 = __funnelshift_r(a1, a2, sh); o2 = __funnelshift_r(a2, a3, sh);
    } else {
        unsigned int v[3] = {0, 0, 0};
#pragma unroll
        for (int j = 0; j < 12; ++j) v[j >> 2] |= (unsigned int)__ldg(row + refl_col(X0 + j, w)) << (8 * (j & 3));
        o0 = v[0]; o1 = v[1]; o2 = v[2];
    }
}

// Exact warp sum of int32 lane values, returned as the correctly rounded float of the 64-bit total: two REDUX
// (low 16 bits unsigned, high part signed; neither can overflow over 32 lanes) instead of a 5-level shuffle chain.
__device__ __forceinline__ float warp_sum_exact_f(int v)
{
    const unsigned int lo = __reduce_add_sync(0xffffffffu, (unsigned int)v & 0xffffu);
    const int hi = __reduce_add_sync(0xffffffffu, v >> 16);
    return fmaf((float)hi, 65536.f, (float)lo);      // both terms exact in fp32, one rounding
}

// For the lane's 8 pixels: diff = J_k - I_k, both Q5 interpolated values. The dp2a chain starts from
// Cp[k] = 256 - 512*I_k, so ((sum + 256) >> 9) - I_k comes out of the shift directly (512*I_k is a multiple of 512).
#define LKF_FOR_PIXELS(T0, T1, T2, U0, U1, U2, Wt, Wb, BODY)                                     \
    {                                                                                             \
        unsigned int t1_ = __funnelshift_r(T0, T1, 8), t5_ = __funnelshift_r(T1, T2, 8);          \
        unsigned int u1_ = __funnelshift_r(U0, U1, 8), u5_ = __funnelshift_r(U1, U2, 8);          \
        unsigned int tt_[4] = {T0, t1_, T1, t5_};                                                 \
        unsigned int uu_[4] = {U0, u1_, U1, u5_};                                                 \
        _Pragma("unroll") for (int k = 0; k < 8; ++k) {                                           \
            int s_ = ((k >> 2) << 1) | (k & 1);       /* k=0,1,2,3,4,5,6,7 -> 0,1,0,1,2,3,2,3 */  \
            int diff;                                                                             \
            if ((k & 2) == 0) { diff = dp2a_lo(Wt, tt_[s_], Cp[k]); diff = dp2a_lo(Wb, uu_[s_], diff); } \
            else { diff = dp2a_hi(Wt, tt_[s_], Cp[k]); diff = dp2a_hi(Wb, uu_[s_], diff); }       \
            diff >>= 9;                                                                           \
            BODY                                                                                  \
        }                                                                                         \
    }

__device__ __forceinline__ unsigned int prmt(unsigned int a, unsigned int b, unsigned int sel) { return __byte_perm(a, b, sel); }

// Register-resident LK kernel. lane = (row r = lane>>1, half hh = lane&1): the lane owns the 8 window pixels (8hh+k, r),
// k=0..7, for the whole track. Everything a lane needs sits in 12-byte row segments (three 32-bit words after re-alignment
// with funnel shifts): no shared memory, no byte-granular traffic. Row r+1 of the window comes from lane+2 by shuffle (the
// two lanes of row 15 only feed their neighbours). Per level:
//   * Scharr under the window with two columns per instruction (packed 16-bit halves, biased so that no half ever
//     borrows from its neighbour); the gradients stay biased by +4096 through the bilinear interpolation, whose weights
//     sum to exactly 2^14, so the bias leaves in the rounding constant;
//   * the row below comes through 10 shuffles of column PAIRS;
//   * the template value and the Newton steps use the same Q14 bilinear taps: two dp2a (16-bit weights x u8 pixels) per
//     pixel, a funnel shift yields the byte pairs of pixels k and k+2 at once;
//   * per-level parameters are one packed record in constant memory, the level scale is built from its exponent, and
//     the convergence test |delta|^2 <= eps^2 is decided in fp32 unless it falls within 1e-6 of the threshold (the fp64
//     evaluation OpenCV uses is only needed there).
// One feature = one warp = one CTA: no shared memory and no block barrier, and features differ in their number of Newton
// steps -- with four warps per CTA the three that finished early kept their slots until the slowest one was done
// (0.854 -> 0.805 ms per 128 pairs with one). 32 CTAs per SM.
// FB = the forward-backward check (ofb_pyrlk_fb): a feature whose forward track has status 1 is tracked back from
// where it landed, in the same warp, and keeps status 1 only when the backward track has status 1 too and ends within
// fb_thr of the starting point (max-norm of the fp32 difference, compared in fp64). next_pts and err are the forward
// pass's. FB = false is the plain LK kernel.
template <bool FB>
__global__ void __launch_bounds__(LKF_WARPS * 32, 32 / LKF_WARPS)
lk_track_fast2_kernel(const __grid_constant__ LKParams P, const float* __restrict__ prev_pts, float* __restrict__ next_pts,
                      uint8_t* __restrict__ status, float* __restrict__ err, const int* __restrict__ counts,
                      int counts_stride, int n_uniform, size_t pts_stride, double fb_thr, float* __restrict__ fb_err)
{
    const int lane = threadIdx.x & 31;
    const int pair = blockIdx.y;
    const int n = counts ? counts[(size_t)pair * counts_stride] : n_uniform;
    const int feat = blockIdx.x * LKF_WARPS + (threadIdx.x >> 5);
    if (feat >= n) return;
    const int winW = P.win_w, winH = P.win_h;
    const int r = lane >> 1, hh = lane & 1;
    const size_t po = (size_t)pair * pts_stride + feat;
    float ptx = prev_pts[2 * po], pty = prev_pts[2 * po + 1];
    float nx = 0.f, ny = 0.f;
    if (P.flags & OFB_LK_USE_INITIAL_FLOW) { nx = next_pts[2 * po]; ny = next_pts[2 * po + 1]; }
    const float hwx = P.hwx, hwy = P.hwy;
    const float FLT_SCALE = 1.f / (1 << 20);
    unsigned int vmask = 0;                       // validity of the lane's pixels: column 8hh+k < winW, row r < winH
#pragma unroll
    for (int k = 0; k < 8; ++k) if (8 * hh + k < winW && r < winH) vmask |= 1u << k;
    bool st = true;
    float errv = 0.f;
    const int pimg = P.prev_image0 + pair * P.prev_image_step, nimg = P.next_image0 + pair * P.next_image_step;

    // FB: pass 1 tracks back from the forward result (I and J swap roles; the level geometry is shared, both pyramids
    // have one size), with no initial flow unless OFB_LK_FB_INITIAL_FLOW
#pragma unroll
    for (int pass = 0; pass < (FB ? 2 : 1); ++pass) {
        const bool bwd = FB && pass == 1;
        for (int level = P.nlev - 1; level >= 0; --level) {
            const LKLevel& L = P.lv[level];
            const int w = L.w, h = L.h, ipitch = bwd ? L.jpitch : L.ipitch, jpitch = bwd ? L.ipitch : L.jpitch;
            const uint8_t* __restrict__ I = bwd ? L.J + (size_t)nimg * L.jstride : L.I + (size_t)pimg * L.istride;
            const uint8_t* __restrict__ J = bwd ? L.I + (size_t)pimg * L.istride : L.J + (size_t)nimg * L.jstride;
            const int ilow = ((((unsigned long long)I) & 3ull) == 0 && (ipitch & 3) == 0) ? 0 : 4;   // see load12
            const int jlow = ((((unsigned long long)J) & 3ull) == 0 && (jpitch & 3) == 0) ? 0 : 4;
            const float sc = __int_as_float((127 - level) << 23);        // 2^-level
            const float ppx = ptx * sc, ppy = pty * sc;
            if (level == P.nlev - 1) {
                if (bwd ? (P.flags & OFB_LK_FB_INITIAL_FLOW) : (P.flags & OFB_LK_USE_INITIAL_FLOW)) { nx = nx * sc; ny = ny * sc; }
                else { nx = ppx; ny = ppy; }
            } else { nx = nx * 2.f; ny = ny * 2.f; }
            const float px = ppx - hwx, py = ppy - hwy;
            const int ix = __float2int_rd(px), iy = __float2int_rd(py);
            if (ix < -winW || ix >= w || iy < -winH || iy >= h) {
                if (level == 0) { st = false; errv = 0.f; }
                continue;
            }
            float a = px - (float)ix, b = py - (float)iy;
            int w00, w01, w10, w11;
            bil_weights(a, b, w00, w01, w10, w11);
            // ---- template ---------------------------------------------------------------------------------
            // rows iy+r-1 (A), iy+r (B), iy+r+1 (C); byte j of a row segment <-> column ix + 8hh - 1 + j, j = 0..11
            const bool icol = ix - 1 >= ilow && ix + 8 + 15 <= w, irow = iy - 1 >= 0 && iy + 16 < h;
            const bool ifast = icol && irow;
            const int X0 = ix - 1 + 8 * hh;
            unsigned int A0, A1, A2, B0, B1, B2, C0, C1, C2;
            {
                int ya = iy + r - 1, yb = iy + r, yc = iy + r + 1;
                if (!irow) { ya = refl101(ya, h); yb = refl101(yb, h); yc = refl101(yc, h); }
                load12(I, w, ipitch, X0, ya, icol, A0, A1, A2);
                load12(I, w, ipitch, X0, yb, icol, B0, B1, B2);
                load12(I, w, ipitch, X0, yc, icol, C0, C1, C2);
            }
            // Scharr, two columns per word. pa/pb/pc[i] = columns (2i, 2i+1) of rows A/B/C as 16-bit halves.
            //   t0 = 3 (A + C) + 10 B            <= 4080                      (vertical smoothing, for gx)
            //   t1 = C - A + 256                 in [1, 511]                  (vertical difference, for gy)
            //   gx[k] + 4096 = t0[k+2] - t0[k] + 4096,   gy[k] + 4096 = 3 (t1[k] + t1[k+2]) + 10 t1[k+1]
            unsigned int GX[5], GY[5];                   // (g[2i], g[2i+1]) + 4096 per half, Scharr at column ix + 8hh + k
            {
                unsigned int t0[6], t1[6];
                const unsigned int aw[3] = {A0, A1, A2}, bw[3] = {B0, B1, B2}, cw[3] = {C0, C1, C2};
#pragma unroll
                for (int i = 0; i < 6; ++i) {
                    const unsigned int sel = (i & 1) ? 0x4342u : 0x4140u;
                    const unsigned int pa = prmt(aw[i >> 1], 0u, sel), pb = prmt(bw[i >> 1], 0u, sel), pc = prmt(cw[i >> 1], 0u, sel);
                    t0[i] = 3u * (pa + pc) + 10u * pb;
                    t1[i] = pc + 0x01000100u - pa;
                }
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    GX[i] = t0[i + 1] + 0x10001000u - t0[i];
                    const unsigned int mid = prmt(t1[i], t1[i + 1], 0x5432u);            // (t1[2i+1], t1[2i+2])
                    GY[i] = 3u * (t1[i] + t1[i + 1]) + 10u * mid;
                }
            }
            if (!ifast) {       // OpenCV's derivative images are ZERO outside the image (a zero gradient is 4096 here)
                const bool rowin = (unsigned)(iy + r) < (unsigned)h;
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const bool okl = rowin && (unsigned)(ix + 8 * hh + 2 * i) < (unsigned)w;
                    const bool okh = rowin && (unsigned)(ix + 8 * hh + 2 * i + 1) < (unsigned)w;
                    const unsigned int keep = (okl ? 0x0000ffffu : 0u) | (okh ? 0xffff0000u : 0u);
                    const unsigned int zero = (okl ? 0u : 0x00001000u) | (okh ? 0u : 0x10000000u);
                    GX[i] = (GX[i] & keep) | zero; GY[i] = (GY[i] & keep) | zero;
                }
            }
            int Cp[8], Gx[8], Gy[8];
            int iA11 = 0, iA12 = 0, iA22 = 0;
            {
                // biased gradients of rows r (own) and r+1 (lane + 2), one value per column k = 0..8
                int gxa[9], gya[9], gxb[9], gyb[9];
#pragma unroll
                for (int i = 0; i < 5; ++i) {
                    const unsigned int nxp = __shfl_down_sync(0xffffffffu, GX[i], 2), nyp = __shfl_down_sync(0xffffffffu, GY[i], 2);
                    gxa[2 * i] = (int)(GX[i] & 0xffffu); gya[2 * i] = (int)(GY[i] & 0xffffu);
                    gxb[2 * i] = (int)(nxp & 0xffffu); gyb[2 * i] = (int)(nyp & 0xffffu);
                    if (i < 4) {
                        gxa[2 * i + 1] = (int)(GX[i] >> 16); gya[2 * i + 1] = (int)(GY[i] >> 16);
                        gxb[2 * i + 1] = (int)(nxp >> 16); gyb[2 * i + 1] = (int)(nyp >> 16);
                    }
                }
                // template value: rows B, C from column ix + 8hh on = byte 1 of the segments; the same dp2a taps as the
                // Newton loop (pixel k reads bytes k, k+1 of both rows)
                const int Wt = (w00 & 0xffff) | (w01 << 16), Wb = (w10 & 0xffff) | (w11 << 16);
                const unsigned int tt[4] = {__funnelshift_r(B0, B1, 8), __funnelshift_r(B0, B1, 16), __funnelshift_r(B1, B2, 8), __funnelshift_r(B1, B2, 16)};
                const unsigned int uu[4] = {__funnelshift_r(C0, C1, 8), __funnelshift_r(C0, C1, 16), __funnelshift_r(C1, C2, 8), __funnelshift_r(C1, C2, 16)};
                const int c0 = (1 << 13) - (4096 << 14);          // rounding constant minus the bias times the weight sum 2^14
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int s_ = ((k >> 2) << 1) | (k & 1);
                    int iv;
                    if ((k & 2) == 0) { iv = dp2a_lo(Wt, tt[s_], 1 << 8); iv = dp2a_lo(Wb, uu[s_], iv); }
                    else { iv = dp2a_hi(Wt, tt[s_], 1 << 8); iv = dp2a_hi(Wb, uu[s_], iv); }
                    iv >>= 9;
                    int gx = (gxa[k] * w00 + gxa[k + 1] * w01 + gxb[k] * w10 + gxb[k + 1] * w11 + c0) >> 14;
                    int gy = (gya[k] * w00 + gya[k + 1] * w01 + gyb[k] * w10 + gyb[k + 1] * w11 + c0) >> 14;
                    if (!((vmask >> k) & 1u)) { gx = 0; gy = 0; }
                    Cp[k] = 256 - 512 * iv; Gx[k] = gx; Gy[k] = gy;
                    iA11 += gx * gx; iA12 += gx * gy; iA22 += gy * gy;
                }
            }
            const float A11 = warp_sum_exact_f(iA11) * FLT_SCALE;
            const float A12 = warp_sum_exact_f(iA12) * FLT_SCALE;
            const float A22 = warp_sum_exact_f(iA22) * FLT_SCALE;
            float D2 = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
            const float dd = A11 - A22;
            const float minEig = (A22 + A11 - sqrtf(__fadd_rn(__fmul_rn(dd, dd), __fmul_rn(__fmul_rn(4.f, A12), A12)))) /
                                 (float)(2 * winW * winH);
            if ((double)minEig < P.min_eig_thr || D2 < 1.1920928955078125e-7f) {
                if (level == 0) st = false;
                continue;
            }
            D2 = 1.f / D2;
            float qx = nx - hwx, qy = ny - hwy;
            float pdx = 0.f, pdy = 0.f;
            bool lost = false;
            unsigned int T0 = 0, T1 = 0, T2 = 0, U0 = 0, U1 = 0, U2 = 0;
            int cjx = INT_MIN, cjy = INT_MIN;
            for (int j = 0; j < P.max_count; ++j) {
                const int jx = __float2int_rd(qx), jy = __float2int_rd(qy);
                if (jx < -winW || jx >= w || jy < -winH || jy >= h) { lost = true; break; }
                a = qx - (float)jx; b = qy - (float)jy;
                bil_weights(a, b, w00, w01, w10, w11);
                const int Wt = (w00 & 0xffff) | (w01 << 16), Wb = (w10 & 0xffff) | (w11 << 16);
                if (jx != cjx || jy != cjy) {               // the patch rows stay in registers while the integer position holds
                    const bool jcol = jx >= jlow && jx + 8 + 16 <= w, jrow = jy >= 0 && jy + 15 < h;
                    OFB_DEV_ASSERT(!jrow || (jy + r >= 0 && jy + r < h)); load12(J, w, jpitch, jx + 8 * hh, jrow ? jy + r : refl101(jy + r, h), jcol, T0, T1, T2);
                    U0 = __shfl_down_sync(0xffffffffu, T0, 2); U1 = __shfl_down_sync(0xffffffffu, T1, 2);
                    U2 = __shfl_down_sync(0xffffffffu, T2, 2);
                    cjx = jx; cjy = jy;
                }
                int ib1 = 0, ib2 = 0;
                LKF_FOR_PIXELS(T0, T1, T2, U0, U1, U2, Wt, Wb, {
                    ib1 += diff * Gx[k]; ib2 += diff * Gy[k];
                })
                const float b1 = warp_sum_exact_f(ib1) * FLT_SCALE;
                const float b2 = warp_sum_exact_f(ib2) * FLT_SCALE;
                const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), D2);
                const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), D2);
                qx += dx; qy += dy;
                nx = qx + hwx; ny = qy + hwy;
                // delta.ddot(delta) <= eps^2, evaluated in double by OpenCV: fp32 decides unless it is within 1e-6 of the bound
                const float s2 = __fmaf_rn(dx, dx, __fmul_rn(dy, dy));
                bool conv = s2 < P.eps_lo;
                if (!conv && !(s2 > P.eps_hi)) conv = (double)dx * (double)dx + (double)dy * (double)dy <= P.eps;
                if (conv) break;
                if (j > 0 && fabsf(dx + pdx) < 0.01f && fabsf(dy + pdy) < 0.01f) {
                    nx -= dx * 0.5f; ny -= dy * 0.5f;
                    break;
                }
                pdx = dx; pdy = dy;
            }
            if (lost && level == 0) st = false;
            if (st && level == 0) {
                const float rx = nx - hwx, ry = ny - hwy;
                const int jx = __float2int_rd(rx), jy = __float2int_rd(ry);
                if (jx < -winW || jx >= w || jy < -winH || jy >= h) { st = false; }
                else if (!bwd) {                  // (the backward pass only needs the status of this bounds test)
                    a = rx - (float)jx; b = ry - (float)jy;
                    bil_weights(a, b, w00, w01, w10, w11);
                    const int Wt = (w00 & 0xffff) | (w01 << 16), Wb = (w10 & 0xffff) | (w11 << 16);
                    if (jx != cjx || jy != cjy) {
                        const bool jcol = jx >= jlow && jx + 8 + 16 <= w, jrow = jy >= 0 && jy + 15 < h;
                        OFB_DEV_ASSERT(!jrow || (jy + r >= 0 && jy + r < h)); load12(J, w, jpitch, jx + 8 * hh, jrow ? jy + r : refl101(jy + r, h), jcol, T0, T1, T2);
                        U0 = __shfl_down_sync(0xffffffffu, T0, 2); U1 = __shfl_down_sync(0xffffffffu, T1, 2);
                        U2 = __shfl_down_sync(0xffffffffu, T2, 2);
                    }
                    int ie = 0;
                    LKF_FOR_PIXELS(T0, T1, T2, U0, U1, U2, Wt, Wb, {
                        if ((vmask >> k) & 1u) ie += abs(diff);
                    })
                    errv = (float)__reduce_add_sync(0xffffffffu, ie) * (1.f / (float)(32 * winW * winH));
                }
            }
        }
        if (FB && pass == 0) {
            // the forward result is stored now and the starting point re-read at the end, so that neither stays in
            // registers across the backward pass; likewise the initial flow g is re-read here, before the store
            // overwrites it, rather than kept from the forward pass's load
            float gx = 0.f, gy = 0.f;
            const bool seed = (P.flags & OFB_LK_FB_INITIAL_FLOW) != 0;
            if (seed) { gx = next_pts[2 * po]; gy = next_pts[2 * po + 1]; __syncwarp(); }
            if (lane == 0) {
                OFB_DEV_ASSERT(feat >= 0 && feat < n && (gridDim.y == 1 || po < (size_t)(pair + 1) * pts_stride));
                next_pts[2 * po] = nx; next_pts[2 * po + 1] = ny;
                if (err) err[po] = st ? errv : 0.f;
                if (!st) { status[po] = 0; if (fb_err) fb_err[po] = INFINITY; }
            }
            if (!st) return;
            const float p0x = ptx, p0y = pty;
            ptx = nx; pty = ny;
            if (seed) { nx = nx + (p0x - gx); ny = ny + (p0y - gy); }     // backward initial flow p1 + (p0 - g)
        }
    }
    if (FB) {
        if (lane == 0) {
            const float d = fmaxf(fabsf(prev_pts[2 * po] - nx), fabsf(prev_pts[2 * po + 1] - ny));
            status[po] = st && (double)d < fb_thr ? 1 : 0;
            if (fb_err) fb_err[po] = st ? d : INFINITY;
        }
        return;
    }
    if (lane == 0) {
        OFB_DEV_ASSERT(feat >= 0 && feat < n && (gridDim.y == 1 || po < (size_t)(pair + 1) * pts_stride));   // (one pair: the stride is unused)
        next_pts[2 * po] = nx; next_pts[2 * po + 1] = ny;
        status[po] = st ? 1 : 0;
        if (err) err[po] = st ? errv : 0.f;
    }
}

__global__ void fill_inf_kernel(float* __restrict__ out, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = INFINITY;
}

}  // namespace

size_t ofb_lk_warp_smem(int win_w, int win_h)
{
    int RW = win_w + 3, RH = win_h + 3, RP = (RW + 3) & ~3;
    size_t b = (((size_t)RP * RH + 15) & ~(size_t)15);
    b += sizeof(short) * 2 * (size_t)(win_w + 1) * (win_h + 1) + sizeof(short) * 3 * (size_t)win_w * win_h;
    return (b + 15) & ~(size_t)15;
}

int ofb_lk_device(ofb_ctx* ctx, const ofb_pyr* prev, int prev_image0, int prev_step, const ofb_pyr* next, int next_image0,
                  int next_step, int n_pairs, const float* prev_pts, const int* counts, int counts_stride, int n_uniform,
                  size_t pts_stride, int win_w, int win_h, int max_level, int max_count, double eps, int flags,
                  double min_eig_thr, float* next_pts, uint8_t* status, float* err, double fb_thr, float* fb_err)
{
    OFB_REQUIRE(win_w > 2 && win_h > 2, "pyrlk: winSize must be larger than 2x2");
    const bool fb = fb_thr > 0.0;
    OFB_REQUIRE(win_w * win_h <= 64 * 64, "pyrlk: winSize too large (max 4096 pixels)");
    OFB_REQUIRE(prev->w[0] == next->w[0] && prev->h[0] == next->h[0], "pyrlk: prev/next size mismatch");
    LKParams P;
    memset(&P, 0, sizeof(P));
    int nlev = prev->n_levels < next->n_levels ? prev->n_levels : next->n_levels;
    if (max_level >= 0 && max_level + 1 < nlev) nlev = max_level + 1;
    // OpenCV cuts the pyramid at the first level that is not larger than the window
    int eff = 1;
    for (int l = 1; l < nlev; ++l) {
        if (prev->w[l] <= win_w || prev->h[l] <= win_h) break;
        eff = l + 1;
    }
    P.nlev = eff;
    for (int l = 0; l < eff; ++l) {
        LKLevel& L = P.lv[l];
        if (l == 0) {
            L.I = prev->level0; L.istride = prev->level0_stride; L.ipitch = prev->level0_pitch;
            L.J = next->level0; L.jstride = next->level0_stride; L.jpitch = next->level0_pitch;
        } else {
            L.I = prev->base + prev->level_off[l]; L.istride = prev->image_stride[l]; L.ipitch = prev->pitch[l];
            L.J = next->base + next->level_off[l]; L.jstride = next->image_stride[l]; L.jpitch = next->pitch[l];
        }
        L.w = prev->w[l]; L.h = prev->h[l];
    }
    P.win_w = win_w; P.win_h = win_h;
    P.hwx = (win_w - 1) * 0.5f; P.hwy = (win_h - 1) * 0.5f;
    P.max_count = max_count < 0 ? 0 : (max_count > 100 ? 100 : max_count);
    double e = eps < 0 ? 0 : (eps > 10 ? 10 : eps);
    P.eps = e * e;
    P.eps_lo = (float)(P.eps * (1.0 - 1e-6)); P.eps_hi = (float)(P.eps * (1.0 + 1e-6));
    if (!((double)P.eps_lo < P.eps)) P.eps_lo = 0.f;                 // (eps^2 too small for the bracket: always ask fp64)
    if (!((double)P.eps_hi > P.eps)) P.eps_hi = INFINITY;
    P.min_eig_thr = min_eig_thr;
    P.flags = flags;
    P.prev_image0 = prev_image0; P.prev_image_step = prev_step;
    P.next_image0 = next_image0; P.next_image_step = next_step;
    if (n_uniform <= 0) return OFB_OK;
    const char* env = getenv("OFB_LK_GENERIC");      // parity tests cross-check the two kernels
    if (win_w <= 16 && win_h <= 15 && !(env && env[0] == '1')) {
        dim3 fgrid(ofb_div_up(n_uniform, LKF_WARPS), n_pairs);
        if (fb)
            lk_track_fast2_kernel<true><<<fgrid, LKF_WARPS * 32, 0, ctx->stream>>>(P, prev_pts, next_pts, status, err, counts,
                                                                                  counts_stride, n_uniform, pts_stride,
                                                                                  fb_thr, fb_err);
        else
            lk_track_fast2_kernel<false><<<fgrid, LKF_WARPS * 32, 0, ctx->stream>>>(P, prev_pts, next_pts, status, err, counts,
                                                                                   counts_stride, n_uniform, pts_stride,
                                                                                   0.0, nullptr);
        OFB_LAUNCH_CHECK(ctx);
        return OFB_OK;
    }
    size_t wsm = ofb_lk_warp_smem(win_w, win_h);
    size_t smem = wsm * LK_WARPS;
    if (fb) OFB_TRY(ofb_ensure_smem(ctx, FS_LK_FB, lk_track_kernel<true>, smem));
    else OFB_TRY(ofb_ensure_smem(ctx, FS_LK, lk_track_kernel<false>, smem));
    if (n_uniform <= 0) return OFB_OK;
    dim3 grid(ofb_div_up(n_uniform, LK_WARPS), n_pairs);
    if (fb)
        lk_track_kernel<true><<<grid, LK_WARPS * 32, smem, ctx->stream>>>(P, prev_pts, next_pts, status, err, counts, counts_stride,
                                                                         n_uniform, pts_stride, wsm, fb_thr, fb_err);
    else
        lk_track_kernel<false><<<grid, LK_WARPS * 32, smem, ctx->stream>>>(P, prev_pts, next_pts, status, err, counts, counts_stride,
                                                                          n_uniform, pts_stride, wsm, 0.0, nullptr);
    OFB_LAUNCH_CHECK(ctx);
    return OFB_OK;
}

extern "C" int ofb_pyrlk(ofb_ctx* ctx, const ofb_pyr* prev, int prev_image, const ofb_pyr* next, int next_image,
                         const float* prev_pts, int n, int win_w, int win_h, int max_level,
                         int max_count, double eps, int flags, double min_eig_thr,
                         float* next_pts, uint8_t* status, float* err)
{
    OFB_REQUIRE(ctx && prev && next && next_pts && status, "pyrlk: null argument");
    OFB_REQUIRE(n >= 0, "pyrlk: negative point count");
    OFB_REQUIRE(prev_image >= 0 && prev_image < prev->n_images && next_image >= 0 && next_image < next->n_images,
                "pyrlk: image index out of range");
    if (n == 0) return OFB_OK;
    OFB_REQUIRE(prev_pts, "pyrlk: null prevPts");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void* dpts;
    OFB_TRY(ofb_stage_in(ctx, SC_PTS0, prev_pts, sizeof(float) * 2 * (size_t)n, &dpts));
    OutStage o[3];
    OFB_TRY(ofb_stage_out(ctx, SC_PTS1, next_pts, sizeof(float) * 2 * (size_t)n, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_STAT, status, (size_t)n, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_ERR, err, sizeof(float) * (size_t)n, &o[2]));
    if ((flags & OFB_LK_USE_INITIAL_FLOW) && o[0].copy_back)
        OFB_CUDA(cudaMemcpyAsync(o[0].dev, next_pts, sizeof(float) * 2 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    OFB_TRY(ofb_lk_device(ctx, prev, prev_image, 0, next, next_image, 0, 1, (const float*)dpts, nullptr, 0, n, 0, win_w, win_h,
                          max_level, max_count, eps, flags, min_eig_thr, (float*)o[0].dev, (uint8_t*)o[1].dev,
                          (float*)o[2].dev));
    return ofb_finish_out(ctx, o, 3);
}

extern "C" int ofb_pyrlk_fb(ofb_ctx* ctx, const ofb_pyr* prev, int prev_image, const ofb_pyr* next, int next_image,
                            const float* prev_pts, int n, int win_w, int win_h, int max_level, int max_count, double eps,
                            double min_eig_thr, double fb_max_err, float* next_pts, uint8_t* status, float* err, float* fb_err)
{
    OFB_REQUIRE(ctx && prev && next && next_pts && status, "pyrlk_fb: null argument");
    OFB_REQUIRE(ofb_fb_thr_ok(fb_max_err), "pyrlk_fb: fb_max_err must be >= 0 (0 = no check)");
    OFB_REQUIRE(n >= 0, "pyrlk_fb: negative point count");
    OFB_REQUIRE(prev_image >= 0 && prev_image < prev->n_images && next_image >= 0 && next_image < next->n_images,
                "pyrlk_fb: image index out of range");
    if (n == 0) return OFB_OK;
    OFB_REQUIRE(prev_pts, "pyrlk_fb: null prevPts");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void* dpts;
    OFB_TRY(ofb_stage_in(ctx, SC_PTS0, prev_pts, sizeof(float) * 2 * (size_t)n, &dpts));
    OutStage o[4];
    OFB_TRY(ofb_stage_out(ctx, SC_PTS1, next_pts, sizeof(float) * 2 * (size_t)n, &o[0]));
    OFB_TRY(ofb_stage_out(ctx, SC_STAT, status, (size_t)n, &o[1]));
    OFB_TRY(ofb_stage_out(ctx, SC_ERR, err, sizeof(float) * (size_t)n, &o[2]));
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, fb_err, sizeof(float) * (size_t)n, &o[3]));
    if (fb_max_err == 0.0 && o[3].dev) {     // no check, no backward pass: no distance either
        fill_inf_kernel<<<ofb_div_up(n, 256), 256, 0, ctx->stream>>>((float*)o[3].dev, n);
        OFB_LAUNCH_CHECK(ctx);
    }
    OFB_TRY(ofb_lk_device(ctx, prev, prev_image, 0, next, next_image, 0, 1, (const float*)dpts, nullptr, 0, n, 0, win_w, win_h,
                          max_level, max_count, eps, 0, min_eig_thr, (float*)o[0].dev, (uint8_t*)o[1].dev, (float*)o[2].dev,
                          fb_max_err, (float*)o[3].dev));
    return ofb_finish_out(ctx, o, 4);
}
