/*
 * of_oracle.c -- CPU ORACLE (test infrastructure, NOT product code).
 *
 * Scalar C restatement of the image stages of the reference's velocity-measurement
 * hot path. The reference (liquidcronos/Drone-stabilisation-...) does not own this
 * arithmetic: it calls OpenCV, which is an un-vendored, un-pinned third-party
 * dependency (no requirements file in /root/reference; the only build available is
 * the image's cv2 4.13.0 wheel). Reference call sites this follows:
 *   cv2.cvtColor(..., COLOR_BGR2GRAY)   velocity_measurment_node:113, evaluate_exp.py:65,85
 *   cv2.goodFeaturesToTrack             velocity_measurment_node:120,163, evaluate_exp.py:66,106,
 *                                       of_module.py:44,86, of_library.py:238
 *   cv2.calcOpticalFlowPyrLK            velocity_measurment_node:133, evaluate_exp.py:98,
 *                                       of_module.py:88, of_library.py:249
 * The algorithms restated are OpenCV's published ones (imgproc pyrDown, cornerMinEigenVal,
 * goodFeaturesToTrack, video calcOpticalFlowPyrLK) as summarised in SURVEY.md App. B.
 *
 * PARITY PIN: the reference holds no golden vectors for these stages (SURVEY.md 8c), so
 * the oracle is pinned against cv2 4.13.0 itself on identical inputs
 * (tests/test_oracle_vs_cv2.py) and against fixtures generated from cv2
 * (tests/golden/, generator tools/make_golden.py).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <float.h>

#define ORC_API __attribute__((visibility("default")))

/* OpenCV borderInterpolate(p, len, BORDER_REFLECT_101) */
static int refl101(int p, int len)
{
    if (len == 1) return 0;
    while ((unsigned)p >= (unsigned)len) {
        if (p < 0) p = -p;
        else p = 2 * len - 2 - p;
    }
    return p;
}

/* ---- BGR -> grey: (3735 B + 19235 G + 9798 R + 2^14) >> 15  (SURVEY App. B.1) ---- */
ORC_API void orc_bgr2gray(const uint8_t* bgr, int w, int h, int pitch, uint8_t* gray, int gpitch)
{
    for (int y = 0; y < h; ++y) {
        const uint8_t* s = bgr + (size_t)y * pitch;
        uint8_t* d = gray + (size_t)y * gpitch;
        for (int x = 0; x < w; ++x)
            d[x] = (uint8_t)((3735 * s[3 * x] + 19235 * s[3 * x + 1] + 9798 * s[3 * x + 2] + (1 << 14)) >> 15);
    }
}

/* ---- pyrDown u8: [1 4 6 4 1]^2 / 256, decimate by 2, reflect-101 (App. B.2) ---- */
ORC_API void orc_pyr_down(const uint8_t* src, int w, int h, int pitch, uint8_t* dst, int dpitch)
{
    static const int k[5] = {1, 4, 6, 4, 1};
    int dw = (w + 1) / 2, dh = (h + 1) / 2;
    for (int y = 0; y < dh; ++y)
        for (int x = 0; x < dw; ++x) {
            int acc = 0;
            for (int j = -2; j <= 2; ++j) {
                const uint8_t* row = src + (size_t)refl101(2 * y + j, h) * pitch;
                int racc = 0;
                for (int i = -2; i <= 2; ++i) racc += k[i + 2] * row[refl101(2 * x + i, w)];
                acc += k[j + 2] * racc;
            }
            dst[(size_t)y * dpitch + x] = (uint8_t)((acc + 128) >> 8);
        }
}

/* ---- cornerMinEigenVal, aperture 3, u8 input (App. B.5) ---------------------------
 * OpenCV: scaled Sobel -> products -> box SUM (reflect-101 on the product images) -> lambda_min, all in fp32 with a
 * running column sum. The Sobel outputs are integers, so the products and the blockSize x blockSize window sums are
 * integers too (< 2^31 for blockSize <= 45): orc_min_eig_map takes them EXACTLY and rounds only where the result is
 * formed -- a = (float)Sxx * (scale^2/2), b = (float)Sxy * scale^2, c = (float)Syy * (scale^2/2),
 * (a + c) - sqrt((a - c)^2 + b^2) -- which makes the map independent of the summation order (and symmetric wherever
 * the window sums are, e.g. rows 0 and 1 for an even blockSize, as OpenCV's own running sums happen to be). It differs
 * from OpenCV's fp32 accumulation by its summation noise, a few ulp of a + c ("documented float tie").
 * orc_min_eig_map_fp32sum keeps the plain fp32 accumulation (window order) for comparison.
 */
ORC_API void orc_min_eig_map(const uint8_t* src, int w, int h, int pitch, int block_size, float* eig)
{
    const float scale = (float)(1.0 / (4.0 * 255.0 * block_size));
    const float scale2 = scale * scale, h2 = 0.5f * scale2;
    const int bs = block_size, a0 = bs / 2;
    const int pw = w + bs, ph = h + bs;                     /* padded product images + one zero row/column */
    long long* I = (long long*)calloc((size_t)3 * (pw + 1) * (ph + 1), sizeof(long long));
    long long* Ixx = I; long long* Ixy = I + (size_t)(pw + 1) * (ph + 1); long long* Iyy = Ixy + (size_t)(pw + 1) * (ph + 1);
    /* integral images of the products at the reflected POSITIONS y - a0 + j, x - a0 + i */
    for (int py = 0; py < ph - 1; ++py) {
        const int y = refl101(py - a0, h);
        const uint8_t* r0 = src + (size_t)refl101(y - 1, h) * pitch;
        const uint8_t* r1 = src + (size_t)y * pitch;
        const uint8_t* r2 = src + (size_t)refl101(y + 1, h) * pitch;
        long long rxx = 0, rxy = 0, ryy = 0;
        for (int px = 0; px < pw - 1; ++px) {
            const int x = refl101(px - a0, w);
            const int xm = refl101(x - 1, w), xp = refl101(x + 1, w);
            const int gx = (r0[xp] - r0[xm]) + 2 * (r1[xp] - r1[xm]) + (r2[xp] - r2[xm]);
            const int gy = (r2[xm] + 2 * r2[x] + r2[xp]) - (r0[xm] + 2 * r0[x] + r0[xp]);
            rxx += (long long)gx * gx; rxy += (long long)gx * gy; ryy += (long long)gy * gy;
            const size_t o = (size_t)(py + 1) * (pw + 1) + (px + 1), up = o - (pw + 1);
            Ixx[o] = Ixx[up] + rxx; Ixy[o] = Ixy[up] + rxy; Iyy[o] = Iyy[up] + ryy;
        }
    }
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const size_t o00 = (size_t)y * (pw + 1) + x, o01 = o00 + bs, o10 = o00 + (size_t)bs * (pw + 1), o11 = o10 + bs;
            const int sxx = (int)(Ixx[o11] - Ixx[o01] - Ixx[o10] + Ixx[o00]);
            const int sxy = (int)(Ixy[o11] - Ixy[o01] - Ixy[o10] + Ixy[o00]);
            const int syy = (int)(Iyy[o11] - Iyy[o01] - Iyy[o10] + Iyy[o00]);
            const float a = (float)sxx * h2, b = (float)sxy * scale2, c = (float)syy * h2;
            const float dac = a - c;
            const float t1 = dac * dac, t2 = b * b;
            eig[(size_t)y * w + x] = (a + c) - sqrtf(t1 + t2);
        }
    free(I);
}

ORC_API void orc_min_eig_map_fp32sum(const uint8_t* src, int w, int h, int pitch, int block_size, float* eig)
{
    float scale = (float)(1.0 / (4.0 * 255.0 * block_size));
    float* dxx = (float*)malloc(sizeof(float) * 3 * (size_t)w * h);
    float* dxy = dxx + (size_t)w * h;
    float* dyy = dxy + (size_t)w * h;
    for (int y = 0; y < h; ++y) {
        const uint8_t* r0 = src + (size_t)refl101(y - 1, h) * pitch;
        const uint8_t* r1 = src + (size_t)y * pitch;
        const uint8_t* r2 = src + (size_t)refl101(y + 1, h) * pitch;
        for (int x = 0; x < w; ++x) {
            int xm = refl101(x - 1, w), xp = refl101(x + 1, w);
            int gx = (r0[xp] - r0[xm]) + 2 * (r1[xp] - r1[xm]) + (r2[xp] - r2[xm]);
            int gy = (r2[xm] + 2 * r2[x] + r2[xp]) - (r0[xm] + 2 * r0[x] + r0[xp]);
            float fx = (float)gx * scale, fy = (float)gy * scale;
            dxx[(size_t)y * w + x] = fx * fx;
            dxy[(size_t)y * w + x] = fx * fy;
            dyy[(size_t)y * w + x] = fy * fy;
        }
    }
    int a0 = block_size / 2;
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            float sxx = 0.f, sxy = 0.f, syy = 0.f;
            for (int j = 0; j < block_size; ++j) {
                size_t ro = (size_t)refl101(y - a0 + j, h) * w;
                for (int i = 0; i < block_size; ++i) {
                    size_t o = ro + refl101(x - a0 + i, w);
                    sxx += dxx[o]; sxy += dxy[o]; syy += dyy[o];
                }
            }
            float a = sxx * 0.5f, b = sxy, c = syy * 0.5f;
            eig[(size_t)y * w + x] = (a + c) - sqrtf((a - c) * (a - c) + b * b);
        }
    free(dxx);
}

/* ---- goodFeaturesToTrack selection on a given eig map (App. B.5) ----------------- */
typedef struct { float v; int addr; } orc_cand;
static int cand_cmp(const void* pa, const void* pb)
{
    const orc_cand* a = (const orc_cand*)pa; const orc_cand* b = (const orc_cand*)pb;
    if (a->v > b->v) return -1;
    if (a->v < b->v) return 1;
    return (a->addr > b->addr) ? -1 : (a->addr < b->addr) ? 1 : 0;   /* tie: larger address first */
}

/* returns number of corners written to xy (capacity cap pairs); eig is not modified */
ORC_API int orc_select_features(const float* eig, int w, int h, const uint8_t* mask, int mpitch,
                                int max_corners, double quality, double min_distance,
                                float* xy, int cap)
{
    double max_val = 0; int have = 0;
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            if (mask && !mask[(size_t)y * mpitch + x]) continue;
            float v = eig[(size_t)y * w + x];
            if (!have || v > max_val) { max_val = v; have = 1; }
        }
    if (!have) max_val = 0;
    float thr = (float)(max_val * quality);
    size_t ncand = 0, ccap = 1024;
    orc_cand* c = (orc_cand*)malloc(ccap * sizeof(orc_cand));
#define TH(v) ((v) > thr ? (v) : 0.f)
    for (int y = 1; y < h - 1; ++y)
        for (int x = 1; x < w - 1; ++x) {
            float v = TH(eig[(size_t)y * w + x]);
            if (v == 0.f) continue;
            if (mask && !mask[(size_t)y * mpitch + x]) continue;
            float m = v;
            for (int j = -1; j <= 1; ++j)
                for (int i = -1; i <= 1; ++i) {
                    float q = TH(eig[(size_t)(y + j) * w + (x + i)]);
                    if (q > m) m = q;
                }
            if (v != m) continue;
            if (ncand == ccap) { ccap *= 2; c = (orc_cand*)realloc(c, ccap * sizeof(orc_cand)); }
            c[ncand].v = v; c[ncand].addr = y * w + x; ++ncand;
        }
#undef TH
    qsort(c, ncand, sizeof(orc_cand), cand_cmp);
    int n = 0;
    if (min_distance >= 1) {
        int cell = (int)lrint(min_distance);       /* cvRound: half to even */
        int gw = (w + cell - 1) / cell, gh = (h + cell - 1) / cell;
        double md2 = min_distance * min_distance;
        /* per-cell singly linked lists of accepted corners */
        int* head = (int*)malloc(sizeof(int) * (size_t)gw * gh);
        int* next = (int*)malloc(sizeof(int) * (ncand ? ncand : 1));
        int* ax = (int*)malloc(sizeof(int) * (ncand ? ncand : 1));
        int* ay = (int*)malloc(sizeof(int) * (ncand ? ncand : 1));
        int nacc = 0;
        for (int i = 0; i < gw * gh; ++i) head[i] = -1;
        for (size_t i = 0; i < ncand; ++i) {
            int y = c[i].addr / w, x = c[i].addr - y * w;
            int xc = x / cell, yc = y / cell;
            int x1 = xc - 1 < 0 ? 0 : xc - 1, y1 = yc - 1 < 0 ? 0 : yc - 1;
            int x2 = xc + 1 > gw - 1 ? gw - 1 : xc + 1, y2 = yc + 1 > gh - 1 ? gh - 1 : yc + 1;
            int good = 1;
            for (int yy = y1; yy <= y2 && good; ++yy)
                for (int xx = x1; xx <= x2 && good; ++xx)
                    for (int e = head[yy * gw + xx]; e >= 0; e = next[e]) {
                        float dx = (float)(x - ax[e]), dy = (float)(y - ay[e]);
                        if ((double)(dx * dx + dy * dy) < md2) { good = 0; break; }
                    }
            if (!good) continue;
            ax[nacc] = x; ay[nacc] = y; next[nacc] = head[yc * gw + xc]; head[yc * gw + xc] = nacc; ++nacc;
            if (n < cap) { xy[2 * n] = (float)x; xy[2 * n + 1] = (float)y; }
            ++n;
            if (max_corners > 0 && n == max_corners) break;
        }
        free(head); free(next); free(ax); free(ay);
    } else {
        for (size_t i = 0; i < ncand; ++i) {
            int y = c[i].addr / w, x = c[i].addr - y * w;
            if (n < cap) { xy[2 * n] = (float)x; xy[2 * n + 1] = (float)y; }
            ++n;
            if (max_corners > 0 && n == max_corners) break;
        }
    }
    free(c);
    return n;
}

ORC_API int orc_good_features(const uint8_t* src, int w, int h, int pitch, const uint8_t* mask, int mpitch,
                              int max_corners, double quality, double min_distance, int block_size,
                              float* xy, int cap)
{
    float* eig = (float*)malloc(sizeof(float) * (size_t)w * h);
    orc_min_eig_map(src, w, h, pitch, block_size, eig);
    int n = orc_select_features(eig, w, h, mask, mpitch, max_corners, quality, min_distance, xy, cap);
    free(eig);
    return n;
}

/* ---- pyramidal Lucas-Kanade (App. B.3 / B.4) --------------------------------------- */
typedef struct { int w, h; uint8_t* img; int16_t* dx; int16_t* dy; } orc_level;

static inline int img_pad(const orc_level* L, int x, int y)
{   /* image level padded by winSize with reflect-101 */
    return L->img[(size_t)refl101(y, L->h) * L->w + refl101(x, L->w)];
}
static inline int der_pad(const orc_level* L, const int16_t* d, int x, int y)
{   /* derivative level padded with zeros */
    if ((unsigned)x >= (unsigned)L->w || (unsigned)y >= (unsigned)L->h) return 0;
    return d[(size_t)y * L->w + x];
}

static void scharr(orc_level* L)
{
    int w = L->w, h = L->h;
    L->dx = (int16_t*)malloc(sizeof(int16_t) * (size_t)w * h);
    L->dy = (int16_t*)malloc(sizeof(int16_t) * (size_t)w * h);
    for (int y = 0; y < h; ++y) {
        const uint8_t* r0 = L->img + (size_t)refl101(y - 1, h) * w;
        const uint8_t* r1 = L->img + (size_t)y * w;
        const uint8_t* r2 = L->img + (size_t)refl101(y + 1, h) * w;
        for (int x = 0; x < w; ++x) {
            int xm = refl101(x - 1, w), xp = refl101(x + 1, w);
            L->dx[(size_t)y * w + x] = (int16_t)(3 * (r0[xp] - r0[xm]) + 10 * (r1[xp] - r1[xm]) + 3 * (r2[xp] - r2[xm]));
            L->dy[(size_t)y * w + x] = (int16_t)(3 * (r2[xm] - r0[xm]) + 10 * (r2[x] - r0[x]) + 3 * (r2[xp] - r0[xp]));
        }
    }
}

static int build_pyr(const uint8_t* img, int w, int h, int pitch, int max_level, int win_w, int win_h,
                     orc_level* lv, int with_deriv)
{
    int n = 0;
    for (int l = 0; l <= max_level; ++l) {
        orc_level* L = &lv[l];
        if (l == 0) {
            L->w = w; L->h = h;
            L->img = (uint8_t*)malloc((size_t)w * h);
            for (int y = 0; y < h; ++y) memcpy(L->img + (size_t)y * w, img + (size_t)y * pitch, w);
        } else {
            L->w = (lv[l - 1].w + 1) / 2; L->h = (lv[l - 1].h + 1) / 2;
            /* level cut: a level must stay larger than the window */
            if (L->w <= win_w || L->h <= win_h) break;
            L->img = (uint8_t*)malloc((size_t)L->w * L->h);
            orc_pyr_down(lv[l - 1].img, lv[l - 1].w, lv[l - 1].h, lv[l - 1].w, L->img, L->w);
        }
        L->dx = L->dy = NULL;
        if (with_deriv) scharr(L);
        ++n;
    }
    return n;   /* number of levels built (maxLevel_eff + 1) */
}
static void free_pyr(orc_level* lv, int n)
{
    for (int l = 0; l < n; ++l) { free(lv[l].img); free(lv[l].dx); free(lv[l].dy); }
}

static inline void bil_weights(float a, float b, int* w00, int* w01, int* w10, int* w11)
{
    const int W_BITS = 14;
    *w00 = (int)lrintf((1.f - a) * (1.f - b) * (1 << W_BITS));
    *w01 = (int)lrintf(a * (1.f - b) * (1 << W_BITS));
    *w10 = (int)lrintf((1.f - a) * b * (1 << W_BITS));
    *w11 = (1 << W_BITS) - *w00 - *w01 - *w10;
}

/* flags: ORC_LK_EXACT_SUMS sums A, b and the L1 error as exact int64 integers and rounds each sum to fp32 once, as
 * the device kernels do (their per-lane partials are exact integers, reduced in 64 bits); the error is then scaled by
 * the fp32 reciprocal of 32 * win_w * win_h, as there. Without it the sums are OpenCV's running fp32 additions in
 * window order and the error is divided, as lkpyramid.cpp does. */
#define ORC_LK_EXACT_SUMS (1 << 16)

ORC_API int orc_pyrlk(const uint8_t* prev, const uint8_t* next, int w, int h, int pitch,
                      const float* prev_pts, int n, int win_w, int win_h, int max_level,
                      int max_count, double eps_in, int flags, double min_eig_thr,
                      float* next_pts, uint8_t* status, float* err)
{
    const int exact = (flags & ORC_LK_EXACT_SUMS) != 0;
    if (max_count < 0) max_count = 0; if (max_count > 100) max_count = 100;
    double e = eps_in < 0 ? 0 : eps_in > 10 ? 10 : eps_in;
    double eps = e * e;
    orc_level pl[16], nl[16];
    if (max_level > 15) max_level = 15;
    int nlev_p = build_pyr(prev, w, h, pitch, max_level, win_w, win_h, pl, 1);
    int nlev_n = build_pyr(next, w, h, pitch, max_level, win_w, win_h, nl, 0);
    int nlev = nlev_p < nlev_n ? nlev_p : nlev_n;
    const float FLT_SCALE = 1.f / (1 << 20);
    const int W_BITS = 14, W_BITS1 = 14;
    float hwx = (win_w - 1) * 0.5f, hwy = (win_h - 1) * 0.5f;
    int npx = win_w * win_h;
    int16_t* Ip = (int16_t*)malloc(sizeof(int16_t) * 3 * npx);
    int16_t* Dx = Ip + npx; int16_t* Dy = Dx + npx;

    for (int i = 0; i < n; ++i) { status[i] = 1; err[i] = 0; }
    for (int level = nlev - 1; level >= 0; --level) {
        const orc_level* I = &pl[level]; const orc_level* J = &nl[level];
        float sc = 1.f / (float)(1 << level);
        for (int i = 0; i < n; ++i) {
            float ppx = prev_pts[2 * i] * sc, ppy = prev_pts[2 * i + 1] * sc;
            float npx_, npy_;
            if (level == nlev - 1) { npx_ = ppx; npy_ = ppy; }
            else { npx_ = next_pts[2 * i] * 2.f; npy_ = next_pts[2 * i + 1] * 2.f; }
            next_pts[2 * i] = npx_; next_pts[2 * i + 1] = npy_;

            float px = ppx - hwx, py = ppy - hwy;
            int ix = (int)floorf(px), iy = (int)floorf(py);
            if (ix < -win_w || ix >= I->w || iy < -win_h || iy >= I->h) {
                if (level == 0) { status[i] = 0; err[i] = 0; }
                continue;
            }
            float a = px - ix, b = py - iy;
            int w00, w01, w10, w11; bil_weights(a, b, &w00, &w01, &w10, &w11);
            float A11 = 0, A12 = 0, A22 = 0;
            long long iA11 = 0, iA12 = 0, iA22 = 0;
            for (int y = 0; y < win_h; ++y)
                for (int x = 0; x < win_w; ++x) {
                    int X = ix + x, Y = iy + y;
                    int iv = (img_pad(I, X, Y) * w00 + img_pad(I, X + 1, Y) * w01 +
                              img_pad(I, X, Y + 1) * w10 + img_pad(I, X + 1, Y + 1) * w11 + (1 << (W_BITS1 - 5 - 1))) >> (W_BITS1 - 5);
                    int gx = (der_pad(I, I->dx, X, Y) * w00 + der_pad(I, I->dx, X + 1, Y) * w01 +
                              der_pad(I, I->dx, X, Y + 1) * w10 + der_pad(I, I->dx, X + 1, Y + 1) * w11 + (1 << (W_BITS1 - 1))) >> W_BITS1;
                    int gy = (der_pad(I, I->dy, X, Y) * w00 + der_pad(I, I->dy, X + 1, Y) * w01 +
                              der_pad(I, I->dy, X, Y + 1) * w10 + der_pad(I, I->dy, X + 1, Y + 1) * w11 + (1 << (W_BITS1 - 1))) >> W_BITS1;
                    Ip[y * win_w + x] = (int16_t)iv; Dx[y * win_w + x] = (int16_t)gx; Dy[y * win_w + x] = (int16_t)gy;
                    if (exact) { iA11 += gx * gx; iA12 += gx * gy; iA22 += gy * gy; }
                    else { A11 += (float)(gx * gx); A12 += (float)(gx * gy); A22 += (float)(gy * gy); }
                }
            if (exact) { A11 = (float)iA11; A12 = (float)iA12; A22 = (float)iA22; }
            A11 *= FLT_SCALE; A12 *= FLT_SCALE; A22 *= FLT_SCALE;
            float D = A11 * A22 - A12 * A12;
            float minEig = (A22 + A11 - sqrtf((A11 - A22) * (A11 - A22) + 4.f * A12 * A12)) / (float)(2 * win_w * win_h);
            if (minEig < min_eig_thr || D < FLT_EPSILON) {
                if (level == 0) status[i] = 0;
                continue;
            }
            D = 1.f / D;
            float qx = npx_ - hwx, qy = npy_ - hwy;
            float pdx = 0, pdy = 0;
            for (int j = 0; j < max_count; ++j) {
                int jx = (int)floorf(qx), jy = (int)floorf(qy);
                if (jx < -win_w || jx >= J->w || jy < -win_h || jy >= J->h) {
                    if (level == 0) status[i] = 0;
                    break;
                }
                a = qx - jx; b = qy - jy;
                bil_weights(a, b, &w00, &w01, &w10, &w11);
                float b1 = 0, b2 = 0;
                long long ib1 = 0, ib2 = 0;
                for (int y = 0; y < win_h; ++y)
                    for (int x = 0; x < win_w; ++x) {
                        int X = jx + x, Y = jy + y;
                        int jv = (img_pad(J, X, Y) * w00 + img_pad(J, X + 1, Y) * w01 +
                                  img_pad(J, X, Y + 1) * w10 + img_pad(J, X + 1, Y + 1) * w11 + (1 << (W_BITS - 5 - 1))) >> (W_BITS - 5);
                        int diff = jv - Ip[y * win_w + x];
                        if (exact) { ib1 += diff * Dx[y * win_w + x]; ib2 += diff * Dy[y * win_w + x]; }
                        else { b1 += (float)(diff * Dx[y * win_w + x]); b2 += (float)(diff * Dy[y * win_w + x]); }
                    }
                if (exact) { b1 = (float)ib1; b2 = (float)ib2; }
                b1 *= FLT_SCALE; b2 *= FLT_SCALE;
                float dx = (float)((A12 * b2 - A22 * b1) * D);
                float dy = (float)((A12 * b1 - A11 * b2) * D);
                qx += dx; qy += dy;
                next_pts[2 * i] = qx + hwx; next_pts[2 * i + 1] = qy + hwy;
                if ((double)dx * dx + (double)dy * dy <= eps) break;
                if (j > 0 && fabsf(dx + pdx) < 0.01f && fabsf(dy + pdy) < 0.01f) {
                    next_pts[2 * i] -= dx * 0.5f; next_pts[2 * i + 1] -= dy * 0.5f;
                    break;
                }
                pdx = dx; pdy = dy;
            }
            if (status[i] && level == 0) {
                float rx = next_pts[2 * i] - hwx, ry = next_pts[2 * i + 1] - hwy;
                int jx = (int)floorf(rx), jy = (int)floorf(ry);
                if (jx < -win_w || jx >= J->w || jy < -win_h || jy >= J->h) { status[i] = 0; continue; }
                a = rx - jx; b = ry - jy;
                bil_weights(a, b, &w00, &w01, &w10, &w11);
                float errval = 0;
                long long ierr = 0;
                for (int y = 0; y < win_h; ++y)
                    for (int x = 0; x < win_w; ++x) {
                        int X = jx + x, Y = jy + y;
                        int jv = (img_pad(J, X, Y) * w00 + img_pad(J, X + 1, Y) * w01 +
                                  img_pad(J, X, Y + 1) * w10 + img_pad(J, X + 1, Y + 1) * w11 + (1 << (W_BITS - 5 - 1))) >> (W_BITS - 5);
                        if (exact) ierr += abs(jv - Ip[y * win_w + x]);
                        else errval += (float)abs(jv - Ip[y * win_w + x]);
                    }
                err[i] = exact ? (float)ierr * (1.f / (float)(32 * win_w * win_h)) : errval * 1.f / (32 * win_w * win_h);
            }
        }
    }
    free(Ip);
    free_pyr(pl, nlev_p);
    free_pyr(nl, nlev_n);
    return nlev - 1;   /* effective maxLevel */
}
