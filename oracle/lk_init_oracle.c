/*
 * lk_init_oracle.c -- CPU ORACLE (test infrastructure, NOT product code) for the gyro prediction of the LK tracks.
 *
 * orc_pyrlk_init is of_oracle.c's orc_pyrlk with OPTFLOW_USE_INITIAL_FLOW: next_pts holds the initial guess on entry,
 * and at the top level LK starts from it scaled by 1/2^L, as cv2 4.13 does (lkpyramid.cpp:
 * nextPt = nextPts[i] * (float)(1./(1 << level))). Everything else -- pyramid, Scharr derivatives, bilinear weights,
 * Newton iterations, exits, error -- is orc_pyrlk's line for line, and the helpers are of_oracle.c's own (included).
 * Pinned against cv2 4.13 by tests/golden/gyro_golden.npz (tests/test_host_gyro.py).
 *
 * Built on first use by oracle/gyro_oracle.py (gcc, of_oracle's flags) into a temporary directory.
 */
#include "of_oracle.c"

ORC_API int orc_pyrlk_init(const uint8_t* prev, const uint8_t* next, int w, int h, int pitch,
                           const float* prev_pts, int n, int win_w, int win_h, int max_level,
                           int max_count, double eps_in, double min_eig_thr,
                           float* next_pts, uint8_t* status, float* err)
{
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
            if (level == nlev - 1) { npx_ = next_pts[2 * i] * sc; npy_ = next_pts[2 * i + 1] * sc; }   /* the guess */
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
                    A11 += (float)(gx * gx); A12 += (float)(gx * gy); A22 += (float)(gy * gy);
                }
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
                for (int y = 0; y < win_h; ++y)
                    for (int x = 0; x < win_w; ++x) {
                        int X = jx + x, Y = jy + y;
                        int jv = (img_pad(J, X, Y) * w00 + img_pad(J, X + 1, Y) * w01 +
                                  img_pad(J, X, Y + 1) * w10 + img_pad(J, X + 1, Y + 1) * w11 + (1 << (W_BITS - 5 - 1))) >> (W_BITS - 5);
                        int diff = jv - Ip[y * win_w + x];
                        b1 += (float)(diff * Dx[y * win_w + x]);
                        b2 += (float)(diff * Dy[y * win_w + x]);
                    }
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
                for (int y = 0; y < win_h; ++y)
                    for (int x = 0; x < win_w; ++x) {
                        int X = jx + x, Y = jy + y;
                        int jv = (img_pad(J, X, Y) * w00 + img_pad(J, X + 1, Y) * w01 +
                                  img_pad(J, X, Y + 1) * w10 + img_pad(J, X + 1, Y + 1) * w11 + (1 << (W_BITS - 5 - 1))) >> (W_BITS - 5);
                        errval += (float)abs(jv - Ip[y * win_w + x]);
                    }
                err[i] = errval * 1.f / (32 * win_w * win_h);
            }
        }
    }
    free(Ip);
    free_pyr(pl, nlev_p);
    free_pyr(nl, nlev_n);
    return nlev - 1;   /* effective maxLevel */
}
