// pyrlk.cuh -- shared declarations of the Lucas-Kanade stage.
#pragma once
#include "common.cuh"

// one pyramid level of both images, packed so that the register-resident kernel fetches it with three 16-byte loads
struct LKLevel {
    const uint8_t* I; const uint8_t* J;          // image 0 of the batch at this level
    unsigned long long istride, jstride;         // bytes between images of the batch
    int w, h, ipitch, jpitch;
};

struct LKParams {
    LKLevel lv[OFB_MAX_LEVELS];
    int nlev;                     // levels actually used (after OpenCV's window-size cut)
    int win_w, win_h, max_count, flags;
    double eps;                   // squared, clamped
    double min_eig_thr;
    float eps_lo, eps_hi;         // fp32 brackets of eps: |delta|^2 below eps_lo / above eps_hi decides without fp64
    float hwx, hwy;               // (win - 1) / 2
    int prev_image0, prev_image_step, next_image0, next_image_step;   // image of pair p = image0 + p*step
};

// Device-pointer core. counts (optional): per-pair feature count at counts[pair*counts_stride];
// n_uniform = upper bound of the per-pair count (grid size).
// fb_thr > 0: forward-backward check (ofb_pyrlk_fb) folded into status; fb_err (optional) gets the distance where both
// passes had status 1, +inf elsewhere. fb_thr == 0: plain LK (fb_err is not written). The caller validates fb_thr.
int ofb_lk_device(ofb_ctx* ctx, const ofb_pyr* prev, int prev_image0, int prev_step, const ofb_pyr* next, int next_image0,
                  int next_step, int n_pairs, const float* prev_pts, const int* counts, int counts_stride, int n_uniform,
                  size_t pts_stride, int win_w, int win_h, int max_level, int max_count, double eps, int flags,
                  double min_eig_thr, float* next_pts, uint8_t* status, float* err, double fb_thr = 0.0,
                  float* fb_err = nullptr);

// threshold of the forward-backward check: 0 = off, > 0 (+inf included) = on; negative values and NaN are invalid
static inline bool ofb_fb_thr_ok(double t) { return t >= 0.0; }
