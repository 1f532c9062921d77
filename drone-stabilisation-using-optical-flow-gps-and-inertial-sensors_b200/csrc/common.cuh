// common.cuh -- context, error plumbing and host<->device staging shared by every stage.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <vector>
#include <utility>
#include "../../include/ofb200.h"

void ofb_set_error(const char* fmt, ...);

#define OFB_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            ofb_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return OFB_E_CUDA;                                                                  \
        }                                                                                       \
    } while (0)

#define OFB_REQUIRE(cond, ...)                                                                  \
    do {                                                                                        \
        if (!(cond)) { ofb_set_error(__VA_ARGS__); return OFB_E_INVALID; }                      \
    } while (0)

#define OFB_TRY(call)                                                                           \
    do { int r__ = (call); if (r__ != OFB_OK) return r__; } while (0)

// grow-only device buffer
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return OFB_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            ofb_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
            p = nullptr;
            return OFB_E_NOMEM;
        }
        cap = want;
        return OFB_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return (T*)p; }
};

// grow-only pinned host buffer (staging for host-pointer outputs)
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return OFB_OK;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) {
            ofb_set_error("cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
            p = nullptr;
            return OFB_E_NOMEM;
        }
        cap = want;
        return OFB_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// Debug build (-DOFB_DEBUG_BOUNDS=1, `python -m ofb200._build --debug` -> libofb200_dbg.so, selected with OFB200_LIB): the
// index arithmetic of the kernels is checked where it is computed; a violation prints its location and traps, which
// surfaces as a CUDA error of the call. compute-sanitizer is not available on the GPU pool, this is the substitute.
#ifdef OFB_DEBUG_BOUNDS
#define OFB_DEV_ASSERT(c)                                                                                              \
    do {                                                                                                               \
        if (!(c)) {                                                                                                    \
            printf("OFB_DEV_ASSERT %s:%d: %s (block %d,%d,%d thread %d)\n", __FILE__, __LINE__, #c, (int)blockIdx.x,     \
                   (int)blockIdx.y, (int)blockIdx.z, (int)threadIdx.x);                                                \
            __trap();                                                                                                  \
        }                                                                                                              \
    } while (0)
#else
#define OFB_DEV_ASSERT(c) ((void)0)
#endif

enum { OFB_NSCRATCH = 26, OFB_NSTAGES = 5, OFB_NSTAGE_EV = 6, OFB_NFUNC_SLOTS = 32 };

struct ofb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    uint64_t launches = 0;
    // what a caller may have put on the stream besides API calls that launch kernels: asynchronous copies into device memory
    // (ofb_memcpy_async) and anything at all once the stream handle was handed out (ofb_ctx_stream). The tracker moves its
    // ingest to an internal stream only when neither happened since its previous step (see tracker_step_launches).
    uint64_t async_writes = 0;
    bool stream_exported = false;
    // streams of objects living on this context (a tracker's split solve) that must be joined before the context's
    // stream counts as "done": ofb_ctx_sync, ofb_timer_stop and the memcpy calls wait for them (ofb_join_aux)
    std::vector<std::pair<cudaStream_t, cudaEvent_t>> aux_join;
    // cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel: what this context has already
    // requested for each kernel that needs more than 48 KB (slot = FS_* below). Per context, hence per device.
    size_t func_smem[OFB_NFUNC_SLOTS] = {};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    DevBuf scratch[OFB_NSCRATCH];   // role-indexed scratch arenas (see each stage)
    PinBuf pin[4];
    std::vector<ofb_pyr*> pyramids;
    ofb_pyr* pair_pyr[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // [slot][prev|next] workspace pyramids of ofb_frame_pairs
    // host-input pipelining of ofb_frame_pairs: H2D of sub-batch i+1 on copy_stream overlaps compute of sub-batch i
    cudaStream_t copy_stream = nullptr;
    cudaStream_t upload_stream = nullptr;        // stream level-0 uploads go to (nullptr = stream)
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> ev_piece;           // one per uploaded sub-batch of a call
    // the ordered-selection kernel occupies one CTA per image; the pyramid kernels of the same batch run beside
    // it on aux_stream (fork after the lambda_min kernel, join before LK)
    cudaStream_t aux_stream = nullptr, aux2_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr;
    const int* feat_active = nullptr;            // per-image flags (device): the lambda_min kernels skip images whose flag is 0
    bool feat_prezeroed = false;                 // the caller reset the per-image state and cell grids of the next features call
    bool fork_after_eig = false;                 // ofb_features_device records ev_fork after the lambda_min launch
    // second context (own stream + scratch) that takes every other chunk of a resident ofb_frame_pairs batch
    ofb_ctx* twin = nullptr;
    cudaEvent_t ev_twin_fork = nullptr, ev_twin_join = nullptr;
    // optional per-stage CUDA-event timing of ofb_frame_pairs (ofb_ctx_set_profile)
    bool profile = false;
    cudaEvent_t stage_ev[OFB_NSTAGE_EV] = {};
    float stage_ms[OFB_NSTAGES] = {};
    uint64_t stage_calls = 0;
};

// scratch roles
enum {
    SC_IN0 = 0, SC_IN1, SC_IN2, SC_IN3, SC_IN4, SC_IN5,      // staged host inputs
    SC_OUT0, SC_OUT1, SC_OUT2, SC_OUT3,                      // staged outputs
    SC_CAND, SC_CANDCNT, SC_SEL, SC_GRID, SC_PTS0, SC_PTS1, SC_STAT, SC_ERR,
    SC_MC0, SC_MC1, SC_MC2, SC_TMP0, SC_TMP1, SC_TMP2,
    SC_FRAMES,                                               // device staging of host frames (ofb_frame_pairs)
    SC_CALIB                                                 // calibrated tracks of ofb_frame_pairs_cam
};

struct ofb_pyr {
    int n_images = 0, n_levels = 0;       // n_images = capacity
    int n_active = 0;                     // images in use (<= n_images): launches and uploads cover these
    int w[OFB_MAX_LEVELS], h[OFB_MAX_LEVELS], pitch[OFB_MAX_LEVELS];
    size_t level_off[OFB_MAX_LEVELS];     // byte offset of level l (image 0) inside `base`
    size_t image_stride[OFB_MAX_LEVELS];  // byte stride between images at level l
    uint8_t* base = nullptr;              // owned storage for levels >= 1 (and level 0 when copied)
    const uint8_t* level0 = nullptr;      // level 0 (may alias caller memory when it was device-resident)
    int level0_pitch = 0;
    size_t level0_stride = 0;
    bool level0_owned = false;
    size_t bytes = 0;
};

// order the context's stream behind everything enqueued on the registered auxiliary streams
static inline cudaError_t ofb_join_aux(ofb_ctx* ctx)
{
    for (auto& sj : ctx->aux_join) {
        cudaError_t e = cudaEventRecord(sj.second, sj.first);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, sj.second, 0);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

static inline bool ofb_is_device_ptr(const void* p)
{
    if (!p) return false;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Returns a device view of `p` (bytes long): p itself when device-resident, else a staged copy
// in scratch[role] (async H2D on the context stream).
static inline int ofb_stage_in(ofb_ctx* ctx, int role, const void* p, size_t bytes, const void** dev)
{
    if (!p || bytes == 0) { *dev = nullptr; return OFB_OK; }
    if (ofb_is_device_ptr(p)) { *dev = p; return OFB_OK; }
    OFB_TRY(ctx->scratch[role].reserve(bytes));
    OFB_CUDA(cudaMemcpyAsync(ctx->scratch[role].p, p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dev = ctx->scratch[role].p;
    return OFB_OK;
}

// Output staging: returns device pointer to write to; remember if a copy-back is needed.
struct OutStage {
    void* user = nullptr; void* dev = nullptr; size_t bytes = 0; bool copy_back = false;
};
static inline int ofb_stage_out(ofb_ctx* ctx, int role, void* p, size_t bytes, OutStage* o)
{
    o->user = p; o->bytes = bytes; o->copy_back = false; o->dev = nullptr;
    if (!p || bytes == 0) return OFB_OK;
    if (ofb_is_device_ptr(p)) { o->dev = p; return OFB_OK; }
    OFB_TRY(ctx->scratch[role].reserve(bytes));
    o->dev = ctx->scratch[role].p; o->copy_back = true;
    return OFB_OK;
}
// enqueue copy-backs; returns true in *need_sync if any host output was written
static inline int ofb_finish_out(ofb_ctx* ctx, OutStage* outs, int n)
{
    bool any = false;
    for (int i = 0; i < n; ++i)
        if (outs[i].copy_back) {
            OFB_CUDA(cudaMemcpyAsync(outs[i].user, outs[i].dev, outs[i].bytes, cudaMemcpyDeviceToHost, ctx->stream));
            any = true;
        }
    if (any) OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    return OFB_OK;
}

#define OFB_LAUNCH_CHECK(ctx)                                                                   \
    do { (ctx)->launches++; OFB_CUDA(cudaGetLastError()); } while (0)

static inline int ofb_div_up(int a, int b) { return (a + b - 1) / b; }

// kernels launched with more than 48 KB of dynamic shared memory (slots of ofb_ctx::func_smem)
enum {
    FS_MARCH = 0,            // + 2 * {bs 3, 7, 12} + write_map          (6 slots)
    FS_TILE = 6,             // + 2 * {bs 3, 7, runtime} + write_map     (6 slots)
    FS_CAND = 12,            // + write_map                              (2 slots)
    FS_SELECT = 14,          // + {256, 512, 1024 threads}               (3 slots)
    FS_LK = 17,
    FS_PYR_TOP = 18,
    FS_SELECT16 = 19,        // + {256, 512, 1024 threads}: non-portable cluster size (16) allowed     (3 slots)
    FS_MARCH_LEAN = 22,      // + 2 * {bs 3, 7, 12} + write_map: the marching kernel without the general row loop (6 slots)
    FS_LK_FB = 28            // the generic LK kernel with the forward-backward check
};
// Raises a kernel's dynamic shared-memory limit on the context's device when this context has not done so yet.
template <class F>
static inline int ofb_ensure_smem(ofb_ctx* ctx, int slot, F func, size_t smem)
{
    if (smem <= 48 * 1024 || smem <= ctx->func_smem[slot]) return OFB_OK;
    OFB_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ctx->func_smem[slot] = smem;
    return OFB_OK;
}

// stage entry points implemented in the per-stage translation units (device pointers only)
int ofb_pyr_build_device(ofb_ctx* ctx, ofb_pyr* pyr);
int ofb_pyr_build_from(ofb_ctx* ctx, ofb_pyr* pyr, int first_level);
int ofb_pyr_ingest_bgr(ofb_ctx* ctx, ofb_pyr* pyr, const uint8_t* bgr, int bpitch, size_t bstride);
int ofb_pyr_alloc(ofb_ctx* ctx, const uint8_t* img, int w, int h, int pitch, size_t image_stride, int n_images,
                  int max_level, ofb_pyr** out);
int ofb_pyr_prepare(ofb_ctx* ctx, ofb_pyr** slot, const uint8_t* img, int w, int h, int pitch, size_t image_stride,
                    int n_images, int capacity, int max_level, bool build);
