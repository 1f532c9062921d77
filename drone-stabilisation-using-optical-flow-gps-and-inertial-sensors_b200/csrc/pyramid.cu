// pyramid.cu -- stage 0/1: BGR->grey and the Gaussian image pyramid.
//
// Replaces cv2.cvtColor(COLOR_BGR2GRAY) (velocity_measurment_node:113) and the pyramid that
// cv2.calcOpticalFlowPyrLK builds internally on every call (velocity_measurment_node:133,
// flight_experiments/evaluate_exp.py:98, optical_flow_experiments/of_module.py:88): pyrDown =
// separable [1 4 6 4 1]/16 in both axes, decimate by two, reflect-101 borders, integer
// (sum + 128) >> 8 -- bit-exact with OpenCV (SURVEY App. B.2).
//
// Persistent CTAs walk the 64x32 output tiles of the whole batch. The 160x67-byte source footprint of a tile is
// staged in shared memory by the TMA engine (cp.async.bulk.tensor through a 3-D tensor map {x, y, image}, completion on an mbarrier) into
// one of two stages, so the copy of the next tile overlaps the filtering of the current one (border tiles: 128-bit
// loads plus a reflect-101 byte gather for the groups that cross the image edge). Every thread then produces a 4x2
// block of outputs: the horizontal 5-tap filter of four adjacent outputs is eight dp4a on re-aligned
// words (funnel shifts) per source row, seven source rows feed both output rows, and each output row is
// written with one 32-bit store. Source bytes are read from HBM exactly once per level (plus halo):
// algorithmic bytes per level = w*h read + ((w+1)/2)*((h+1)/2) written.
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>

namespace {

constexpr int PT_W = 64, PT_H = 32;                 // output tile
constexpr int PS_W = 2 * PT_W + 32;                 // staged source columns: 2*X0-16 .. 2*X0+143 (10 x 16 bytes)
constexpr int PS_H = 2 * PT_H + 3;                  // staged source rows:    2*Y0-2 .. 2*Y0+64
constexpr int PS_PITCH = PS_W;                      // bytes, multiple of 16
constexpr int PYR_THREADS = 256;                    // threads of the two down-sampling kernels (the filter uses 128)

__device__ __forceinline__ int refl101(int p, int len)
{
    if (len == 1) return 0;
    while ((unsigned)p >= (unsigned)len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}

// Branch-free reflect-101 + clamp: exact wherever one reflection suffices (|overshoot| < len), which covers
// every source position a needed output reads when len >= 3; positions beyond that are never consumed.
__device__ __forceinline__ int refl101_bf(int p, int len)
{
    p = p < 0 ? -p : p;
    p = p >= len ? 2 * len - 2 - p : p;
    return max(0, min(p, len - 1));
}

// ---- TMA (bulk-copy) + mbarrier helpers: raw PTX, sm_90+/sm_100a ---------------------------------------
__device__ __forceinline__ unsigned int smem_u32(const void* p) { return (unsigned int)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned int bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned int parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one tile (PS_W x PS_H bytes of image z at (x,y)) : global -> shared through the tensor map, completion
// counted in bytes on the mbarrier (SASS: UTMALDG)
__device__ __forceinline__ void tma_tile_g2s(void* dst, const CUtensorMap* tmap, int x, int y, int z, unsigned long long* bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_u32(dst)), "l"(tmap), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Stage the source footprint of tile (X0,Y0) into `tile`: interior tiles by the TMA engine (one bulk copy per
// row, completion on `bar`), border tiles by a reflect-101 gather. Returns true when the copy is asynchronous.
__device__ __forceinline__ bool pyr_stage_tile(const CUtensorMap* tmap, bool use_tma, int img, const uint8_t* __restrict__ s,
                                               int sw, int sh, int spitch, int X0, int Y0, uint8_t* tile,
                                               unsigned long long* bar, bool aligned, bool tiny)
{
    const int sx0 = 2 * X0 - 16, sy0 = 2 * Y0 - 2;   // source coordinate of tile[0][0]
    const bool interior = use_tma && sx0 >= 0 && sx0 + PS_W <= sw && sy0 >= 0 && sy0 + PS_H <= sh;
    if (interior) {
        if (threadIdx.x == 0) {
            mbar_expect_tx(bar, PS_H * PS_W);
            tma_tile_g2s(tile, tmap, sx0, sy0, img, bar);
        }
        return true;
    }
    // 16-byte groups: a group inside its (reflected) source row is one 128-bit load; only groups that cross
    // the image edge gather bytes (independent loads: a border tile costs one memory latency, not one per byte)
    uint4* t128 = (uint4*)tile;
    constexpr int GPR = PS_W / 16;
    for (int i = threadIdx.x; i < PS_H * GPR; i += (int)blockDim.x) {
        const int r = i / GPR, c = i - r * GPR;
        const int yy = tiny ? refl101(sy0 + r, sh) : refl101_bf(sy0 + r, sh);
        const int gx0 = sx0 + 16 * c;
        const uint8_t* row = s + (size_t)yy * spitch;
        uint4 v;
        if (aligned && gx0 >= 0 && gx0 + 16 <= sw) {
            v = __ldg((const uint4*)(row + gx0));
        } else {
            unsigned int wv[4] = {0, 0, 0, 0};
            // the filter never reads tile bytes 0..13 and 145..159 (outputs 4tx+k read bytes 8tx+14+2k .. +4):
            // the first group needs its last two bytes, the last group its first byte
            if (c == 0 && !tiny) {
                wv[3] = ((unsigned int)__ldg(row + refl101_bf(gx0 + 14, sw)) << 16) | ((unsigned int)__ldg(row + refl101_bf(gx0 + 15, sw)) << 24);
            } else if (c == GPR - 1 && !tiny) {
                wv[0] = (unsigned int)__ldg(row + refl101_bf(gx0, sw));
            } else if (tiny) {
                for (int j = 0; j < 16; ++j) wv[j >> 2] |= (unsigned int)__ldg(row + refl101(gx0 + j, sw)) << (8 * (j & 3));
            } else {
                unsigned int bv[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) bv[j] = __ldg(row + refl101_bf(gx0 + j, sw));
#pragma unroll
                for (int j = 0; j < 16; ++j) wv[j >> 2] |= bv[j] << (8 * (j & 3));
            }
            v = make_uint4(wv[0], wv[1], wv[2], wv[3]);
        }
        t128[r * (PS_PITCH / 16) + c] = v;
    }
    return false;
}

// Filters one staged tile: 128 of the CTA's 256 threads produce a 4x4 block of outputs each. An output row needs five input
// rows, two adjacent output rows share three of them: a thread that owns four output rows runs the horizontal pass over 11
// input rows (2.75 per output row; 3.5 with the 4x2 blocks of round 1, which cost 14 % more instructions per output). The
// vertical taps are accumulated as the rows come, so only the 16 running sums stay in registers.
__device__ __forceinline__ void pyr_filter_tile(const uint8_t* tile, uint8_t* __restrict__ d, int X0, int Y0, int dw, int dh,
                                                int dpitch)
{
    if (threadIdx.x >= 128) return;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // 16 x 8 threads, 4x4 outputs each
    const int ox = X0 + 4 * tx, oy = Y0 + 4 * ty;
    if (ox < dw && oy < dh) {
        // outputs ox..ox+3 need source columns 2ox-2 .. 2ox+8 = tile bytes 8tx+14 .. 8tx+24: words 2tx+3 .. 2tx+6
        // (local bytes j=0..15 <-> tile byte 8tx+12+j; taps of output k are j = 2+2k .. 6+2k);
        // output rows oy .. oy+3 need tile rows 8ty .. 8ty+10
        OFB_DEV_ASSERT((8 * ty + 10) * PS_PITCH + 4 * (2 * tx + 3 + 3) + 3 < PS_H * PS_PITCH);
        const uint32_t* t32 = (const uint32_t*)tile + (8 * ty) * (PS_PITCH / 4) + 2 * tx + 3;
        unsigned int acc[4][4];
#pragma unroll
        for (int rr = 0; rr < 4; ++rr)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[rr][k] = 0u;
#pragma unroll
        for (int r = 0; r < 11; ++r) {
            const uint32_t* row = t32 + r * (PS_PITCH / 4);
            const unsigned int w0 = row[0], w1 = row[1], w2 = row[2], w3 = row[3];
            const unsigned int f01 = __funnelshift_r(w0, w1, 16), f12 = __funnelshift_r(w1, w2, 16), f23 = __funnelshift_r(w2, w3, 16);
            unsigned int hs[4];
            hs[0] = __dp4a(f12, 0x00000001u, __dp4a(f01, 0x04060401u, 0u));
            hs[1] = __dp4a(w2, 0x00000001u, __dp4a(w1, 0x04060401u, 0u));
            hs[2] = __dp4a(f23, 0x00000001u, __dp4a(f12, 0x04060401u, 0u));
            hs[3] = __dp4a(w3, 0x00000001u, __dp4a(w2, 0x04060401u, 0u));
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int t = r - 2 * rr;                          // tap index of input row r in output row rr (compile time)
                if (t < 0 || t > 4) continue;
                const unsigned int wgt = (t == 0 || t == 4) ? 1u : (t == 2 ? 6u : 4u);
#pragma unroll
                for (int k = 0; k < 4; ++k) acc[rr][k] += wgt * hs[k];
            }
        }
        const bool vec_ok = ox + 3 < dw && ((dpitch & 3) == 0) && ((((size_t)d) & 3) == 0);
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
            if (oy + rr >= dh) break;
            unsigned int packed = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) packed |= ((acc[rr][k] + 128u) >> 8) << (8 * k);
            OFB_DEV_ASSERT(oy + rr >= 0 && oy + rr < dh && ox >= 0 && ox < dw && (!vec_ok || ox + 3 < dpitch));
            uint8_t* drow = d + (size_t)(oy + rr) * dpitch + ox;
            if (vec_ok) *(uint32_t*)drow = packed;
            else
                for (int k = 0; k < 4 && ox + k < dw; ++k) drow[k] = (uint8_t)(packed >> (8 * k));
        }
    }
}

// One tile per CTA, staged with direct loads (no mbarrier set-up): used for the small upper levels, which are
// latency-bound launches.
__global__ void __launch_bounds__(PYR_THREADS)
pyr_down_small_kernel(const uint8_t* __restrict__ src, int sw, int sh, int spitch, size_t sstride, uint8_t* __restrict__ dst,
                      int dw, int dh, int dpitch, size_t dstride)
{
    __shared__ __align__(16) uint8_t tile[PS_H * PS_PITCH];
    const uint8_t* s = src + (size_t)blockIdx.z * sstride;
    const bool aligned = ((spitch & 15) == 0) && ((((size_t)s) & 15) == 0);
    const bool tiny = sw < 4 || sh < 4;
    const int X0 = blockIdx.x * PT_W, Y0 = blockIdx.y * PT_H;
    pyr_stage_tile(nullptr, false, 0, s, sw, sh, spitch, X0, Y0, tile, nullptr, aligned, tiny);
    __syncthreads();
    pyr_filter_tile(tile, dst + (size_t)blockIdx.z * dstride, X0, Y0, dw, dh, dpitch);
}

// BGR frames (cv2.cvtColor(frame, COLOR_BGR2GRAY) at velocity_measurment_node:113 in front of the pyramid): one kernel
// converts the source footprint of a level-1 tile to grey in shared memory, writes the tile's own 128x64 block of the
// grey level 0 (LK tracks on it) and filters level 1 from shared memory -- the grey image is written once and never
// read back for the first pyramid level (the separate ingest + pyr_down pair wrote P and re-read P bytes per frame).
// A 16-pixel group is 48 BGR bytes = three 128-bit loads; a pixel's (B, G, R) is re-aligned to the low bytes of a word
// with one funnel shift and weighted by two dp2a: (3735 B + 19235 G) + (9798 R) + 2^14 >> 15, cv2's fixed-point rule.
__device__ __forceinline__ int dp2a_lo_u(unsigned int w16x2, unsigned int bytes, int c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w16x2), "r"(bytes), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi_u(unsigned int w16x2, unsigned int bytes, int c)
{
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w16x2), "r"(bytes), "r"(c));
    return d;
}
__device__ __forceinline__ unsigned int bgr_to_gray_word(unsigned int px)      // bytes 0..2 = B, G, R (byte 3 ignored)
{
    int v = dp2a_lo_u(3735u | (19235u << 16), px, 1 << 14);
    v = dp2a_hi_u(9798u, px, v);                                               // 9798 R + 0 * byte 3
    return (unsigned int)v >> 15;
}

__global__ void __launch_bounds__(256)
ingest_bgr_pyr_kernel(const uint8_t* __restrict__ bgr, int w, int h, int bpitch, size_t bstride,
                      uint8_t* __restrict__ gray, int gpitch, size_t gstride,
                      uint8_t* __restrict__ dst, int dw, int dh, int dpitch, size_t dstride)
{
    __shared__ __align__(16) uint8_t tile[PS_H * PS_PITCH];
    const uint8_t* __restrict__ src = bgr + (size_t)blockIdx.z * bstride;
    uint8_t* __restrict__ g0 = gray + (size_t)blockIdx.z * gstride;
    const int X0 = blockIdx.x * PT_W, Y0 = blockIdx.y * PT_H;
    const int sx0 = 2 * X0 - 16, sy0 = 2 * Y0 - 2;                 // source pixel of tile[0][0]
    const bool aligned = ((bpitch & 15) == 0) && ((((size_t)src) & 15) == 0) && ((gpitch & 15) == 0) && ((((size_t)g0) & 15) == 0);
    constexpr int GPR = PS_W / 16;                                 // 16-pixel groups per tile row
    // groups 1 .. GPR-2 = the tile's own 128 columns; of the two outer groups the filter reads only the last two /
    // the first pixel (see pyr_stage_tile), handled below
    for (int i = threadIdx.x; i < PS_H * (GPR - 2); i += 256) {
        const int r = i / (GPR - 2), c = 1 + i - r * (GPR - 2);
        const int y = sy0 + r, gx0 = sx0 + 16 * c;
        const int yy = refl101_bf(y, h);
        const uint8_t* __restrict__ row = src + (size_t)yy * bpitch;
        unsigned int out[4];
        if (aligned && gx0 + 16 <= w) {                            // (gx0 >= 0 for these groups)
            const uint4* __restrict__ q = (const uint4*)(row + 3 * gx0);
            const uint4 a = __ldg(q), b = __ldg(q + 1), d = __ldg(q + 2);
            const unsigned int wd[13] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, d.x, d.y, d.z, d.w, 0u};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                unsigned int packed = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int p = 4 * j + k, byte = 3 * p;          // pixel p starts at byte 3p of the 48-byte group
                    const unsigned int px = __funnelshift_r(wd[byte >> 2], wd[(byte >> 2) + 1], 8 * (byte & 3));
                    packed |= bgr_to_gray_word(px) << (8 * k);
                }
                out[j] = packed;
            }
        } else {                                                   // right image edge: per pixel, reflect-101 columns
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                unsigned int packed = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint8_t* __restrict__ p = row + 3 * refl101_bf(gx0 + 4 * j + k, w);
                    const unsigned int px = (unsigned int)__ldg(p) | ((unsigned int)__ldg(p + 1) << 8) | ((unsigned int)__ldg(p + 2) << 16);
                    packed |= bgr_to_gray_word(px) << (8 * k);
                }
                out[j] = packed;
            }
        }
        *(uint4*)(tile + r * PS_PITCH + 16 * c) = make_uint4(out[0], out[1], out[2], out[3]);
        // this tile's own block of the grey level 0: source rows 2Y0 .. 2Y0+63 of these columns
        if (r >= 2 && r < PS_H - 1 && y < h && gx0 < w) {
            uint8_t* __restrict__ o = g0 + (size_t)y * gpitch + gx0;
            if (aligned && gx0 + 16 <= w) *(uint4*)o = make_uint4(out[0], out[1], out[2], out[3]);
            else
                for (int k = 0; k < 16 && gx0 + k < w; ++k) o[k] = (uint8_t)(out[k >> 2] >> (8 * (k & 3)));
        }
    }
    for (int i = threadIdx.x; i < PS_H * 3; i += 256) {            // halo columns: tile bytes 14, 15 and 144
        const int r = i / 3, e = i - r * 3;
        const int j = e < 2 ? 14 + e : 16 * (GPR - 1);
        const uint8_t* __restrict__ p = src + (size_t)refl101_bf(sy0 + r, h) * bpitch + 3 * refl101_bf(sx0 + j, w);
        const unsigned int px = (unsigned int)__ldg(p) | ((unsigned int)__ldg(p + 1) << 8) | ((unsigned int)__ldg(p + 2) << 16);
        tile[r * PS_PITCH + j] = (uint8_t)bgr_to_gray_word(px);
    }
    __syncthreads();
    pyr_filter_tile(tile, dst + (size_t)blockIdx.z * dstride, X0, Y0, dw, dh, dpitch);
}

// Persistent kernel: each CTA walks tiles t = blockIdx.x, +gridDim.x, ... of the whole batch with two shared-
// memory stages: the TMA copy of tile i+1 is in flight while tile i is filtered.
__global__ void __launch_bounds__(PYR_THREADS)
pyr_down_kernel(const __grid_constant__ CUtensorMap tmap, int use_tma, const uint8_t* __restrict__ src, int sw, int sh, int spitch,
                size_t sstride, uint8_t* __restrict__ dst, int dw, int dh, int dpitch, size_t dstride, int tiles_x, int tiles_y,
                int n_tiles)
{
    constexpr int STAGE_BYTES = (PS_H * PS_PITCH + 127) & ~127;    // TMA destinations must be 128-byte aligned
    __shared__ __align__(128) uint8_t tiles[2][STAGE_BYTES];
    __shared__ __align__(8) unsigned long long bars[2];
    const bool aligned = ((spitch & 15) == 0) && ((((size_t)src) & 15) == 0) && ((sstride & 15) == 0);
    const bool tiny = sw < 4 || sh < 4;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int per_img = tiles_x * tiles_y;
    unsigned int phase[2] = {0, 0};
    bool async_[2] = {false, false};
    int t = blockIdx.x;
    if (t >= n_tiles) return;
    // tile coordinates advance by gridDim.x tiles per step: one division up front, carries afterwards
    const int G = gridDim.x;
    const int d_img = G / per_img, d_rem = G - d_img * per_img, d_ty = d_rem / tiles_x, d_tx = d_rem - d_ty * tiles_x;
    int img = t / per_img, ty_, tx_;
    { const int rem = t - img * per_img; ty_ = rem / tiles_x; tx_ = rem - ty_ * tiles_x; }
    int nimg = img, nty = ty_, ntx = tx_;
    auto advance = [&](int& im, int& y, int& x) {
        x += d_tx; if (x >= tiles_x) { x -= tiles_x; ++y; }
        y += d_ty; if (y >= tiles_y) { y -= tiles_y; ++im; }
        im += d_img;
    };
    async_[0] = pyr_stage_tile(&tmap, use_tma != 0, img, src + (size_t)img * sstride, sw, sh, spitch, tx_ * PT_W, ty_ * PT_H, tiles[0],
                               &bars[0], aligned, tiny);
    for (int it = 0; t < n_tiles; t += G, ++it) {
        const int st = it & 1;
        advance(nimg, nty, ntx);
        if (t + G < n_tiles)         // prefetch the next tile into the other stage (free since the barrier at loop end)
            async_[st ^ 1] = pyr_stage_tile(&tmap, use_tma != 0, nimg, src + (size_t)nimg * sstride, sw, sh, spitch, ntx * PT_W,
                                            nty * PT_H, tiles[st ^ 1], &bars[st ^ 1], aligned, tiny);
        if (async_[st]) { mbar_wait(&bars[st], phase[st]); phase[st] ^= 1; }
        else __syncthreads();        // gathered tile: make the generic-proxy stores visible
        pyr_filter_tile(tiles[st], dst + (size_t)img * dstride, tx_ * PT_W, ty_ * PT_H, dw, dh, dpitch);
        img = nimg; ty_ = nty; tx_ = ntx;
        fence_proxy_async();         // this stage is refilled by the async proxy two tiles from now
        __syncthreads();
    }
}

__global__ void bgr2gray_kernel(const uint8_t* __restrict__ bgr, int w, int h, int pitch, uint8_t* __restrict__ gray,
                                int gpitch)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w || y >= h) return;
    const uint8_t* p = bgr + (size_t)y * pitch + 3 * x;
    gray[(size_t)y * gpitch + x] = (uint8_t)((3735 * p[0] + 19235 * p[1] + 9798 * p[2] + (1 << 14)) >> 15);
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
static PFN_cuTensorMapEncodeTiled tensor_map_encoder()
{
    static PFN_cuTensorMapEncodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_cuTensorMapEncodeTiled)f;
        else cudaGetLastError();
    }
    return fn;
}

int ofb_pyr_build_device(ofb_ctx* ctx, ofb_pyr* p) { return ofb_pyr_build_from(ctx, p, 1); }

// Fused first step for BGR frames: grey level 0 (into `gray`, which must be the pyramid's level 0) and level 1 from one
// read of the BGR frames, then the remaining levels as usual. Images too small for the fused tile kernel's single
// reflection (or pyramids without a level 1) are converted by the caller and built with ofb_pyr_build_device.
int ofb_pyr_ingest_bgr(ofb_ctx* ctx, ofb_pyr* p, const uint8_t* bgr, int bpitch, size_t bstride)
{
    OFB_REQUIRE(p->n_levels >= 2 && p->w[0] >= 4 && p->h[0] >= 4, "pyr_ingest_bgr: needs a level 1 and an image of at least 4x4");
    const int tiles_x = ofb_div_up(p->w[1], PT_W), tiles_y = ofb_div_up(p->h[1], PT_H);
    dim3 g3(tiles_x, tiles_y, p->n_active);
    ingest_bgr_pyr_kernel<<<g3, 256, 0, ctx->stream>>>(bgr, p->w[0], p->h[0], bpitch, bstride, (uint8_t*)p->level0, p->level0_pitch,
                                                      p->level0_stride, p->base + p->level_off[1], p->w[1], p->h[1], p->pitch[1],
                                                      p->image_stride[1]);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_pyr_build_from(ctx, p, 2);
}

int ofb_pyr_build_from(ofb_ctx* ctx, ofb_pyr* p, int first_level)
{
    for (int l = first_level; l < p->n_levels; ++l) {
        const uint8_t* s; int sp; size_t ss;
        if (l == 1) { s = p->level0; sp = p->level0_pitch; ss = p->level0_stride; }
        else { s = p->base + p->level_off[l - 1]; sp = p->pitch[l - 1]; ss = p->image_stride[l - 1]; }
        const int tiles_x = ofb_div_up(p->w[l], PT_W), tiles_y = ofb_div_up(p->h[l], PT_H);
        const long long n_tiles = (long long)tiles_x * tiles_y * p->n_active;
        OFB_REQUIRE(n_tiles < (1ll << 31), "pyramid: batch too large");
        // persistent CTAs: 5 per SM are resident (48 registers x 256 threads, 21.5 KB of shared memory each);
        // fewer tiles -> one CTA per tile
        // (the in-CTA double buffering pays once a CTA owns several tiles; a level with fewer than ~4 tiles per
        // resident CTA runs one tile per CTA and relies on the 5 co-resident CTAs to overlap copy and filter)
        long long grid = (long long)ctx->sm_count * (5 * 256 / PYR_THREADS);
        if (n_tiles < grid * 4) grid = n_tiles;
        if (grid == n_tiles) {
            // small level: latency-bound, one tile per CTA with direct loads
            dim3 g3(tiles_x, tiles_y, p->n_active);
            pyr_down_small_kernel<<<g3, PYR_THREADS, 0, ctx->stream>>>(s, p->w[l - 1], p->h[l - 1], sp, ss, p->base + p->level_off[l],
                                                              p->w[l], p->h[l], p->pitch[l], p->image_stride[l]);
            OFB_LAUNCH_CHECK(ctx);
            continue;
        }
        CUtensorMap tmap;
        memset(&tmap, 0, sizeof(tmap));
        int use_tma = 0;
        if (PFN_cuTensorMapEncodeTiled enc = tensor_map_encoder()) {
            // source level as a 3-D u8 tensor {x, y, image}; strides must be multiples of 16 bytes
            if ((((size_t)s) & 15) == 0 && (sp & 15) == 0 && (ss & 15) == 0 && p->w[l - 1] >= PS_W && p->h[l - 1] >= PS_H) {
                cuuint64_t gdim[3] = {(cuuint64_t)p->w[l - 1], (cuuint64_t)p->h[l - 1], (cuuint64_t)p->n_active};
                cuuint64_t gstr[2] = {(cuuint64_t)sp, (cuuint64_t)(p->n_active > 1 ? ss : (size_t)sp * p->h[l - 1])};
                if (gstr[1] < gstr[0] * gdim[1]) gstr[1] = gstr[0] * gdim[1];
                cuuint32_t box[3] = {(cuuint32_t)PS_W, (cuuint32_t)PS_H, 1};
                cuuint32_t estr[3] = {1, 1, 1};
                CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)s, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                 CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                use_tma = (r == CUDA_SUCCESS) ? 1 : 0;
            }
        }
        pyr_down_kernel<<<(unsigned int)grid, PYR_THREADS, 0, ctx->stream>>>(tmap, use_tma, s, p->w[l - 1], p->h[l - 1], sp, ss,
                                                                    p->base + p->level_off[l], p->w[l], p->h[l], p->pitch[l],
                                                                    p->image_stride[l], tiles_x, tiles_y, (int)n_tiles);
        OFB_LAUNCH_CHECK(ctx);
    }
    return OFB_OK;
}

static int pyr_upload_level0(ofb_ctx* ctx, ofb_pyr* p, const uint8_t* img, int pitch, size_t image_stride)
{
    cudaStream_t s = ctx->upload_stream ? ctx->upload_stream : ctx->stream;
    if (pitch == p->pitch[0] && image_stride == p->image_stride[0]) {       // same layout on both sides: one copy
        OFB_CUDA(cudaMemcpyAsync(p->base + p->level_off[0], img, image_stride * (size_t)(p->n_active - 1) +
                                 (size_t)pitch * (p->h[0] - 1) + p->w[0], cudaMemcpyHostToDevice, s));
        return OFB_OK;
    }
    for (int i = 0; i < p->n_active; ++i)
        OFB_CUDA(cudaMemcpy2DAsync(p->base + p->level_off[0] + (size_t)i * p->image_stride[0], p->pitch[0],
                                   img + (size_t)i * image_stride, pitch, p->w[0], p->h[0], cudaMemcpyHostToDevice, s));
    return OFB_OK;
}

// Allocates the pyramid object and its level storage. When `img` is device memory level 0 aliases
// it (the caller keeps it alive while the pyramid is in use); host images are copied in.
static int ofb_pyr_alloc_cap(ofb_ctx* ctx, const uint8_t* img, int w, int h, int pitch, size_t image_stride, int n_active,
                             int n_images, int max_level, ofb_pyr** out, bool upload = true)
{
    ofb_pyr* p = new ofb_pyr();
    p->n_images = n_images;
    p->n_active = n_active;
    bool dev = upload && ofb_is_device_ptr(img);         // (!upload: level 0 is owned and filled by a kernel)
    int lw = w, lh = h, nl = 1;
    p->w[0] = w; p->h[0] = h;
    for (int l = 1; l <= max_level && l < OFB_MAX_LEVELS; ++l) {
        lw = (lw + 1) / 2; lh = (lh + 1) / 2;
        p->w[l] = lw; p->h[l] = lh; nl = l + 1;
        if (lw == 1 && lh == 1) break;
    }
    p->n_levels = nl;
    size_t off = 0;
    for (int l = 0; l < nl; ++l) {
        if (l == 0 && dev) { p->pitch[0] = pitch; p->level_off[0] = 0; p->image_stride[0] = image_stride; continue; }
        // level 0 (host frames copied in): tight 16-aligned pitch, so that frames whose width is a multiple
        // of 16 and whose size is a multiple of 256 land with ONE contiguous H2D copy per sub-batch
        p->pitch[l] = (int)align_up((size_t)p->w[l] + (l == 0 ? 0 : 4), 16);
        p->image_stride[l] = align_up((size_t)p->pitch[l] * p->h[l], 256);
        p->level_off[l] = off;
        off += p->image_stride[l] * n_images;
    }
    p->bytes = off + 256;
    cudaError_t e = cudaMalloc((void**)&p->base, p->bytes);
    if (e != cudaSuccess) {
        ofb_set_error("pyramid: cudaMalloc(%zu) failed: %s", p->bytes, cudaGetErrorString(e));
        delete p;
        return OFB_E_NOMEM;
    }
    if (dev) {
        p->level0 = img; p->level0_pitch = pitch; p->level0_stride = image_stride; p->level0_owned = false;
    } else {
        p->level0 = p->base + p->level_off[0]; p->level0_pitch = p->pitch[0]; p->level0_stride = p->image_stride[0];
        p->level0_owned = true;
        int r = upload ? pyr_upload_level0(ctx, p, img, pitch, image_stride) : OFB_OK;
        if (r != OFB_OK) { cudaFree(p->base); delete p; return r; }
    }
    *out = p;
    return OFB_OK;
}

int ofb_pyr_alloc(ofb_ctx* ctx, const uint8_t* img, int w, int h, int pitch, size_t image_stride, int n_images,
                  int max_level, ofb_pyr** out)
{
    return ofb_pyr_alloc_cap(ctx, img, w, h, pitch, image_stride, n_images, n_images, max_level, out);
}

// Workspace pyramid for the fused path: reuses *slot when geometry and residency match (capacity >= n_images),
// so a steady stream of frame pairs never reallocates. build=false only refreshes level 0 (upload on
// ctx->upload_stream when set); the caller then runs ofb_pyr_build_device on the compute stream.
int ofb_pyr_prepare(ofb_ctx* ctx, ofb_pyr** slot, const uint8_t* img, int w, int h, int pitch, size_t image_stride,
                    int n_images, int capacity, int max_level, bool build)
{
    ofb_pyr* p = *slot;
    bool dev = ofb_is_device_ptr(img);
    if (capacity < n_images) capacity = n_images;
    int want_levels = 1; { int lw = w, lh = h; for (int l = 1; l <= max_level && l < OFB_MAX_LEVELS; ++l) { lw = (lw + 1) / 2; lh = (lh + 1) / 2; want_levels = l + 1; if (lw == 1 && lh == 1) break; } }
    if (p && p->n_images >= n_images && p->n_images <= 2 * capacity && p->w[0] == w && p->h[0] == h &&
        p->n_levels == want_levels && p->level0_owned == !dev) {
        p->n_active = n_images;
        if (dev) { p->level0 = img; p->level0_pitch = pitch; p->level0_stride = image_stride; p->pitch[0] = pitch; p->image_stride[0] = image_stride; }
        else OFB_TRY(pyr_upload_level0(ctx, p, img, pitch, image_stride));
    } else {
        if (p) { cudaDeviceSynchronize(); cudaFree(p->base); delete p; *slot = nullptr; }
        // allocate for `capacity` images, use n_images of them
        OFB_TRY(ofb_pyr_alloc_cap(ctx, img, w, h, pitch, image_stride, n_images, capacity, max_level, &p));
        *slot = p;
    }
    return build ? ofb_pyr_build_device(ctx, p) : OFB_OK;
}

extern "C" int ofb_pyramid(ofb_ctx* ctx, const uint8_t* img, int w, int h, int pitch, size_t image_stride,
                           int n_images, int max_level, ofb_pyr** out)
{
    OFB_REQUIRE(ctx && img && out, "pyramid: null argument");
    OFB_REQUIRE(w > 0 && h > 0 && pitch >= w, "pyramid: bad image geometry %dx%d pitch %d", w, h, pitch);
    OFB_REQUIRE(n_images > 0 && n_images <= 65535, "pyramid: n_images must be in 1..65535");
    OFB_REQUIRE(max_level >= 0, "pyramid: max_level must be >= 0");
    OFB_REQUIRE(n_images == 1 || image_stride >= (size_t)pitch * (h - 1) + w, "pyramid: image_stride too small");
    OFB_CUDA(cudaSetDevice(ctx->device));
    ofb_pyr* p = nullptr;
    OFB_TRY(ofb_pyr_alloc(ctx, img, w, h, pitch, image_stride, n_images, max_level, &p));
    int r = ofb_pyr_build_device(ctx, p);
    if (r != OFB_OK) { cudaFree(p->base); delete p; return r; }
    ctx->pyramids.push_back(p);
    *out = p;
    return OFB_OK;
}

extern "C" int ofb_pyramid_bgr(ofb_ctx* ctx, const uint8_t* bgr, int w, int h, int pitch, size_t image_stride,
                               int n_images, int max_level, ofb_pyr** out)
{
    OFB_REQUIRE(ctx && bgr && out, "pyramid_bgr: null argument");
    OFB_REQUIRE(w > 0 && h > 0 && pitch >= 3 * w, "pyramid_bgr: bad image geometry %dx%d pitch %d", w, h, pitch);
    OFB_REQUIRE(n_images > 0 && n_images <= 65535, "pyramid_bgr: n_images must be in 1..65535");
    OFB_REQUIRE(max_level >= 0, "pyramid_bgr: max_level must be >= 0");
    OFB_REQUIRE(n_images == 1 || image_stride >= (size_t)pitch * (h - 1) + 3 * (size_t)w, "pyramid_bgr: image_stride too small");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void* dsrc;
    const size_t bytes = image_stride * (size_t)(n_images - 1) + (size_t)pitch * (h - 1) + 3 * (size_t)w;
    OFB_TRY(ofb_stage_in(ctx, SC_FRAMES, bgr, bytes, &dsrc));
    ofb_pyr* p = nullptr;
    OFB_TRY(ofb_pyr_alloc_cap(ctx, nullptr, w, h, 0, 0, n_images, n_images, max_level, &p, false));
    int r;
    if (p->n_levels >= 2 && w >= 4 && h >= 4) r = ofb_pyr_ingest_bgr(ctx, p, (const uint8_t*)dsrc, pitch, image_stride);
    else {
        // no level 1 (or a tiny image): plain conversion, then the generic level kernels
        r = OFB_OK;
        for (int i = 0; i < n_images && r == OFB_OK; ++i) {
            dim3 grid(ofb_div_up(w, 256), h);
            bgr2gray_kernel<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)dsrc + (size_t)i * image_stride, w, h, pitch,
                                                          (uint8_t*)p->level0 + (size_t)i * p->level0_stride, p->level0_pitch);
            ctx->launches++;
            if (cudaGetLastError() != cudaSuccess) { ofb_set_error("pyramid_bgr: conversion launch failed"); r = OFB_E_CUDA; }
        }
        if (r == OFB_OK) r = ofb_pyr_build_device(ctx, p);
    }
    if (r != OFB_OK) { cudaFree(p->base); delete p; return r; }
    ctx->pyramids.push_back(p);
    *out = p;
    return OFB_OK;
}

extern "C" int ofb_pyr_free(ofb_ctx* ctx, ofb_pyr* pyr)
{
    OFB_REQUIRE(ctx && pyr, "pyr_free: null argument");
    for (size_t i = 0; i < ctx->pyramids.size(); ++i)
        if (ctx->pyramids[i] == pyr) {
            ctx->pyramids.erase(ctx->pyramids.begin() + i);
            cudaStreamSynchronize(ctx->stream);
            cudaFree(pyr->base);
            delete pyr;
            return OFB_OK;
        }
    ofb_set_error("pyr_free: pyramid does not belong to this context");
    return OFB_E_INVALID;
}

extern "C" int ofb_pyr_info(const ofb_pyr* pyr, int* n_images, int* n_levels, int* widths, int* heights, int* pitches)
{
    OFB_REQUIRE(pyr, "pyr_info: null pyramid");
    if (n_images) *n_images = pyr->n_images;
    if (n_levels) *n_levels = pyr->n_levels;
    for (int l = 0; l < pyr->n_levels; ++l) {
        if (widths) widths[l] = pyr->w[l];
        if (heights) heights[l] = pyr->h[l];
        if (pitches) pitches[l] = l == 0 ? pyr->level0_pitch : pyr->pitch[l];
    }
    return OFB_OK;
}

extern "C" int ofb_pyr_download(ofb_ctx* ctx, const ofb_pyr* pyr, int image, int level, uint8_t* dst, int dst_pitch)
{
    OFB_REQUIRE(ctx && pyr && dst, "pyr_download: null argument");
    OFB_REQUIRE(image >= 0 && image < pyr->n_images && level >= 0 && level < pyr->n_levels,
                "pyr_download: image/level out of range");
    OFB_REQUIRE(dst_pitch >= pyr->w[level], "pyr_download: dst_pitch too small");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const uint8_t* s; int sp;
    if (level == 0) { s = pyr->level0 + (size_t)image * pyr->level0_stride; sp = pyr->level0_pitch; }
    else { s = pyr->base + pyr->level_off[level] + (size_t)image * pyr->image_stride[level]; sp = pyr->pitch[level]; }
    OFB_CUDA(cudaMemcpy2DAsync(dst, dst_pitch, s, sp, pyr->w[level], pyr->h[level], cudaMemcpyDefault, ctx->stream));
    OFB_CUDA(cudaStreamSynchronize(ctx->stream));
    return OFB_OK;
}

extern "C" int ofb_bgr2gray(ofb_ctx* ctx, const uint8_t* bgr, int w, int h, int pitch, uint8_t* gray, int gray_pitch)
{
    OFB_REQUIRE(ctx && bgr && gray, "bgr2gray: null argument");
    OFB_REQUIRE(w > 0 && h > 0 && pitch >= 3 * w && gray_pitch >= w, "bgr2gray: bad geometry");
    OFB_CUDA(cudaSetDevice(ctx->device));
    const void* din;
    OFB_TRY(ofb_stage_in(ctx, SC_IN0, bgr, (size_t)pitch * h, &din));
    OutStage o;
    OFB_TRY(ofb_stage_out(ctx, SC_OUT0, gray, (size_t)gray_pitch * h, &o));
    dim3 grid(ofb_div_up(w, 256), h);
    bgr2gray_kernel<<<grid, 256, 0, ctx->stream>>>((const uint8_t*)din, w, h, pitch, (uint8_t*)o.dev, gray_pitch);
    OFB_LAUNCH_CHECK(ctx);
    return ofb_finish_out(ctx, &o, 1);
}
