// Flow-driven bilinear backward warps for sm_100a.
//
//  * warp_torch_kernel  -- zero-padded warp, bit-compatible with
//    SpatialTransformation.forward (sff_scripts_unfolding/utils/image_warp_torch.py:97-113).
//  * image_warp_kernel  -- clamp-border warp with numpy image_warp semantics
//    (simu_sff/image_warp.py:3-111), NHWC, uint8 truncation.
//
// Both are HBM-bound gathers: per output pixel 8 B of flow, 4*C B of image
// (each source pixel is touched by ~4 neighbouring outputs, served by L1/L2) and
// 4*C B of output.  One thread owns PX horizontally adjacent pixels so flow
// loads and output stores are 16-byte vectors when the row is aligned; all
// arithmetic uses the non-contracting intrinsics (__fadd_rn/__fmul_rn/__fsub_rn)
// in the reference's operation order, so results are bit-equal to the CPU run of
// the reference, not merely close.
#include "common.cuh"
#include "tma.cuh"
#include <cuda.h>
#include <stdlib.h>
#include <type_traits>

namespace sstem {

struct BilinearTap {
    int x0, x1, y0, y1;  // coordinates in the 1-px zero-padded image, clamped to it
    float wa, wb, wc, wd;
};

// image_warp_torch.py:43-57,82-91: x = (fx + j) + 1, floor, +1, clamp, weights from the clamped x1/y1
__device__ __forceinline__ BilinearTap torch_tap(float fx, float fy, int i, int j, int H, int W) {
    BilinearTap t;
    const float x = __fadd_rn(__fadd_rn(fx, (float)j), 1.0f);
    const float y = __fadd_rn(__fadd_rn(fy, (float)i), 1.0f);
    const float xf = floorf(x), yf = floorf(y);
    const float mx = (float)(W + 1), my = (float)(H + 1);
    // clamp(floor(x)) and clamp(floor(x) + 1) -- done in float so huge |flow| cannot overflow
    const float x0c = fminf(fmaxf(xf, 0.f), mx), x1c = fminf(fmaxf(__fadd_rn(xf, 1.0f), 0.f), mx);
    const float y0c = fminf(fmaxf(yf, 0.f), my), y1c = fminf(fmaxf(__fadd_rn(yf, 1.0f), 0.f), my);
    t.x0 = (int)x0c; t.x1 = (int)x1c; t.y0 = (int)y0c; t.y1 = (int)y1c;
    const float dx = __fsub_rn(x1c, x), dy = __fsub_rn(y1c, y);
    const float ex = __fsub_rn(1.0f, dx), ey = __fsub_rn(1.0f, dy);
    t.wa = __fmul_rn(dx, dy);
    t.wb = __fmul_rn(dx, ey);
    t.wc = __fmul_rn(ex, dy);
    t.wd = __fmul_rn(ex, ey);
    return t;
}

// sample of the zero-padded image at padded coordinates (py, px)
__device__ __forceinline__ float padded_at(const float* __restrict__ im, int py, int px, int H, int W) {
    const int yy = py - 1, xx = px - 1;
    return ((unsigned)yy < (unsigned)H && (unsigned)xx < (unsigned)W) ? __ldg(im + (int64_t)yy * W + xx) : 0.f;
}

// CT = compile-time channel count (0 = runtime loop).  With CT > 0 all 4*CT*PX gathers of a
// thread are independent straight-line loads, so they are in flight together.
#ifndef SSTEM_WARP_PX
#define SSTEM_WARP_PX 1
#endif
#ifndef SSTEM_WARP_MINB
#define SSTEM_WARP_MINB 6
#endif
template <int PX, bool NHWC, int CT>
__global__ void __launch_bounds__(256, SSTEM_WARP_MINB)
warp_torch_kernel(const float* __restrict__ moving, const float* __restrict__ flow,
                  int64_t fs_b, int64_t fs_h, int64_t fs_w, int64_t fs_c,
                  float* __restrict__ out, int C, int H, int W, int groups_per_row, int64_t total_groups) {
    const int64_t gidx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gidx >= total_groups) return;
    const int gx = (int)(gidx % groups_per_row);
    const int i = (int)((gidx / groups_per_row) % H);
    const int64_t b = gidx / ((int64_t)groups_per_row * H);
    const int j0 = gx * PX;
    const int64_t plane = (int64_t)H * W;
    const int nc = CT > 0 ? CT : C;

    const float* frow = flow + b * fs_b + (int64_t)i * fs_h;
    const bool full = (j0 + PX <= W);
    // flow: vector loads when the two components are separate contiguous planes
    // (the layout at every reference call site) or interleaved pairs
    float fxv[PX], fyv[PX];
    if (PX == 4 && full && fs_w == 1 && (((uintptr_t)(frow + j0) | (uintptr_t)(frow + fs_c + j0)) & 15u) == 0) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(frow + j0));
        const float4 c = __ldcs(reinterpret_cast<const float4*>(frow + fs_c + j0));
        fxv[0] = a.x; fxv[1 % PX] = a.y; fxv[2 % PX] = a.z; fxv[3 % PX] = a.w;
        fyv[0] = c.x; fyv[1 % PX] = c.y; fyv[2 % PX] = c.z; fyv[3 % PX] = c.w;
    } else if (PX == 2 && full && fs_w == 1 && (((uintptr_t)(frow + j0) | (uintptr_t)(frow + fs_c + j0)) & 7u) == 0) {
        const float2 a = __ldcs(reinterpret_cast<const float2*>(frow + j0));
        const float2 c = __ldcs(reinterpret_cast<const float2*>(frow + fs_c + j0));
        fxv[0] = a.x; fxv[1 % PX] = a.y; fyv[0] = c.x; fyv[1 % PX] = c.y;
    } else if (PX == 4 && full && fs_w == 2 && fs_c == 1 && ((uintptr_t)(frow + 2 * j0) & 15u) == 0) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(frow + 2 * j0));
        const float4 c = __ldcs(reinterpret_cast<const float4*>(frow + 2 * j0 + 4));
        fxv[0] = a.x; fyv[0] = a.y; fxv[1 % PX] = a.z; fyv[1 % PX] = a.w;
        fxv[2 % PX] = c.x; fyv[2 % PX] = c.y; fxv[3 % PX] = c.z; fyv[3 % PX] = c.w;
    } else {
#pragma unroll
        for (int p = 0; p < PX; ++p) {
            const int j = min(j0 + p, W - 1);
            fxv[p] = __ldg(frow + (int64_t)j * fs_w);
            fyv[p] = __ldg(frow + (int64_t)j * fs_w + fs_c);
        }
    }
    // per pixel: the 4 source offsets inside a plane (or -1 when the tap lies in the zero border)
    int oa[PX], ob[PX], oc[PX], od[PX];
    float wa[PX], wb[PX], wc[PX], wd[PX];
#pragma unroll
    for (int p = 0; p < PX; ++p) {
        const BilinearTap t = torch_tap(fxv[p], fyv[p], i, j0 + p, H, W);
        const int xa = t.x0 - 1, xb = t.x1 - 1, ya = t.y0 - 1, yb = t.y1 - 1;
        const bool vxa = (unsigned)xa < (unsigned)W, vxb = (unsigned)xb < (unsigned)W;
        const bool vya = (unsigned)ya < (unsigned)H, vyb = (unsigned)yb < (unsigned)H;
        oa[p] = (vya && vxa) ? ya * W + xa : -1;      // (y0, x0)
        ob[p] = (vyb && vxa) ? yb * W + xa : -1;      // (y1, x0)
        oc[p] = (vya && vxb) ? ya * W + xb : -1;      // (y0, x1)
        od[p] = (vyb && vxb) ? yb * W + xb : -1;      // (y1, x1)
        wa[p] = t.wa; wb[p] = t.wb; wc[p] = t.wc; wd[p] = t.wd;
    }
    auto channel = [&](int c) {
        const float* im = moving + (b * nc + c) * plane;
        float Ia[PX], Ib[PX], Ic[PX], Id[PX];
#pragma unroll
        for (int p = 0; p < PX; ++p) {
            Ia[p] = oa[p] >= 0 ? __ldg(im + oa[p]) : 0.f;
            Ib[p] = ob[p] >= 0 ? __ldg(im + ob[p]) : 0.f;
            Ic[p] = oc[p] >= 0 ? __ldg(im + oc[p]) : 0.f;
            Id[p] = od[p] >= 0 ? __ldg(im + od[p]) : 0.f;
        }
        float res[PX];
#pragma unroll
        for (int p = 0; p < PX; ++p) {
            // image_warp_torch.py:93: sum over the stacked [wa*Ia, wb*Ib, wc*Ic, wd*Id]
            float r = __fadd_rn(__fmul_rn(wa[p], Ia[p]), __fmul_rn(wb[p], Ib[p]));
            r = __fadd_rn(r, __fmul_rn(wc[p], Ic[p]));
            r = __fadd_rn(r, __fmul_rn(wd[p], Id[p]));
            res[p] = r;
        }
        if (NHWC) {
#pragma unroll
            for (int p = 0; p < PX; ++p)
                if (j0 + p < W) out[((b * H + i) * (int64_t)W + j0 + p) * nc + c] = res[p];
        } else {
            float* orow = out + (b * nc + c) * plane + (int64_t)i * W + j0;
            if (PX == 4 && full && ((uintptr_t)orow & 15u) == 0) {
                __stcs(reinterpret_cast<float4*>(orow), make_float4(res[0], res[1 % PX], res[2 % PX], res[3 % PX]));
            } else if (PX == 2 && full && ((uintptr_t)orow & 7u) == 0) {
                __stcs(reinterpret_cast<float2*>(orow), make_float2(res[0], res[1 % PX]));
            } else {
#pragma unroll
                for (int p = 0; p < PX; ++p)
                    if (j0 + p < W) orow[p] = res[p];
            }
        }
    };
    if (CT > 0) {
#pragma unroll
        for (int c = 0; c < CT; ++c) channel(c);
    } else {
        for (int c = 0; c < C; ++c) channel(c);
    }
}

// ---- TMA-tiled variant ------------------------------------------------------------------------
// A CTA owns a TH x TW output tile.  Thread 0 pulls the tile's two flow planes into shared memory
// with TMA (cp.async.bulk.tensor, completion on an mbarrier); every thread derives its taps, a
// redux-based block reduction gives the bounding box of all in-image taps, and when that box fits
// BH x BW the source window of all channels arrives with ONE more TMA load (out-of-image parts of
// the box are zero-filled by the hardware = the reference's zero padding); the gathers then hit
// shared memory.  Tiles whose taps spread further (fold lines, very rough flows) gather from
// global memory instead.  No registers are tied up by bytes in flight, which is what lets an
// HBM-bound gather approach copy bandwidth.  Needs W % 4 == 0, planar flow (stride 1 along x) and
// 16-byte aligned bases (tensor-map rules); otherwise the direct kernel above runs.
#ifndef SSTEM_WARP_TH
#define SSTEM_WARP_TH 8
#endif
#ifndef SSTEM_WARP_BH
#define SSTEM_WARP_BH 24
#endif
constexpr int WT_TH = SSTEM_WARP_TH, WT_TW = 64;      // output tile; WT_TH * 16 threads, 4 pixels each
constexpr int WT_BH = SSTEM_WARP_BH, WT_BW = 96;      // source window (box of the image tensor map)
constexpr int WT_SH = WT_TH + 4, WT_SW = 72;          // small window, tried first (smooth flows): 1.7x the tile
constexpr int WT_MH = WT_TH + 8, WT_MW = 80;          // medium window: 2.5x the tile
constexpr int WT_THREADS = WT_TH * 16;
constexpr int WT_HALF = WT_TH / 2;                    // a thread's two rows are WT_HALF apart

// A tile whose taps spread beyond the largest window.  Out of line on purpose: it is the rare path, and inlined it
// cost the common path registers (72-register budget at 7 CTAs per SM: measured -4 % on the fold flow).
template <int CT>
__device__ __noinline__ void warp_partial_tile(const float* s_fx, const float* s_fy, float* s_im, int* s_box, uint64_t* bar1,
                                               const CUtensorMap* map_im, const float* __restrict__ moving,
                                               float* __restrict__ obase, int b, int i0, int j00, int H, int W) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t plane = (int64_t)H * W;
    // the taps are derived again from the flow tile (still in shared memory): passing the caller's arrays would force them
    // into local memory for the common path too (measured: -10 % on every flow)
    int xa[4], ya[4], dxs[4], dys[4];
    float wa[4], wb[4], wc[4], wd[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int r = warp + WT_HALF * (q >> 1), cidx = lane + 32 * (q & 1);
        const BilinearTap t = torch_tap(s_fx[r * WT_TW + cidx], s_fy[r * WT_TW + cidx], i0 + r, j00 + cidx, H, W);
        xa[q] = t.x0 - 1; ya[q] = t.y0 - 1;
        dxs[q] = t.x1 - t.x0; dys[q] = t.y1 - t.y0;
        wa[q] = t.wa; wb[q] = t.wb; wc[q] = t.wc; wd[q] = t.wd;
    }
        int sx = 0, sy = 0, cnt = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = i0 + warp + WT_HALF * (q >> 1), j = j00 + lane + 32 * (q & 1);
            if (i < H && j < W) {                           // taps relative to the tile origin: sums cannot overflow
                sx += min(max(xa[q] - j00, -4096), 4096);
                sy += min(max(ya[q] - i0, -4096), 4096);
                ++cnt;
            }
        }
        sx = __reduce_add_sync(0xffffffffu, sx); sy = __reduce_add_sync(0xffffffffu, sy); cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0) { atomicAdd(&s_box[4], sx); atomicAdd(&s_box[5], sy); atomicAdd(&s_box[6], cnt); }
        __syncthreads();
        const int n_in = max(s_box[6], 1);
        // window origin: mean tap position minus half the window (x rounded down to 4 floats = 16 bytes)
        const int wx0 = (j00 + s_box[4] / n_in - WT_BW / 2 + 1) & ~3, wy0 = i0 + s_box[5] / n_in - WT_BH / 2 + 1;
        constexpr bool use_window = true;                  // (the caller sends tiles with a huge bounding box elsewhere)
        if (tid == 0) {
            mbar_expect_tx(bar1, (unsigned)(CT * WT_BH * WT_BW * sizeof(float)));
            tma_load_3d(s_im, map_im, bar1, wx0, wy0, b * CT);
        }
        bool in_win[4];
        int o00[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int rx = xa[q] - wx0, ry = ya[q] - wy0;
            in_win[q] = use_window && rx >= 0 && rx + dxs[q] < WT_BW && ry >= 0 && ry + dys[q] < WT_BH;
            o00[q] = ry * WT_BW + rx;
        }
        mbar_wait(bar1, 0);
#pragma unroll                                              // all channels' global gathers of a pixel in flight together
        for (int c = 0; c < CT; ++c) {
            const float* im = moving + ((int64_t)b * CT + c) * plane;
            const float* sc = s_im + c * (WT_BH * WT_BW);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float Ia, Ib, Ic, Id;
                if (in_win[q]) {                            // out-of-image parts of the window were zero-filled by the TMA unit
                    const float* p0 = sc + o00[q];
                    Ia = p0[0]; Ic = p0[dxs[q]];
                    Ib = p0[dys[q] * WT_BW]; Id = p0[dys[q] * WT_BW + dxs[q]];
                } else {
                    const int x0 = xa[q], y0 = ya[q], x1 = x0 + dxs[q], y1 = y0 + dys[q];
                    const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)x1 < (unsigned)W;
                    const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)y1 < (unsigned)H;
                    Ia = (vy0 && vx0) ? __ldg(im + (int64_t)y0 * W + x0) : 0.f;
                    Ib = (vy1 && vx0) ? __ldg(im + (int64_t)y1 * W + x0) : 0.f;
                    Ic = (vy0 && vx1) ? __ldg(im + (int64_t)y0 * W + x1) : 0.f;
                    Id = (vy1 && vx1) ? __ldg(im + (int64_t)y1 * W + x1) : 0.f;
                }
                float r = __fadd_rn(__fmul_rn(wa[q], Ia), __fmul_rn(wb[q], Ib));
                r = __fadd_rn(r, __fmul_rn(wc[q], Ic));
                r = __fadd_rn(r, __fmul_rn(wd[q], Id));
                const int i = i0 + warp + WT_HALF * (q >> 1), j = j00 + lane + 32 * (q & 1);
                if (i < H && j < W) __stcs(obase + c * plane + (int64_t)i * W + j, r);
            }
        }
}

#ifndef SSTEM_WARP_PARTIAL
#define SSTEM_WARP_PARTIAL 1
#endif
#ifndef SSTEM_WARP_TMA_MINB
#define SSTEM_WARP_TMA_MINB 7
#endif
// STITCH: the output assembly of the correction module as the kernel's epilogue -- sff_scripts_fusion/inference.py:163-171:
// (warped * 255).astype(uint8) -> PIL 'L' -> stitch with the interpolated section where the warped one is < 2 -- so the
// float32 warped image is never written (12 B/pixel at C = 3) nor read back by a separate kernel; only uint8 leaves.
struct WarpStitch {
    const uint8_t* interp;                              // [B,H,W] uint8, the interpolated section
    uint8_t* gray;                                      // [B,H,W] uint8 out (nullable): the warped section, 'L'
    uint8_t* stitch;                                    // [B,H,W] uint8 out
};
template <int CT>
__device__ __forceinline__ unsigned luma_term(int c, float r) {
    const unsigned u = (unsigned)(uint8_t)(int)__fmul_rn(r, 255.0f);        // astype(np.uint8)
    return CT == 3 ? (c == 0 ? 19595u : (c == 1 ? 38470u : 7471u)) * u : u; // PIL RGB -> L, fixed point
}
template <int CT, bool STITCH = false>
__global__ void __launch_bounds__(WT_THREADS, SSTEM_WARP_TMA_MINB)
warp_torch_tma_kernel(const __grid_constant__ CUtensorMap map_fx, const __grid_constant__ CUtensorMap map_fy,
                      const __grid_constant__ CUtensorMap map_im, const __grid_constant__ CUtensorMap map_im_small,
                      const __grid_constant__ CUtensorMap map_im_mid, const float* __restrict__ moving,
                      float* __restrict__ out, int H, int W, const WarpStitch st) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* s_im = reinterpret_cast<float*>(smem_raw);                       // [CT][BH][BW]
    float* s_fx = s_im + CT * WT_BH * WT_BW;                                // [TH][TW]
    float* s_fy = s_fx + WT_TH * WT_TW;
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_fy + WT_TH * WT_TW);      // 2 barriers
    int* s_box = reinterpret_cast<int*>(bar + 2);                           // min x, min y, max x, max y, sum x, sum y, count

    const int tid = threadIdx.x;
    const int j00 = blockIdx.x * WT_TW, i0 = blockIdx.y * WT_TH;
    const int b = blockIdx.z;
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        s_box[0] = INT32_MAX; s_box[1] = INT32_MAX; s_box[2] = INT32_MIN; s_box[3] = INT32_MIN;
        s_box[4] = 0; s_box[5] = 0; s_box[6] = 0;
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(&bar[0], 2u * WT_TH * WT_TW * sizeof(float));
        tma_load_3d(s_fx, &map_fx, &bar[0], j00, i0, b);
        tma_load_3d(s_fy, &map_fy, &bar[0], j00, i0, b);
    }
    // thread -> 4 pixels: rows (warp, warp + WT_HALF) x columns (lane, lane + 32).  Lanes walk along x,
    // so shared-memory reads are bank-conflict free and every global store is a full 128-byte line.
    const int warp = tid >> 5, lane = tid & 31;
    mbar_wait(&bar[0], 0);

    int offa[4];                                        // (y0, x0) relative to the window origin, filled in below
    int xa[4], ya[4], dxs[4], dys[4];                   // x0 / y0 in image coordinates (-1 .. W / H); x1-x0, y1-y0
    float wa[4], wb[4], wc[4], wd[4];
    int mnx = INT32_MAX, mny = INT32_MAX, mxx = INT32_MIN, mxy = INT32_MIN;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int r = warp + WT_HALF * (q >> 1), cidx = lane + 32 * (q & 1);
        const int i = i0 + r, j = j00 + cidx;
        const BilinearTap t = torch_tap(s_fx[r * WT_TW + cidx], s_fy[r * WT_TW + cidx], i, j, H, W);
        xa[q] = t.x0 - 1; ya[q] = t.y0 - 1;
        dxs[q] = t.x1 - t.x0; dys[q] = t.y1 - t.y0;
        wa[q] = t.wa; wb[q] = t.wb; wc[q] = t.wc; wd[q] = t.wd;
        if (i < H && j < W) {
            // the window must cover every tap, including those in the zero border (-1 / W / H):
            // TMA zero-fills whatever lies outside the image, which IS the reference's padding
            mnx = min(mnx, xa[q]); mxx = max(mxx, xa[q] + dxs[q]);
            mny = min(mny, ya[q]); mxy = max(mxy, ya[q] + dys[q]);
        }
    }
    mnx = __reduce_min_sync(0xffffffffu, mnx); mny = __reduce_min_sync(0xffffffffu, mny);
    mxx = __reduce_max_sync(0xffffffffu, mxx); mxy = __reduce_max_sync(0xffffffffu, mxy);
    if (lane == 0) {
        atomicMin(&s_box[0], mnx); atomicMin(&s_box[1], mny); atomicMax(&s_box[2], mxx); atomicMax(&s_box[3], mxy);
    }
    __syncthreads();
    // the box must start on a 16-byte boundary in global memory: round the left edge down to 4 floats
    const int bx0 = s_box[0] & ~3, by0 = s_box[1], bx1 = s_box[2], by1 = s_box[3];
    const bool small = (bx1 - bx0 < WT_SW) && (by1 - by0 < WT_SH);
    const bool mid = !small && (bx1 - bx0 < WT_MW) && (by1 - by0 < WT_MH);
    const bool fits = small || mid || ((bx1 - bx0 < WT_BW) && (by1 - by0 < WT_BH));
    const int pitch = small ? WT_SW : (mid ? WT_MW : WT_BW);            // block-uniform
    const int cstride = small ? WT_SH * WT_SW : (mid ? WT_MH * WT_MW : WT_BH * WT_BW);
    if (fits && tid == 0) {
        mbar_expect_tx(&bar[1], (unsigned)(CT * cstride * sizeof(float)));
        tma_load_3d(s_im, small ? &map_im_small : (mid ? &map_im_mid : &map_im), &bar[1], bx0, by0, b * CT);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) offa[q] = (ya[q] - by0) * pitch + (xa[q] - bx0);
    const int64_t plane = (int64_t)H * W;
    float* obase = out + (int64_t)b * CT * plane;
    [[maybe_unused]] unsigned lum[4] = {0u, 0u, 0u, 0u};  // STITCH: fixed-point luma of the thread's 4 pixels
    [[maybe_unused]] auto stitch_store = [&]() {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = i0 + warp + WT_HALF * (q >> 1), j = j00 + lane + 32 * (q & 1);
            if (i < H && j < W) {
                const unsigned L = CT == 3 ? (lum[q] + 0x8000u) >> 16 : lum[q];
                const int64_t idx = (int64_t)b * plane + (int64_t)i * W + j;
                if (st.gray) st.gray[idx] = (uint8_t)L;
                st.stitch[idx] = L >= 2u ? (uint8_t)L : st.interp[idx];
            }
        }
    };
    if (fits) {
        // word offsets of the four taps of each pixel inside one channel plane of the window, and the
        // pixel's offset inside one output plane: computed once, shared by all channels
        int a00[4], a01[4], a10[4], a11[4];
        unsigned ooff[4];
        bool ok[4];
        float2 wa2[2], wb2[2], wc2[2], wd2[2];          // pixels (0,1) and (2,3) side by side for the packed FP32 ops
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int i = i0 + warp + WT_HALF * (q >> 1), j = j00 + lane + 32 * (q & 1);
            ok[q] = i < H && j < W;
            // A pixel outside the image (last tile row / column of a ragged shape) is not in the box, so its taps can lie
            // anywhere -- far outside the window and the CTA's shared memory when the flow moves the tile's taps far.  It
            // reads the window's first words instead; its result is never stored.
            a00[q] = ok[q] ? offa[q] : 0;
            a01[q] = a00[q] + dxs[q];
            a10[q] = a00[q] + dys[q] * pitch;
            a11[q] = a10[q] + dxs[q];
            ooff[q] = (unsigned)(i * W + j);
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            wa2[h] = make_float2(wa[2 * h], wa[2 * h + 1]); wb2[h] = make_float2(wb[2 * h], wb[2 * h + 1]);
            wc2[h] = make_float2(wc[2 * h], wc[2 * h + 1]); wd2[h] = make_float2(wd[2 * h], wd[2 * h + 1]);
        }
        mbar_wait(&bar[1], 0);
        // the channel stride is a compile-time constant inside each branch, so every LDS below is
        // [register + immediate]: no integer work per load
        auto blend = [&](auto cstride_tag) {
            constexpr int CS = decltype(cstride_tag)::value;
#pragma unroll
            for (int c = 0; c < CT; ++c) {
                const float* sc = s_im + c * CS;
                float* oc = obase + c * plane;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int q0 = 2 * h, q1 = 2 * h + 1;
                    const float2 Ia = make_float2(sc[a00[q0]], sc[a00[q1]]), Ib = make_float2(sc[a10[q0]], sc[a10[q1]]);
                    const float2 Ic = make_float2(sc[a01[q0]], sc[a01[q1]]), Id = make_float2(sc[a11[q0]], sc[a11[q1]]);
                    // image_warp_torch.py:93, per component: ((wa*Ia + wb*Ib) + wc*Ic) + wd*Id without
                    // contraction.  The products are packed (FMUL2); the sums stay scalar because ptxas 12.9
                    // fuses mul.rn.f32x2 + add.rn.f32x2 into FFMA2 despite the .rn (even with -fmad=false).
                    const float2 pa = __fmul2_rn(wa2[h], Ia), pb = __fmul2_rn(wb2[h], Ib);
                    const float2 pc = __fmul2_rn(wc2[h], Ic), pd = __fmul2_rn(wd2[h], Id);
                    const float rx = __fadd_rn(__fadd_rn(__fadd_rn(pa.x, pb.x), pc.x), pd.x);
                    const float ry = __fadd_rn(__fadd_rn(__fadd_rn(pa.y, pb.y), pc.y), pd.y);
                    if constexpr (STITCH) { lum[q0] += luma_term<CT>(c, rx); lum[q1] += luma_term<CT>(c, ry); }
                    else {
                        if (ok[q0]) __stcs(oc + ooff[q0], rx);
                        if (ok[q1]) __stcs(oc + ooff[q1], ry);
                    }
                }
            }
        };
        if (small) blend(std::integral_constant<int, WT_SH * WT_SW>{});
        else if (mid) blend(std::integral_constant<int, WT_MH * WT_MW>{});
        else blend(std::integral_constant<int, WT_BH * WT_BW>{});
        if constexpr (STITCH) stitch_store();
    } else {
        // The taps of this tile spread beyond the largest window (a fold line crosses it, or the flow is rough).  All-or-
        // nothing would send every pixel of the tile to global-memory gathers (measured 1.1 TB/s on an N(0, 5 px) flow);
        // instead the largest window is centred on the tile's mean tap position, fetched with the same single TMA box,
        // and each PIXEL decides: all four taps inside the window -> shared memory, else -> its own global gathers.
        // A fold line through the tile splits its taps into two clusters tens of pixels apart: no window serves both, and
        // these few tiles (1.7 % on the SFF fold flow) set the kernel's tail -- they take the plain global gathers below.
        // Only a bounding box that outruns the window moderately (a rough but zero-mean flow: N(0, 5 px) gives ~38 x 98) goes to
        // the out-of-line path; tiles next to a fold line (100-200 columns wide) were measured faster on the plain gathers.
        const bool moderate = SSTEM_WARP_PARTIAL && !STITCH && (bx1 - bx0 < WT_BW + 32) && (by1 - by0 < 2 * WT_BH);
        if (moderate) {
            warp_partial_tile<CT>(s_fx, s_fy, s_im, s_box, &bar[1], &map_im, moving, obase, b, i0, j00, H, W);
            return;
        }
#pragma unroll 1
        for (int c = 0; c < CT; ++c) {
            const float* im = moving + ((int64_t)b * CT + c) * plane;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int x0 = xa[q], y0 = ya[q], x1 = x0 + dxs[q], y1 = y0 + dys[q];
                const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)x1 < (unsigned)W;
                const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)y1 < (unsigned)H;
                const float Ia = (vy0 && vx0) ? __ldg(im + (int64_t)y0 * W + x0) : 0.f;
                const float Ib = (vy1 && vx0) ? __ldg(im + (int64_t)y1 * W + x0) : 0.f;
                const float Ic = (vy0 && vx1) ? __ldg(im + (int64_t)y0 * W + x1) : 0.f;
                const float Id = (vy1 && vx1) ? __ldg(im + (int64_t)y1 * W + x1) : 0.f;
                float r = __fadd_rn(__fmul_rn(wa[q], Ia), __fmul_rn(wb[q], Ib));
                r = __fadd_rn(r, __fmul_rn(wc[q], Ic));
                r = __fadd_rn(r, __fmul_rn(wd[q], Id));
                const int i = i0 + warp + WT_HALF * (q >> 1), j = j00 + lane + 32 * (q & 1);
                if constexpr (STITCH) lum[q] += luma_term<CT>(c, r);
                else if (i < H && j < W) __stcs(obase + c * plane + (int64_t)i * W + j, r);
            }
        }
        if constexpr (STITCH) stitch_store();
    }
}

// 3-D fp32 tensor map over (x: W, y: H, z: n) with strides (1, row, slab) in elements
static bool make_map3(CUtensorMap* m, const float* base, int64_t W, int64_t H, int64_t n, int64_t row, int64_t slab,
                      int bw, int bh, int bn) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n};
    const cuuint64_t strides[2] = {(cuuint64_t)row * 4, (cuuint64_t)slab * 4};
    const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// returns 0 on launch, >0 cuda error, PATH_NOT_APPLICABLE when the TMA path does not apply (caller falls back)
template <int CT, bool STITCH = false>
static int try_launch_warp_tma(const float* moving, const float* flow, const int64_t* fs, float* out,
                               int64_t B, int64_t H, int64_t W, cudaStream_t s, WarpStitch st = WarpStitch{nullptr, nullptr, nullptr}) {
    if ((W & 3) || fs[2] != 1 || !aligned16(moving) || !aligned16(flow) || (!STITCH && !aligned16(out))) return PATH_NOT_APPLICABLE;
    if ((fs[0] & 3) || (fs[1] & 3) || (fs[3] & 3) || fs[1] < W || B > 65535 || (H + WT_TH - 1) / WT_TH > 65535) return PATH_NOT_APPLICABLE;
    CUtensorMap mfx, mfy, mim, mims, mimm;
    if (!make_map3(&mfx, flow, W, H, B, fs[1], fs[0], WT_TW, WT_TH, 1)) return PATH_NOT_APPLICABLE;
    if (!make_map3(&mfy, flow + fs[3], W, H, B, fs[1], fs[0], WT_TW, WT_TH, 1)) return PATH_NOT_APPLICABLE;
    if (!make_map3(&mim, moving, W, H, B * CT, W, H * W, WT_BW, WT_BH, CT)) return PATH_NOT_APPLICABLE;
    if (!make_map3(&mims, moving, W, H, B * CT, W, H * W, WT_SW, WT_SH, CT)) return PATH_NOT_APPLICABLE;
    if (!make_map3(&mimm, moving, W, H, B * CT, W, H * W, WT_MW, WT_MH, CT)) return PATH_NOT_APPLICABLE;
    const size_t smem = (size_t)(CT * WT_BH * WT_BW + 2 * WT_TH * WT_TW) * sizeof(float) + 64;   // 2 barriers + 7 ints of tile statistics
    static PerDeviceOnce done;
    int dev = 0;
    cudaGetDevice(&dev);
    if (!done.test(dev)) {
        cudaError_t e = cudaFuncSetAttribute(warp_torch_tma_kernel<CT, STITCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        done.set(dev);
    }
    dim3 grid((unsigned)((W + WT_TW - 1) / WT_TW), (unsigned)((H + WT_TH - 1) / WT_TH), (unsigned)B);
    warp_torch_tma_kernel<CT, STITCH><<<grid, WT_THREADS, smem, s>>>(mfx, mfy, mim, mims, mimm, moving, out, (int)H, (int)W, st);
    count_launch();
    return finish_launch();
}

// ---- numpy image_warp semantics -------------------------------------------------
// One thread owns 4 consecutive pixels of the flat [B*H*W] index space: the flow arrives as two
// 16-byte loads, the uint8 / float results leave as 4-byte (16-byte) words, and the 16*C gathers of
// the thread are independent.  CT = compile-time channel count (0 = runtime loop).
template <typename PixT, bool NEAREST, int CT>
__global__ void __launch_bounds__(256)
image_warp_kernel(const PixT* __restrict__ im, const float* __restrict__ flow,
                  uint8_t* __restrict__ out_u8, float* __restrict__ out_f32,
                  int C, int H, int W, int64_t total) {
    constexpr int PX = 4;
    const int64_t idx0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * PX;   // first pixel of this thread
    if (idx0 >= total) return;
    const int nc = CT > 0 ? CT : C;
    const bool full = idx0 + PX <= total;
    float fx[PX], fy[PX];
    // idx0 is a multiple of 4, so flow + 2*idx0 is 32-byte aligned exactly when the flow base is 16-byte aligned;
    // an 8-byte aligned base (the ABI minimum: e.g. flows[i] of a [N,H,W,2] tensor with H*W odd) takes 8-byte loads
    const bool flow16 = (reinterpret_cast<uintptr_t>(flow) & 15u) == 0;
    if (full && flow16) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(flow + 2 * idx0));
        const float4 c = __ldcs(reinterpret_cast<const float4*>(flow + 2 * idx0) + 1);
        fx[0] = a.x; fy[0] = a.y; fx[1] = a.z; fy[1] = a.w; fx[2] = c.x; fy[2] = c.y; fx[3] = c.z; fy[3] = c.w;
    } else if (full) {
#pragma unroll
        for (int p = 0; p < PX; ++p) {
            const float2 f = __ldcs(reinterpret_cast<const float2*>(flow + 2 * (idx0 + p)));
            fx[p] = f.x; fy[p] = f.y;
        }
    } else {
#pragma unroll
        for (int p = 0; p < PX; ++p) {
            const int64_t q = min(idx0 + p, total - 1);
            fx[p] = __ldg(flow + 2 * q); fy[p] = __ldg(flow + 2 * q + 1);
        }
    }
    int j = (int)(idx0 % W);
    int i = (int)((idx0 / W) % H);
    int64_t b = idx0 / ((int64_t)W * H);
    int oa[PX], ob[PX], oc[PX], od[PX];                 // pixel offsets (in pixels) of the 4 taps inside image b
    int64_t boff[PX];
    float wa[PX], wb[PX], wc[PX], wd[PX];
#pragma unroll
    for (int p = 0; p < PX; ++p) {
        const float ffx = floorf(fx[p]), ffy = floorf(fy[p]);
        // image_warp.py:45-57: integer displacement, then clip (bounded first so the add cannot overflow)
        const float lim = 1073741824.0f;
        const int dxi = (int)fminf(fmaxf(ffx, -lim), lim), dyi = (int)fminf(fmaxf(ffy, -lim), lim);
        const int x0 = min(max(j + dxi, 0), W - 1);
        const int y0 = min(max(i + dyi, 0), H - 1);
        // :84-88 -- x1 is taken from the CLIPPED x0
        const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
        oa[p] = y0 * W + x0; ob[p] = y1 * W + x0; oc[p] = y0 * W + x1; od[p] = y1 * W + x1;
        boff[p] = b * (int64_t)H * W;
        // :72-82 -- weights from frac(flow), independent of clipping
        const float xw = __fsub_rn(fx[p], ffx), yw = __fsub_rn(fy[p], ffy);
        const float ax = __fsub_rn(1.0f, xw), ay = __fsub_rn(1.0f, yw);
        wa[p] = __fmul_rn(ax, ay); wb[p] = __fmul_rn(ax, yw); wc[p] = __fmul_rn(xw, ay); wd[p] = __fmul_rn(xw, yw);
        if (++j == W) { j = 0; if (++i == H) { i = 0; ++b; } }
    }
    // results of the 4 pixels, channel-interleaved exactly as they lie in NHWC memory
    constexpr int MAXV = CT > 0 ? PX * CT : 1;
    float res[MAXV];
    auto one = [&](int p, int c) -> float {
        const PixT* base = im + boff[p] * nc + c;
        if (NEAREST) return (float)__ldg(base + (int64_t)oa[p] * nc);
        const float Ia = (float)__ldg(base + (int64_t)oa[p] * nc), Ib = (float)__ldg(base + (int64_t)ob[p] * nc);
        const float Ic = (float)__ldg(base + (int64_t)oc[p] * nc), Id = (float)__ldg(base + (int64_t)od[p] * nc);
        float r = __fadd_rn(__fmul_rn(wa[p], Ia), __fmul_rn(wb[p], Ib));
        r = __fadd_rn(r, __fmul_rn(wc[p], Ic));
        return __fadd_rn(r, __fmul_rn(wd[p], Id));
    };
    if (CT > 0 && full) {
#pragma unroll
        for (int p = 0; p < PX; ++p)
#pragma unroll
            for (int c = 0; c < CT; ++c) res[p * CT + c] = one(p, c);
        const int64_t o = idx0 * CT;                     // 4*CT consecutive elements, 4*CT-aligned
        if (out_f32) {
#pragma unroll
            for (int k = 0; k < CT; ++k)
                __stcs(reinterpret_cast<float4*>(out_f32 + o) + k, make_float4(res[4 * k], res[4 * k + 1], res[4 * k + 2], res[4 * k + 3]));
        }
        if (out_u8) {
#pragma unroll
            for (int k = 0; k < CT; ++k) {               // :110 astype(uint8): truncation
                const uchar4 q = make_uchar4((uint8_t)(int)res[4 * k], (uint8_t)(int)res[4 * k + 1],
                                             (uint8_t)(int)res[4 * k + 2], (uint8_t)(int)res[4 * k + 3]);
                __stcs(reinterpret_cast<uchar4*>(out_u8 + o) + k, q);
            }
        }
    } else {
        for (int p = 0; p < PX; ++p) {
            if (idx0 + p >= total) break;
            for (int c = 0; c < nc; ++c) {
                const float r = one(p, c);
                if (out_f32) out_f32[(idx0 + p) * nc + c] = r;
                if (out_u8) out_u8[(idx0 + p) * nc + c] = (uint8_t)(int)r;
            }
        }
    }
}

}  // namespace sstem

using namespace sstem;

extern "C" int sstem_warp_forward(const float* moving, const float* flow, const int64_t flow_strides[4],
                                  float* out, int64_t B, int64_t C, int64_t H, int64_t W,
                                  int32_t out_layout, void* stream) {
    if (!moving || !flow || !flow_strides || !out) return SSTEM_E_NULL;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || H > (1 << 24) || W > (1 << 24)) return SSTEM_E_SHAPE;
    if (!aligned4(moving) || !aligned4(flow) || !aligned4(out)) return SSTEM_E_ALIGN;
    if (out_layout != SSTEM_LAYOUT_NCHW && out_layout != SSTEM_LAYOUT_NHWC) return SSTEM_E_FLAG;
    DeviceGuard guard(out);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    if (H * W > INT32_MAX) return SSTEM_E_SHAPE;       // in-plane offsets are 32-bit
    static const bool no_tma = getenv("SSTEM_WARP_NO_TMA") != nullptr;   // experiments: force the direct kernel
    if (out_layout == SSTEM_LAYOUT_NCHW && (C == 1 || C == 3) && !no_tma) {
        const int r = (C == 3) ? try_launch_warp_tma<3>(moving, flow, flow_strides, out, B, H, W, s)
                               : try_launch_warp_tma<1>(moving, flow, flow_strides, out, B, H, W, s);
        if (r != PATH_NOT_APPLICABLE) return r;
    }
    constexpr int PX = SSTEM_WARP_PX;
    const int gpr = (int)((W + PX - 1) / PX);
    const int64_t groups = B * H * gpr;
    const unsigned blocks = (unsigned)((groups + 255) / 256);
#define SSTEM_WARP_LAUNCH(NHWC_, CT_)                                                                        \
    warp_torch_kernel<PX, NHWC_, CT_><<<blocks, 256, 0, s>>>(moving, flow, flow_strides[0], flow_strides[1],  \
                                                             flow_strides[2], flow_strides[3], out, (int)C,   \
                                                             (int)H, (int)W, gpr, groups)
    const bool nhwc = out_layout == SSTEM_LAYOUT_NHWC;
    if (C == 3) { if (nhwc) SSTEM_WARP_LAUNCH(true, 3); else SSTEM_WARP_LAUNCH(false, 3); }
    else if (C == 1) { if (nhwc) SSTEM_WARP_LAUNCH(true, 1); else SSTEM_WARP_LAUNCH(false, 1); }
    else { if (nhwc) SSTEM_WARP_LAUNCH(true, 0); else SSTEM_WARP_LAUNCH(false, 0); }
#undef SSTEM_WARP_LAUNCH
    count_launch();
    return finish_launch();
}

// ---- backward of the torch-semantics warp ----------------------------------------------------------------------------
// The reference's SpatialTransformation is differentiable through its ATen ops (image_warp_torch.py:32-95); no reference
// call site uses that (main_fusion.py:227-235 runs it under no_grad / detach), so this is a plain one-thread-per-pixel
// kernel, not a tuned one.  With out = wa Ia + wb Ib + wc Ic + wd Id, wa = dx dy, wb = dx (1-dy), wc = (1-dx) dy,
// wd = (1-dx)(1-dy), dx = x1_clamped - x, dy = y1_clamped - y (floor, clamp and the gather indices carry no gradient):
//   d out / d fx = dy (Ic - Ia) + (1-dy) (Id - Ib),   d out / d fy = dx (Ib - Ia) + (1-dx) (Id - Ic),
//   d out / d I(tap) = the tap's weight (scattered with atomics; taps in the 1-px zero border give nothing).
namespace sstem {
__global__ void __launch_bounds__(256)
warp_torch_backward_kernel(const float* __restrict__ moving, const float* __restrict__ flow,
                           int64_t fs_b, int64_t fs_h, int64_t fs_w, int64_t fs_c, const float* __restrict__ grad_out,
                           float* __restrict__ grad_moving, float* __restrict__ grad_flow, int C, int H, int W, int64_t total) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int j = (int)(idx % W), i = (int)((idx / W) % H);
    const int64_t b = idx / ((int64_t)W * H);
    const float* fp = flow + b * fs_b + (int64_t)i * fs_h + (int64_t)j * fs_w;
    const float fx = __ldg(fp), fy = __ldg(fp + fs_c);
    const BilinearTap t = torch_tap(fx, fy, i, j, H, W);
    // dx, dy exactly as torch_tap forms them
    const float x = __fadd_rn(__fadd_rn(fx, (float)j), 1.0f), y = __fadd_rn(__fadd_rn(fy, (float)i), 1.0f);
    const float dx = __fsub_rn((float)t.x1, x), dy = __fsub_rn((float)t.y1, y);
    const float ex = __fsub_rn(1.0f, dx), ey = __fsub_rn(1.0f, dy);
    const int xa = t.x0 - 1, xb = t.x1 - 1, ya = t.y0 - 1, yb = t.y1 - 1;
    const bool vxa = (unsigned)xa < (unsigned)W, vxb = (unsigned)xb < (unsigned)W;
    const bool vya = (unsigned)ya < (unsigned)H, vyb = (unsigned)yb < (unsigned)H;
    const int64_t plane = (int64_t)H * W;
    float gfx = 0.f, gfy = 0.f;
    for (int c = 0; c < C; ++c) {
        const int64_t pb = (b * C + c) * plane;
        const float g = __ldg(grad_out + pb + (int64_t)i * W + j);
        if (grad_flow) {
            const float* im = moving + pb;
            const float Ia = (vya && vxa) ? __ldg(im + (int64_t)ya * W + xa) : 0.f, Ib = (vyb && vxa) ? __ldg(im + (int64_t)yb * W + xa) : 0.f;
            const float Ic = (vya && vxb) ? __ldg(im + (int64_t)ya * W + xb) : 0.f, Id = (vyb && vxb) ? __ldg(im + (int64_t)yb * W + xb) : 0.f;
            gfx += g * (dy * (Ic - Ia) + ey * (Id - Ib));
            gfy += g * (dx * (Ib - Ia) + ex * (Id - Ic));
        }
        if (grad_moving) {
            float* gm = grad_moving + pb;
            if (vya && vxa) atomicAdd(gm + (int64_t)ya * W + xa, t.wa * g);
            if (vyb && vxa) atomicAdd(gm + (int64_t)yb * W + xa, t.wb * g);
            if (vya && vxb) atomicAdd(gm + (int64_t)ya * W + xb, t.wc * g);
            if (vyb && vxb) atomicAdd(gm + (int64_t)yb * W + xb, t.wd * g);
        }
    }
    if (grad_flow) {
        grad_flow[2 * idx] = gfx;
        grad_flow[2 * idx + 1] = gfy;
    }
}
}  // namespace sstem

extern "C" int sstem_warp_backward(const float* moving, const float* flow, const int64_t flow_strides[4], const float* grad_out,
                                   float* grad_moving, float* grad_flow, int64_t B, int64_t C, int64_t H, int64_t W, void* stream) {
    if (!moving || !flow || !flow_strides || !grad_out || (!grad_moving && !grad_flow)) return SSTEM_E_NULL;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || H > (1 << 24) || W > (1 << 24) || H * W > INT32_MAX) return SSTEM_E_SHAPE;
    if (!aligned4(moving) || !aligned4(flow) || !aligned4(grad_out) || !aligned4(grad_moving) || !aligned4(grad_flow)) return SSTEM_E_ALIGN;
    DeviceGuard guard(grad_moving ? (const void*)grad_moving : (const void*)grad_flow);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    if (grad_moving) {
        cudaError_t e = cudaMemsetAsync(grad_moving, 0, (size_t)(B * C * H * W) * sizeof(float), s);
        if (e != cudaSuccess) return (int)e;
    }
    const int64_t total = B * H * W;
    warp_torch_backward_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(moving, flow, flow_strides[0], flow_strides[1], flow_strides[2],
                                                                             flow_strides[3], grad_out, grad_moving, grad_flow, (int)C, (int)H, (int)W, total);
    count_launch();
    return finish_launch();
}

extern "C" int sstem_warp_stitch_u8(const float* warped, const uint8_t* interp, uint8_t* gray_out, uint8_t* stitch_out,
                                    int64_t B, int64_t C, int64_t H, int64_t W, void* stream);

extern "C" int sstem_warp_stitch_forward(const float* moving, const float* flow, const int64_t flow_strides[4],
                                         const uint8_t* interp, uint8_t* gray_out, uint8_t* stitch_out,
                                         int64_t B, int64_t C, int64_t H, int64_t W, void* stream) {
    if (!moving || !flow || !flow_strides || !interp || !stitch_out) return SSTEM_E_NULL;
    if (B <= 0 || H <= 0 || W <= 0 || (C != 1 && C != 3) || H > (1 << 24) || W > (1 << 24)) return SSTEM_E_SHAPE;
    if (!aligned4(moving) || !aligned4(flow)) return SSTEM_E_ALIGN;
    DeviceGuard guard(stitch_out);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    if (H * W > INT32_MAX) return SSTEM_E_SHAPE;
    const WarpStitch st{interp, gray_out, stitch_out};
    const int r = (C == 3) ? try_launch_warp_tma<3, true>(moving, flow, flow_strides, nullptr, B, H, W, s, st)
                           : try_launch_warp_tma<1, true>(moving, flow, flow_strides, nullptr, B, H, W, s, st);
    if (r != PATH_NOT_APPLICABLE) return r;
    // shapes the TMA kernel does not take: the two steps one after the other through a stream-ordered scratch image
    float* tmp = nullptr;
    if (workspace_alloc(reinterpret_cast<void**>(&tmp), (size_t)(B * C * H * W) * sizeof(float), s)) return (int)cudaErrorMemoryAllocation;
    int e = sstem_warp_forward(moving, flow, flow_strides, tmp, B, C, H, W, SSTEM_LAYOUT_NCHW, stream);
    if (!e) e = sstem_warp_stitch_u8(tmp, interp, gray_out, stitch_out, B, C, H, W, stream);
    cudaFreeAsync(tmp, s);
    return e;
}

extern "C" int sstem_image_warp(const void* im, int32_t pix_type, const float* flow,
                                uint8_t* out_u8, float* out_f32,
                                int64_t B, int64_t H, int64_t W, int64_t C, int32_t mode, void* stream) {
    if (!im || !flow || (!out_u8 && !out_f32)) return SSTEM_E_NULL;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return SSTEM_E_SHAPE;
    if (pix_type != SSTEM_PIX_U8 && pix_type != SSTEM_PIX_F32) return SSTEM_E_FLAG;
    if (mode != SSTEM_WARP_BILINEAR && mode != SSTEM_WARP_NEAREST) return SSTEM_E_FLAG;
    if ((reinterpret_cast<uintptr_t>(flow) & 7u) != 0) return SSTEM_E_ALIGN;
    if (pix_type == SSTEM_PIX_F32 && !aligned4(im)) return SSTEM_E_ALIGN;
    if (out_f32 && !aligned4(out_f32)) return SSTEM_E_ALIGN;
    DeviceGuard guard(out_u8 ? (const void*)out_u8 : (const void*)out_f32);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    if (H * W > INT32_MAX) return SSTEM_E_SHAPE;       // in-image pixel offsets are 32-bit
    const int64_t total = B * H * W;
    const unsigned blocks = (unsigned)(((total + 3) / 4 + 255) / 256);
    const bool nearest = mode == SSTEM_WARP_NEAREST;
    // the vector stores need 4-byte (uint8) / 16-byte (float) aligned outputs and 16-byte aligned flow
    const bool vec_ok = aligned16(flow) && (!out_u8 || aligned4(out_u8)) && (!out_f32 || aligned16(out_f32));
#define SSTEM_IW_LAUNCH(T_, N_, CT_)                                                                              \
    image_warp_kernel<T_, N_, CT_><<<blocks, 256, 0, s>>>((const T_*)im, flow, out_u8, out_f32, (int)C, (int)H, (int)W, total)
#define SSTEM_IW_DISPATCH(T_, N_)                                                    \
    {                                                                                \
        if (vec_ok && C == 1) SSTEM_IW_LAUNCH(T_, N_, 1);                            \
        else if (vec_ok && C == 3) SSTEM_IW_LAUNCH(T_, N_, 3);                       \
        else SSTEM_IW_LAUNCH(T_, N_, 0);                                             \
    }
    if (pix_type == SSTEM_PIX_U8) {
        if (nearest) SSTEM_IW_DISPATCH(uint8_t, true) else SSTEM_IW_DISPATCH(uint8_t, false)
    } else {
        if (nearest) SSTEM_IW_DISPATCH(float, true) else SSTEM_IW_DISPATCH(float, false)
    }
#undef SSTEM_IW_DISPATCH
#undef SSTEM_IW_LAUNCH
    count_launch();
    return finish_launch();
}
