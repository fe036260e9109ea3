// Launchers of the third-generation tap-gradient kernel (device code in sepconv_k51_v3.cuh): repack the input
// channel-interleaved into a stream-ordered workspace, encode the four tensor maps, launch the persistent grid,
// release the workspace.  Also the tap gradients on the tile-major tap layout of SURVEY 8f N2
// (sstem_sepconv_backward_tiled; the layout conversions are in sepconv_layout.cu).
#include "sepconv_k51_v3.cuh"

#include <stdlib.h>

namespace sstem {
namespace {

template <bool WV, bool WH, bool ACCUM>
int launch_v3_kernel(const CUtensorMap& min, const CUtensorMap& mv, const CUtensorMap& mh, const CUtensorMap& mg,
                     float* gv, float* gh, int* counter, const V3Shape& sh, cudaStream_t s) {
    static PerDeviceOnce done;
    auto kern = sepconv_bwd_taps_k51_v3_kernel<WV, WH, ACCUM>;
    if (int e = set_smem_once(kern, V3_SMEM, done)) return e;
    const int ctas = std::min<int64_t>(2 * (int64_t)sm_count(), (int64_t)sh.ntiles);
    kern<<<ctas, V3_WARPS * 32, V3_SMEM, s>>>(min, mv, mh, mg, gv, gh, counter, sh, g_gate.ptr, g_gate.want);
    count_launch();
    return finish_launch();
}

// tensor maps of the persistent kernel: window groups, vertical-tap groups, horizontal taps, upstream gradient
bool make_v3_maps(CUtensorMap* min, CUtensorMap* mv, CUtensorMap* mh, CUtensorMap* mg, const float* ws, const float* v,
                  const float* h, const float* g, int64_t B, int64_t C, int64_t c0, int64_t H, int64_t W) {
    const int64_t IH = H + K51 - 1, IW = W + K51 - 1, plane = H * W;
    {
        // a repacked row is 4 * IW contiguous floats: the box's inner extent is a whole 960-byte row segment (an inner
        // extent of one pixel = 16 bytes makes the TMA unit issue 240 tiny requests per box: measured 1.5x slower)
        const int64_t dims[3] = {4 * IW, IH, B}, strides[3] = {1, 4 * IW, 4 * IW * IH};
        const int box[3] = {4 * V3_WIN_COLS, V3_GROUP, 1};
        if (!make_map_f32(min, ws, 3, dims, strides, box)) return false;
    }
    const int64_t tdims[4] = {W, H, K51, B}, tstrides[4] = {1, W, plane, (int64_t)K51 * plane};
    if (v) {
        const int box[4] = {V3_COLS, B3_R, V3_GROUP, 1};
        if (!make_map_f32(mv, v, 4, tdims, tstrides, box)) return false;
    }
    if (h) {
        // tap and row dimensions swapped: the box lands as [row][tap][col], whose per-lane register copy hits 32 different
        // banks (as [tap][row][col] the four tap groups of a column collide in one bank)
        const int64_t rdims[4] = {W, K51, H, B}, rstrides[4] = {1, plane, W, (int64_t)K51 * plane};
        const int box[4] = {V3_COLS, K51, B3_R, 1};
        if (!make_map_f32(mh, h, 4, rdims, rstrides, box)) return false;
    }
    {
        const int64_t dims[4] = {W, H, 3, B}, strides[4] = {1, W, plane, C * plane};
        const int box[4] = {V3_COLS, B3_R, 3, 1};
        if (!make_map_f32(mg, g + c0 * plane, 4, dims, strides, box)) return false;
    }
    return true;
}

template <bool WV, bool WH, bool ACCUM, int CC>
int launch_v3_tiled_kernel(const CUtensorMap& min, const CUtensorMap& mv, const CUtensorMap& mh, const CUtensorMap& mg,
                           float* gv, float* gh, int* counter, const V3Shape& sh, cudaStream_t s) {
    static PerDeviceOnce done;
    auto kern = sepconv_bwd_taps_k51_v3_tiled_kernel<WV, WH, ACCUM, CC>;
    if (int e = set_smem_once(kern, V3_SMEM, done)) return e;
    const int ctas = std::min<int64_t>(2 * (int64_t)sm_count(), (int64_t)sh.ntiles);
    kern<<<ctas, V3_WARPS * 32, V3_SMEM, s>>>(min, mv, mh, mg, gv, gh, counter, sh, g_gate.ptr, g_gate.want);
    count_launch();
    return finish_launch();
}

// The upstream gradient as the tiled kernel reads it: planes of W floats, rows `gpitch` floats apart (a multiple of 4),
// planes `gplane` and images `gbatch` floats apart, base 16-byte aligned.
struct TiledGrad {
    const float* g;
    int64_t gpitch, gplane, gbatch;
};

// One channel chunk (CC planes from c0) of the tiled tap gradients; later chunks accumulate.
template <int CC>
int launch_tiled_chunk(const TiledGrad& tg, const float* in, const float* vt, const float* ht, float* gvt, float* ght,
                       int64_t B, int C, int c0, int H, int W, bool accum, cudaStream_t s) {
    const int64_t tiles_x = (W + V3_COLS * V3_WARPS - 1) / (V3_COLS * V3_WARPS);
    const int64_t tiles_y = 2 * (int64_t)((H + 7) / 8);     // half tiles; ceil(H/4) would miss the bottom half of the last tile row
    const int64_t tiles_x8 = (W + 7) / 8, tiles_y8 = (H + 7) / 8;
    const int64_t IH = H + K51 - 1, IW = W + K51 - 1, IWP = (IW + 3) & ~(int64_t)3;
    float* ws = nullptr;
    const size_t ws_bytes = CC == 3 ? (size_t)(B * IH * IW) * 16 : (size_t)(B * IH * IWP) * 4;
    if (workspace_alloc(reinterpret_cast<void**>(&ws), ws_bytes + 256, s)) return cudaErrorMemoryAllocation;
    int* counter = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + ws_bytes);   // dynamic tile scheduler ticket
    cudaMemsetAsync(counter, 0, 256, s);
    int e = CC == 3 ? launch_repack_nhwc4(in, ws, B, C, c0, IH, IW, s) : launch_repack_plane_pitch(in, ws, B, C, c0, IH, IW, IWP, s);
    CUtensorMap min, mv, mh, mg;
    if (!e) {
        const int64_t row = CC == 3 ? 4 * IW : IWP;
        const int64_t dims[3] = {row, IH, B}, strides[3] = {1, row, row * IH};
        const int box[3] = {(CC == 3 ? 4 : 1) * V3_WIN_COLS, V3_GROUP, 1};
        // tile-major taps: the tile row and the batch merge into one dimension; v lands as [plane][row][col], h as
        // [row][tap][col] -- the ring-slot and tap-buffer layouts of the [B,51,H,W] maps
        const int64_t tstride = tiles_x8 * K51 * 64;
        const int64_t vdims[5] = {8, 8, K51, tiles_x8, tiles_y8 * B}, vstrides[5] = {1, 8, 64, K51 * 64, tstride};
        const int64_t hdims[5] = {8, K51, 8, tiles_x8, tiles_y8 * B}, hstrides[5] = {1, 64, 8, K51 * 64, tstride};
        const int vbox[5] = {V3_COLS, B3_R, V3_GROUP, 1, 1}, hbox[5] = {V3_COLS, K51, B3_R, 1, 1};
        const int64_t gdims[4] = {W, H, CC, B}, gstrides[4] = {1, tg.gpitch, tg.gplane, tg.gbatch};
        const int gbox[4] = {V3_COLS, B3_R, CC, 1};
        if (!make_map_f32(&min, ws, 3, dims, strides, box) || !make_map_f32(&mg, tg.g + c0 * tg.gplane, 4, gdims, gstrides, gbox))
            e = SSTEM_E_SHAPE;
        mv = mh = min;                                     // unused by a kernel that does not want them, but must be valid objects
        if (!e && ght && !make_map_f32(&mv, vt, 5, vdims, vstrides, vbox)) e = SSTEM_E_SHAPE;
        if (!e && gvt && !make_map_f32(&mh, ht, 5, hdims, hstrides, hbox)) e = SSTEM_E_SHAPE;
    }
    if (!e) {
        V3Shape sh{H, W, (int)tiles_x, (int)tiles_y, (int)(tiles_x * tiles_y * B), C, c0};
#define SSTEM_V3T_LAUNCH(WV_, WH_)                                                                                  \
        e = accum ? launch_v3_tiled_kernel<WV_, WH_, true, CC>(min, mv, mh, mg, gvt, ght, counter, sh, s)          \
                  : launch_v3_tiled_kernel<WV_, WH_, false, CC>(min, mv, mh, mg, gvt, ght, counter, sh, s)
        if (gvt && ght) SSTEM_V3T_LAUNCH(true, true);
        else if (gvt) SSTEM_V3T_LAUNCH(true, false);
        else SSTEM_V3T_LAUNCH(false, true);
#undef SSTEM_V3T_LAUNCH
    }
    cudaFreeAsync(ws, s);
    return e;
}

// Tap gradients on tile-major taps, always on the persistent kernel.  gray: one one-plane launch with the channel-summed
// gradient; otherwise 3-channel chunks, then single planes.  The gradient's tensor map needs W % 4 == 0 and a 16-byte
// aligned base: otherwise, and always for gray, it is staged at a 4-float row pitch first (a few floats per pixel,
// against ~840 B per pixel that the kernel itself moves).
int launch_bwd_taps_tiled(const float* g, const float* in, const float* vt, const float* ht, float* gvt, float* ght,
                          int64_t B, int C, int H, int W, bool gray, cudaStream_t s) {
    const int64_t tiles_x = (W + V3_COLS * V3_WARPS - 1) / (V3_COLS * V3_WARPS), tiles_y = 2 * (int64_t)((H + 7) / 8);
    if (tiles_x * tiles_y * B > INT32_MAX / 2) return SSTEM_E_SHAPE;
    const int64_t plane = (int64_t)H * W;
    TiledGrad tg{g, W, plane, (int64_t)C * plane};
    float* staged = nullptr;
    if (gray || (W & 3) || !aligned16(g)) {
        const int64_t WP = (W + 3) & ~3, nplanes = gray ? 1 : C;
        if (workspace_alloc(reinterpret_cast<void**>(&staged), (size_t)(B * nplanes * H * WP) * 4, s)) return cudaErrorMemoryAllocation;
        if (int e = launch_stage_grad_planes(g, staged, B, C, H, W, WP, gray, s)) { cudaFreeAsync(staged, s); return e; }
        tg = TiledGrad{staged, WP, H * WP, nplanes * H * WP};
    }
    int e = 0;
    if (gray) {
        e = launch_tiled_chunk<1>(tg, in, vt, ht, gvt, ght, B, C, 0, H, W, false, s);
    } else {
        for (int c0 = 0; c0 < C && !e;) {
            if (C - c0 >= 3) { e = launch_tiled_chunk<3>(tg, in, vt, ht, gvt, ght, B, C, c0, H, W, c0 > 0, s); c0 += 3; }
            else { e = launch_tiled_chunk<1>(tg, in, vt, ht, gvt, ght, B, C, c0, H, W, c0 > 0, s); c0 += 1; }
        }
    }
    if (staged) cudaFreeAsync(staged, s);
    return e;
}

}  // namespace

// returns 0 on launch, > 0 CUDA error, -1000 when the path does not apply (caller runs the first-generation kernel)
int try_launch_bwd_taps_k51_v3(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                               int64_t B, int C, int c0, int H, int W, int accumulate, cudaStream_t s) {
    if ((W & 3) || !aligned16(v) || !aligned16(h) || !aligned16(g) || ((int64_t)H * W * c0 & 3)) return -1000;
    const int64_t tiles_x = (W + V3_COLS * V3_WARPS - 1) / (V3_COLS * V3_WARPS), tiles_y = (H + B3_R - 1) / B3_R;
    if (tiles_x * tiles_y * B > INT32_MAX / 2) return -1000;
    // a persistent grid needs several tiles per warp to balance; small problems stay on the CTA-per-tile kernel
    static const int64_t min_tiles = getenv("SSTEM_V3_MIN_TILES") ? atoll(getenv("SSTEM_V3_MIN_TILES")) : 6;    // measured crossover: ~6 tiles per warp (tap gradients), ~10 (forward)
    if (tiles_x * tiles_y * B < min_tiles * 2 * sm_count()) return -1000;
    const int64_t IH = H + K51 - 1, IW = W + K51 - 1;
    float* ws = nullptr;
    const size_t ws_bytes = (size_t)(B * IH * IW) * 16;
    if (workspace_alloc(reinterpret_cast<void**>(&ws), ws_bytes + 256, s)) return -1000;
    int* counter = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + ws_bytes);   // dynamic tile scheduler ticket
    cudaMemsetAsync(counter, 0, 256, s);
    int e = launch_repack_nhwc4(in, ws, B, C, c0, IH, IW, s);
    CUtensorMap min, mv, mh, mg;
    if (!e && !make_v3_maps(&min, &mv, &mh, &mg, ws, gh ? v : nullptr, gv ? h : nullptr, g, B, C, c0, H, W)) e = -1000;
    if (!e) {
        if (!gh) mv = min;                                 // unused by the kernel, but must be a valid object to copy
        if (!gv) mh = min;
        V3Shape sh{H, W, (int)tiles_x, (int)tiles_y, (int)(tiles_x * tiles_y * B), C, c0};
#define SSTEM_V3_LAUNCH(WV_, WH_)                                                                   \
        e = accumulate ? launch_v3_kernel<WV_, WH_, true>(min, mv, mh, mg, gv, gh, counter, sh, s)           \
                       : launch_v3_kernel<WV_, WH_, false>(min, mv, mh, mg, gv, gh, counter, sh, s)
        if (gv && gh) SSTEM_V3_LAUNCH(true, true);
        else if (gv) SSTEM_V3_LAUNCH(true, false);
        else SSTEM_V3_LAUNCH(false, true);
#undef SSTEM_V3_LAUNCH
    }
    cudaFreeAsync(ws, s);
    return e;
}

}  // namespace sstem

using namespace sstem;

extern "C" int sstem_sepconv_backward_tiled(const float* grad_output, const float* input,
                                            const float* vertical_tiled, const float* horizontal_tiled,
                                            float* grad_input, float* grad_vertical_tiled, float* grad_horizontal_tiled,
                                            int64_t B, int64_t C, int64_t H, int64_t W, int32_t K, uint32_t flags, void* stream) {
    if (!grad_output || !input || !vertical_tiled || !horizontal_tiled) return SSTEM_E_NULL;
    if (!grad_input && !grad_vertical_tiled && !grad_horizontal_tiled) return SSTEM_E_NULL;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || C > 65535 || H > (1 << 24) || W > (1 << 24)) return SSTEM_E_SHAPE;
    if (K != K51) return SSTEM_E_SHAPE;                    // the tiled layout is defined for the reference's 51 taps
    if (flags & ~SSTEM_SEPCONV_GRAY_REPLICATED) return SSTEM_E_FLAG;
    if (!aligned4(grad_output) || !aligned4(input) || !aligned4(grad_input)) return SSTEM_E_ALIGN;
    if (!aligned16(vertical_tiled) || !aligned16(horizontal_tiled) || !aligned16(grad_vertical_tiled) || !aligned16(grad_horizontal_tiled))
        return SSTEM_E_ALIGN;
    const void* any_out = grad_vertical_tiled ? grad_vertical_tiled : (grad_horizontal_tiled ? grad_horizontal_tiled : grad_input);
    DeviceGuard guard(any_out);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    if (grad_vertical_tiled || grad_horizontal_tiled) {
        const bool gray = (flags & SSTEM_SEPCONV_GRAY_REPLICATED) && C > 1;
        if (int e = launch_bwd_taps_tiled(grad_output, input, vertical_tiled, horizontal_tiled, grad_vertical_tiled, grad_horizontal_tiled,
                                          B, (int)C, (int)H, (int)W, gray, s))
            return e;
    }
    if (!grad_input) return 0;
    // grad_input is not a tuned path here: the taps go back to [B,51,H,W] in the workspace (2 x 204 B per pixel, ~816 B
    // per pixel of conversion traffic) and the [B,51,H,W] kernel runs
    const int64_t n = B * K51 * H * W;
    float* taps = nullptr;
    if (workspace_alloc(reinterpret_cast<void**>(&taps), (size_t)n * 2 * sizeof(float), s)) return cudaErrorMemoryAllocation;
    int e = launch_taps_from_tiled(vertical_tiled, taps, B, H, W, s);
    if (!e) e = launch_taps_from_tiled(horizontal_tiled, taps + n, B, H, W, s);
    if (!e) e = launch_sepconv_bwd_input_k51(grad_output, taps, taps + n, grad_input, B, C, H, W, s);
    cudaFreeAsync(taps, s);
    return e;
}

#ifdef SSTEM_V3_PHASES
// diagnostic builds only (tools/v3_phases.py): clock64 ticks per tile phase, summed over the warps of every launch
extern "C" int sstem_v3_phases_bwd(unsigned long long* out, int reset) { return sstem::v3_phases_read(out, reset); }
#endif
