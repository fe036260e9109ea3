// Launcher of the third-generation tap-gradient kernel (device code in sepconv_k51_v3.cuh): repack the input
// channel-interleaved into a stream-ordered workspace, encode the four tensor maps, launch the persistent grid,
// release the workspace.
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

#ifdef SSTEM_V3_PHASES
// diagnostic builds only (tools/v3_phases.py): clock64 ticks per tile phase, summed over the warps of every launch
extern "C" int sstem_v3_phases_bwd(unsigned long long* out, int reset) { return sstem::v3_phases_read(out, reset); }
#endif
