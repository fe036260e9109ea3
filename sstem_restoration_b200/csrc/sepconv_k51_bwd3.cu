// Launchers of the third-generation tap-gradient kernel (device code and the shared launch steps in
// sepconv_k51_v3.cuh): the 3-channel chunks on [B,51,H,W] taps that the generation-1 dispatcher hands over
// (try_launch_bwd_taps_k51_v3), and the tap gradients on the tile-major tap layout of SURVEY 8f N2
// (sstem_sepconv_backward_tiled; the layout conversions are in sepconv_layout.cu).
#include "sepconv_k51_v3.cuh"

namespace sstem {
namespace {

// The upstream gradient as the kernel reads it: planes of W floats, rows `pitch` floats apart (a multiple of 4), planes
// `plane` and images `batch` floats apart, base 16-byte aligned.
struct GradPlanes {
    const float* g;
    int64_t pitch, plane, batch;
};

// One channel chunk (CC planes from sh.c0) of grad_vertical and / or grad_horizontal (null when not wanted); `accum`
// adds to them (the chunks after the first).  TILED: taps and tap gradients are tile-major; otherwise [B,51,H,W], CC = 3.
template <int CC, bool TILED>
int launch_bwd_chunk(const GradPlanes& gp, const float* in, const float* v, const float* h, float* gv, float* gh,
                     int64_t B, const V3Shape& sh, bool accum, cudaStream_t s) {
    static_assert(TILED || CC == 3, "the [B,51,H,W] tap-gradient kernel reads three channels");
    V3Window<CC> win(in, B, sh, s);
    if (win.err) return win.err;
    // both tap maps are encoded: the one the kernel does not read (no gv or no gh) must still be a valid object to copy
    CUtensorMap mv, mh, mg;
    const int64_t gdims[4] = {sh.W, sh.H, CC, B}, gstrides[4] = {1, gp.pitch, gp.plane, gp.batch};
    const int gbox[4] = {V3_COLS, B3_R, CC, 1};
    if (!make_map_f32(&mg, gp.g + sh.c0 * gp.plane, 4, gdims, gstrides, gbox)) return SSTEM_E_SHAPE;
    if constexpr (TILED) {
        // tile-major taps: the tile row and the batch merge into one dimension; v lands as [plane][row][col], h as
        // [row][tap][col] -- the ring-slot and tap-buffer layouts of the [B,51,H,W] maps
        const int64_t tiles_x8 = (sh.W + 7) / 8, tiles_y8 = (sh.H + 7) / 8, tstride = tiles_x8 * K51 * 64;
        const int64_t vdims[5] = {8, 8, K51, tiles_x8, tiles_y8 * B}, vstrides[5] = {1, 8, 64, K51 * 64, tstride};
        const int64_t hdims[5] = {8, K51, 8, tiles_x8, tiles_y8 * B}, hstrides[5] = {1, 64, 8, K51 * 64, tstride};
        const int vbox[5] = {V3_COLS, B3_R, V3_GROUP, 1, 1}, hbox[5] = {V3_COLS, K51, B3_R, 1, 1};
        if (!make_map_f32(&mv, v, 5, vdims, vstrides, vbox) || !make_map_f32(&mh, h, 5, hdims, hstrides, hbox)) return SSTEM_E_SHAPE;
    } else if (!make_v3_tap_maps(&mv, &mh, v, h, B, sh.H, sh.W, B3_R)) {
        return SSTEM_E_SHAPE;
    }
    // one kernel per combination of gradients written (gv, gh or both) and accumulation
    auto launch = [&](auto wv, auto wh, auto acc) {
        constexpr bool WV = decltype(wv)::value, WH = decltype(wh)::value, ACCUM = decltype(acc)::value;
        if constexpr (TILED)
            return launch_persistent<sepconv_bwd_taps_k51_v3_tiled_kernel<WV, WH, ACCUM, CC>>(V3_SMEM, sh.ntiles, s, win.map, mv, mh,
                                                                                             mg, gv, gh, win.counter, sh);
        else
            return launch_persistent<sepconv_bwd_taps_k51_v3_kernel<WV, WH, ACCUM>>(V3_SMEM, sh.ntiles, s, win.map, mv, mh, mg, gv, gh,
                                                                                   win.counter, sh);
    };
    using T = std::true_type;
    using F = std::false_type;
    auto with_accum = [&](auto wv, auto wh) { return accum ? launch(wv, wh, T{}) : launch(wv, wh, F{}); };
    if (gv && gh) return with_accum(T{}, T{});
    if (gv) return with_accum(T{}, F{});
    return with_accum(F{}, T{});
}

// Tap gradients on tile-major taps, always on the persistent kernel.  gray: one one-plane launch with the channel-summed
// gradient; otherwise 3-channel chunks, then single planes.  The gradient's tensor map needs W % 4 == 0 and a 16-byte
// aligned base: otherwise, and always for gray, it is staged at a 4-float row pitch first (a few floats per pixel,
// against ~840 B per pixel that the kernel itself moves).
int launch_bwd_taps_tiled(const float* g, const float* in, const float* vt, const float* ht, float* gvt, float* ght,
                          int64_t B, int C, int H, int W, bool gray, cudaStream_t s) {
    V3Shape sh;   // half tiles: ceil(H/4) rows of warp tiles would miss the bottom half of the last tile row
    if (!v3_shape(sh, B, C, 0, H, W, 2 * (int64_t)((H + 7) / 8))) return SSTEM_E_SHAPE;
    const int64_t plane = (int64_t)H * W;
    GradPlanes gp{g, W, plane, (int64_t)C * plane};
    float* staged = nullptr;
    if (gray || (W & 3) || !aligned16(g)) {
        const int64_t WP = (W + 3) & ~3, nplanes = gray ? 1 : C;
        if (workspace_alloc(reinterpret_cast<void**>(&staged), (size_t)(B * nplanes * H * WP) * 4, s)) return cudaErrorMemoryAllocation;
        if (int e = launch_stage_grad_planes(g, staged, B, C, H, W, WP, gray, s)) { cudaFreeAsync(staged, s); return e; }
        gp = GradPlanes{staged, WP, H * WP, nplanes * H * WP};
    }
    int e = 0;
    if (gray) {
        e = launch_bwd_chunk<1, true>(gp, in, vt, ht, gvt, ght, B, sh, false, s);
    } else {
        for (int c0 = 0; c0 < C && !e;) {
            sh.c0 = c0;
            if (C - c0 >= 3) { e = launch_bwd_chunk<3, true>(gp, in, vt, ht, gvt, ght, B, sh, c0 > 0, s); c0 += 3; }
            else { e = launch_bwd_chunk<1, true>(gp, in, vt, ht, gvt, ght, B, sh, c0 > 0, s); c0 += 1; }
        }
    }
    if (staged) cudaFreeAsync(staged, s);
    return e;
}

}  // namespace

int try_launch_bwd_taps_k51_v3(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                               int64_t B, int C, int c0, int H, int W, int accumulate, cudaStream_t s) {
    // measured crossover: ~6 CTA tiles per CTA (the forward's is ~10)
    return try_v3(aligned16(v) && aligned16(h) && aligned16(g) && !((int64_t)H * W * c0 & 3), B, C, c0, H, W, B3_R, 6,
                  [&](const V3Shape& sh) {
                      const GradPlanes gp{g, W, (int64_t)H * W, (int64_t)C * H * W};
                      return launch_bwd_chunk<3, false>(gp, in, v, h, gv, gh, B, sh, accumulate != 0, s);
                  });
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
