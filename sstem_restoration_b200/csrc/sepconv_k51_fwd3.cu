// Launchers of the third-generation forward kernel (device code and the shared launch steps in sepconv_k51_v3.cuh): the
// 3-channel chunks on [B,51,H,W] taps that the generation-1 dispatcher hands over (try_launch_fwd_k51_v3), and the
// forward on the tile-major tap layout of SURVEY 8f N2 (sstem_sepconv_forward_tiled; the layout conversion
// sstem_taps_to_tiled is in sepconv_layout.cu).
#include "sepconv_k51_v3.cuh"

namespace sstem {
namespace {

// One channel chunk (CC planes from sh.c0).  TILED: the taps are tile-major and arrive by bulk copies, not tensor maps.
// `replicas`: output planes written per computed plane (gray x3); `accum`: add to the output instead of overwriting it.
template <int CC, bool TILED>
int launch_fwd_v3(const V3Shape& sh, const float* in, const float* v, const float* h, float* out, int64_t B, int replicas,
                  bool accum, cudaStream_t s) {
    V3Window<CC> win(in, B, sh, s);
    if (win.err) return win.err;
    CUtensorMap mv = win.map, mh = win.map;                // TILED: unused by the kernel, but must be valid objects to copy
    if (!TILED && !make_v3_tap_maps(&mv, &mh, v, h, B, sh.H, sh.W, F3_R)) return SSTEM_E_SHAPE;
    const F3Tiled tl{TILED ? v : nullptr, TILED ? h : nullptr, (sh.W + 7) / 8, (sh.H + 7) / 8, accum ? 1 : 0};
    return launch_persistent<sepconv_fwd_k51_v3_kernel<CC, TILED>>(F3_SMEM, sh.ntiles, s, win.map, mv, mh, tl, out, win.counter,
                                                                   sh, replicas);
}

}  // namespace

int try_launch_fwd_k51_v3(const float* in, const float* v, const float* h, float* out,
                          int64_t B, int C, int c0, int H, int W, cudaStream_t s) {
    // measured crossover: ~10 CTA tiles per CTA (the tap gradients' is ~6)
    return try_v3(aligned16(v) && aligned16(h), B, C, c0, H, W, F3_R, 10,
                  [&](const V3Shape& sh) { return launch_fwd_v3<3, false>(sh, in, v, h, out, B, 1, false, s); });
}

}  // namespace sstem

using namespace sstem;

extern "C" int sstem_sepconv_forward_tiled(const float* input, const float* vertical_tiled, const float* horizontal_tiled,
                                           float* output, int64_t B, int64_t C, int64_t H, int64_t W,
                                           int32_t K, uint32_t flags, void* stream) {
    if (!input || !vertical_tiled || !horizontal_tiled || !output) return SSTEM_E_NULL;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || C > 65535 || H > (1 << 24) || W > (1 << 24)) return SSTEM_E_SHAPE;
    if (K != K51) return SSTEM_E_SHAPE;                    // the tiled layout is defined for the reference's 51 taps
    if (flags & ~(SSTEM_SEPCONV_GRAY_REPLICATED | SSTEM_SEPCONV_ACCUMULATE)) return SSTEM_E_FLAG;
    // the replicated planes are written from one register: nothing to add them to
    if ((flags & SSTEM_SEPCONV_GRAY_REPLICATED) && (flags & SSTEM_SEPCONV_ACCUMULATE) && C > 1) return SSTEM_E_FLAG;
    if (!aligned4(input) || !aligned4(output)) return SSTEM_E_ALIGN;
    DeviceGuard guard(output);
    if (guard.err) return guard.err;
    if (!aligned16(vertical_tiled) || !aligned16(horizontal_tiled)) return SSTEM_E_ALIGN;
    V3Shape sh;
    if (!v3_shape(sh, B, (int)C, 0, (int)H, (int)W, (H + F3_R - 1) / F3_R)) return SSTEM_E_SHAPE;
    cudaStream_t s = (cudaStream_t)stream;
    const bool accum = flags & SSTEM_SEPCONV_ACCUMULATE;
    if ((flags & SSTEM_SEPCONV_GRAY_REPLICATED) && C > 1)
        return launch_fwd_v3<1, true>(sh, input, vertical_tiled, horizontal_tiled, output, B, (int)C, false, s);
    int e = 0;
    for (int c0 = 0; c0 < C && !e;) {                      // channel chunks of 3, then single planes
        sh.c0 = c0;
        if (C - c0 >= 3) { e = launch_fwd_v3<3, true>(sh, input, vertical_tiled, horizontal_tiled, output, B, 1, accum, s); c0 += 3; }
        else { e = launch_fwd_v3<1, true>(sh, input, vertical_tiled, horizontal_tiled, output, B, 1, accum, s); c0 += 1; }
    }
    return e;
}

#ifdef SSTEM_V3_PHASES
// diagnostic builds only (tools/v3_phases.py): clock64 ticks per tile phase, summed over the warps of every launch
extern "C" int sstem_v3_phases_fwd(unsigned long long* out, int reset) { return sstem::v3_phases_read(out, reset); }
#endif
