// Tap-gradient launchers of the tuned 51-tap kernel (device code in sepconv_k51.cuh).
// Compiled four times (-DSSTEM_BWD_PART=0..3) so the 72 instantiations build in parallel:
// part 0 = dispatcher, 1 = gv + gh, 2 = gv only, 3 = gh only.
#include "sepconv_k51.cuh"

#ifndef SSTEM_BWD_PART
#error "compile with -DSSTEM_BWD_PART=0..3"
#endif

namespace sstem {

int launch_bwd_taps_k51_vh(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                           int64_t B, int C, int H, int W, bool gray, cudaStream_t s);
int launch_bwd_taps_k51_v(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                          int64_t B, int C, int H, int W, bool gray, cudaStream_t s);
int launch_bwd_taps_k51_h(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                          int64_t B, int C, int H, int W, bool gray, cudaStream_t s);

#if SSTEM_BWD_PART == 0
int launch_sepconv_bwd_taps_k51(const float* g, const float* in, const float* v, const float* h,
                                float* gv, float* gh, int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s) {
    if (B > 65535 || (H + SSTEM_BWD_R - 1) / SSTEM_BWD_R > 65535)
        return launch_sepconv_bwd_taps_generic(g, in, v, h, gv, gh, B, C, H, W, 51, s);
    if (gv && gh) return launch_bwd_taps_k51_vh(g, in, v, h, gv, gh, B, (int)C, (int)H, (int)W, gray, s);
    if (gv) return launch_bwd_taps_k51_v(g, in, v, h, gv, gh, B, (int)C, (int)H, (int)W, gray, s);
    return launch_bwd_taps_k51_h(g, in, v, h, gv, gh, B, (int)C, (int)H, (int)W, gray, s);
}
#else
namespace {

template <int CC, bool VEC, bool PAIR, bool WV, bool WH>
int launch_bwd_variant(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                       int64_t B, int C, int c0, int H, int W, int accumulate, int replicas, cudaStream_t s) {
    constexpr int G = SSTEM_BWD_G, R = SSTEM_BWD_R;
    constexpr size_t smem = smem_bytes<G, R, CC>();
    static PerDeviceOnce done;
    dim3 grid((unsigned)((W + Geo<G, R>::TILE_W - 1) / Geo<G, R>::TILE_W), (unsigned)((H + R - 1) / R), (unsigned)B);
    if (accumulate) {
        static PerDeviceOnce done_a;
        auto kern = sepconv_bwd_taps_k51_kernel<CC, G, R, VEC, PAIR, WV, WH, true>;
        if (int e = set_smem_once(kern, smem, done_a)) return e;
        kern<<<grid, 128, smem, s>>>(g, in, v, h, gv, gh, C, c0, H, W, replicas, (int64_t)0, 1, 1, 1.f, g_gate.ptr, g_gate.want);
    } else {
        auto kern = sepconv_bwd_taps_k51_kernel<CC, G, R, VEC, PAIR, WV, WH, false>;
        if (int e = set_smem_once(kern, smem, done)) return e;
        kern<<<grid, 128, smem, s>>>(g, in, v, h, gv, gh, C, c0, H, W, replicas, (int64_t)0, 1, 1, 1.f, g_gate.ptr, g_gate.want);
    }
    count_launch();
    return finish_launch();
}

template <int CC, bool WV, bool WH>
int launch_bwd_chunk(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                     int64_t B, int C, int c0, int H, int W, int accumulate, int replicas, cudaStream_t s) {
    const bool vec = ((W & 3) == 0) && aligned16(v);
    const bool pair = (((W + K51 - 1) & 1) == 0) && ((reinterpret_cast<uintptr_t>(in) & 7u) == 0);
    if (vec && pair) return launch_bwd_variant<CC, true, true, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, accumulate, replicas, s);
    if (vec) return launch_bwd_variant<CC, true, false, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, accumulate, replicas, s);
    if (pair) return launch_bwd_variant<CC, false, true, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, accumulate, replicas, s);
    return launch_bwd_variant<CC, false, false, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, accumulate, replicas, s);
}

template <bool WV, bool WH>
int launch_bwd_all(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                   int64_t B, int C, int H, int W, bool gray, cudaStream_t s) {
    if (gray && C > 1)                                     // identical planes: one channel, summed upstream gradient
        return launch_bwd_chunk<1, WV, WH>(g, in, v, h, gv, gh, B, C, 0, H, W, 0, C, s);
    int c0 = 0;
    while (c0 < C) {                                       // channel chunks of <= 3; later chunks accumulate
        const int cc = (C - c0) < 3 ? (C - c0) : 3;
        const int acc = c0 > 0;
        int e;
        if (cc == 3) {
            // third-generation kernel (persistent warps, TMA-streamed, channel-interleaved window) when its layout rules hold
            e = try_launch_bwd_taps_k51_v3(g, in, v, h, WV ? gv : nullptr, WH ? gh : nullptr, B, C, c0, H, W, acc, s);
            if (e == PATH_NOT_APPLICABLE) e = launch_bwd_chunk<3, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, acc, 1, s);
        }
        else if (cc == 2) e = launch_bwd_chunk<2, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, acc, 1, s);
        else e = launch_bwd_chunk<1, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, acc, 1, s);
        if (e) return e;
        c0 += cc;
    }
    return 0;
}

}  // namespace

#if SSTEM_BWD_PART == 1
int launch_bwd_taps_k51_vh(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                           int64_t B, int C, int H, int W, bool gray, cudaStream_t s) {
    return launch_bwd_all<true, true>(g, in, v, h, gv, gh, B, C, H, W, gray, s);
}
#elif SSTEM_BWD_PART == 2
int launch_bwd_taps_k51_v(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                          int64_t B, int C, int H, int W, bool gray, cudaStream_t s) {
    return launch_bwd_all<true, false>(g, in, v, h, gv, gh, B, C, H, W, gray, s);
}
#else
int launch_bwd_taps_k51_h(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                          int64_t B, int C, int H, int W, bool gray, cudaStream_t s) {
    return launch_bwd_all<false, true>(g, in, v, h, gv, gh, B, C, H, W, gray, s);
}
#endif
#endif

}  // namespace sstem
