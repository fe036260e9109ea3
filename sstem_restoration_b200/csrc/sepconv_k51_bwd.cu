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
    if (!fits_grid<BWD_R>(B, H)) return launch_sepconv_bwd_taps_generic(g, in, v, h, gv, gh, B, C, H, W, 51, s);
    if (gv && gh) return launch_bwd_taps_k51_vh(g, in, v, h, gv, gh, B, (int)C, (int)H, (int)W, gray, s);
    if (gv) return launch_bwd_taps_k51_v(g, in, v, h, gv, gh, B, (int)C, (int)H, (int)W, gray, s);
    return launch_bwd_taps_k51_h(g, in, v, h, gv, gh, B, (int)C, (int)H, (int)W, gray, s);
}
#else
namespace {

template <int CC, bool WV, bool WH>
int launch_bwd_chunk(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                     int64_t B, int C, int c0, int H, int W, bool accumulate, int replicas, cudaStream_t s) {
    return dispatch([&](auto vec, auto pair, auto acc) {
        constexpr size_t smem = smem_bytes<BWD_G, BWD_R, CC>();
        return launch_k51<sepconv_bwd_taps_k51_kernel<CC, BWD_G, BWD_R, decltype(vec)::value, decltype(pair)::value, WV, WH,
                                                      decltype(acc)::value>, BWD_G, BWD_R>(
            smem, smem, B, H, W, s, g, in, v, h, gv, gh, C, c0, H, W, replicas, (int64_t)0, 1, 1, 1.f, g_gate.ptr, g_gate.want);
    }, ring_vec(W, v), window_pair(W, in), accumulate);
}

template <bool WV, bool WH>
int launch_bwd_all(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                   int64_t B, int C, int H, int W, bool gray, cudaStream_t s) {
    if (gray && C > 1)                                     // identical planes: one channel, summed upstream gradient
        return launch_bwd_chunk<1, WV, WH>(g, in, v, h, gv, gh, B, C, 0, H, W, false, C, s);
    return for_each_chunk(C, [&](auto cc, int c0) {       // later chunks accumulate
        constexpr int CC = decltype(cc)::value;
        if constexpr (CC == 3) {
            // third-generation kernel (persistent warps, TMA-streamed, channel-interleaved window) when its layout rules hold
            const int e = try_launch_bwd_taps_k51_v3(g, in, v, h, WV ? gv : nullptr, WH ? gh : nullptr, B, C, c0, H, W, c0 > 0, s);
            if (e != PATH_NOT_APPLICABLE) return e;
        }
        return launch_bwd_chunk<CC, WV, WH>(g, in, v, h, gv, gh, B, C, c0, H, W, c0 > 0, 1, s);
    });
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
