// Forward launchers of the tuned 51-tap kernel (device code in sepconv_k51.cuh).
#include "sepconv_k51.cuh"

namespace sstem {
namespace {

template <int CC>
int launch_fwd_chunk(const float* in, const float* v, const float* h, float* out,
                     int64_t B, int C, int c0, int H, int W, int replicas, cudaStream_t s) {
    return dispatch([&](auto vec, auto pair) {
        constexpr size_t smem = smem_bytes<FWD_G, FWD_R, CC>();
        return launch_k51<sepconv_fwd_k51_kernel<CC, FWD_G, FWD_R, decltype(vec)::value, decltype(pair)::value>, FWD_G, FWD_R>(
            smem, smem, B, H, W, s, in, v, h, out, C, c0, H, W, replicas, g_gate.ptr, g_gate.want);
    }, ring_vec(W, v), window_pair(W, in));
}

}  // namespace

int launch_sepconv_fwd_k51(const float* in, const float* v, const float* h, float* out,
                           int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s) {
    if (!fits_grid<FWD_R>(B, H)) return launch_sepconv_fwd_generic(in, v, h, out, B, C, H, W, 51, false, s);
    if (gray && C > 1)                                     // identical planes: compute one, write C copies
        return launch_fwd_chunk<1>(in, v, h, out, B, (int)C, 0, (int)H, (int)W, (int)C, s);
    return for_each_chunk(C, [&](auto cc, int c0) {       // taps re-read per chunk
        constexpr int CC = decltype(cc)::value;
        if constexpr (CC == 3) {
            // third-generation kernel (persistent warps, TMA-streamed, channel-interleaved window) when its layout rules hold
            const int e = try_launch_fwd_k51_v3(in, v, h, out, B, (int)C, c0, (int)H, (int)W, s);
            if (e != PATH_NOT_APPLICABLE) return e;
        }
        return launch_fwd_chunk<CC>(in, v, h, out, B, (int)C, c0, (int)H, (int)W, 1, s);
    });
}

}  // namespace sstem
