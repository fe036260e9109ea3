// Forward launchers of the tuned 51-tap kernel (device code in sepconv_k51.cuh).
#include "sepconv_k51.cuh"

namespace sstem {
namespace {

template <int CC, bool VEC, bool PAIR>
int launch_fwd_variant(const float* in, const float* v, const float* h, float* out,
                       int64_t B, int C, int c0, int H, int W, int replicas, cudaStream_t s) {
    constexpr int G = SSTEM_FWD_G, R = SSTEM_FWD_R;
    constexpr size_t smem = smem_bytes<G, R, CC>();
    static PerDeviceOnce done;
    auto kern = sepconv_fwd_k51_kernel<CC, G, R, VEC, PAIR>;
    if (int e = set_smem_once(kern, smem, done)) return e;
    dim3 grid((unsigned)((W + Geo<G, R>::TILE_W - 1) / Geo<G, R>::TILE_W), (unsigned)((H + R - 1) / R), (unsigned)B);
    kern<<<grid, 128, smem, s>>>(in, v, h, out, C, c0, H, W, replicas, g_gate.ptr, g_gate.want);
    count_launch();
    return finish_launch();
}

template <int CC>
int launch_fwd_chunk(const float* in, const float* v, const float* h, float* out,
                     int64_t B, int C, int c0, int H, int W, int replicas, cudaStream_t s) {
    const bool vec = ((W & 3) == 0) && aligned16(v);
    const bool pair = (((W + K51 - 1) & 1) == 0) && ((reinterpret_cast<uintptr_t>(in) & 7u) == 0);
    if (vec && pair) return launch_fwd_variant<CC, true, true>(in, v, h, out, B, C, c0, H, W, replicas, s);
    if (vec) return launch_fwd_variant<CC, true, false>(in, v, h, out, B, C, c0, H, W, replicas, s);
    if (pair) return launch_fwd_variant<CC, false, true>(in, v, h, out, B, C, c0, H, W, replicas, s);
    return launch_fwd_variant<CC, false, false>(in, v, h, out, B, C, c0, H, W, replicas, s);
}

}  // namespace

int launch_sepconv_fwd_k51(const float* in, const float* v, const float* h, float* out,
                           int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s) {
    if (B > 65535 || (H + SSTEM_FWD_R - 1) / SSTEM_FWD_R > 65535)   // grid.y / grid.z limits
        return launch_sepconv_fwd_generic(in, v, h, out, B, C, H, W, 51, false, s);
    if (gray && C > 1)                                     // identical planes: compute one, write C copies
        return launch_fwd_chunk<1>(in, v, h, out, B, (int)C, 0, (int)H, (int)W, (int)C, s);
    int c0 = 0;
    while (c0 < C) {                                       // channels in chunks of <= 3 (taps re-read per chunk)
        const int cc = (C - c0) < 3 ? (int)(C - c0) : 3;
        int e;
        if (cc == 3) {
            // third-generation kernel (persistent warps, TMA-streamed, channel-interleaved window) when its layout rules hold
            e = try_launch_fwd_k51_v3(in, v, h, out, B, (int)C, c0, (int)H, (int)W, s);
            if (e == PATH_NOT_APPLICABLE) e = launch_fwd_chunk<3>(in, v, h, out, B, (int)C, c0, (int)H, (int)W, 1, s);
        }
        else if (cc == 2) e = launch_fwd_chunk<2>(in, v, h, out, B, (int)C, c0, (int)H, (int)W, 1, s);
        else e = launch_fwd_chunk<1>(in, v, h, out, B, (int)C, c0, (int)H, (int)W, 1, s);
        if (e) return e;
        c0 += cc;
    }
    return 0;
}

}  // namespace sstem
