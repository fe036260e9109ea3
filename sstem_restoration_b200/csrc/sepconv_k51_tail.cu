// Launchers of the fused interpolation tail (device code in sepconv_k51.cuh).
#include "sepconv_k51.cuh"

namespace sstem {
namespace {

// up to 3 channel planes are staged side by side: the kernel's attribute allows 3, a launch uses `nplanes`
template <int G, int R>
size_t tail_smem_used(int nplanes) {
    return nplanes == 1 ? smem_bytes<G, R, 1>() : (nplanes == 2 ? smem_bytes<G, R, 2>() : smem_bytes<G, R, 3>());
}

}  // namespace

int launch_interp_tail_fwd_k51(const float* frame1, const float* frame2, int64_t frame_bstride,
                               const float* k1v, const float* k1h, const float* k2v, const float* k2h, float* out,
                               int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s) {
    if (!fits_grid<FWD_R>(B, H)) return SSTEM_E_SHAPE;
    const int cs = gray ? 1 : (int)C;
    const int nplanes = cs <= 3 ? cs : 1;
    const float scale = gray ? 1.f : 1.f / (float)C;
    const TailFrames fa = {{frame2, frame1}, {k2v, k1v}, {k2h, k1h}};   // frame 2 first, as the reference's expression
    return dispatch([&](auto vec) {
        return launch_k51<interp_tail_fwd_k51_kernel<FWD_G, FWD_R, decltype(vec)::value>, FWD_G, FWD_R>(
            smem_bytes<FWD_G, FWD_R, 3>(), tail_smem_used<FWD_G, FWD_R>(nplanes), B, (int)H, (int)W, s,
            fa, frame_bstride, cs, nplanes, out, scale, (int)H, (int)W);
    }, ring_vec(W, k1v) && ring_vec(W, k2v));
}

// tap gradients of ONE frame of the fused tail (the two frames are independent)
int launch_interp_tail_bwd_k51(const float* g, const float* frame, int64_t frame_bstride, const float* v, const float* h,
                               float* gv, float* gh, int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s) {
    if (!fits_grid<BWD_R>(B, H)) return SSTEM_E_SHAPE;
    const int cs = gray ? 1 : (int)C;
    const int nplanes = cs <= 3 ? cs : 1;
    const float gscale = gray ? 1.f : 1.f / (float)C;
    auto launch = [&](auto vec, auto wv, auto wh) {
        return launch_k51<sepconv_bwd_taps_k51_kernel<1, BWD_G, BWD_R, decltype(vec)::value, false, decltype(wv)::value,
                                                      decltype(wh)::value, false, true>, BWD_G, BWD_R>(
            smem_bytes<BWD_G, BWD_R, 3>(), tail_smem_used<BWD_G, BWD_R>(nplanes), B, (int)H, (int)W, s,
            g, frame, v, h, gv, gh, 1, 0, (int)H, (int)W, 1, frame_bstride, cs, nplanes, gscale, nullptr, 0);
    };
    // one kernel per combination of gradients written: gv and gh, gv only, gh only
    using T = std::true_type;
    using F = std::false_type;
    return dispatch([&](auto vec) {
        if (gv && gh) return launch(vec, T{}, T{});
        if (gv) return launch(vec, T{}, F{});
        return launch(vec, F{}, T{});
    }, ring_vec(W, v));
}

}  // namespace sstem
