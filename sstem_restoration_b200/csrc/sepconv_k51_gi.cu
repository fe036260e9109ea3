// Launcher of the tuned grad_input kernel (device code in sepconv_k51.cuh).
#include "sepconv_k51.cuh"

namespace sstem {

int launch_sepconv_bwd_input_k51(const float* g, const float* v, const float* h, float* gi,
                                 int64_t B, int64_t C, int64_t H, int64_t W, cudaStream_t s) {
    if (!fits_grid<FWD_R>(B, H)) return launch_sepconv_bwd_input_generic(g, v, h, gi, B, C, H, W, 51, s);
    cudaError_t e = cudaMemsetAsync(gi, 0, (size_t)B * C * (H + K51 - 1) * (W + K51 - 1) * sizeof(float), s);
    if (e != cudaSuccess) return (int)e;
    return for_each_chunk(C, [&](auto cc, int c0) {
        return dispatch([&](auto vec) {
            constexpr size_t smem = smem_bytes<FWD_G, FWD_R, decltype(cc)::value>();
            return launch_k51<sepconv_bwd_input_k51_kernel<decltype(cc)::value, FWD_R, decltype(vec)::value>, FWD_G, FWD_R>(
                smem, smem, B, (int)H, (int)W, s, g, v, h, gi, (int)C, c0, (int)H, (int)W);
        }, ring_vec(W, v));
    });
}

}  // namespace sstem
