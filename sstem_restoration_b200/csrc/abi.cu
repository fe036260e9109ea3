// C-ABI entry points for the sepconv path (argument checks + dispatch) and the
// small ABI utilities.  See include/sstem_b200.h for the contract.
#include "common.cuh"

namespace sstem {
std::atomic<int64_t> g_launches{0};
thread_local LaunchGate g_gate;
}
using namespace sstem;

static int check_sepconv_dims(int64_t B, int64_t C, int64_t H, int64_t W, int K) {
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return SSTEM_E_SHAPE;
    if (K < 1 || K > 64) return SSTEM_E_SHAPE;
    if (H + K - 1 > INT32_MAX / 2 || W + K - 1 > INT32_MAX / 2 || C > 65535) return SSTEM_E_SHAPE;
    return 0;
}

extern "C" int sstem_sepconv_forward(const float* input, const float* vertical, const float* horizontal,
                                     float* output, int64_t B, int64_t C, int64_t H, int64_t W,
                                     int32_t K, uint32_t flags, void* stream) {
    if (!input || !vertical || !horizontal || !output) return SSTEM_E_NULL;
    if (int e = check_sepconv_dims(B, C, H, W, K)) return e;
    if (flags & ~(SSTEM_SEPCONV_STRICT_ORDER | SSTEM_SEPCONV_GRAY_REPLICATED)) return SSTEM_E_FLAG;
    if (!aligned4(input) || !aligned4(vertical) || !aligned4(horizontal) || !aligned4(output)) return SSTEM_E_ALIGN;
    DeviceGuard guard(output);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    const bool strict = flags & SSTEM_SEPCONV_STRICT_ORDER;
    const bool gray = flags & SSTEM_SEPCONV_GRAY_REPLICATED;
    if (K == 51 && !strict) return launch_sepconv_fwd_k51(input, vertical, horizontal, output, B, C, H, W, gray, s);
    return launch_sepconv_fwd_generic(input, vertical, horizontal, output, B, C, H, W, K, strict, s);
}

extern "C" int sstem_sepconv_backward(const float* grad_output, const float* input,
                                      const float* vertical, const float* horizontal,
                                      float* grad_input, float* grad_vertical, float* grad_horizontal,
                                      int64_t B, int64_t C, int64_t H, int64_t W,
                                      int32_t K, uint32_t flags, void* stream) {
    if (!grad_output || !input || !vertical || !horizontal) return SSTEM_E_NULL;
    if (!grad_input && !grad_vertical && !grad_horizontal) return SSTEM_E_NULL;
    if (int e = check_sepconv_dims(B, C, H, W, K)) return e;
    if (flags & ~(SSTEM_SEPCONV_STRICT_ORDER | SSTEM_SEPCONV_GRAY_REPLICATED)) return SSTEM_E_FLAG;
    if (!aligned4(grad_output) || !aligned4(input) || !aligned4(vertical) || !aligned4(horizontal) ||
        !aligned4(grad_input) || !aligned4(grad_vertical) || !aligned4(grad_horizontal))
        return SSTEM_E_ALIGN;
    const void* any_out = grad_vertical ? grad_vertical : (grad_horizontal ? grad_horizontal : grad_input);
    DeviceGuard guard(any_out);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    int e = 0;
    if (grad_vertical || grad_horizontal) {
        if (K == 51)
            e = launch_sepconv_bwd_taps_k51(grad_output, input, vertical, horizontal, grad_vertical, grad_horizontal, B, C, H, W,
                                            (flags & SSTEM_SEPCONV_GRAY_REPLICATED) != 0, s);
        else
            e = launch_sepconv_bwd_taps_generic(grad_output, input, vertical, horizontal, grad_vertical, grad_horizontal, B, C, H, W, K, s);
        if (e) return e;
    }
    if (grad_input) {
        if (K == 51) e = launch_sepconv_bwd_input_k51(grad_output, vertical, horizontal, grad_input, B, C, H, W, s);
        else e = launch_sepconv_bwd_input_generic(grad_output, vertical, horizontal, grad_input, B, C, H, W, K, s);
    }
    return e;
}

// ---- gray x3 detection on the device (no host round trip) ------------------------------------------------------------
extern "C" int sstem_sepconv_forward_detect(const float* input, const float* vertical, const float* horizontal,
                                            float* output, int64_t B, int64_t C, int64_t H, int64_t W,
                                            int32_t K, uint32_t flags, int32_t* gray_flag, void* stream) {
    if (!gray_flag) return SSTEM_E_NULL;
    if (!aligned4(gray_flag)) return SSTEM_E_ALIGN;
    if (flags & ~SSTEM_SEPCONV_STRICT_ORDER) return SSTEM_E_FLAG;      // GRAY_REPLICATED is what this call decides itself
    const bool detect = K == 51 && !(flags & SSTEM_SEPCONV_STRICT_ORDER) && C > 1;
    if (!detect) {                                                      // nothing to gain: general path, flag = 0
        const int e = sstem_sepconv_forward(input, vertical, horizontal, output, B, C, H, W, K, flags, stream);
        if (e) return e;
        DeviceGuard guard(output);
        return (int)cudaMemsetAsync(gray_flag, 0, sizeof(int32_t), (cudaStream_t)stream);
    }
    if (!input || !vertical || !horizontal || !output) return SSTEM_E_NULL;
    if (int e = check_sepconv_dims(B, C, H, W, K)) return e;
    {
        DeviceGuard guard(output);
        if (guard.err) return guard.err;
        if (int e = launch_planes_equal(input, B, C, (H + K - 1) * (W + K - 1), gray_flag, (cudaStream_t)stream)) return e;
    }
    {   // identical planes: one plane computed, C written
        GateScope gate(gray_flag, 1);
        if (int e = sstem_sepconv_forward(input, vertical, horizontal, output, B, C, H, W, K, SSTEM_SEPCONV_GRAY_REPLICATED, stream)) return e;
    }
    GateScope gate(gray_flag, 0);
    return sstem_sepconv_forward(input, vertical, horizontal, output, B, C, H, W, K, 0, stream);
}

extern "C" int sstem_sepconv_backward_detect(const float* grad_output, const float* input,
                                             const float* vertical, const float* horizontal,
                                             float* grad_input, float* grad_vertical, float* grad_horizontal,
                                             int64_t B, int64_t C, int64_t H, int64_t W,
                                             int32_t K, uint32_t flags, const int32_t* gray_flag, void* stream) {
    if (!gray_flag) return SSTEM_E_NULL;
    if (flags & ~SSTEM_SEPCONV_STRICT_ORDER) return SSTEM_E_FLAG;
    const bool detect = K == 51 && C > 1 && (grad_vertical || grad_horizontal);
    if (!detect)
        return sstem_sepconv_backward(grad_output, input, vertical, horizontal, grad_input, grad_vertical, grad_horizontal, B, C, H, W, K, flags, stream);
    // grad_input does not depend on the input: computed once, ungated
    if (grad_input)
        if (int e = sstem_sepconv_backward(grad_output, input, vertical, horizontal, grad_input, nullptr, nullptr, B, C, H, W, K, flags, stream)) return e;
    {
        GateScope gate(gray_flag, 1);
        if (int e = sstem_sepconv_backward(grad_output, input, vertical, horizontal, nullptr, grad_vertical, grad_horizontal, B, C, H, W, K,
                                           flags | SSTEM_SEPCONV_GRAY_REPLICATED, stream))
            return e;
    }
    GateScope gate(gray_flag, 0);
    return sstem_sepconv_backward(grad_output, input, vertical, horizontal, nullptr, grad_vertical, grad_horizontal, B, C, H, W, K, flags, stream);
}

static int check_tail_args(int64_t B, int64_t C, int64_t H, int64_t W, int32_t K, uint32_t flags, int64_t bstride) {
    if (int e = check_sepconv_dims(B, C, H, W, K)) return e;
    if (K != 51) return SSTEM_E_SHAPE;                  // the reference's only tap count; no generic tail
    if (flags & ~SSTEM_SEPCONV_GRAY_REPLICATED) return SSTEM_E_FLAG;
    if (bstride < C * H * W) return SSTEM_E_SHAPE;
    return 0;
}

extern "C" int sstem_interp_tail_forward(const float* frame1, const float* frame2, int64_t frame_batch_stride,
                                         const float* k1v, const float* k1h, const float* k2v, const float* k2h,
                                         float* output, int64_t B, int64_t C, int64_t H, int64_t W,
                                         int32_t K, uint32_t flags, void* stream) {
    if (!frame1 || !frame2 || !k1v || !k1h || !k2v || !k2h || !output) return SSTEM_E_NULL;
    if (int e = check_tail_args(B, C, H, W, K, flags, frame_batch_stride)) return e;
    if (!aligned4(frame1) || !aligned4(frame2) || !aligned4(k1v) || !aligned4(k1h) || !aligned4(k2v) || !aligned4(k2h) ||
        !aligned4(output))
        return SSTEM_E_ALIGN;
    DeviceGuard guard(output);
    if (guard.err) return guard.err;
    return launch_interp_tail_fwd_k51(frame1, frame2, frame_batch_stride, k1v, k1h, k2v, k2h, output, B, C, H, W,
                                      (flags & SSTEM_SEPCONV_GRAY_REPLICATED) != 0, (cudaStream_t)stream);
}

extern "C" int sstem_interp_tail_backward(const float* grad_output, const float* frame1, const float* frame2,
                                          int64_t frame_batch_stride,
                                          const float* k1v, const float* k1h, const float* k2v, const float* k2h,
                                          float* g_k1v, float* g_k1h, float* g_k2v, float* g_k2h,
                                          int64_t B, int64_t C, int64_t H, int64_t W,
                                          int32_t K, uint32_t flags, void* stream) {
    if (!grad_output || !frame1 || !frame2 || !k1v || !k1h || !k2v || !k2h) return SSTEM_E_NULL;
    if (!g_k1v && !g_k1h && !g_k2v && !g_k2h) return SSTEM_E_NULL;
    if (int e = check_tail_args(B, C, H, W, K, flags, frame_batch_stride)) return e;
    if (!aligned4(grad_output) || !aligned4(frame1) || !aligned4(frame2) || !aligned4(k1v) || !aligned4(k1h) ||
        !aligned4(k2v) || !aligned4(k2h) || !aligned4(g_k1v) || !aligned4(g_k1h) || !aligned4(g_k2v) || !aligned4(g_k2h))
        return SSTEM_E_ALIGN;
    const void* any_out = g_k1v ? g_k1v : (g_k1h ? g_k1h : (g_k2v ? g_k2v : g_k2h));
    DeviceGuard guard(any_out);
    if (guard.err) return guard.err;
    const bool gray = (flags & SSTEM_SEPCONV_GRAY_REPLICATED) != 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (g_k2v || g_k2h)
        if (int e = launch_interp_tail_bwd_k51(grad_output, frame2, frame_batch_stride, k2v, k2h, g_k2v, g_k2h, B, C, H, W, gray, s))
            return e;
    if (g_k1v || g_k1h)
        if (int e = launch_interp_tail_bwd_k51(grad_output, frame1, frame_batch_stride, k1v, k1h, g_k1v, g_k1h, B, C, H, W, gray, s))
            return e;
    return 0;
}

extern "C" int64_t sstem_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" int sstem_abi_version(void) { return SSTEM_ABI_VERSION; }

extern "C" const char* sstem_error_string(int code) {
    switch (code) {
        case 0: return "success";
        case SSTEM_E_NULL: return "sstem: a required pointer is NULL";
        case SSTEM_E_SHAPE: return "sstem: non-positive size or unsupported tap count (1..64)";
        case SSTEM_E_ALIGN: return "sstem: pointer is not sufficiently aligned";
        case SSTEM_E_DEVICE: return "sstem: pointer is not CUDA device memory";
        case SSTEM_E_FLAG: return "sstem: unknown flag, layout or mode";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "sstem: unknown error code";
}
