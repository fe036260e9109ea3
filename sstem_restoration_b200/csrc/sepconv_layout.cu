// Layout kernels around the 51-tap kernels, each compiled once: the input repacks that the third-generation kernels'
// tensor maps read (sepconv_k51_fwd3.cu, sepconv_k51_bwd3.cu) in a stream-ordered workspace, the gray x3 plane
// comparison (abi.cu), the tile-major tap layout of SURVEY 8f N2 (sstem_taps_to_tiled, sstem_taps_from_tiled) and the
// upstream-gradient staging of the tiled tap gradients (sepconv_k51_bwd3.cu).
#include "sepconv_k51.cuh"

namespace sstem {
namespace {

// NCHW planes c0..c0+2 of `in` [B,C,IH,IW] -> out [B,IH,IW] float4 (x, y, z = the three channels, w = 0)
template <bool VEC4>
__global__ void __launch_bounds__(256)
repack_nchw3_to_nhwc4_kernel(const float* __restrict__ in, float4* __restrict__ out, int C, int c0, int64_t plane, int64_t total,
                             const int* gate, int gate_want) {
    SSTEM_GATE_RETURN(gate, gate_want);
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    if (VEC4) {                                           // plane % 4 == 0 and 16-byte aligned base: 4 pixels per thread
        const int64_t n4 = total >> 2, p4 = plane >> 2;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += step) {
            const int64_t b = i / p4, p = i - b * p4;
            const float4* s = reinterpret_cast<const float4*>(in + (b * C + c0) * plane) + p;
            const float4 a = __ldcs(s), bb = __ldcs(s + p4), c = __ldcs(s + 2 * p4);
            float4* d = out + 4 * i;
            d[0] = make_float4(a.x, bb.x, c.x, 0.f);
            d[1] = make_float4(a.y, bb.y, c.y, 0.f);
            d[2] = make_float4(a.z, bb.z, c.z, 0.f);
            d[3] = make_float4(a.w, bb.w, c.w, 0.f);
        }
    } else {
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
            const int64_t b = i / plane, p = i - b * plane;
            const float* s = in + (b * C + c0) * plane + p;
            out[i] = make_float4(__ldg(s), __ldg(s + plane), __ldg(s + 2 * plane), 0.f);
        }
    }
}

// One plane (channel c0) of in [B,C,IH,IW] -> out [B,IH,IWP] with the row pitch IWP rounded up to 4 floats, so that
// the copy can be the source of a tensor map (16-byte strides); the pad columns are zero.
__global__ void __launch_bounds__(256)
repack_plane_pitch_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int c0, int IH, int IW, int IWP, int64_t total,
                          const int* gate, int gate_want) {
    SSTEM_GATE_RETURN(gate, gate_want);
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const int x = (int)(i % IWP);
        const int64_t r = i / IWP;
        const int y = (int)(r % IH);
        const int64_t b = r / IH;
        out[i] = x < IW ? __ldg(in + ((b * C + c0) * IH + y) * (int64_t)IW + x) : 0.f;
    }
}

// flag = 1 iff every channel plane of in [B,C,plane] is bit-identical to plane 0 of its image (gray sections replicated
// x3: sff_scripts_interp/data/data_provider.py:136-137).  *flag must be 1 on entry; any mismatch clears it.
__global__ void __launch_bounds__(256)
planes_equal_kernel(const float* __restrict__ in, int C, int64_t plane, int64_t total /* B * plane */, int* __restrict__ flag) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    bool same = true;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total && same; i += step) {
        const int64_t b = i / plane, p = i - b * plane;
        const unsigned* s = reinterpret_cast<const unsigned*>(in) + b * C * plane + p;
        const unsigned ref = __ldg(s);
        for (int c = 1; c < C; ++c) same = same && (__ldg(s + c * plane) == ref);
    }
    if (!__all_sync(0xffffffffu, same) && (threadIdx.x & 31) == 0) *flag = 0;
}

// NCHW taps [B,51,H,W] -> tile-major [B][ceil(H/8)][ceil(W/8)][51][8][8] (zero outside the image): the layout the
// TILED kernels consume (SURVEY 8f N2).  One thread per output element; reads are 32-byte row segments.
__global__ void __launch_bounds__(256)
taps_to_tiled_kernel(const float* __restrict__ taps, float* __restrict__ tiled, int H, int W, int ty8, int tx8, int64_t total) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const int col = (int)(i & 7), row = (int)((i >> 3) & 7);
        int64_t r = i >> 6;
        const int tap = (int)(r % K51); r /= K51;
        const int tx = (int)(r % tx8); r /= tx8;
        const int ty = (int)(r % ty8);
        const int64_t b = r / ty8;
        const int y = ty * 8 + row, x = tx * 8 + col;
        tiled[i] = (y < H && x < W) ? __ldg(taps + ((b * K51 + tap) * H + y) * (int64_t)W + x) : 0.f;
    }
}

// The inverse: tile-major -> [B,51,H,W] (the padding entries are not read).  One thread per output element.
__global__ void __launch_bounds__(256)
taps_from_tiled_kernel(const float* __restrict__ tiled, float* __restrict__ taps, int H, int W, int ty8, int tx8, int64_t total) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const int x = (int)(i % W);
        int64_t r = i / W;
        const int y = (int)(r % H); r /= H;
        const int tap = (int)(r % K51);
        const int64_t b = r / K51;
        taps[i] = __ldg(tiled + (((b * ty8 + (y >> 3)) * tx8 + (x >> 3)) * K51 + tap) * 64 + (y & 7) * 8 + (x & 7));
    }
}

// grad_output planes at a 16-byte row pitch for the tiled tap-gradient kernel's tensor map: out [B,nplanes,H,WP] holds the
// C planes of g [B,C,H,W], or (sum) their channel sum, the gray x3 shortcut's upstream gradient.  Pad columns are zero.
__global__ void __launch_bounds__(256)
stage_grad_planes_kernel(const float* __restrict__ g, float* __restrict__ out, int C, int nplanes, int H, int W, int WP, int64_t total) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    const int64_t plane = (int64_t)H * W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const int x = (int)(i % WP);
        int64_t r = i / WP;
        const int y = (int)(r % H); r /= H;
        const int p = (int)(r % nplanes);
        const int64_t b = r / nplanes;
        float v = 0.f;
        if (x < W) {
            const float* src = g + (b * C + (nplanes == C ? p : 0)) * plane + (int64_t)y * W + x;
            v = __ldg(src);
            if (nplanes != C)
                for (int c = 1; c < C; ++c) v += __ldg(src + c * plane);
        }
        out[i] = v;
    }
}

}  // namespace

// Stream-ordered scratch memory (released with cudaFreeAsync on the same stream).  The device's default pool hands
// freed blocks back to the driver at every synchronisation unless told otherwise -- each call then paid a real
// allocation (measured: +1.5 ms per 80 MB) -- so its release threshold is raised once per device.
int workspace_alloc(void** p, size_t bytes, cudaStream_t s) {
    static PerDeviceOnce tuned;
    int dev = 0;
    cudaGetDevice(&dev);
    if (!tuned.test(dev)) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
        tuned.set(dev);
    }
    if (cudaMallocAsync(p, bytes, s) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    return 0;
}

// Repacks channels c0..c0+2 of in [B,C,IH,IW] into ws [B,IH,IW,4].
int launch_repack_nhwc4(const float* in, float* ws, int64_t B, int C, int c0, int64_t IH, int64_t IW, cudaStream_t s) {
    const int64_t plane = IH * IW, total = B * plane;
    const bool vec = (plane % 4 == 0) && aligned16(in) && ((int64_t)C * plane % 4 == 0) && ((int64_t)c0 * plane % 4 == 0);
    const int64_t work = vec ? total / 4 : total;
    const unsigned blocks = (unsigned)std::min<int64_t>((work + 255) / 256, (int64_t)sm_count() * 16);
    if (vec) repack_nchw3_to_nhwc4_kernel<true><<<blocks, 256, 0, s>>>(in, reinterpret_cast<float4*>(ws), C, c0, plane, total, g_gate.ptr, g_gate.want);
    else repack_nchw3_to_nhwc4_kernel<false><<<blocks, 256, 0, s>>>(in, reinterpret_cast<float4*>(ws), C, c0, plane, total, g_gate.ptr, g_gate.want);
    count_launch();
    return finish_launch();
}

// Copies plane c0 of in [B,C,IH,IW] into ws [B,IH,IWP] (IWP >= IW, a multiple of 4; zero pad columns).
int launch_repack_plane_pitch(const float* in, float* ws, int64_t B, int C, int c0, int64_t IH, int64_t IW, int64_t IWP, cudaStream_t s) {
    const int64_t total = B * IH * IWP;
    const unsigned blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 16);
    repack_plane_pitch_kernel<<<blocks, 256, 0, s>>>(in, ws, C, c0, (int)IH, (int)IW, (int)IWP, total, g_gate.ptr, g_gate.want);
    count_launch();
    return finish_launch();
}

int launch_stage_grad_planes(const float* g, float* out, int64_t B, int64_t C, int64_t H, int64_t W, int64_t WP, bool sum,
                             cudaStream_t s) {
    const int nplanes = sum ? 1 : (int)C;
    const int64_t total = B * nplanes * H * WP;
    const unsigned blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 16);
    stage_grad_planes_kernel<<<blocks, 256, 0, s>>>(g, out, (int)C, nplanes, (int)H, (int)W, (int)WP, total);
    count_launch();
    return finish_launch();
}

int launch_taps_from_tiled(const float* tiled, float* taps, int64_t B, int64_t H, int64_t W, cudaStream_t s) {
    const int64_t total = B * K51 * H * W;
    const unsigned blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 32);
    taps_from_tiled_kernel<<<blocks, 256, 0, s>>>(tiled, taps, (int)H, (int)W, (int)((H + 7) / 8), (int)((W + 7) / 8), total);
    count_launch();
    return finish_launch();
}

int launch_planes_equal(const float* in, int64_t B, int64_t C, int64_t plane, int* flag, cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(flag, 1, sizeof(int), s);      // non-zero = "identical planes" until a mismatch clears it
    if (e != cudaSuccess) return (int)e;
    const int64_t total = B * plane;
    const unsigned blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 16);
    planes_equal_kernel<<<blocks, 256, 0, s>>>(in, (int)C, plane, total, flag);
    count_launch();
    return finish_launch();
}

}  // namespace sstem

using namespace sstem;

// ---- tile-major taps (SURVEY 8f N2) ---------------------------------------------------------------------------------
extern "C" int64_t sstem_taps_tiled_elems(int64_t B, int64_t H, int64_t W) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    return B * ((H + 7) / 8) * ((W + 7) / 8) * K51 * 64;
}

extern "C" int sstem_taps_to_tiled(const float* taps, float* tiled, int64_t B, int64_t H, int64_t W, void* stream) {
    if (!taps || !tiled) return SSTEM_E_NULL;
    if (B <= 0 || H <= 0 || W <= 0 || H > (1 << 24) || W > (1 << 24)) return SSTEM_E_SHAPE;
    if (!aligned4(taps) || !aligned16(tiled)) return SSTEM_E_ALIGN;
    DeviceGuard guard(tiled);
    if (guard.err) return guard.err;
    const int64_t total = sstem_taps_tiled_elems(B, H, W);
    const unsigned blocks = (unsigned)std::min<int64_t>((total + 255) / 256, (int64_t)sm_count() * 32);
    taps_to_tiled_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(taps, tiled, (int)H, (int)W, (int)((H + 7) / 8), (int)((W + 7) / 8), total);
    count_launch();
    return finish_launch();
}

extern "C" int sstem_taps_from_tiled(const float* tiled, float* taps, int64_t B, int64_t H, int64_t W, void* stream) {
    if (!tiled || !taps) return SSTEM_E_NULL;
    if (B <= 0 || H <= 0 || W <= 0 || H > (1 << 24) || W > (1 << 24)) return SSTEM_E_SHAPE;
    if (!aligned16(tiled) || !aligned4(taps)) return SSTEM_E_ALIGN;
    DeviceGuard guard(taps);
    if (guard.err) return guard.err;
    return launch_taps_from_tiled(tiled, taps, B, H, W, (cudaStream_t)stream);
}
