// Shared host-side helpers for the C-ABI translation units (no torch, no THC).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>

#include "../../include/sstem_b200.h"

namespace sstem {

extern std::atomic<int64_t> g_launches;

inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// Switches the calling thread to the device that owns `ptr` for the lifetime of
// the guard (nn.DataParallel replica threads call in with their own current
// device, but a stray call from another thread must still land correctly).
struct DeviceGuard {
    int prev = -1;
    int err = 0;
    explicit DeviceGuard(const void* ptr) {
        cudaPointerAttributes at;
        cudaError_t e = cudaPointerGetAttributes(&at, ptr);
        if (e != cudaSuccess) { cudaGetLastError(); err = SSTEM_E_DEVICE; return; }
        if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) { err = SSTEM_E_DEVICE; return; }
        int cur = 0;
        cudaGetDevice(&cur);
        if (cur != at.device) { prev = cur; cudaSetDevice(at.device); }
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

inline bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

inline int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
        cached_dev = dev;
    }
    return cached;
}

inline int finish_launch() { return (int)cudaGetLastError(); }

// Device-side launch gate (gray x3 detection without a host round trip): a kernel launched while a gate is set reads
// `*ptr` first and returns at once unless it equals `want`.  The C-ABI *_detect entry points launch BOTH candidate paths,
// each under its gate; the flag is written by planes_equal_kernel earlier on the same stream.  Thread-local, so replica
// threads do not see each other's gates.
struct LaunchGate {
    const int* ptr = nullptr;
    int want = 0;
};
extern thread_local LaunchGate g_gate;
struct GateScope {
    LaunchGate prev;
    GateScope(const int* ptr, int want) : prev(g_gate) { g_gate.ptr = ptr; g_gate.want = want; }
    ~GateScope() { g_gate = prev; }
};
#define SSTEM_GATE_RETURN(gate, want) do { if ((gate) != nullptr && ((*(gate) != 0) != ((want) != 0))) return; } while (0)

// One bit per device ordinal: "this kernel's function attributes have been set on that device".
// Replica threads (nn.DataParallel) race here, so the flag is atomic; setting an attribute twice is
// harmless, skipping it is not -- ordinals >= 64 simply set it on every call.
struct PerDeviceOnce {
    std::atomic<uint64_t> mask{0};
    bool test(int dev) const { return dev < 64 && ((mask.load(std::memory_order_acquire) >> dev) & 1u); }
    void set(int dev) { if (dev < 64) mask.fetch_or(uint64_t(1) << dev, std::memory_order_release); }
};

// ---- launchers implemented in the per-op translation units -----------------
int launch_sepconv_fwd_generic(const float* in, const float* v, const float* h, float* out,
                               int64_t B, int64_t C, int64_t H, int64_t W, int K, bool strict,
                               cudaStream_t s);
int launch_sepconv_fwd_k51(const float* in, const float* v, const float* h, float* out,
                           int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s);
int launch_sepconv_bwd_taps_generic(const float* g, const float* in, const float* v, const float* h,
                                    float* gv, float* gh,
                                    int64_t B, int64_t C, int64_t H, int64_t W, int K, cudaStream_t s);
int launch_sepconv_bwd_taps_k51(const float* g, const float* in, const float* v, const float* h,
                                float* gv, float* gh,
                                int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s);
int launch_interp_tail_fwd_k51(const float* frame1, const float* frame2, int64_t frame_bstride,
                               const float* k1v, const float* k1h, const float* k2v, const float* k2h, float* out,
                               int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s);
int launch_interp_tail_bwd_k51(const float* g, const float* frame, int64_t frame_bstride, const float* v, const float* h,
                               float* gv, float* gh, int64_t B, int64_t C, int64_t H, int64_t W, bool gray, cudaStream_t s);
int launch_sepconv_bwd_input_k51(const float* g, const float* v, const float* h, float* gi,
                                 int64_t B, int64_t C, int64_t H, int64_t W, cudaStream_t s);
int launch_sepconv_bwd_input_generic(const float* g, const float* v, const float* h, float* gi,
                                     int64_t B, int64_t C, int64_t H, int64_t W, int K, cudaStream_t s);

// Returned by a try_launch_* launcher whose fast path does not apply to the call; the caller runs its general kernel.
// Distinct from every CUDA error (positive) and SSTEM_E_* code, and never returned through the C ABI.
constexpr int PATH_NOT_APPLICABLE = INT32_MIN;

// third-generation 51-tap kernels on a 3-channel chunk of [B,51,H,W] taps (sepconv_k51_bwd3.cu, sepconv_k51_fwd3.cu):
// 0, a CUDA error, or PATH_NOT_APPLICABLE (the caller runs generation 1)
int try_launch_bwd_taps_k51_v3(const float* g, const float* in, const float* v, const float* h, float* gv, float* gh,
                               int64_t B, int C, int c0, int H, int W, int accumulate, cudaStream_t s);
int try_launch_fwd_k51_v3(const float* in, const float* v, const float* h, float* out,
                          int64_t B, int C, int c0, int H, int W, cudaStream_t s);

// layout kernels (sepconv_layout.cu): stream-ordered workspace, input repacks, gray x3 plane comparison
int workspace_alloc(void** p, size_t bytes, cudaStream_t s);
int launch_repack_nhwc4(const float* in, float* ws, int64_t B, int C, int c0, int64_t IH, int64_t IW, cudaStream_t s);
int launch_repack_plane_pitch(const float* in, float* ws, int64_t B, int C, int c0, int64_t IH, int64_t IW, int64_t IWP,
                              cudaStream_t s);
int launch_planes_equal(const float* in, int64_t B, int64_t C, int64_t plane, int* flag, cudaStream_t s);
// grad_output [B,C,H,W] -> out [B,nplanes,H,WP] (WP >= W a multiple of 4, zero pad columns): all C planes, or with `sum`
// their channel sum as one plane
int launch_stage_grad_planes(const float* g, float* out, int64_t B, int64_t C, int64_t H, int64_t W, int64_t WP, bool sum,
                             cudaStream_t s);
// tile-major taps -> [B,51,H,W]
int launch_taps_from_tiled(const float* tiled, float* taps, int64_t B, int64_t H, int64_t W, cudaStream_t s);

}  // namespace sstem
