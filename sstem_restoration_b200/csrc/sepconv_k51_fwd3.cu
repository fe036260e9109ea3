// Launchers of the third-generation forward kernel (device code in sepconv_k51_v3.cuh): copy the input into the layout
// the window loads want (channel-interleaved for 3 channels, 16-byte pitch for 1) in a stream-ordered workspace, encode
// the tensor maps, launch the persistent grid.  Also the forward on the tile-major tap layout of SURVEY 8f N2
// (sstem_sepconv_forward_tiled; the layout conversion sstem_taps_to_tiled is in sepconv_layout.cu).
#include "sepconv_k51_v3.cuh"

#include <stdlib.h>

namespace sstem {
namespace {

// returns 0 on launch, > 0 CUDA error, -1000 when the path does not apply
template <int CC, bool TILED>
int launch_fwd_v3(const float* in, const float* v, const float* h, float* out,
                  int64_t B, int C, int c0, int H, int W, int replicas, bool force, cudaStream_t s, bool accum = false) {
    if (!TILED && ((W & 3) || !aligned16(v) || !aligned16(h))) return -1000;
    if (TILED && (!aligned16(v) || !aligned16(h))) return SSTEM_E_ALIGN;
    const int64_t tiles_x = (W + V3_COLS * V3_WARPS - 1) / (V3_COLS * V3_WARPS), tiles_y = (H + F3_R - 1) / F3_R;
    if (tiles_x * tiles_y * B > INT32_MAX / 2) return -1000;
    // a persistent grid needs several tiles per warp to balance; small problems stay on the CTA-per-tile kernel
    static const int64_t min_tiles = getenv("SSTEM_V3_MIN_TILES") ? atoll(getenv("SSTEM_V3_MIN_TILES")) : 10;   // measured crossover: ~10 tiles per warp (forward), ~6 (tap gradients)
    if (!force && tiles_x * tiles_y * B < min_tiles * 2 * sm_count()) return -1000;
    const int64_t IH = H + K51 - 1, IW = W + K51 - 1, plane = (int64_t)H * W;
    const int64_t IWP = (IW + 3) & ~(int64_t)3;              // CC == 1: row pitch of the plane copy
    float* ws = nullptr;
    const size_t ws_bytes = CC == 3 ? (size_t)(B * IH * IW) * 16 : (size_t)(B * IH * IWP) * 4;
    if (workspace_alloc(reinterpret_cast<void**>(&ws), ws_bytes + 256, s)) return -1000;
    int* counter = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + ws_bytes);   // dynamic tile scheduler ticket
    cudaMemsetAsync(counter, 0, 256, s);
    int e = CC == 3 ? launch_repack_nhwc4(in, ws, B, C, c0, IH, IW, s) : launch_repack_plane_pitch(in, ws, B, C, c0, IH, IW, IWP, s);
    CUtensorMap min, mv, mh;
    if (!e) {
        const int64_t row = CC == 3 ? 4 * IW : IWP;
        const int64_t dims[3] = {row, IH, B}, strides[3] = {1, row, row * IH};
        const int box[3] = {(CC == 3 ? 4 : 1) * V3_WIN_COLS, V3_GROUP, 1};
        if (!make_map_f32(&min, ws, 3, dims, strides, box)) e = -1000;
        if (!e && !TILED) {
            // h with its tap and row dimensions swapped: the box lands as [row][tap][col] (conflict-free register copy)
            const int64_t tdims[4] = {W, H, K51, B}, tstrides[4] = {1, W, plane, (int64_t)K51 * plane};
            const int64_t rdims[4] = {W, K51, H, B}, rstrides[4] = {1, plane, W, (int64_t)K51 * plane};
            const int vbox[4] = {V3_COLS, F3_R, V3_GROUP, 1}, hbox[4] = {V3_COLS, K51, F3_R, 1};
            if (!make_map_f32(&mv, v, 4, tdims, tstrides, vbox) || !make_map_f32(&mh, h, 4, rdims, rstrides, hbox)) e = -1000;
        } else if (!e) {
            mv = min;                                      // unused by the kernel, but must be valid objects to copy
            mh = min;
        }
    }
    if (!e) {
        static PerDeviceOnce done;
        auto kern = sepconv_fwd_k51_v3_kernel<CC, TILED>;
        e = set_smem_once(kern, F3_SMEM, done);
        if (!e) {
            V3Shape sh{H, W, (int)tiles_x, (int)tiles_y, (int)(tiles_x * tiles_y * B), C, c0};
            F3Tiled tl{TILED ? v : nullptr, TILED ? h : nullptr, (int)((W + 7) / 8), (int)((H + 7) / 8), accum ? 1 : 0};
            const int ctas = (int)std::min<int64_t>(2 * (int64_t)sm_count(), (int64_t)sh.ntiles);
            kern<<<ctas, V3_WARPS * 32, F3_SMEM, s>>>(min, mv, mh, tl, out, counter, sh, replicas, g_gate.ptr, g_gate.want);
            count_launch();
            e = finish_launch();
        }
    }
    cudaFreeAsync(ws, s);
    return e;
}

}  // namespace

int try_launch_fwd_k51_v3(const float* in, const float* v, const float* h, float* out,
                          int64_t B, int C, int c0, int H, int W, cudaStream_t s) {
    return launch_fwd_v3<3, false>(in, v, h, out, B, C, c0, H, W, 1, false, s);
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
    cudaStream_t s = (cudaStream_t)stream;
    const bool accum = flags & SSTEM_SEPCONV_ACCUMULATE;
    int e = 0;
    if ((flags & SSTEM_SEPCONV_GRAY_REPLICATED) && C > 1) {
        e = launch_fwd_v3<1, true>(input, vertical_tiled, horizontal_tiled, output, B, (int)C, 0, (int)H, (int)W, (int)C, true, s);
    } else {
        int c0 = 0;
        while (c0 < C && !e) {                             // channel chunks of 3, then single planes
            if (C - c0 >= 3) { e = launch_fwd_v3<3, true>(input, vertical_tiled, horizontal_tiled, output, B, (int)C, c0, (int)H, (int)W, 1, true, s, accum); c0 += 3; }
            else { e = launch_fwd_v3<1, true>(input, vertical_tiled, horizontal_tiled, output, B, (int)C, c0, (int)H, (int)W, 1, true, s, accum); c0 += 1; }
        }
    }
    return e == -1000 ? SSTEM_E_SHAPE : e;
}

#ifdef SSTEM_V3_PHASES
// diagnostic builds only (tools/v3_phases.py): clock64 ticks per tile phase, summed over the warps of every launch
extern "C" int sstem_v3_phases_fwd(unsigned long long* out, int reset) { return sstem::v3_phases_read(out, reset); }
#endif
