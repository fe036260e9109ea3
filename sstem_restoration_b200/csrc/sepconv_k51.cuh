// Tuned 51-tap adaptive separable convolution for sm_100a: device code shared by the
// translation units sepconv_k51_{fwd,bwd,gi,tail}.cu (split so that nvcc compiles the ~130
// kernel instantiations in parallel): forward, the fused gradient w.r.t. the vertical /
// horizontal taps, the gradient w.r.t. the input and the fused interpolation tail.
//
//   out[b,c,y,x] = sum_fy v[b,fy,y,x] * ( sum_fx in[b,c,y+fy,x+fx] * h[b,fx,y,x] )
//
// (same sum as libs/sepconv/src/SeparableConvolution_kernel.cu:45-49 of the
// reference, factored: 2*C*K*(K+1) flop per pixel instead of 3*C*K*K; tap
// gradients per kernel.cu:97-111 and :134-149, sharing t = sum_c g_c * in_c.)
//
// This is a per-pixel bilinear form v^T P h with no operand shared between
// pixels except the image window P, so it runs on the FP32 FMA pipe, not on the
// tensor cores.  The design problem is operand bandwidth: one LDS per FMA caps
// at 1/4 of the FMA rate.  Mapping (G = tap groups per pixel, R = rows per lane):
//
//   * CTA = 4 warps = one R-row x (128/G)-column output tile of one image, all
//     channels; 2 CTAs per SM (255 registers each) so one CTA's loads hide
//     behind the other's arithmetic.
//   * The input window of the tile, (R+50) x (128/G+50) per channel, is staged
//     once in shared memory with cp.async (the reference layout's row pitch,
//     (W+50)*4 B, is not a multiple of 16 B, which rules out a TMA tensor map).
//   * A warp owns 32/G columns x R rows.  Lane = (column pg = lane/G, tap group
//     g = lane%G); the lane keeps the taps fx = G*t+g of all R rows of its column
//     in registers for the whole tile.
//   * Step s = 0..R+49 walks the input rows.  One LDS.32 of P[s][col+fx] feeds
//     the R rows' FMAs (row p uses it with fy = s-p): R FMAs per shared-memory
//     word, issued as packed FFMA2 (fma.rn.f32x2, scalar-broadcast operand) on
//     row pairs.
//   * Vertical taps are consumed once each, diagonally (row p needs fy = s-p):
//     they stream through a warp-private cp.async ring, VDEPTH steps ahead.
//   * The G tap groups of a pixel are summed with a transpose-reduce over
//     shuffles: once per tile (forward) or once per step for gv (backward).
#pragma once
#include "common.cuh"
#include <type_traits>
#include <utility>

namespace sstem {

namespace {

constexpr int K51 = 51;
constexpr int VDEPTH = 8;                  // steps of vertical taps in flight per warp

constexpr int FWD_G = 4, FWD_R = 8;        // forward, grad_input and the fused tail forward
constexpr int BWD_G = 4, BWD_R = 4;        // tap gradients
constexpr int FWD_NPRE = 13;               // taps of the next row (channel 0) preloaded during the current step;
                                           // 3-channel kernel (measured: +2 % there; 13 at C = 1 costs 5 %)
constexpr int FWD_NPRE1 = 4;               // the same for the one- / two-channel kernels and the fused tail (measured:
                                           // gray x3 forward +5 %, tail +0.4 %; 8 is no better)
constexpr int BWD_NPRE = 7;                // taps of the next row preloaded during the current step
constexpr int MIN_CTAS = 2;                // CTAs per SM in every __launch_bounds__ (3 spills in the step loop: DESIGN 7)

// ---- geometry of one configuration --------------------------------------------------------
template <int G, int R>
struct Geo {
    static constexpr int NT = (K51 + G - 1) / G;        // taps per lane (slot NT-1 may not exist)
    static constexpr int LAST_VALID_G = K51 - G * (NT - 1);  // lanes g >= this have no tap in slot NT-1
    static constexpr int COLS = 32 / G;                 // columns per warp
    static constexpr int TILE_W = 4 * COLS;             // columns per CTA
    static constexpr int ROWS = R + K51 - 1;            // input rows of the window
    static constexpr int PITCH = ((TILE_W + G * NT + 3) / 4) * 4;  // smem row pitch (floats)
    static constexpr int NP = R / 2;                    // row pairs
    static constexpr int SLOT = R * COLS;               // floats per v-ring slot
    static_assert(R % 2 == 0 && (32 % G) == 0 && COLS % 4 == 0, "unsupported geometry");
};

__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    const int n = valid ? 4 : 0;           // src-size 0 => zero fill
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(src), "r"(n));
}
__device__ __forceinline__ void cp_async8(float* dst_smem, const float* src, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    const int n = valid ? 8 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(src), "r"(n));
}
__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
    const int n = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(src), "r"(n));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// Stage the input window of the tile: a thread owns one column (pair) and walks down the
// rows, so the loop has no div/mod.  PAIR: (W+50) even and `in` 8-byte aligned.
template <int CC, int ROWS, int PITCH, bool PAIR>
__device__ __forceinline__ void stage_window(float* tile, const float* __restrict__ in, int64_t img_off,
                                             int x0, int y0, int IH, int IW, int tid) {
    constexpr int CPR = PAIR ? PITCH / 2 : PITCH;       // copies per row
    constexpr int RSTEP = 128 / CPR;                    // rows covered per pass
    static_assert(RSTEP >= 1, "window too wide for 128 threads");
    const int cidx = tid % CPR, r0 = tid / CPR;
    const int col = PAIR ? 2 * cidx : cidx;
    const int gx = x0 + col;
    if (r0 < RSTEP) {
        const bool colok = gx < IW;                     // PAIR: IW and gx even, a pair never straddles
        const float* src = in + img_off + (int64_t)(y0 + r0) * IW + (colok ? gx : 0);
        float* dst = tile + r0 * PITCH + col;
#pragma unroll 1
        for (int c = 0; c < CC; ++c) {
            const float* sp = src;
            float* dp = dst;
#pragma unroll 2
            for (int r = r0; r < ROWS; r += RSTEP) {
                const bool ok = colok && (y0 + r < IH);
                if (PAIR) cp_async8(dp, ok ? sp : in, ok); else cp_async4(dp, ok ? sp : in, ok);
                sp += (int64_t)RSTEP * IW;
                dp += RSTEP * PITCH;
            }
            src += (int64_t)IH * IW;
            dst += ROWS * PITCH;
        }
    }
    cp_async_commit();                                  // group 0: the window
}

// Fused-tail staging (no padded copy of the frame exists): window element (r, col) is pixel
// (clamp(y0 + r - 25), clamp(x0 + col - 25)) of the UNPADDED frame -- ReplicationPad2d(25) folded into
// the load (model_interp.py:46,90-91) -- summed over `cs` channel planes (the channel mean of the
// tail commutes with the convolution, which is linear in the image).  cs <= 3: every plane is
// fetched with asynchronous 4-byte copies into its own shared-memory plane (`nplanes` = cs of
// them) and tail_window_reduce() folds them into plane 0 once they have landed, each thread
// summing exactly the words it copied; cs > 3: plain loads, channel sum, st.shared.
template <int ROWS, int PITCH>
__device__ __forceinline__ void stage_window_tail(float* tile, const float* __restrict__ fr, int cs, int nplanes,
                                                  int x0, int y0, int H, int W, int tid) {
    constexpr int HALO = K51 / 2;
    constexpr int CPR = PITCH / 2;                      // a thread owns two adjacent columns
    constexpr int RSTEP = 128 / CPR;
    static_assert(PITCH % 2 == 0 && RSTEP >= 1, "window too wide for 128 threads");
    const int cidx = tid % CPR, r0 = tid / CPR;
    if (r0 < RSTEP) {
        const int ca = min(max(x0 + 2 * cidx - HALO, 0), W - 1), cb = min(max(x0 + 2 * cidx + 1 - HALO, 0), W - 1);
        float* dst = tile + r0 * PITCH + 2 * cidx;
        const int64_t plane = (int64_t)H * W;
        if (nplanes == cs) {
#pragma unroll 2
            for (int r = r0; r < ROWS; r += RSTEP) {
                const float* row = fr + (int64_t)min(max(y0 + r - HALO, 0), H - 1) * W;
                for (int c = 0; c < nplanes; ++c) {
                    cp_async4(dst + c * (ROWS * PITCH), row + c * plane + ca, true);
                    cp_async4(dst + c * (ROWS * PITCH) + 1, row + c * plane + cb, true);
                }
                dst += RSTEP * PITCH;
            }
        } else {
#pragma unroll 2
            for (int r = r0; r < ROWS; r += RSTEP) {
                const float* row = fr + (int64_t)min(max(y0 + r - HALO, 0), H - 1) * W;
                float sa = __ldg(row + ca), sb = __ldg(row + cb);
                for (int c = 1; c < cs; ++c) { sa += __ldg(row + c * plane + ca); sb += __ldg(row + c * plane + cb); }
                dst[0] = sa;
                dst[1] = sb;
                dst += RSTEP * PITCH;
            }
        }
    }
    cp_async_commit();                                  // group 0: the window (possibly empty)
}

// after the window's cp.async group has completed for THIS thread, before the block barrier
template <int ROWS, int PITCH>
__device__ __forceinline__ void tail_window_reduce(float* tile, int nplanes, int tid) {
    constexpr int CPR = PITCH / 2, RSTEP = 128 / CPR;
    if (nplanes < 2) return;
    const int cidx = tid % CPR, r0 = tid / CPR;
    if (r0 >= RSTEP) return;
    float2* dst = reinterpret_cast<float2*>(tile + r0 * PITCH + 2 * cidx);
#pragma unroll 4
    for (int r = r0; r < ROWS; r += RSTEP) {
        float2 a = dst[0];
        for (int c = 1; c < nplanes; ++c) {
            const float2 q = dst[c * (ROWS * PITCH / 2)];
            a.x += q.x;
            a.y += q.y;
        }
        dst[0] = a;
        dst += RSTEP * PITCH / 2;
    }
}

// Warp-private ring of vertical taps.  Step st holds, for every row p of the tile,
// v[fy = st - p][y0 + p][columns of this warp]; invalid fy / rows / columns are zero filled,
// which also makes the prologue / epilogue contributions vanish.
template <int G, int R, bool VEC>
struct VRing {
    using Gm = Geo<G, R>;
    static constexpr int NCHUNK = VEC ? R * (Gm::COLS / 4) : R * Gm::COLS;   // copy jobs per step
    static constexpr int NJOB = (NCHUNK + 31) / 32;                          // per lane
    float* ring;
    const float* src[NJOB];
    const float* dummy;
    int p_[NJOB];
    bool ok_[NJOB], act_[NJOB];
    int dst_[NJOB];
    int64_t plane;
    int slot_w = 0, step_w = 0, slot_r = 0, pg;

    __device__ __forceinline__ void init(float* ring_, const float* __restrict__ v, int64_t vb_off, int64_t plane_,
                                         int y0, int xw0, int H, int W, int lane) {
        ring = ring_;
        plane = plane_;
        dummy = v;
        pg = lane / G;
#pragma unroll
        for (int j = 0; j < NJOB; ++j) {
            const int e = lane + 32 * j;
            const int p = VEC ? e / (Gm::COLS / 4) : e / Gm::COLS;
            const int col = VEC ? 4 * (e % (Gm::COLS / 4)) : e % Gm::COLS;
            act_[j] = e < NCHUNK;
            p_[j] = p;
            ok_[j] = act_[j] && (y0 + p < H) && (xw0 + col < W);
            dst_[j] = p * Gm::COLS + col;
            src[j] = v + vb_off + (int64_t)min(y0 + p, H - 1) * W + min(xw0 + col, W - 1) - (int64_t)p * plane;
        }
    }
    __device__ __forceinline__ void issue() {           // fetch the next step
        float* slot = ring + slot_w * Gm::SLOT;
#pragma unroll
        for (int j = 0; j < NJOB; ++j) {
            const int fy = step_w - p_[j];
            const bool ok = ok_[j] && fy >= 0 && fy < K51;
            if (act_[j]) {
                if (VEC) cp_async16(slot + dst_[j], ok ? src[j] : dummy, ok);
                else cp_async4(slot + dst_[j], ok ? src[j] : dummy, ok);
            }
            src[j] += plane;
        }
        cp_async_commit();
        ++step_w;
        slot_w = (slot_w + 1 == VDEPTH) ? 0 : slot_w + 1;
    }
    __device__ __forceinline__ void read(float2 (&dst)[R / 2]) {
        const float* slot = ring + slot_r * Gm::SLOT + pg;
#pragma unroll
        for (int pp = 0; pp < R / 2; ++pp)
            dst[pp] = make_float2(slot[(2 * pp) * Gm::COLS], slot[(2 * pp + 1) * Gm::COLS]);
        slot_r = (slot_r + 1 == VDEPTH) ? 0 : slot_r + 1;
    }
    __device__ __forceinline__ void advance(float2 (&dst)[R / 2]) {   // make the next step readable, refill the ring
        cp_async_wait<VDEPTH - 3>();
        __syncwarp();
        issue();
        read(dst);
    }
};

// Transpose-reduce over the G tap-group lanes of a pixel: on return lane g holds, in
// val[0 .. N/G-1], the group totals of the original values with index g*(N/G) + j.
template <int G, int N>
__device__ __forceinline__ void group_reduce(float (&val)[N], int g) {
    static_assert(N % G == 0, "N must be a multiple of G");
    int n = N;
#pragma unroll
    for (int m = G / 2; m >= 1; m >>= 1) {
        const int half = n / 2;
        const bool up = (g & m) != 0;
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            if (i < half) {
                const float send = up ? val[i] : val[i + half];
                const float keep = up ? val[i + half] : val[i];
                val[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
            }
        }
        n = half;
    }
}

// per-tile load of the horizontal taps of this lane: h2[pp][t] = (row 2pp, row 2pp+1), tap G*t+g
template <int G, int R>
__device__ __forceinline__ void load_h(float2 (&h2)[R / 2][Geo<G, R>::NT], const float* __restrict__ h,
                                       int64_t hb_off, int64_t plane, int y0, int x, int H, int W, int g) {
    using Gm = Geo<G, R>;
    const float* hp[R];
#pragma unroll
    for (int p = 0; p < R; ++p) hp[p] = h + hb_off + g * plane + (int64_t)min(y0 + p, H - 1) * W + x;
    const int64_t tstep = (int64_t)G * plane;
    const bool novalid = g >= Gm::LAST_VALID_G;         // slot NT-1 does not exist for this lane
#pragma unroll
    for (int t = 0; t < Gm::NT; ++t) {
        const bool last = (t == Gm::NT - 1);            // masked by P = 0; read the previous tap again
#pragma unroll
        for (int pp = 0; pp < R / 2; ++pp) {
            const float* pa = (last && novalid) ? hp[2 * pp] - tstep : hp[2 * pp];
            const float* pb = (last && novalid) ? hp[2 * pp + 1] - tstep : hp[2 * pp + 1];
            h2[pp][t] = make_float2(__ldg(pa), __ldg(pb));
            hp[2 * pp] += tstep;
            hp[2 * pp + 1] += tstep;
        }
    }
}

template <int S0, class Step, int... I>
__device__ __forceinline__ void edge_steps(Step& step, std::integer_sequence<int, I...>) {
    (step(std::integral_constant<int, S0 + I>{}, S0 + I), ...);
}

// The R + 50 steps of a window.  The edge steps 0 .. R-2 and 51 .. R+49, where some rows have fy = s - p outside
// [0, 50], are compile-time steps; the steady steps R-1 .. 50 between them run in a loop.  step(S, s, vuse, vfill)
// runs step s from the vertical taps in vuse and fills vfill with the next step's; S is an integral_constant, the step
// at an edge and -1 in the steady loop.  TWO_STEP: two steady steps per iteration, vcur and vnext swapping roles (no
// register copies).  The one-channel kernels use it (measured +8 % on the gray forward, +2-6 % on the tail kernels);
// the others keep one step per iteration (two-step at three channels: 0 % forward, -3 % on the tap gradients).
template <int R, bool TWO_STEP, class Step>
__device__ __forceinline__ void walk_steps(Step&& step, float2 (&vcur)[R / 2], float2 (&vnext)[R / 2]) {
    auto one_step = [&](auto S, int s) {
        step(S, s, vcur, vnext);
#pragma unroll
        for (int pp = 0; pp < R / 2; ++pp) vcur[pp] = vnext[pp];
    };
    edge_steps<0>(one_step, std::make_integer_sequence<int, R - 1>{});
    constexpr std::integral_constant<int, -1> STEADY{};
    if constexpr (TWO_STEP) {
        static_assert((K51 - R + 1) % 2 == 0, "the two-step steady loop needs an even number of steady steps");
#pragma unroll 1
        for (int s = R - 1; s < K51; s += 2) {
            step(STEADY, s, vcur, vnext);
            step(STEADY, s + 1, vnext, vcur);
        }
    } else {
#pragma unroll 1
        for (int s = R - 1; s < K51; ++s) one_step(STEADY, s);
    }
    edge_steps<K51>(one_step, std::make_integer_sequence<int, R - 1>{});
}

// =====================================================================================
// Forward
// =====================================================================================
// One input row for all CC channels.  S >= 0: compile-time step (prologue / epilogue, where
// some rows have fy = s - p outside [0, 50] -- inactive pairs vanish at compile time);
// S < 0: steady state, runtime step, every row active.
template <int CC, int G, int R, int S>
__device__ __forceinline__ void fwd_step(const float* __restrict__ prow0, bool novalid,
                                         const float2 (&h2)[R / 2][Geo<G, R>::NT], const float2 (&v2)[R / 2],
                                         float2 (&acc)[CC][R / 2], float (&pre)[FWD_NPRE + 1]) {
    using Gm = Geo<G, R>;
    constexpr int NPRE = (CC >= 3) ? FWD_NPRE : FWD_NPRE1;   // channel 0's first taps were loaded during the previous step
#pragma unroll
    for (int c = 0; c < CC; ++c) {
        const float* prow = prow0 + c * Gm::ROWS * Gm::PITCH;
        float2 part[Gm::NP];
#pragma unroll
        for (int pp = 0; pp < Gm::NP; ++pp) part[pp] = make_float2(0.f, 0.f);
#pragma unroll
        for (int t = 0; t < Gm::NT; ++t) {
            float P = (c == 0 && t < NPRE) ? pre[t] : prow[G * t];
            if (t == Gm::NT - 1) P = novalid ? 0.f : P;  // this tap does not exist for the lane
#pragma unroll
            for (int pp = 0; pp < Gm::NP; ++pp) {
                if (S >= 0 && (S < 2 * pp || S > 2 * pp + K51)) continue;   // pair entirely outside
                part[pp] = __ffma2_rn(make_float2(P, P), h2[pp][t], part[pp]);
            }
        }
#pragma unroll
        for (int pp = 0; pp < Gm::NP; ++pp) {
            if (S >= 0) {
                if (S < 2 * pp || S > 2 * pp + K51) continue;
                // a row whose fy is out of range must not even see part (NaN/Inf safety)
                if (S - 2 * pp > K51 - 1) part[pp].x = 0.f;
                if (S - 2 * pp - 1 < 0) part[pp].y = 0.f;
            }
            acc[c][pp] = __ffma2_rn(v2[pp], part[pp], acc[c][pp]);
        }
    }
#pragma unroll
    for (int t = 0; t < NPRE; ++t) pre[t] = prow0[Gm::PITCH + G * t];   // next row (one row of slack follows the window)
}

// VEC: W % 4 == 0 and v 16-byte aligned -> the ring is fed with 16-byte cp.async.
template <int CC, int G, int R, bool VEC, bool PAIR>
__global__ void __launch_bounds__(128, MIN_CTAS)
sepconv_fwd_k51_kernel(const float* __restrict__ in, const float* __restrict__ v,
                       const float* __restrict__ h, float* __restrict__ out,
                       int C, int c0, int H, int W, int replicas, const int* gate, int gate_want) {
    SSTEM_GATE_RETURN(gate, gate_want);
    using Gm = Geo<G, R>;
    extern __shared__ __align__(16) float tile[];      // [CC][ROWS][PITCH] + 4 warps x v ring
    const int IW = W + K51 - 1, IH = H + K51 - 1;
    const int x0 = blockIdx.x * Gm::TILE_W, y0 = blockIdx.y * R;
    const int64_t b = blockIdx.z;
    const int64_t plane = (int64_t)H * W;
    const int tid = threadIdx.x;

    const int warp = tid >> 5, lane = tid & 31;
    const int pg = lane / G, g = lane % G;
    const int xl = warp * Gm::COLS + pg;                // column inside the tile
    const int x = min(x0 + xl, W - 1);                  // clamped for loads; stores are masked
    const bool novalid = g >= Gm::LAST_VALID_G;

    float2 h2[Gm::NP][Gm::NT];
    stage_window<CC, Gm::ROWS, Gm::PITCH, PAIR>(tile, in, (b * C + c0) * (int64_t)IH * IW, x0, y0, IH, IW, tid);

    VRing<G, R, VEC> vr;
    vr.init(tile + CC * Gm::ROWS * Gm::PITCH + warp * (VDEPTH * Gm::SLOT), v, b * K51 * plane, plane,
            y0, x0 + warp * Gm::COLS, H, W, lane);
#pragma unroll
    for (int st = 0; st < VDEPTH - 1; ++st) vr.issue();

    load_h<G, R>(h2, h, b * K51 * plane, plane, y0, x, H, W, g);   // (issuing these before the window costs 6-10 % here)

    float2 acc[CC][Gm::NP];
#pragma unroll
    for (int c = 0; c < CC; ++c)
#pragma unroll
        for (int pp = 0; pp < Gm::NP; ++pp) acc[c][pp] = make_float2(0.f, 0.f);

    cp_async_wait<VDEPTH - 2>();                        // window + step 0 have landed (this thread's part)
    __syncthreads();                                    // ... and everybody else's part of the window

    float2 vcur[Gm::NP], vnext[Gm::NP];
    vr.read(vcur);
    const float* prow = tile + xl + g;                  // P column of tap slot t is xl + g + G*t
    float pre[FWD_NPRE + 1];
#pragma unroll
    for (int t = 0; t < ((CC >= 3) ? FWD_NPRE : FWD_NPRE1); ++t) pre[t] = prow[G * t];
    walk_steps<R, CC == 1>([&](auto S, int, auto& vuse, auto& vfill) {
        vr.advance(vfill);
        fwd_step<CC, G, R, decltype(S)::value>(prow, novalid, h2, vuse, acc, pre);
        prow += Gm::PITCH;
    }, vcur, vnext);

    // ---- sum the G tap groups of each pixel: lane g ends up with rows g*(R/G).. of every channel
    constexpr int NV = (R >= G) ? R : G;
    constexpr int PER = NV / G;                         // rows per lane after the reduce
#pragma unroll
    for (int c = 0; c < CC; ++c) {
        float val[NV];
#pragma unroll
        for (int pp = 0; pp < Gm::NP; ++pp) { val[2 * pp] = acc[c][pp].x; val[2 * pp + 1] = acc[c][pp].y; }
#pragma unroll
        for (int i = R; i < NV; ++i) val[i] = 0.f;
        group_reduce<G, NV>(val, g);
        if (x0 + xl < W) {
            float* ob = out + ((b * C + c0 + c) * (int64_t)H + y0) * W + x0 + xl;
#pragma unroll
            for (int j = 0; j < PER; ++j) {
                const int p = g * PER + j;
                if (p < R && y0 + p < H) {
                    ob[(int64_t)p * W] = val[j];
                    // gray x3 shortcut: the input planes are identical copies, so are the outputs
                    for (int rc = 1; rc < replicas; ++rc) ob[(int64_t)rc * H * W + (int64_t)p * W] = val[j];
                }
            }
        }
    }
}

// =====================================================================================
// Backward w.r.t. the taps, fused:
//   t[fy][fx]  = sum_c g[c] * in[c][y+fy][x+fx]
//   gv[fy]     = sum_fx t[fy][fx] * h[fx]
//   gh[fx]     = sum_fy t[fy][fx] * v[fy]
// 2*(C+2)*K*K flop per pixel.  A lane keeps h and the gh accumulators of its taps for R
// rows in registers; every step it forms t for its taps from NT*C shared-memory words,
// accumulates gh in place, and the gv partial sums of the G tap groups are
// transpose-reduced over shuffles so that lane g stores gv[fy = s-g] of row g.
// =====================================================================================
template <int CC, int G, int R, int S, bool WV, bool WH>
__device__ __forceinline__ void bwd_step(const float* __restrict__ prow0, bool novalid,
                                         const float2 (&g2)[CC][R / 2], const float2 (&h2)[R / 2][Geo<G, R>::NT],
                                         const float2 (&v2)[R / 2], float2 (&gh2)[R / 2][Geo<G, R>::NT],
                                         float2 (&gvp)[R / 2], float (&pre)[CC][BWD_NPRE + 1]) {
    using Gm = Geo<G, R>;
    constexpr int NP = Gm::NP, NT = Gm::NT;
    constexpr int NPRE = BWD_NPRE;                       // first taps of the NEXT row are loaded one step early
    if (CC == 1) {
        // One channel (also the gray x3 shortcut): t = g * P, so g factors out of both sums --
        //   gv[fy] = g * sum_fx P h[fx],   gh[fx] = g * sum_fy P v[fy]
        // 2 FMAs per (fy, fx) instead of 3; the caller multiplies by g (gv per step, gh once per tile).
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) gvp[pp] = make_float2(0.f, 0.f);
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            float P = (t < NPRE) ? pre[0][t] : prow0[G * t];
            if (t == NT - 1) P = novalid ? 0.f : P;
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) {
                float2 P2 = make_float2(P, P);
                if (S >= 0) {                            // a row whose fy is out of range must not see P
                    if (S < 2 * pp || S > 2 * pp + K51) continue;
                    if (S - 2 * pp > K51 - 1) P2.x = 0.f;
                    if (S - 2 * pp - 1 < 0) P2.y = 0.f;
                }
                if (WV) gvp[pp] = __ffma2_rn(P2, h2[pp][t], gvp[pp]);
                if (WH) gh2[pp][t] = __ffma2_rn(P2, v2[pp], gh2[pp][t]);
            }
        }
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) gvp[pp] = __fmul2_rn(gvp[pp], g2[0][pp]);
#pragma unroll
        for (int t = 0; t < NPRE; ++t) pre[0][t] = prow0[Gm::PITCH + G * t];
        return;
    }
    constexpr int TB = (NT + 1) / 2;                     // taps per block: NP*TB independent FFMA2 chains
    float2 gva[NP], gvb[NP];                             // two partial sums per row pair
#pragma unroll
    for (int pp = 0; pp < NP; ++pp) gva[pp] = gvb[pp] = make_float2(0.f, 0.f);
#pragma unroll
    for (int tb = 0; tb < NT; tb += TB) {
        float2 t2[TB][NP];
#pragma unroll
        for (int j = 0; j < TB; ++j)
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) t2[j][pp] = make_float2(0.f, 0.f);
        // the channel sum is the dependent direction: channel-outer / tap-inner
#pragma unroll
        for (int c = 0; c < CC; ++c) {
#pragma unroll
            for (int j = 0; j < TB; ++j) {
                const int t = tb + j;
                if (t >= NT) continue;
                float P = (t < NPRE) ? pre[c][t] : prow0[c * Gm::ROWS * Gm::PITCH + G * t];
                if (t == NT - 1) P = novalid ? 0.f : P;
#pragma unroll
                for (int pp = 0; pp < NP; ++pp) {
                    if (S >= 0 && (S < 2 * pp || S > 2 * pp + K51)) continue;
                    t2[j][pp] = __ffma2_rn(make_float2(P, P), g2[c][pp], t2[j][pp]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < TB; ++j) {
            const int t = tb + j;
            if (t >= NT) continue;
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) {
                if (S >= 0) {                            // rows whose fy is out of range contribute nothing
                    if (S < 2 * pp || S > 2 * pp + K51) continue;
                    if (S - 2 * pp > K51 - 1) t2[j][pp].x = 0.f;
                    if (S - 2 * pp - 1 < 0) t2[j][pp].y = 0.f;
                }
                if (WH) gh2[pp][t] = __ffma2_rn(t2[j][pp], v2[pp], gh2[pp][t]);
                if (WV) {
                    if (t & 1) gvb[pp] = __ffma2_rn(t2[j][pp], h2[pp][t], gvb[pp]);
                    else gva[pp] = __ffma2_rn(t2[j][pp], h2[pp][t], gva[pp]);
                }
            }
        }
    }
#pragma unroll
    for (int pp = 0; pp < NP; ++pp) gvp[pp] = make_float2(gva[pp].x + gvb[pp].x, gva[pp].y + gvb[pp].y);
    if (NPRE > 0) {                                      // next row's first taps (the row after the last is smem slack)
#pragma unroll
        for (int c = 0; c < CC; ++c)
#pragma unroll
            for (int t = 0; t < NPRE; ++t) pre[c][t] = prow0[c * Gm::ROWS * Gm::PITCH + Gm::PITCH + G * t];
    }
}

// TAIL (fused interpolation tail, CC == 1): `in` is the UNPADDED frame [B, cs.., H, W] with batch
// stride `in_bstride`; the window is its replicate-padded channel sum, gout is [B,1,H,W] and is
// scaled by `gscale` (= 1/C of the channel mean) -- see interp_tail_fwd_k51_kernel.
template <int CC, int G, int R, bool VEC, bool PAIR, bool WV, bool WH, bool ACCUM, bool TAIL = false>
__global__ void __launch_bounds__(128, MIN_CTAS)
sepconv_bwd_taps_k51_kernel(const float* __restrict__ gout, const float* __restrict__ in,
                            const float* __restrict__ v, const float* __restrict__ h,
                            float* __restrict__ gv, float* __restrict__ gh,
                            int C, int c0, int H, int W, int replicas,
                            int64_t in_bstride, int cs, int nplanes, float gscale, const int* gate, int gate_want) {
    SSTEM_GATE_RETURN(gate, gate_want);
    static_assert(!TAIL || CC == 1, "the fused tail works on one (channel-summed) plane");
    constexpr bool accumulate = ACCUM;                   // later channel chunks (C > 3) add into gv / gh
    using Gm = Geo<G, R>;
    constexpr int NP = Gm::NP, NT = Gm::NT;
    static_assert(R == G, "the per-step gv reduce maps row p to lane g == p");
    extern __shared__ __align__(16) float tile[];
    const int IW = W + K51 - 1, IH = H + K51 - 1;
    const int x0 = blockIdx.x * Gm::TILE_W, y0 = blockIdx.y * R;
    const int64_t b = blockIdx.z;
    const int64_t plane = (int64_t)H * W;
    const int tid = threadIdx.x;

    const int warp = tid >> 5, lane = tid & 31;
    const int pg = lane / G, g = lane % G;
    const int xl = warp * Gm::COLS + pg;
    const int x = min(x0 + xl, W - 1);
    const bool novalid = g >= Gm::LAST_VALID_G;
    const bool col_ok = (x0 + xl < W);

    // Fused tail: its window staging (4-byte copies, clamped addresses) is slow to issue, so the tap loads -- the
    // long pole of the prologue -- go first (+3-4 %); with the padded input's 8-byte window copies the opposite
    // order is faster (tap loads first: -6 % at three channels, -3..-10 % at one).
    constexpr bool HFIRST = TAIL;
    float2 h2[NP][NT], gh2[NP][NT], g2[CC][NP];
    if (WV && HFIRST) load_h<G, R>(h2, h, b * K51 * plane, plane, y0, x, H, W, g);
    if (TAIL) stage_window_tail<Gm::ROWS, Gm::PITCH>(tile, in + b * in_bstride, cs, nplanes, x0, y0, H, W, tid);
    else stage_window<CC, Gm::ROWS, Gm::PITCH, PAIR>(tile, in, (b * C + c0) * (int64_t)IH * IW, x0, y0, IH, IW, tid);

    VRing<G, R, VEC> vr;
    vr.init(tile + (TAIL ? nplanes : CC) * Gm::ROWS * Gm::PITCH + warp * (VDEPTH * Gm::SLOT), v, b * K51 * plane, plane,
            y0, x0 + warp * Gm::COLS, H, W, lane);
#pragma unroll
    for (int st = 0; st < VDEPTH - 1; ++st) {
        if (WH) vr.issue(); else cp_async_commit();
    }

    if (WV && !HFIRST) load_h<G, R>(h2, h, b * K51 * plane, plane, y0, x, H, W, g);
#pragma unroll
    for (int pp = 0; pp < NP; ++pp)
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            gh2[pp][t] = make_float2(0.f, 0.f);
            if (!WV) h2[pp][t] = make_float2(0.f, 0.f);
        }
#pragma unroll
    for (int c = 0; c < CC; ++c)
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) {
            const float* gp = gout + (b * C + c0 + c) * plane + x;
            const int ya = y0 + 2 * pp, yb = ya + 1;
            // rows / columns outside the image get g = 0: they then contribute nothing
            g2[c][pp].x = (col_ok && ya < H) ? __ldg(gp + (int64_t)ya * W) : 0.f;
            g2[c][pp].y = (col_ok && yb < H) ? __ldg(gp + (int64_t)yb * W) : 0.f;
            // gray x3 shortcut: identical input planes => t = (sum_c g_c) * P
            for (int rc = 1; rc < replicas; ++rc) {
                g2[c][pp].x += (col_ok && ya < H) ? __ldg(gp + rc * plane + (int64_t)ya * W) : 0.f;
                g2[c][pp].y += (col_ok && yb < H) ? __ldg(gp + rc * plane + (int64_t)yb * W) : 0.f;
            }
            if (TAIL) { g2[c][pp].x *= gscale; g2[c][pp].y *= gscale; }
        }

    cp_async_wait<VDEPTH - 2>();
    if (TAIL) tail_window_reduce<Gm::ROWS, Gm::PITCH>(tile, nplanes, tid);
    __syncthreads();

    float2 vcur[NP], vnext[NP];
    if (WH) vr.read(vcur);
    else {
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) vcur[pp] = vnext[pp] = make_float2(0.f, 0.f);
    }
    const float* prow = tile + xl + g;
    // gv[fy = s - g][y0 + g][x]: pointer for s = 0, advanced by one plane per step
    float* gv_ptr = WV ? gv + b * K51 * plane + (int64_t)min(y0 + g, H - 1) * W + x - (int64_t)g * plane : nullptr;
    const bool gv_row_ok = col_ok && (y0 + g < H);
    auto store_gv = [&](int s, float2 (&gvp)[NP]) {
        if (WV) {
            float val[R];
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) { val[2 * pp] = gvp[pp].x; val[2 * pp + 1] = gvp[pp].y; }
            group_reduce<G, R>(val, g);                  // lane g now holds the total of row g
            const int fy = s - g;
            if (gv_row_ok && fy >= 0 && fy < K51) *gv_ptr = accumulate ? (*gv_ptr + val[0]) : val[0];
            gv_ptr += plane;
        }
    };
    float2 gvp[NP];
    float pre[CC][BWD_NPRE + 1];
#pragma unroll
    for (int c = 0; c < CC; ++c)
#pragma unroll
        for (int t = 0; t < BWD_NPRE; ++t) pre[c][t] = prow[c * Gm::ROWS * Gm::PITCH + G * t];
    walk_steps<R, CC == 1>([&](auto S, int s, auto& vuse, auto& vfill) {
        if (WH) {
            vr.advance(vfill);
        } else {                                         // no v taps: keep the cp.async group arithmetic
            cp_async_wait<VDEPTH - 3>();
            __syncwarp();
            cp_async_commit();
        }
        bwd_step<CC, G, R, decltype(S)::value, WV, WH>(prow, novalid, g2, h2, vuse, gh2, gvp, pre);
        store_gv(s, gvp);
        prow += Gm::PITCH;
    }, vcur, vnext);

    // ---- gh: complete per lane (the sum over fy happened in registers) ---------------------------
    if (WH && col_ok) {
        float* gp = gh + (b * K51 + g) * plane + x0 + xl;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            if (t == NT - 1 && novalid) break;
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) {
                const int ya = y0 + 2 * pp, yb = ya + 1;
                float* da = gp + (int64_t)(G * t) * plane + (int64_t)ya * W;
                float* db = gp + (int64_t)(G * t) * plane + (int64_t)yb * W;
                const float2 val = (CC == 1) ? __fmul2_rn(gh2[pp][t], g2[0][pp]) : gh2[pp][t];   // CC == 1: g was factored out
                if (ya < H) *da = accumulate ? (*da + val.x) : val.x;
                if (yb < H) *db = accumulate ? (*db + val.y) : val.y;
            }
        }
    }
}

// =====================================================================================
// Backward w.r.t. the input (the adjoint of the forward; the reference never computes it):
//   gi[c][y+fy][x+fx] += g[c][y][x] * v[fy][y][x] * h[fx][y][x]
// The forward's lane mapping run "in reverse": at step s the lane forms, for each of its taps,
//   q = sum over its R rows of h[row][tap] * (g[row] * v[fy = s-row][row])
// (all operands in registers) and adds q to word x+fx of row s of a shared gi tile.
// The adds are plain read-modify-writes, made race-free by construction:
//   * inside a warp the 4 tap groups walk their taps in rotated order (group g starts 2g taps
//     in), so the 32 lanes of one instruction always hit 32 different words;
//   * the 4 warps run one step apart (warp w does step tau - w at time tau, a barrier per
//     step), so at any time they work on 4 different rows.
// The tile, (R+50) x (TILE_W+50) per channel, overlaps its neighbours' by 50, so it is
// flushed with global atomics into a zero-initialised gi (the order of those few adds, hence
// the last bit, may vary run to run).  2*C*K*(K+1) flop per pixel, like the forward.
// =====================================================================================
template <int CC, int R, int S>
__device__ __forceinline__ void gi_step(float* __restrict__ trowA, int thr, bool g3,
                                        const float2 (&g2)[CC][R / 2], const float2 (&h2)[R / 2][13],
                                        const float2 (&v2)[R / 2]) {
    using Gm = Geo<4, R>;
    constexpr int NT = 13;
    constexpr int CH = Gm::ROWS * Gm::PITCH;            // channel stride of the tile
    // slot t of tap group g holds tap 4*((t + 2g) mod 13) + g; its word is trowA[4t] before the
    // wrap (t < thr = 13 - 2g) and trowA[4t - 52] after it
    float* trowB = trowA - 52;
    float2 a2[CC][Gm::NP];
#pragma unroll
    for (int c = 0; c < CC; ++c)
#pragma unroll
        for (int pp = 0; pp < Gm::NP; ++pp) {
            a2[c][pp] = __fmul2_rn(g2[c][pp], v2[pp]);   // v = 0 where fy is out of range ...
            if (S >= 0) {                                // ... but 0 * NaN is NaN: a row outside its 51 steps must not leak one
                if (S - 2 * pp > K51 - 1 || S - 2 * pp < 0) a2[c][pp].x = 0.f;
                if (S - 2 * pp - 1 < 0 || S - 2 * pp - 1 > K51 - 1) a2[c][pp].y = 0.f;
            }
        }
    // One slot at a time: within a slot the 32 lanes (and the CC channel planes) hit distinct
    // words, so the read-modify-writes below are race free; ACROSS slots lanes do revisit words,
    // which is safe because a warp's shared-memory accesses execute in program order -- the
    // __syncwarp() keeps the compiler from hoisting the next slot's loads above these stores.
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        float* wp = (t < thr ? trowA : trowB) + 4 * t;
        float old[CC];
#pragma unroll
        for (int c = 0; c < CC; ++c) old[c] = wp[c * CH];
#pragma unroll
        for (int c = 0; c < CC; ++c) {
            float2 q2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int pp = 0; pp < Gm::NP; ++pp) {
                if (S >= 0 && (S < 2 * pp || S > 2 * pp + K51)) continue;
                q2 = __ffma2_rn(h2[pp][t], a2[c][pp], q2);
            }
            old[c] += q2.x + q2.y;
        }
        if (!(t == 6 && g3)) {                          // (g == 3, slot 6) would be tap 51
#pragma unroll
            for (int c = 0; c < CC; ++c) wp[c * CH] = old[c];
        }
        __syncwarp();                                   // the next slot may read words other lanes just wrote
    }
}

template <int CC, int R, bool VEC>
__global__ void __launch_bounds__(128, MIN_CTAS)
sepconv_bwd_input_k51_kernel(const float* __restrict__ gout, const float* __restrict__ v,
                             const float* __restrict__ h, float* __restrict__ gi,
                             int C, int c0, int H, int W) {
    constexpr int G = FWD_G;
    using Gm = Geo<G, R>;
    static_assert(Gm::NT == 13, "rotation scheme is written for 4 tap groups of 13");
    extern __shared__ __align__(16) float tile[];      // [CC][ROWS][PITCH] gi accumulators + 4 warps x v ring
    const int IW = W + K51 - 1, IH = H + K51 - 1;
    const int x0 = blockIdx.x * Gm::TILE_W, y0 = blockIdx.y * R;
    const int64_t b = blockIdx.z;
    const int64_t plane = (int64_t)H * W;
    const int tid = threadIdx.x;
    for (int i = tid; i < CC * Gm::ROWS * Gm::PITCH; i += 128) tile[i] = 0.f;
    cp_async_commit();                                  // group 0 (empty): keeps the ring's group arithmetic

    const int warp = tid >> 5, lane = tid & 31;
    const int pg = lane / G, g = lane % G;
    const int xl = warp * Gm::COLS + pg;
    const int x = min(x0 + xl, W - 1);
    const bool g3 = (g == 3);
    const bool col_ok = (x0 + xl < W);

    VRing<G, R, VEC> vr;
    vr.init(tile + CC * Gm::ROWS * Gm::PITCH + warp * (VDEPTH * Gm::SLOT), v, b * K51 * plane, plane,
            y0, x0 + warp * Gm::COLS, H, W, lane);
#pragma unroll
    for (int st = 0; st < VDEPTH - 1; ++st) vr.issue();

    // horizontal taps in rotated slot order: slot t <- tap 4*((t + 2g) mod 13) + g
    float2 h2[Gm::NP][13], g2[CC][Gm::NP];
    {
        const float* hp[R];
#pragma unroll
        for (int p = 0; p < R; ++p) hp[p] = h + (b * K51 + g) * plane + (int64_t)min(y0 + p, H - 1) * W + x;
#pragma unroll
        for (int t = 0; t < 13; ++t) {
            int m = t + 2 * g;
            m = m >= 13 ? m - 13 : m;
            m = (m == 12 && g3) ? 11 : m;               // tap 51 does not exist: read tap 47, its q is discarded
            const int64_t off = (int64_t)(4 * m) * plane;
#pragma unroll
            for (int pp = 0; pp < Gm::NP; ++pp)
                h2[pp][t] = make_float2(__ldg(hp[2 * pp] + off), __ldg(hp[2 * pp + 1] + off));
        }
    }
#pragma unroll
    for (int c = 0; c < CC; ++c)
#pragma unroll
        for (int pp = 0; pp < Gm::NP; ++pp) {
            const float* gp = gout + (b * C + c0 + c) * plane + x;
            const int ya = y0 + 2 * pp, yb = ya + 1;
            g2[c][pp].x = (col_ok && ya < H) ? __ldg(gp + (int64_t)ya * W) : 0.f;   // outside the image: no contribution
            g2[c][pp].y = (col_ok && yb < H) ? __ldg(gp + (int64_t)yb * W) : 0.f;
        }
    cp_async_wait<VDEPTH - 2>();
    __syncthreads();                                    // tile zeroed

    float2 vcur[Gm::NP], vnext[Gm::NP];
    vr.read(vcur);
    float* trow = tile + xl + g + 8 * g;                // word of slot 0: x + g + 4*(2g)
    const int thr = 13 - 2 * g;
    for (int i = 0; i < warp; ++i) __syncthreads();     // skew: warp w runs w steps behind warp 0
    walk_steps<R, false>([&](auto S, int, auto& vuse, auto& vfill) {
        vr.advance(vfill);
        gi_step<CC, R, decltype(S)::value>(trow, thr, g3, g2, h2, vuse);
        trow += Gm::PITCH;
        __syncthreads();
    }, vcur, vnext);
    for (int i = warp; i < 3; ++i) __syncthreads();     // every warp passes the same number of barriers
    __syncthreads();

    // ---- flush: the tile overlaps its neighbours', so add into the (pre-zeroed) gradient -----------
    constexpr int FW = Gm::TILE_W + K51 - 1;            // columns that can be non-zero
    if (tid < FW && x0 + tid < IW) {                    // a thread owns one column and walks down the rows
#pragma unroll 1
        for (int c = 0; c < CC; ++c) {
            const float* tp = tile + c * Gm::ROWS * Gm::PITCH + tid;
            float* gp = gi + ((b * C + c0 + c) * (int64_t)IH + y0) * IW + x0 + tid;
            const int rmax = min(Gm::ROWS, IH - y0);
#pragma unroll 2
            for (int r = 0; r < rmax; ++r) {
                const float val = tp[r * Gm::PITCH];
                if (val != 0.f) atomicAdd(gp + (int64_t)r * IW, val);
            }
        }
    }
}

// =====================================================================================
// Fused interpolation tail -- IFNet.forward, sff_scripts_interp/model/model_interp.py:90-97
// (sp_scripts_train/networks.py:116-123 runs the same expression twice):
//   y   = sepconv(ReplicationPad2d(25)(i2), k2v, k2h) + sepconv(ReplicationPad2d(25)(i1), k1v, k1h)
//   out = mean_c y                                                           -> [B,1,H,W]
// One launch instead of 2 pads + 2 sepconvs + add + mean: the padding is folded into the window
// load (clamped coordinates), the channel mean is taken on the IMAGE side (the convolution is
// linear in the image: mean_c sepconv(i_c) = sepconv(mean_c i_c)), so each frame costs one plane
// of FMAs instead of C, and both frames accumulate into the same registers.  With
// SSTEM_SEPCONV_GRAY_REPLICATED the planes are identical copies (what every reference caller
// feeds: data_provider.py:136-137) and plane 0 is used as is.
// Same lane mapping / step loop as sepconv_fwd_k51_kernel<1, ...>, run once per frame.
// =====================================================================================
struct TailFrames {                                     // indexed by the frame loop straight from the constant bank,
    const float* frame[2];                              // so the six pointers hold no registers across it
    const float* v[2];
    const float* h[2];
};

template <int G, int R, bool VEC>
__global__ void __launch_bounds__(128, MIN_CTAS)
interp_tail_fwd_k51_kernel(const __grid_constant__ TailFrames fa, int64_t frame_bstride, int cs, int nplanes,
                           float* __restrict__ out, float scale, int H, int W) {
    using Gm = Geo<G, R>;
    extern __shared__ __align__(16) float tile[];      // [nplanes][ROWS][PITCH] + 4 warps x v ring
    const int x0 = blockIdx.x * Gm::TILE_W, y0 = blockIdx.y * R;
    const int64_t b = blockIdx.z;
    const int64_t plane = (int64_t)H * W;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int pg = lane / G, g = lane % G;
    const int xl = warp * Gm::COLS + pg;
    const int x = min(x0 + xl, W - 1);
    const bool novalid = g >= Gm::LAST_VALID_G;

    float2 acc[1][Gm::NP];
#pragma unroll
    for (int pp = 0; pp < Gm::NP; ++pp) acc[0][pp] = make_float2(0.f, 0.f);

#pragma unroll 1
    for (int f = 0; f < 2; ++f) {                       // frame 2 first, as the reference's expression
        const float* __restrict__ fr = fa.frame[f] + b * frame_bstride;
        const float* __restrict__ v = fa.v[f];
        const float* __restrict__ h = fa.h[f];
        float2 h2[Gm::NP][Gm::NT];
        load_h<G, R>(h2, h, b * K51 * plane, plane, y0, x, H, W, g);   // the long pole of the prologue goes first
        if (f > 0) {
            cp_async_wait<0>();                         // the previous frame's look-ahead ring copies have landed ...
            __syncthreads();                            // ... and nobody reads its window any more
        }
        stage_window_tail<Gm::ROWS, Gm::PITCH>(tile, fr, cs, nplanes, x0, y0, H, W, tid);

        VRing<G, R, VEC> vr;
        vr.init(tile + nplanes * Gm::ROWS * Gm::PITCH + warp * (VDEPTH * Gm::SLOT), v, b * K51 * plane, plane,
                y0, x0 + warp * Gm::COLS, H, W, lane);
#pragma unroll
        for (int st = 0; st < VDEPTH - 1; ++st) vr.issue();


        cp_async_wait<VDEPTH - 2>();
        tail_window_reduce<Gm::ROWS, Gm::PITCH>(tile, nplanes, tid);
        __syncthreads();

        float2 vcur[Gm::NP], vnext[Gm::NP];
        vr.read(vcur);
        const float* prow = tile + xl + g;
        float pre[FWD_NPRE + 1];
#pragma unroll
        for (int t = 0; t < FWD_NPRE1; ++t) pre[t] = prow[G * t];
        walk_steps<R, true>([&](auto S, int, auto& vuse, auto& vfill) {
            vr.advance(vfill);
            fwd_step<1, G, R, decltype(S)::value>(prow, novalid, h2, vuse, acc, pre);
            prow += Gm::PITCH;
        }, vcur, vnext);
    }

    constexpr int NV = (R >= G) ? R : G;
    constexpr int PER = NV / G;
    float val[NV];
#pragma unroll
    for (int pp = 0; pp < Gm::NP; ++pp) { val[2 * pp] = acc[0][pp].x; val[2 * pp + 1] = acc[0][pp].y; }
#pragma unroll
    for (int i = R; i < NV; ++i) val[i] = 0.f;
    group_reduce<G, NV>(val, g);
    if (x0 + xl < W) {
        float* ob = out + (b * H + y0) * (int64_t)W + x0 + xl;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int p = g * PER + j;
            if (p < R && y0 + p < H) ob[(int64_t)p * W] = val[j] * scale;
        }
    }
}

// ---- host side ------------------------------------------------------------------------------
template <typename Kern>
int set_smem_once(Kern kern, size_t smem, PerDeviceOnce& done) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (!done.test(dev)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        done.set(dev);
    }
    return 0;
}

template <int G, int R, int CC>
constexpr size_t smem_bytes() {
    return ((size_t)CC * Geo<G, R>::ROWS * Geo<G, R>::PITCH + 4 * VDEPTH * Geo<G, R>::SLOT) * sizeof(float);
}

// grid.y (row tiles) and grid.z (images) of a generation-1 launch are limited to 65535
template <int R>
bool fits_grid(int64_t B, int64_t H) { return B <= 65535 && (H + R - 1) / R <= 65535; }

// VEC: the v ring is fed with 16-byte copies (W % 4 == 0, v 16-byte aligned)
inline bool ring_vec(int64_t W, const float* v) { return (W & 3) == 0 && aligned16(v); }
// PAIR: the padded input window is staged with 8-byte copies ((W + 50) even, `in` 8-byte aligned)
inline bool window_pair(int64_t W, const float* in) {
    return ((W + K51 - 1) & 1) == 0 && (reinterpret_cast<uintptr_t>(in) & 7u) == 0;
}

// f(std::true_type or std::false_type for each flag, in order): the runtime flags become template arguments
template <class F>
int dispatch(F&& f) { return f(); }
template <class F, class... Flags>
int dispatch(F&& f, bool flag, Flags... rest) {
    if (flag) return dispatch([&](auto... t) { return f(std::true_type{}, t...); }, rest...);
    return dispatch([&](auto... t) { return f(std::false_type{}, t...); }, rest...);
}

// One launch of a generation-1 kernel on 128 threads per R-row x TILE_W-column tile of each of B images.  `smem` is the
// most the kernel may use (its attribute, set once per device; one PerDeviceOnce per kernel, as launch_persistent),
// `smem_used` what this launch uses.
template <auto Kern, int G, int R, class... Args>
int launch_k51(size_t smem, size_t smem_used, int64_t B, int H, int W, cudaStream_t s, const Args&... args) {
    static PerDeviceOnce done;
    if (int e = set_smem_once(Kern, smem, done)) return e;
    const dim3 grid((unsigned)((W + Geo<G, R>::TILE_W - 1) / Geo<G, R>::TILE_W), (unsigned)((H + R - 1) / R), (unsigned)B);
    Kern<<<grid, 128, smem_used, s>>>(args...);
    count_launch();
    return finish_launch();
}

// Channel chunks of at most three planes, in order: f(std::integral_constant<int, CC>, c0) for each, until one fails.
template <class F>
int for_each_chunk(int64_t C, F&& f) {
    for (int c0 = 0; c0 < C;) {
        const int cc = C - c0 < 3 ? (int)(C - c0) : 3;
        const int e = cc == 3 ? f(std::integral_constant<int, 3>{}, c0)
                              : (cc == 2 ? f(std::integral_constant<int, 2>{}, c0) : f(std::integral_constant<int, 1>{}, c0));
        if (e) return e;
        c0 += cc;
    }
    return 0;
}

}  // namespace
}  // namespace sstem
