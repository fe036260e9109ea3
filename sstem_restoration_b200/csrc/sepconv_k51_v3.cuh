// Third-generation tap-gradient kernel: persistent warps fed entirely by TMA.
//
// Measured on a second generation (CTA per tile, removed; DESIGN §4.1 and §7): with the window and the vertical taps
// of a tile arriving as two big TMA boxes the step loop itself became 15 % faster, but the tile's prologue -- waiting
// for ~130 KB per tile to cross the SM's L2 port, then for the horizontal taps -- grew to 16 % of all warp time,
// because a CTA cannot prefetch its next tile and only one other CTA is there to cover.  Here nothing waits:
//
//   * a WARP, not a CTA, owns a tile (8 columns x 4 rows) and walks a sequence of tiles (persistent grid, two
//     4-warp CTAs per SM); warps never synchronise with each other, so they drift apart and cover each other's
//     tile switches;
//   * the window streams through a 3-slot ring in groups of 4 input rows: one TMA box {4 channels, 60 columns, 4 rows}
//     of the input repacked channel-interleaved, [B][H+50][W+50][4] with the 4th lane zero (sepconv_layout.cu: its
//     rows are 16-byte multiples and a lane reads all three channels of a tap with one LDS.128), plus one box
//     {8 columns, 4 rows, 4 planes} of vertical taps per group,
//     requested two groups (8 steps) ahead by lane 0, completion on the slot's mbarrier.  A step's vertical taps sit
//     in the current or the previous group's slot at compile-time offsets; tap planes outside 0..50 and pixels
//     outside the image are zero-filled by the TMA unit;
//   * the horizontal taps and the upstream gradient of the NEXT tile are prefetched into shared memory by two more
//     boxes issued right after the current tile copied its own into registers, a whole tile (~30 us) ahead.
//
// Per step a lane issues 130 FFMA2, 13 LDS.128 (window), 4 LDS (v), the gv transpose-reduce and one store; the
// ring costs ~10 instructions per 4 steps.  The forward's operation order is that of generation 1 (bit-identical
// results); grad_vertical sums its 13 tap terms in one chain instead of two (same tolerance against the oracle).
#pragma once
#include "sepconv_k51.cuh"
#include "tma.cuh"
#include <stdlib.h>
#include <type_traits>

namespace sstem {
namespace {

constexpr int V3_COLS = 8;                                   // columns per warp tile
constexpr int V3_WIN_COLS = 60;                              // 8 + 52 tap slots
constexpr int V3_GROUP = 4;                                  // input rows per ring slot
constexpr int V3_NGROUPS = 14;                               // 56 >= 54 input rows per tile
constexpr int B3_R = 4;                                      // rows per warp tile of the tap-gradient kernel
constexpr int B3_ROWS = B3_R + K51 - 1;                      // 54 input rows per tile
constexpr unsigned V3_WIN_BYTES = V3_GROUP * V3_WIN_COLS * 16;   // 3840
constexpr unsigned V3_V_BYTES = V3_GROUP * B3_R * V3_COLS * 4;   // 512: [plane][row][col]
constexpr unsigned V3_SLOT_BYTES = V3_WIN_BYTES + V3_V_BYTES;    // 4352 = 34 * 128
constexpr unsigned V3_H_BYTES = K51 * B3_R * V3_COLS * 4;        // 6528: [row][tap][col]
constexpr unsigned V3_G_BYTES = 3 * B3_R * V3_COLS * 4;          // 384:  [channel][row][col]
constexpr unsigned V3_OFF_H = 3 * V3_SLOT_BYTES;                 // 13056
constexpr unsigned V3_OFF_G = V3_OFF_H + V3_H_BYTES;             // 19584
constexpr unsigned V3_OFF_BAR = V3_OFF_G + V3_G_BYTES;           // 19968: full[3], hbar
constexpr unsigned V3_WARP_BYTES = V3_OFF_BAR + 128;             // 20096 = 157 * 128
constexpr int V3_WARPS = 4;
constexpr size_t V3_SMEM = (size_t)V3_WARPS * V3_WARP_BYTES + 128;

struct V3Shape {
    int H, W, tiles_x, tiles_y, ntiles, C, c0;
};

// L2 policies: a window row is read by ~14 tile rows within a few tens of microseconds (evict last) and must not be
// pushed out by the 1.7 GB of taps streaming past it.  The taps keep the normal policy: a warp tile reads 32 bytes of
// each 64-byte DRAM sector and its neighbour the other half -- marked evict-first the sector was often gone before
// the neighbour asked (measured: +0.5 GB of DRAM reads per launch).
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_load_4d_a(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2, int c3,
                                              uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_load_3d_a(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(policy) : "memory");
}
// Ordered variant for the tile-start copies of the tap / gradient buffers: the "memory" clobber keeps the compiler from
// sinking the load below the TMA request that refills the buffer (it did: the values are first used deep inside the
// first step, and 5 pixels in 500 000 came out wrong).
__device__ __forceinline__ float lds_f32_ordered(unsigned addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ float4 lds_f32x4(unsigned addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

// SSTEM_V3_PHASES (diagnostic builds only, off in the shipped library; tools/v3_phases.py): every warp adds the clock64
// ticks it spends in each phase of a tile to counters in the unused tail of its barrier block (no extra registers but
// the last timestamp), and lane 0 adds them to v3_phase_ticks when the warp leaves.  One array per translation unit:
// the forward's in sepconv_k51_fwd3.cu, the tap gradients' in sepconv_k51_bwd3.cu.
enum V3Phase { V3P_START, V3P_FIRST, V3P_STEADY, V3P_LAST, V3P_STORE, V3P_BARRIER, V3P_COUNT };
#ifdef SSTEM_V3_PHASES
__device__ unsigned long long v3_phase_ticks[V3P_COUNT];
struct V3PhaseClock {
    unsigned long long* acc;                               // V3P_COUNT counters in this warp's shared memory
    long long last;
    __device__ V3PhaseClock(unsigned char* warp_smem, unsigned off, bool lead) : acc(reinterpret_cast<unsigned long long*>(warp_smem + off)) {
        if (lead)
            for (int i = 0; i < V3P_COUNT; ++i) acc[i] = 0;
        last = clock64();
    }
    __device__ __forceinline__ void mark(int phase, bool lead) {
        const long long now = clock64();
        if (lead) acc[phase] += (unsigned long long)(now - last);
        last = now;
    }
    __device__ void flush(bool lead) {
        if (lead)
            for (int i = 0; i < V3P_COUNT; ++i) atomicAdd(&v3_phase_ticks[i], acc[i]);
    }
};
// copies (and optionally clears) this translation unit's totals; 0 or a CUDA error
inline int v3_phases_read(unsigned long long* out, int reset) {
    if (cudaError_t e = cudaMemcpyFromSymbol(out, v3_phase_ticks, sizeof(v3_phase_ticks))) return (int)e;
    if (reset) {
        const unsigned long long zero[V3P_COUNT] = {};
        if (cudaError_t e = cudaMemcpyToSymbol(v3_phase_ticks, zero, sizeof(zero))) return (int)e;
    }
    return 0;
}
#define V3_PHASE_INIT(warp_smem, off) V3PhaseClock v3_clock(warp_smem, off, lead)
#define V3_PHASE(p) v3_clock.mark(p, lead)
#define V3_PHASE_FLUSH() v3_clock.flush(lead)
#else
#define V3_PHASE_INIT(warp_smem, off) ((void)0)
#define V3_PHASE(p) ((void)0)
#define V3_PHASE_FLUSH() ((void)0)
#endif

// One input row: per tap slot t and row pair, t2 = sum_c g_c P_c, then gh += t2 v and gv += t2 h.  gv sums its 13 tap
// terms in one chain (generation 1 uses two partial sums; one chain measured 0.8 % faster here, 4 fewer FADD per step).
// Operands are addressed by shared-memory byte addresses:
//   pa            window row of this step, already offset to the lane's first tap column
//   va[p]         address of v[fy = s - p][row p][column of the lane]   (only read when the row is active)
// CC = 3: channel-interleaved window, one LDS.128 per tap; CC = 1: one plane at a 16-byte row pitch, one LDS.32 per tap
// and t2 = P g (26 products instead of 78 FFMA2).
template <int S, bool WV, bool WH, int CC>
__device__ __forceinline__ void bwd3_step(unsigned pa, unsigned pa_last, const unsigned (&va)[4],
                                          const float2 (&g2)[CC][2], const float2 (&h2)[2][13],
                                          float2 (&gh2)[2][13], float2 (&gvp)[2]) {
    constexpr int NP = 2, NT = 13;
    float2 v2[NP];
#pragma unroll
    for (int pp = 0; pp < NP; ++pp) {
        // S >= 0: a row whose fy = S - p is outside 0..50 gets v = 0 without touching shared memory
        const bool a_ok = (S < 0) || (S - 2 * pp >= 0 && S - 2 * pp < K51);
        const bool b_ok = (S < 0) || (S - 2 * pp - 1 >= 0 && S - 2 * pp - 1 < K51);
        v2[pp].x = (WH && a_ok) ? lds_f32(va[2 * pp]) : 0.f;
        v2[pp].y = (WH && b_ok) ? lds_f32(va[2 * pp + 1]) : 0.f;
    }
#pragma unroll
    for (int pp = 0; pp < NP; ++pp) gvp[pp] = make_float2(0.f, 0.f);
    float2 t2[NT][NP];
    float4 P[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) {                         // channels x, y, z of column x + g + 4t; slot 12 of the lanes
        const unsigned a = t == NT - 1 ? pa_last : pa + (CC == 3 ? 64 : 16) * t;   // g == 3 (tap 51 does not exist) rereads
        P[t] = CC == 3 ? lds_f32x4(a) : make_float4(lds_f32(a), 0.f, 0.f, 0.f);   // tap 47, h = 0 there
    }
#pragma unroll
    for (int c = 0; c < CC; ++c)
#pragma unroll
        for (int t = 0; t < NT; ++t)
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) {
                if (S >= 0 && (S < 2 * pp || S > 2 * pp + K51)) continue;
                const float p = c == 0 ? P[t].x : (c == 1 ? P[t].y : P[t].z);
                t2[t][pp] = __ffma2_rn(make_float2(p, p), g2[c][pp], c == 0 ? make_float2(0.f, 0.f) : t2[t][pp]);
            }
#pragma unroll
    for (int t = 0; t < NT; ++t)
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) {
            if (S >= 0) {
                if (S < 2 * pp || S > 2 * pp + K51) continue;
                if (S - 2 * pp > K51 - 1) t2[t][pp].x = 0.f;
                if (S - 2 * pp - 1 < 0) t2[t][pp].y = 0.f;
            }
            if (WH) gh2[pp][t] = __ffma2_rn(t2[t][pp], v2[pp], gh2[pp][t]);
            if (WV) gvp[pp] = __ffma2_rn(t2[t][pp], h2[pp][t], gvp[pp]);
        }
}

__device__ __forceinline__ void tma_load_5d_a(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2, int c3,
                                              int c4, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6, %7}], [%2], %8;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "l"(policy) : "memory");
}

#ifndef SSTEM_BWD3_MINB
#define SSTEM_BWD3_MINB 2
#endif
// The tap-gradient kernels' body.  CC = 3: channel-interleaved window [B][H+50][W+50][4], upstream gradient box
// {8 columns, 4 rows, 3 channels}; CC = 1: one plane copied to a 16-byte row pitch, one gradient plane (the gray x3
// shortcut with the channel-summed gradient, single remainder planes, the one-plane frames of the tiled tail).
// TILED: the taps and their gradients are tile-major [B][H/8][W/8][51][8][8] (sstem_taps_to_tiled).  A warp tile is half
// of an 8x8 tile; map_v / map_h are 5-D maps over that layout that land exactly as the [B,51,H,W] maps do
// ([plane][row][col] and [row][tap][col]), so only the coordinates and the stores differ.  Every element of a tile inside
// the tensor is written, entries outside the image as explicit zeros (g is zero there but the window may hold Inf).
template <bool WV, bool WH, bool ACCUM, int CC, bool TILED>
__device__ __forceinline__ void bwd3_taps_body(const CUtensorMap& map_in, const CUtensorMap& map_v, const CUtensorMap& map_h,
                                               const CUtensorMap& map_g, float* __restrict__ gv, float* __restrict__ gh,
                                               int* __restrict__ next_tile_counter, const V3Shape& sh, const int* gate, int gate_want) {
    SSTEM_GATE_RETURN(gate, gate_want);
    constexpr int G = 4, R = 4, NP = 2, NT = 13;
    constexpr unsigned WIN_BYTES = CC == 3 ? V3_WIN_BYTES : V3_WIN_BYTES / 4;   // 4 rows x 60 pixels x (16 | 4) bytes
    constexpr unsigned PIX = CC == 3 ? 16u : 4u;
    constexpr unsigned G_BYTES = CC * B3_R * V3_COLS * 4;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // the shuffle tells the compiler that `warp` -- and with it every ring / barrier address and TMA coordinate below --
    // is warp-uniform, so those live in uniform registers and a TMA issue needs no R2UR moves
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int pg = lane / G, g = lane % G;
    const bool novalid = (g == 3);
    const bool lead = (lane == 0);
    // Tiles are handed out dynamically: SMs do not run at the same speed (L2 distance, DRAM refresh), and with a static
    // round-robin the kernel waited for the slowest warp while 14 % of the warp slots sat empty (ncu: warps_active 6.9
    // of 8).  The unit is a CTA tile = 4 adjacent warp tiles (32 columns): the four warps then request the same 128-byte
    // lines of taps at the same time from the same SM -- with per-warp tickets neighbouring tiles ran up to a tile
    // apart on different SMs and half-used lines were fetched twice (ncu: +0.6 GB of DRAM reads per launch).  One
    // named barrier per tile keeps the four warps on the same ticket; inside a tile they never synchronise.  The first
    // two tiles of a CTA are static, so the prefetch of the next tile's taps never waits for an atomic: the ticket drawn
    // at the start of tile k is tile k+2.
    __shared__ int s_ticket[2];
    const int nctas = gridDim.x;
    int tile = blockIdx.x;
    if (tile >= sh.ntiles) return;
    int ntile = tile + nctas;
    int tile_no = 0;

    const unsigned base = ((unsigned)__cvta_generic_to_shared(smem_raw) + 127u & ~127u) + warp * V3_WARP_BYTES;
    const unsigned bar0 = base + V3_OFF_BAR;               // full[slot] at bar0 + 8 * slot, hbar at bar0 + 24
    const unsigned hbar = bar0 + 24;
    if (lead) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            mbar_init(bar0 + 8 * i, 1);
        mbar_fence_init();
    }
    __syncwarp();
    const uint64_t pol_once = l2_policy_evict_normal(), pol_keep = l2_policy_evict_last();

    const int64_t plane = (int64_t)sh.H * sh.W;
    // TILED: 8x8 tiles per row / column of the tile-major tensors (the row tiles of sh.tiles_y are half tiles)
    const int tiles_x8 = TILED ? (sh.W + 7) >> 3 : 0, tiles_y8 = TILED ? (sh.H + 7) >> 3 : 0;
    auto decode = [&](int t, int& b, int& y0, int& x0) {
        const int tx = t % sh.tiles_x, r = t / sh.tiles_x;
        x0 = (tx * V3_WARPS + warp) * V3_COLS;
        y0 = (r % sh.tiles_y) * R;
        b = r / sh.tiles_y;
    };
    // ring slots travel in registers: slot byte address, its barrier address and the parity of its next completion
    unsigned s_cur = base, s_nxt = base + V3_SLOT_BYTES, s_prv = base + 2 * V3_SLOT_BYTES;
    unsigned b_cur = bar0, b_nxt = bar0 + 8, b_prv = bar0 + 16;
    unsigned p_cur = 0, p_nxt = 0, p_prv = 0, p_h = 0;
    auto issue_group = [&](unsigned slot, unsigned bar, int b, int y0, int x0, int gi) {
        if (lead) {
            mbar_expect_tx(bar, WIN_BYTES + (WH ? V3_V_BYTES : 0u));
            // rows of 60 pixels x 4 floats (CC = 3: 960 contiguous bytes) or x 1 float
            tma_load_3d_a(slot, &map_in, bar, (CC == 3 ? 4 : 1) * x0, y0 + V3_GROUP * gi, b, pol_keep);
            if (WH) {
                // tiled box {8 col, 4 row, 4 tap}: starts at column 0 and row 0 or 4 of its 8x8 tile (32-byte aligned)
                if constexpr (TILED) tma_load_5d_a(slot + V3_WIN_BYTES, &map_v, bar, 0, y0 & 7, V3_GROUP * gi, x0 >> 3, b * tiles_y8 + (y0 >> 3), pol_once);
                else tma_load_4d_a(slot + V3_WIN_BYTES, &map_v, bar, x0, y0, V3_GROUP * gi, b, pol_once);
            }
        }
    };
    auto issue_hg = [&](int b, int y0, int x0) {
        if (lead) {
            mbar_expect_tx(hbar, (WV ? V3_H_BYTES : 0u) + G_BYTES);
            if (WV) {                                      // [row][tap][col]
                if constexpr (TILED) tma_load_5d_a(base + V3_OFF_H, &map_h, hbar, 0, 0, y0 & 7, x0 >> 3, b * tiles_y8 + (y0 >> 3), pol_once);
                else tma_load_4d_a(base + V3_OFF_H, &map_h, hbar, x0, 0, y0, b, pol_once);
            }
            tma_load_4d_a(base + V3_OFF_G, &map_g, hbar, x0, y0, 0, b, pol_once);
        }
    };
    auto rotate = [&]() {                                  // (cur, nxt, prv) <- (nxt, prv, cur)
        unsigned t;
        t = s_cur; s_cur = s_nxt; s_nxt = s_prv; s_prv = t;
        t = b_cur; b_cur = b_nxt; b_nxt = b_prv; b_prv = t;
        t = p_cur; p_cur = p_nxt; p_nxt = p_prv; p_prv = t;
    };

    int tb, ty0, tx0;
    decode(tile, tb, ty0, tx0);
    issue_hg(tb, ty0, tx0);
    issue_group(s_cur, b_cur, tb, ty0, tx0, 0);
    issue_group(s_nxt, b_nxt, tb, ty0, tx0, 1);

    const unsigned lane_win = (unsigned)(pg + g) * PIX;    // lane's first tap column inside a window row
    const unsigned lane_last = lane_win + (novalid ? 11u : 12u) * 4u * PIX;   // its slot 12 (g == 3: tap 47 again, see the h copy)
    const unsigned lane_v = V3_WIN_BYTES + (unsigned)pg * 4u;
    V3_PHASE_INIT(smem_raw + (base - (unsigned)__cvta_generic_to_shared(smem_raw)), V3_OFF_BAR + 32);

#pragma unroll 1
    for (;;) {
        const bool has_next = ntile < sh.ntiles;
        int nb = 0, ny0 = 0, nx0 = 0;
        if (has_next) decode(ntile, nb, ny0, nx0);
        if (has_next && warp == 0 && lead) s_ticket[tile_no & 1] = atomicAdd(next_tile_counter, 1);   // read after this tile's barrier

        // ---- this tile's horizontal taps and upstream gradient: shared memory -> registers
        float2 h2[NP][NT], gh2[NP][NT], g2[CC][NP];
        mbar_wait(hbar, p_h);
        p_h ^= 1;
        {
            // [row][tap][col]: the lanes of one load sit in banks 8 * ((3 * row + g) mod 4) + pg, one wavefront
            const unsigned ha = base + V3_OFF_H + (unsigned)pg * 4u;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const int tap = (t == NT - 1 && novalid) ? (G * (NT - 2) + g) : (G * t + g);   // tap 51: reread tap 47 (masked by P = 0)
#pragma unroll
                for (int pp = 0; pp < NP; ++pp) {
                    gh2[pp][t] = make_float2(0.f, 0.f);
                    h2[pp][t] = WV ? make_float2(lds_f32_ordered(ha + ((2 * pp * K51 + tap) * V3_COLS) * 4),
                                                 lds_f32_ordered(ha + (((2 * pp + 1) * K51 + tap) * V3_COLS) * 4))
                                   : make_float2(0.f, 0.f);
                    // tap 51 does not exist: its window value is tap 47's (finite whenever the lane's own taps are), its weight 0,
                    // its gh accumulator is never stored
                    if (t == NT - 1 && novalid) h2[pp][t] = make_float2(0.f, 0.f);
                }
            }
            const unsigned ga = base + V3_OFF_G + (unsigned)pg * 4u;
#pragma unroll
            for (int c = 0; c < CC; ++c)
#pragma unroll
                for (int pp = 0; pp < NP; ++pp)
                    g2[c][pp] = make_float2(lds_f32_ordered(ga + ((c * R + 2 * pp) * V3_COLS) * 4), lds_f32_ordered(ga + ((c * R + 2 * pp + 1) * V3_COLS) * 4));
        }
        V3_PHASE(V3P_START);
        // The two buffers are refilled (next tile's taps) only after the first group below: they may be overwritten once
        // every lane's copy has ARRIVED in registers, not merely been issued -- the 64 loads queue behind the other warps'
        // shared-memory traffic, and a TMA write issued right here overtook them now and then (grad_vertical wrong in
        // ~5 of 500 000 pixels, differently from run to run).  After group 0 every copied value has been an FFMA2 operand.

        const int x = tx0 + pg;
        const bool col_ok = x < sh.W;
        // TILED: this warp tile's 8x8 tile (none when the CTA tile reaches past the tensor's last tile column)
        const bool tile_ok = !TILED || (tx0 >> 3) < tiles_x8;
        const int64_t tile_base = TILED ? (((int64_t)tb * tiles_y8 + (ty0 >> 3)) * tiles_x8 + (tx0 >> 3)) * (K51 * 64) : 0;
        float* gv_ptr = !WV ? nullptr
                      : TILED ? gv + tile_base + ((ty0 & 7) + g) * V3_COLS + pg - g * 64   // plane fy = -g
                              : gv + (int64_t)tb * K51 * plane + (int64_t)min(ty0 + g, sh.H - 1) * sh.W + min(x, sh.W - 1) - (int64_t)g * plane;
        const bool gv_row_ok = col_ok && (ty0 + g < sh.H);
        float2 gvp[NP];
        auto store_gv = [&](int fy) {                      // fy = s - g for this lane
            if (WV) {
                float val[R];
#pragma unroll
                for (int pp = 0; pp < NP; ++pp) { val[2 * pp] = gvp[pp].x; val[2 * pp + 1] = gvp[pp].y; }
                group_reduce<G, R>(val, g);                // lane g now holds the total of row g
                if constexpr (TILED) {                     // a tap's 4 rows x 8 columns are 128 contiguous bytes
                    if (tile_ok && fy >= 0 && fy < K51) __stcs(gv_ptr, gv_row_ok ? (ACCUM ? (*gv_ptr + val[0]) : val[0]) : 0.f);
                    gv_ptr += 64;
                } else {
                    if (gv_row_ok && fy >= 0 && fy < K51) __stcs(gv_ptr, ACCUM ? (*gv_ptr + val[0]) : val[0]);
                    gv_ptr += plane;
                }
            }
        };
        // One group of 4 input rows.  GI >= 0: compile-time group index (first / last groups of the tile, whose steps
        // are partially active); GI < 0: steady state, runtime group index gi.
        auto run_step = [&](auto gi_tag, auto u_tag, int gi, unsigned wa, unsigned wl, unsigned vc, unsigned vp) {
            constexpr int GI = decltype(gi_tag)::value, U = decltype(u_tag)::value;
            constexpr int S = GI < 0 ? -1 : GI * V3_GROUP + U;            // compile-time step of the partial groups
            if (GI >= 0 && GI * V3_GROUP + U >= B3_ROWS) return;          // rows 54, 55 of the last group: nothing to do
            unsigned va[4];
#pragma unroll
            for (int p = 0; p < 4; ++p)                    // plane s - p: this group's slot or the previous one's
                va[p] = (U - p >= 0 ? vc + ((U - p) * R + p) * V3_COLS * 4 : vp + ((V3_GROUP + U - p) * R + p) * V3_COLS * 4);
            bwd3_step<S, WV, WH, CC>(wa + U * V3_WIN_COLS * PIX, wl + U * V3_WIN_COLS * PIX, va, g2, h2, gh2, gvp);
            store_gv(V3_GROUP * gi + U - g);
        };
        auto run_group = [&](auto gi_tag, int gi) {
            mbar_wait(b_cur, p_cur);
            p_cur ^= 1;
            const unsigned wa = s_cur + lane_win, wl = s_cur + lane_last, vc = s_cur + lane_v, vp = s_prv + lane_v;
            run_step(gi_tag, std::integral_constant<int, 0>{}, gi, wa, wl, vc, vp);
            run_step(gi_tag, std::integral_constant<int, 1>{}, gi, wa, wl, vc, vp);
            run_step(gi_tag, std::integral_constant<int, 2>{}, gi, wa, wl, vc, vp);
            run_step(gi_tag, std::integral_constant<int, 3>{}, gi, wa, wl, vc, vp);
        };
        auto end_group = [&](bool next_tile, int gi_issue) {   // everyone is done with the previous group's slot: refill it
            __syncwarp();
            if (next_tile) { if (has_next) issue_group(s_prv, b_prv, nb, ny0, nx0, gi_issue); }
            else issue_group(s_prv, b_prv, tb, ty0, tx0, gi_issue);
            rotate();
        };

        run_group(std::integral_constant<int, 0>{}, 0);
        end_group(false, 2);
        if (has_next) issue_hg(nb, ny0, nx0);              // see above: h2 / g2 are in registers for sure by now
        V3_PHASE(V3P_FIRST);
#pragma unroll 1
        for (int gi = 1; gi < 12; ++gi) {                  // groups 1..11 = steps 4..47: every row active
            run_group(std::integral_constant<int, -1>{}, gi);
            end_group(false, gi + 2);
        }
        V3_PHASE(V3P_STEADY);
        run_group(std::integral_constant<int, 12>{}, 12);  // steps 48..51
        end_group(true, 0);
        run_group(std::integral_constant<int, 13>{}, 13);  // steps 52, 53 (+ two rows nobody needs)
        end_group(true, 1);
        V3_PHASE(V3P_LAST);

        // ---- gh: complete per lane (the sum over fy happened in registers)
        if constexpr (TILED) if (WH && tile_ok) {
            float* gp = gh + tile_base + g * 64 + (ty0 & 7) * V3_COLS + pg;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                if (t == NT - 1 && novalid) break;
#pragma unroll
                for (int pp = 0; pp < NP; ++pp) {
                    const bool a_ok = col_ok && ty0 + 2 * pp < sh.H, b_ok = col_ok && ty0 + 2 * pp + 1 < sh.H;
                    float* da = gp + G * t * 64 + 2 * pp * V3_COLS;
                    float* db = da + V3_COLS;
                    __stcs(da, a_ok ? (ACCUM ? (*da + gh2[pp][t].x) : gh2[pp][t].x) : 0.f);
                    __stcs(db, b_ok ? (ACCUM ? (*db + gh2[pp][t].y) : gh2[pp][t].y) : 0.f);
                }
            }
        }
        if constexpr (!TILED) if (WH && col_ok) {
            float* gp = gh + ((int64_t)tb * K51 + g) * plane + x;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                if (t == NT - 1 && novalid) break;
#pragma unroll
                for (int pp = 0; pp < NP; ++pp) {
                    const int ya = ty0 + 2 * pp, yb = ya + 1;
                    float* da = gp + (int64_t)(G * t) * plane + (int64_t)ya * sh.W;
                    float* db = gp + (int64_t)(G * t) * plane + (int64_t)yb * sh.W;
                    if (ya < sh.H) __stcs(da, ACCUM ? (*da + gh2[pp][t].x) : gh2[pp][t].x);
                    if (yb < sh.H) __stcs(db, ACCUM ? (*db + gh2[pp][t].y) : gh2[pp][t].y);
                }
            }
        }
        V3_PHASE(V3P_STORE);
        if (!has_next) break;
        asm volatile("bar.sync 1, %0;" ::"n"(V3_WARPS * 32) : "memory");   // the CTA moves to its next tile together
        tile = ntile; tb = nb; ty0 = ny0; tx0 = nx0;
        ntile = 2 * nctas + *reinterpret_cast<volatile int*>(&s_ticket[tile_no & 1]);
        ++tile_no;
        V3_PHASE(V3P_BARRIER);
    }
    V3_PHASE_FLUSH();
}

// [B,51,H,W] taps, three channels
template <bool WV, bool WH, bool ACCUM>
__global__ void __launch_bounds__(V3_WARPS * 32, SSTEM_BWD3_MINB)
sepconv_bwd_taps_k51_v3_kernel(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_v,
                               const __grid_constant__ CUtensorMap map_h, const __grid_constant__ CUtensorMap map_g,
                               float* __restrict__ gv, float* __restrict__ gh, int* __restrict__ next_tile_counter,
                               const V3Shape sh, const int* gate, int gate_want) {
    bwd3_taps_body<WV, WH, ACCUM, 3, false>(map_in, map_v, map_h, map_g, gv, gh, next_tile_counter, sh, gate, gate_want);
}

// tile-major taps and tap gradients, three channels or one (sstem_sepconv_backward_tiled)
template <bool WV, bool WH, bool ACCUM, int CC>
__global__ void __launch_bounds__(V3_WARPS * 32, SSTEM_BWD3_MINB)
sepconv_bwd_taps_k51_v3_tiled_kernel(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_v,
                                     const __grid_constant__ CUtensorMap map_h, const __grid_constant__ CUtensorMap map_g,
                                     float* __restrict__ gv, float* __restrict__ gh, int* __restrict__ next_tile_counter,
                                     const V3Shape sh, const int* gate, int gate_want) {
    bwd3_taps_body<WV, WH, ACCUM, CC, true>(map_in, map_v, map_h, map_g, gv, gh, next_tile_counter, sh, gate, gate_want);
}

// =====================================================================================================================
// Forward, same machinery: a warp owns 8 columns x 8 rows, walks 58 input rows (15 groups of 4) per tile.
//   out[c][p] += v[fy = s - p][p] * sum_t P_c[s][x + g + 4t] * h[4t + g][p]
// Per step: 13 LDS.128 (window), 8 LDS (vertical taps: plane s - p lives in this group's slot or one of the two before
// it), 168 FFMA2.  Ring: 2 window slots, 4 vertical-tap slots, 2 barriers (group parity); the next tile's horizontal
// taps (box {8 columns, 8 rows, 51 taps} = 13 KB) are prefetched while this tile computes.  The four tap groups of a
// pixel are summed once per tile (transpose-reduce), after which lane g holds rows 2g, 2g+1.
// =====================================================================================================================
constexpr int F3_R = 8;
constexpr int F3_ROWS = F3_R + K51 - 1;                          // 58
constexpr unsigned F3_V_BYTES = V3_GROUP * F3_R * V3_COLS * 4;   // 1024: [plane][row][col]
constexpr unsigned F3_H_BYTES = K51 * F3_R * V3_COLS * 4;        // 13056: [row][tap][col] ([tap][row][col] when TILED)
constexpr unsigned F3_OFF_V = 2 * V3_WIN_BYTES;                  // 7680
constexpr unsigned F3_OFF_H = F3_OFF_V + 4 * F3_V_BYTES;         // 11776
constexpr unsigned F3_OFF_BAR = F3_OFF_H + F3_H_BYTES;           // 24832
constexpr unsigned F3_WARP_BYTES = F3_OFF_BAR + 128;             // 24960 = 195 * 128
constexpr size_t F3_SMEM = (size_t)V3_WARPS * F3_WARP_BYTES + 128;

template <int S, int CC>
__device__ __forceinline__ void fwd3_step(unsigned pa, unsigned pa_last, const unsigned (&va)[8],
                                          const float2 (&h2)[4][13], float2 (&acc)[CC][4]) {
    constexpr int NP = 4, NT = 13;
    float2 v2[NP];
#pragma unroll
    for (int pp = 0; pp < NP; ++pp) {                      // S >= 0: rows whose fy = S - p is outside 0..50 get v = 0
        const bool a_ok = (S < 0) || (S - 2 * pp >= 0 && S - 2 * pp < K51);
        const bool b_ok = (S < 0) || (S - 2 * pp - 1 >= 0 && S - 2 * pp - 1 < K51);
        v2[pp].x = a_ok ? lds_f32(va[2 * pp]) : 0.f;
        v2[pp].y = b_ok ? lds_f32(va[2 * pp + 1]) : 0.f;
    }
    float2 part[CC][NP];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        float4 P;                                          // CC == 3: channel-interleaved window, one LDS.128 per tap;
        // slot 12 of the lanes g == 3 (tap 51 does not exist) rereads tap 47's column; h is 0 there
        const unsigned a = t == NT - 1 ? pa_last : pa + (CC == 3 ? 64 : 16) * t;
        if (CC == 3) P = lds_f32x4(a);                     // CC == 1: planar window, one LDS.32
        else P = make_float4(lds_f32(a), 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < CC; ++c) {
            const float p = c == 0 ? P.x : (c == 1 ? P.y : P.z);
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) {
                if (S >= 0 && (S < 2 * pp || S > 2 * pp + K51)) continue;   // pair entirely outside
                part[c][pp] = __ffma2_rn(make_float2(p, p), h2[pp][t], t == 0 ? make_float2(0.f, 0.f) : part[c][pp]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < CC; ++c)
#pragma unroll
        for (int pp = 0; pp < NP; ++pp) {
            if (S >= 0) {
                if (S < 2 * pp || S > 2 * pp + K51) continue;
                // a row whose fy is out of range must not even see part (NaN / Inf safety)
                if (S - 2 * pp > K51 - 1) part[c][pp].x = 0.f;
                if (S - 2 * pp - 1 < 0) part[c][pp].y = 0.f;
            }
            acc[c][pp] = __ffma2_rn(v2[pp], part[c][pp], acc[c][pp]);
        }
}

// CC = 3: channel-interleaved window (float4 per pixel); CC = 1: one plane, copied to a 16-byte pitch (the gray x3
// shortcut runs this and writes `replicas` identical output planes).  TILED: the taps arrive in the tile-major layout
// [B][H/8][W/8][51][8][8] (SURVEY 8f N2: what a tap producer should emit) -- a warp tile's horizontal taps are ONE
// contiguous 13 KB bulk copy and a group of 4 vertical-tap planes one contiguous 1 KB -- instead of 51 x 8 row segments
// of 32 bytes gathered by a tensor map from [B][51][H][W].
struct F3Tiled {
    const float* v;                                        // tile-major vertical / horizontal taps (TILED only)
    const float* h;
    int tiles_x8, tiles_y8;                                // warp tiles per row / column of the tiled layout
    int accum;                                             // add to the output instead of overwriting it (second frame of the interpolation tail)
};
template <int CC, bool TILED>
__global__ void __launch_bounds__(V3_WARPS * 32, 2)
sepconv_fwd_k51_v3_kernel(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_v,
                          const __grid_constant__ CUtensorMap map_h, const F3Tiled tl, float* __restrict__ out,
                          int* __restrict__ next_tile_counter, const V3Shape sh, int replicas, const int* gate, int gate_want) {
    SSTEM_GATE_RETURN(gate, gate_want);
    constexpr int G = 4, R = F3_R, NP = 4, NT = 13;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int pg = lane / G, g = lane % G;
    const bool novalid = (g == 3);
    const bool lead = (lane == 0);
    __shared__ int s_ticket[2];                            // CTA-level dynamic tile tickets: see the tap-gradient kernel
    const int nctas = gridDim.x;
    int tile = blockIdx.x;
    if (tile >= sh.ntiles) return;
    int ntile = tile + nctas;
    int tile_no = 0;

    const unsigned base = ((unsigned)__cvta_generic_to_shared(smem_raw) + 127u & ~127u) + warp * F3_WARP_BYTES;
    const unsigned bar0 = base + F3_OFF_BAR;               // full[group parity] at +0 / +8, hbar at +16
    const unsigned hbar = bar0 + 16;
    if (lead) {
#pragma unroll
        for (int i = 0; i < 3; ++i)
            mbar_init(bar0 + 8 * i, 1);
        mbar_fence_init();
    }
    __syncwarp();
    const uint64_t pol_once = l2_policy_evict_normal(), pol_keep = l2_policy_evict_last();

    const int64_t plane = (int64_t)sh.H * sh.W;
    auto decode = [&](int t, int& b, int& y0, int& x0) {
        const int tx = t % sh.tiles_x, r = t / sh.tiles_x;
        x0 = (tx * V3_WARPS + warp) * V3_COLS;
        y0 = (r % sh.tiles_y) * R;
        b = r / sh.tiles_y;
    };
    // window slots / barriers alternate (a = this group, b = next group); vertical-tap slots rotate through four
    constexpr unsigned WIN_BYTES = CC == 3 ? V3_WIN_BYTES : V3_WIN_BYTES / 4;   // 4 rows x 60 pixels x (16 | 4) bytes
    constexpr unsigned PIX = CC == 3 ? 16u : 4u;
    unsigned w_a = base, w_b = base + V3_WIN_BYTES, b_a = bar0, b_b = bar0 + 8, p_a = 0, p_b = 0, p_h = 0;
    unsigned v_c = base + F3_OFF_V, v_n = v_c + F3_V_BYTES, v_f = v_c + 2 * F3_V_BYTES, v_p = v_c + 3 * F3_V_BYTES;
    // v_c: this group, v_n: next group (in flight), v_f: free -> receives group + 2 at the end of this group... see end_group
    auto issue_group = [&](unsigned wslot, unsigned vslot, unsigned bar, int b, int y0, int x0, int gi) {
        if (lead) {
            // tiled: planes 4gi .. 4gi+3 of this warp tile are contiguous (256 bytes each); planes past the 51st do not exist
            // (nothing reads them: rows with fy > 50 are masked at compile time)
            const int nplanes = TILED ? max(0, min(V3_GROUP, K51 - V3_GROUP * gi)) : V3_GROUP;
            mbar_expect_tx(bar, WIN_BYTES + (unsigned)nplanes * (F3_V_BYTES / V3_GROUP));
            tma_load_3d_a(wslot, &map_in, bar, (CC == 3 ? 4 : 1) * x0, y0 + V3_GROUP * gi, b, pol_keep);
            if (!TILED) tma_load_4d_a(vslot, &map_v, bar, x0, y0, V3_GROUP * gi, b, pol_once);
            else if (nplanes > 0) {
                const float* src = tl.v + (((int64_t)b * tl.tiles_y8 + y0 / F3_R) * tl.tiles_x8 + x0 / V3_COLS) * (K51 * 64) + gi * (V3_GROUP * 64);
                bulk_load(vslot, src, (unsigned)nplanes * (F3_V_BYTES / V3_GROUP), bar);
            }
        }
    };
    auto issue_h = [&](int b, int y0, int x0) {
        if (lead) {
            mbar_expect_tx(hbar, F3_H_BYTES);
            if (!TILED) tma_load_4d_a(base + F3_OFF_H, &map_h, hbar, x0, 0, y0, b, pol_once);   // [row][tap][col]
            else bulk_load(base + F3_OFF_H, tl.h + (((int64_t)b * tl.tiles_y8 + y0 / F3_R) * tl.tiles_x8 + x0 / V3_COLS) * (K51 * 64),
                           F3_H_BYTES, hbar);
        }
    };

    int tb, ty0, tx0;
    decode(tile, tb, ty0, tx0);
    issue_h(tb, ty0, tx0);
    // vertical-tap slots in use at group i: v_c = i, v_p1 = i-1, v_p2 = i-2; v_n = i+1 in flight.  Four registers:
    unsigned v_p1 = v_p, v_p2 = v_f;                       // contents irrelevant before the first groups (never read)
    issue_group(w_a, v_c, b_a, tb, ty0, tx0, 0);
    issue_group(w_b, v_n, b_b, tb, ty0, tx0, 1);

    const unsigned lane_win = (unsigned)(pg + g) * PIX;
    const unsigned lane_last = lane_win + (novalid ? 11u : 12u) * 4u * PIX;
    const unsigned lane_v = (unsigned)pg * 4u;
    V3_PHASE_INIT(smem_raw + (base - (unsigned)__cvta_generic_to_shared(smem_raw)), F3_OFF_BAR + 32);

#pragma unroll 1
    for (;;) {
        const bool has_next = ntile < sh.ntiles;
        int nb = 0, ny0 = 0, nx0 = 0;
        if (has_next) decode(ntile, nb, ny0, nx0);
        if (has_next && warp == 0 && lead) s_ticket[tile_no & 1] = atomicAdd(next_tile_counter, 1);

        float2 h2[NP][NT], acc[CC][NP];
        mbar_wait(hbar, p_h);
        p_h ^= 1;
        {
            // NCHW taps land as [row][tap][col] (banks 8 * ((3 * row + g) mod 4) + pg: one wavefront per load); the tile-major
            // layout is [tap][row][col], an external format (its loads are 4-way bank conflicts)
            const unsigned ha = base + F3_OFF_H + (unsigned)pg * 4u;
            auto h_word = [](int row, int tap) { return TILED ? tap * R + row : row * K51 + tap; };
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const int tap = (t == NT - 1 && novalid) ? (G * (NT - 2) + g) : (G * t + g);
#pragma unroll
                for (int pp = 0; pp < NP; ++pp) {
                    h2[pp][t] = make_float2(lds_f32_ordered(ha + (h_word(2 * pp, tap) * V3_COLS) * 4), lds_f32_ordered(ha + (h_word(2 * pp + 1, tap) * V3_COLS) * 4));
                    if (t == NT - 1 && novalid) h2[pp][t] = make_float2(0.f, 0.f);   // tap 51 does not exist: weight 0 on tap 47's column
                }
            }
        }
#pragma unroll
        for (int c = 0; c < CC; ++c)
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) acc[c][pp] = make_float2(0.f, 0.f);
        V3_PHASE(V3P_START);
        // (the tap buffer is refilled after the second group: see the tap-gradient kernel)

        auto run_step = [&](auto gi_tag, auto u_tag, unsigned wa, unsigned wl, unsigned vc, unsigned vp1, unsigned vp2) {
            constexpr int GI = decltype(gi_tag)::value, U = decltype(u_tag)::value;
            constexpr int S = GI < 0 ? -1 : GI * V3_GROUP + U;
            if (GI >= 0 && GI * V3_GROUP + U >= F3_ROWS) return;          // rows 58, 59 of the last group
            unsigned va[8];
#pragma unroll
            for (int p = 0; p < 8; ++p) {                  // plane s - p: this group's slot or one of the two before
                const int d = U - p;                       // -7 .. 3
                const unsigned slot = d >= 0 ? vc : (d >= -4 ? vp1 : vp2);
                const int pl = d >= 0 ? d : (d >= -4 ? d + 4 : d + 8);
                va[p] = slot + (pl * R + p) * V3_COLS * 4;
            }
            fwd3_step<S, CC>(wa + U * V3_WIN_COLS * PIX, wl + U * V3_WIN_COLS * PIX, va, h2, acc);
        };
        auto run_group = [&](auto gi_tag) {
            mbar_wait(b_a, p_a);
            p_a ^= 1;
            const unsigned wa = w_a + lane_win, wl = w_a + lane_last, vc = v_c + lane_v, vp1 = v_p1 + lane_v, vp2 = v_p2 + lane_v;
            run_step(gi_tag, std::integral_constant<int, 0>{}, wa, wl, vc, vp1, vp2);
            run_step(gi_tag, std::integral_constant<int, 1>{}, wa, wl, vc, vp1, vp2);
            run_step(gi_tag, std::integral_constant<int, 2>{}, wa, wl, vc, vp1, vp2);
            run_step(gi_tag, std::integral_constant<int, 3>{}, wa, wl, vc, vp1, vp2);
        };
        // end of group i: its window slot and the vertical-tap slot of group i-2 are free -> they receive group i+2
        auto end_group = [&](bool next_tile, int gi_issue) {
            __syncwarp();
            if (next_tile) { if (has_next) issue_group(w_a, v_p2, b_a, nb, ny0, nx0, gi_issue); }
            else issue_group(w_a, v_p2, b_a, tb, ty0, tx0, gi_issue);
            unsigned t;
            t = w_a; w_a = w_b; w_b = t;
            t = b_a; b_a = b_b; b_b = t;
            t = p_a; p_a = p_b; p_b = t;
            t = v_p2; v_p2 = v_p1; v_p1 = v_c; v_c = v_n; v_n = t;   // (c, n, p1, p2) <- (n, old p2 [now filling], c, p1)
        };

        run_group(std::integral_constant<int, 0>{});
        end_group(false, 2);
        run_group(std::integral_constant<int, 1>{});
        end_group(false, 3);
        if (has_next) issue_h(nb, ny0, nx0);               // all 8 rows have used their taps by step 7
        V3_PHASE(V3P_FIRST);
#pragma unroll 1
        for (int gi = 2; gi < 12; ++gi) {                  // groups 2..11 = steps 8..47: every row active
            run_group(std::integral_constant<int, -1>{});
            end_group(false, gi + 2);
        }
        V3_PHASE(V3P_STEADY);
        run_group(std::integral_constant<int, 12>{});      // steps 48..51
        end_group(false, 14);
        run_group(std::integral_constant<int, 13>{});      // steps 52..55
        end_group(true, 0);
        run_group(std::integral_constant<int, 14>{});      // steps 56, 57
        end_group(true, 1);
        V3_PHASE(V3P_LAST);

        // ---- sum the 4 tap groups of each pixel: lane g ends up with rows 2g, 2g+1 of every channel
        const int x = tx0 + pg;
#pragma unroll
        for (int c = 0; c < CC; ++c) {
            float val[R];
#pragma unroll
            for (int pp = 0; pp < NP; ++pp) { val[2 * pp] = acc[c][pp].x; val[2 * pp + 1] = acc[c][pp].y; }
            group_reduce<G, R>(val, g);
            if (x < sh.W) {
                float* ob = out + (((int64_t)tb * sh.C + sh.c0 + c) * sh.H + ty0) * sh.W + x;
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int p = 2 * g + j;
                    if (ty0 + p < sh.H) {
                        if (tl.accum) val[j] += ob[(int64_t)p * sh.W];
                        ob[(int64_t)p * sh.W] = val[j];
                        // gray x3 shortcut: the input planes are identical copies, so are the outputs
                        for (int rc = 1; rc < replicas; ++rc) ob[(int64_t)rc * plane + (int64_t)p * sh.W] = val[j];
                    }
                }
            }
        }
        V3_PHASE(V3P_STORE);
        if (!has_next) break;
        asm volatile("bar.sync 1, %0;" ::"n"(V3_WARPS * 32) : "memory");   // the CTA moves to its next tile together
        tile = ntile; tb = nb; ty0 = ny0; tx0 = nx0;
        ntile = 2 * nctas + *reinterpret_cast<volatile int*>(&s_ticket[tile_no & 1]);
        ++tile_no;
        V3_PHASE(V3P_BARRIER);
    }
    V3_PHASE_FLUSH();
}

// =====================================================================================================================
// Host side, shared by the launchers in sepconv_k51_fwd3.cu and sepconv_k51_bwd3.cu.
// =====================================================================================================================

// Tile grid of a persistent launch: CTA tiles of V3_WARPS warp tiles side by side, `tiles_y` warp-tile rows per image.
// false when there are too many tiles for the int tile tickets.
inline bool v3_shape(V3Shape& sh, int64_t B, int C, int c0, int H, int W, int64_t tiles_y) {
    const int64_t tiles_x = (W + V3_COLS * V3_WARPS - 1) / (V3_COLS * V3_WARPS);
    if (tiles_x * tiles_y * B > INT32_MAX / 2) return false;
    sh = V3Shape{H, W, (int)tiles_x, (int)tiles_y, (int)(tiles_x * tiles_y * B), C, c0};
    return true;
}

// The window of one persistent launch, in a stream-ordered workspace: channels sh.c0.. of the input [B,C,H+50,W+50]
// copied to the layout the window boxes read (CC = 3: channel-interleaved [B][H+50][W+50][4]; CC = 1: one plane at a
// 16-byte row pitch), then the dynamic tile scheduler's ticket counter, and the tensor map of the copy.  The workspace
// goes back to the pool on the stream when the object goes out of scope, after the work enqueued on it.
// err: 0, cudaErrorMemoryAllocation when there is no workspace, a CUDA error of the memset or the copy, or SSTEM_E_SHAPE
// when the map cannot be encoded.
template <int CC>
struct V3Window {
    cudaStream_t s;
    float* ws = nullptr;
    int* counter = nullptr;
    CUtensorMap map;
    int err = 0;
    V3Window(const float* in, int64_t B, const V3Shape& sh, cudaStream_t s_) : s(s_) {
        const int64_t IH = sh.H + K51 - 1, IW = sh.W + K51 - 1, IWP = (IW + 3) & ~(int64_t)3;
        const int64_t row = CC == 3 ? 4 * IW : IWP;        // floats per window row
        const size_t bytes = (size_t)(B * IH * row) * 4;
        if (workspace_alloc(reinterpret_cast<void**>(&ws), bytes + 256, s)) { err = cudaErrorMemoryAllocation; return; }
        counter = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + bytes);
        if (cudaError_t e = cudaMemsetAsync(counter, 0, 256, s)) { cudaGetLastError(); err = (int)e; return; }
        err = CC == 3 ? launch_repack_nhwc4(in, ws, B, sh.C, sh.c0, IH, IW, s)
                      : launch_repack_plane_pitch(in, ws, B, sh.C, sh.c0, IH, IW, IWP, s);
        if (err) return;
        // CC = 3: the box's inner extent is a whole 960-byte row segment (an inner extent of one pixel = 16 bytes makes
        // the TMA unit issue 240 tiny requests per box: measured 1.5x slower)
        const int64_t dims[3] = {row, IH, B}, strides[3] = {1, row, row * IH};
        const int box[3] = {(CC == 3 ? 4 : 1) * V3_WIN_COLS, V3_GROUP, 1};
        if (!make_map_f32(&map, ws, 3, dims, strides, box)) err = SSTEM_E_SHAPE;
    }
    ~V3Window() { if (ws) cudaFreeAsync(ws, s); }
};

// Tensor maps of [B,51,H,W] taps for warp tiles of `rows` rows: v in boxes {8 columns, rows, 4 planes}, landing as
// [plane][row][col].  h is described with its tap and row dimensions swapped, {W, 51, H, B}, so that its box
// {8 columns, 51 taps, rows} lands as [row][tap][col]: the per-lane register copy of the taps then hits 32 different
// banks, where as [tap][row][col] the four tap groups of a column collide in one bank.
inline bool make_v3_tap_maps(CUtensorMap* mv, CUtensorMap* mh, const float* v, const float* h, int64_t B, int H, int W, int rows) {
    const int64_t plane = (int64_t)H * W;
    const int64_t vdims[4] = {W, H, K51, B}, vstrides[4] = {1, W, plane, K51 * plane};
    const int64_t hdims[4] = {W, K51, H, B}, hstrides[4] = {1, plane, W, K51 * plane};
    const int vbox[4] = {V3_COLS, rows, V3_GROUP, 1}, hbox[4] = {V3_COLS, K51, rows, 1};
    return make_map_f32(mv, v, 4, vdims, vstrides, vbox) && make_map_f32(mh, h, 4, hdims, hstrides, hbox);
}

// Launches a persistent grid of Kern: two CTAs per SM, fewer when there are fewer CTA tiles.  Templated on the kernel
// itself, not its type: every kernel needs its own PerDeviceOnce, or only the first would get its shared-memory size.
template <auto Kern, class... Args>
int launch_persistent(size_t smem, int ntiles, cudaStream_t s, const Args&... args) {
    static PerDeviceOnce done;
    if (int e = set_smem_once(Kern, smem, done)) return e;
    const int ctas = (int)std::min<int64_t>(2 * (int64_t)sm_count(), (int64_t)ntiles);
    Kern<<<ctas, V3_WARPS * 32, smem, s>>>(args..., g_gate.ptr, g_gate.want);
    count_launch();
    return finish_launch();
}

// When a 3-channel chunk on [B,51,H,W] taps runs on generation 3: `launch(sh)` runs it, or the caller gets
// PATH_NOT_APPLICABLE and runs generation 1.  The tensor maps need W % 4 == 0 and the tensors they read 16-byte aligned
// (`aligned`), the tile tickets must fit an int, and a persistent grid needs several CTA tiles per CTA to balance:
// `min_tiles`, the measured crossover, unless SSTEM_V3_MIN_TILES gives another (A/B runs, tools/sweep_small.py).  A
// launch that returns cudaErrorMemoryAllocation (no workspace; nothing of the chunk has run) or SSTEM_E_SHAPE (a tensor
// map cannot be encoded) falls back too.
template <class Launch>
int try_v3(bool aligned, int64_t B, int C, int c0, int H, int W, int rows, int64_t min_tiles, Launch launch) {
    static const char* env = getenv("SSTEM_V3_MIN_TILES");
    if (env) min_tiles = atoll(env);
    V3Shape sh;
    if ((W & 3) || !aligned || !v3_shape(sh, B, C, c0, H, W, (H + rows - 1) / rows) || sh.ntiles < min_tiles * 2 * sm_count())
        return PATH_NOT_APPLICABLE;
    const int e = launch(sh);
    return e == cudaErrorMemoryAllocation || e == SSTEM_E_SHAPE ? PATH_NOT_APPLICABLE : e;
}

}  // namespace
}  // namespace sstem
