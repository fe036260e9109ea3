// Tap producer (SURVEY 8f, N2 -- the producer side): the last layer pair of the reference's `_kernel_module`,
//     nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True)  ->  nn.Conv2d(51, 51, 3, 1, 1)
// (sff_scripts_interp/model/model_interp.py:18, 130-137; called four times per forward, :86-89), as ONE kernel that
// reads the half-resolution activations, never materialises the upsampled tensor, and writes the taps either NCHW or
// straight into the tile-major layout the consumer streams ([B][H/8][W/8][51][8][8], sstem_sepconv_forward_tiled).
//
// The reference runs this layer through cuDNN with torch's default `allow_tf32 = True`, i.e. in TF32 on the tensor
// cores; so does this kernel, hand-written for sm_100a:
//   * implicit GEMM per output tile of 16 rows x 8 columns: D[128 pixels x 64] += A_tap[128 x 56] * W_tap[64 x 56]^T for
//     the nine taps, 7 K-steps of 8 each = 63 tcgen05.mma (kind::tf32, M = 128, N = 64), accumulator in TMEM
//     (two stages of 64 columns, so the epilogue of tile i overlaps the MMAs of tile i + 1);
//   * the A operand is never gathered per tap: the upsampled 18 x 10 input patch lives in shared memory ONCE, as
//     [channel chunk of 4][patch pixel][4 channels] (16 bytes per pixel and chunk).  In the no-swizzle K-major
//     canonical layout a core matrix is 8 rows x 16 bytes, contiguous: 8 neighbouring pixels of a patch row.  The
//     descriptor of tap (dy, dx) is the same patch with its start address moved by (dy * 10 + dx) * 16 bytes,
//     stride-byte-offset = one patch row (160 B), leading-byte-offset = one chunk (2880 B)
//     (tools/microbench/umma_probe.cu checks exactly this encoding, shifted starts included);
//   * the weights of all nine taps stay resident in shared memory for the life of the CTA (118 KB, bulk copies);
//   * warp roles: 4 epilogue warps (TMEM -> registers -> + bias -> global), 1 MMA warp (uniform descriptor arithmetic,
//     one lane issues), 12 producer warps (thread = patch pixel x chunk parity: half-resolution source window ->
//     shared memory, bilinear blend with ATen's index / weight expressions, round to TF32, write the patch);
//     mbarriers between them, a persistent grid of one CTA per SM.
// Shared memory bandwidth bounds the kernel (each MMA reads 4 KB of A and 2 KB of W for 65 536 FMAs); see DESIGN 4.11
// and profiles/tapconv_r2.md.
// The backward (sstem_tap_conv3x3_backward, DESIGN 4.11b) is at the end of this file: the input gradient reuses this kernel
// on the adjoint weights, the weight gradient is tap_conv3x3_wgrad_kernel.
// The three half-resolution convolutions in front of the producer (sstem_branch_conv3x3, DESIGN 4.11c) follow the
// producer's weight packing, on the same machinery fed by TMA from a chunk-major activation layout; their backward
// (sstem_branch_conv3x3_backward, DESIGN 4.11d) runs that kernel on the adjoint weights and branch_conv3x3_wgrad_kernel.
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "tma.cuh"

namespace sstem {
namespace {

constexpr int TC_MAXC = 52;                                // input channels: 13 chunks of 4
constexpr int TC_WCHUNKS = TC_MAXC / 4;                    // 13 weight chunks per tap (+ one zero chunk shared by all taps)
constexpr int TC_CHUNKS = TC_WCHUNKS + 1;                  // 14 patch chunks = 7 K-steps of 8; chunk 13 is always zero
constexpr int TC_N = 64;                                   // output channels, padded (UMMA N)
constexpr int TC_TH = 16, TC_TW = 8;                       // output tile: 128 pixels = UMMA M
constexpr int TC_PH = TC_TH + 2, TC_PW = TC_TW + 2, TC_NPIX = TC_PH * TC_PW;   // 18 x 10 = 180
// Half-resolution source window: 11 rows x up to 7 columns are used; it is fetched with 16-byte loads (and, in an
// earlier variant, by TMA, which has the same rule), so the first column is rounded down to a multiple of 4 and 12
// columns are loaded (48-byte rows).
constexpr int TC_WIN_H = 11, TC_WIN_W = 12;
constexpr int TC_WIN_CH = TC_WIN_H * TC_WIN_W;             // 132 floats = 528 bytes per channel: [channel][row][column]
constexpr int TC_WIN_GROUPS = 2, TC_WIN_GROUP_CH = 28;     // two channel groups (chunks 0-6, 7-12; a 128-byte aligned start each)
constexpr unsigned TC_WIN_GROUP_BYTES = TC_WIN_GROUP_CH * TC_WIN_CH * 4;       // 14784
constexpr unsigned TC_WIN_GROUP_PITCH = (TC_WIN_GROUP_BYTES + 127) / 128 * 128;   // 14848
constexpr unsigned TC_W_TAP_BYTES = TC_WCHUNKS * TC_N * 16;                    // 13312
constexpr unsigned TC_W_ZERO_OFF = 9 * TC_W_TAP_BYTES;                         // 119808: the zero chunk
constexpr unsigned TC_W_BYTES = TC_W_ZERO_OFF + TC_N * 16;                     // 120832
constexpr unsigned TC_A_BYTES = TC_CHUNKS * TC_NPIX * 16;                      // 40320
constexpr unsigned TC_WIN_BYTES = TC_WIN_GROUPS * TC_WIN_GROUP_PITCH;          // 29696
constexpr unsigned TC_OFF_A = TC_W_BYTES;
constexpr unsigned TC_OFF_WIN = TC_OFF_A + 2 * TC_A_BYTES;
constexpr unsigned TC_OFF_BIAS = TC_OFF_WIN + TC_WIN_BYTES;
constexpr unsigned TC_OFF_BAR = TC_OFF_BIAS + TC_N * 4;
constexpr unsigned TC_SMEM = TC_OFF_BAR + 128 + 128;       // + barriers + alignment slack = 231 680 (of 232 448)
static_assert(TC_SMEM <= 232448, "shared memory budget");
constexpr int TC_EPI_WARPS = 4, TC_PROD_WARPS = 12;
constexpr int TC_THREADS = (TC_EPI_WARPS + 1 + TC_PROD_WARPS) * 32;            // 544
constexpr int TC_PROD_THREADS = TC_PROD_WARPS * 32;                            // 384 = 2 x 192: (patch pixel, chunk parity)
constexpr int TC_PIX_THREADS = TC_PROD_THREADS / 2;                            // 192 >= 180 patch pixels
constexpr unsigned TC_TMEM_COLS = 128;                     // two accumulator stages of 64 columns

struct TapConvShape {
    int B, cin, cout, h, w, H, W;                          // h, w: source; H, W: output (2h, 2w when upsampling)
    int tiles_x, tiles_y, ntiles;
    int k_steps;                                           // ceil(cin / 8)
    float ry, rx;                                          // align_corners scales (in - 1) / (out - 1)
};

// a wait that cannot hang the device: a protocol error traps (the launch fails loudly) instead of spinning for ever.
// try_wait suspends the thread in hardware for up to the hinted time, so a waiting role issues next to nothing.
__device__ __forceinline__ void tc_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return;
    const long long t0 = clock64();
    for (unsigned spins = 1;; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
        if (ok) return;
        if ((spins & 63u) == 0 && clock64() - t0 > 6000000000ll) __trap();   // ~3 s: a deadlock, not a slow tile
    }
}
__device__ __forceinline__ void tc_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_commit(unsigned bar) {   // arrives on `bar` when every MMA issued so far has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint64_t tc_desc(unsigned addr, unsigned lbo, unsigned sbo) {
    // K-major, no swizzle: start >> 4 | leading byte offset (next 16-byte K chunk) | stride byte offset (next 8 rows) | version 1
    return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)((lbo >> 4) & 0x3fffu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3fffu) << 32) | ((uint64_t)1 << 46);
}
// instruction descriptor of tcgen05.mma kind::tf32: D = f32, A = B = tf32, both K-major, M x N
__host__ __device__ constexpr unsigned tc_idesc_tf32(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(n >> 3) << 17) | ((unsigned)(m >> 4) << 24);
}
// D[tmem] (+)= A * B, the accumulate flag as the instruction's predicate
__device__ __forceinline__ void tc_mma(unsigned d_tmem, uint64_t da, uint64_t db, unsigned idesc, bool accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"((unsigned)accumulate) : "memory");
}
// Warp 0 allocates NCOLS columns of tensor memory and writes their address to shared memory at `slot`; every thread
// returns it after the block-wide barrier.
template <unsigned NCOLS>
__device__ __forceinline__ unsigned tmem_alloc(unsigned slot, int warp) {
    if (warp == 0) {
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "n"(NCOLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    return *reinterpret_cast<volatile unsigned*>(__cvta_shared_to_generic(slot));
}
template <unsigned NCOLS>
__device__ __forceinline__ void tmem_dealloc(unsigned tmem, int warp) {   // after every thread's last tensor-memory access
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(NCOLS));
}
__device__ __forceinline__ float to_tf32(float x) {        // round to nearest (the tensor core itself would truncate)
    unsigned u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}
__device__ __forceinline__ void sts128(unsigned addr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// columns taddr .. + 31 of the warp's 32 tensor-memory lanes, one per register; valid after tcgen05.wait::ld
__device__ __forceinline__ void tc_ld32(unsigned taddr, unsigned (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
// The M = 128 epilogues, two accumulator stages of 64 columns: wait until the stage of the CTA's tile `it` is complete
// (barriers b_accfull / b_accempty + 8 * stage), read it from the warp's lanes and release it, so the MMAs of tile
// it + 2 may start.  tmem_lanes = the TMEM base address + the warp's first lane, computed by the caller: there the
// compiler knows the range of warp = tid / 32, and computed here the address arithmetic reschedules the whole kernel.
__device__ __forceinline__ void tc_take_acc(unsigned tmem_lanes, int it, unsigned b_accfull, unsigned b_accempty,
                                            unsigned (&v)[64]) {
    const int as = it & 1;
    tc_wait(b_accfull + 8 * as, (it >> 1) & 1);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned ta = tmem_lanes + as * TC_N;
    tc_ld32(ta, reinterpret_cast<unsigned (&)[32]>(v[0]));
    tc_ld32(ta + 32, reinterpret_cast<unsigned (&)[32]>(v[32]));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    tc_arrive(b_accempty + 8 * as);
}

// The dynamic shared memory from its first 128-byte boundary: shared-window address and generic pointer.
struct AlignedSmem {
    unsigned addr;
    unsigned char* ptr;
};
__device__ __forceinline__ AlignedSmem aligned_smem() {
    extern __shared__ __align__(128) unsigned char tc_smem_raw[];
    const unsigned raw = (unsigned)__cvta_generic_to_shared(tc_smem_raw);
    const unsigned addr = (raw + 127u) & ~127u;
    return {addr, tc_smem_raw + (addr - raw)};
}

// The tiles of a persistent CTA, blockIdx.x, + gridDim.x, ..., as (tile, column, row, image).  The coordinates advance
// by a fixed (column, row) step, so the walk needs no division (two 32-bit divisions per tile and warp were 15 % of all
// instructions issued in tap_conv3x3_kernel).
struct TileIter {
    int tile, tx, ty, b;
};
struct TileWalker {
    int tiles_x, tiles_y, step_tx, step_r;
    __device__ TileWalker(int tiles_x_, int tiles_y_)
        : tiles_x(tiles_x_), tiles_y(tiles_y_), step_tx((int)gridDim.x % tiles_x_), step_r((int)gridDim.x / tiles_x_) {}
    __device__ TileIter first() const {
        TileIter t;
        t.tile = blockIdx.x;
        const int r = t.tile / tiles_x;
        t.tx = t.tile - r * tiles_x;
        t.b = r / tiles_y;
        t.ty = r - t.b * tiles_y;
        return t;
    }
    __device__ void advance(TileIter& t) const {
        t.tile += gridDim.x;
        t.tx += step_tx;
        int dr = step_r;
        if (t.tx >= tiles_x) { t.tx -= tiles_x; ++dr; }
        t.ty += dr;
        while (t.ty >= tiles_y) { t.ty -= tiles_y; ++t.b; }
    }
};

// How the producers read x.
enum class TapSrc {
    NCHW,        // [B][cin][h][w], no upsample
    TILE_MAJOR,  // [B][ceil(h/8)][ceil(w/8)][51][8][8], no upsample (cin == 51: the tap gradients of the tiled consumer, read
                 // by the input gradient of sstem_tap_conv3x3_backward); entries outside the image are never read
    UP,          // NCHW, x2 upsample folded into the producer, source window fetched element by element
    UP_VEC,      // the same with 16-byte loads: w % 4 == 0 and x 16-byte aligned
};

// TILED_OUT: the output is tile-major.  FULL: cin is 49..52, i.e. all 13 chunks exist -- the MMA and blend loops then
// have no per-chunk checks.
template <TapSrc SRC, bool TILED_OUT, bool FULL>
__global__ void __launch_bounds__(TC_THREADS, 1)
tap_conv3x3_kernel(const float* __restrict__ x, const float* __restrict__ wpacked,
                   const float* __restrict__ bias, float* __restrict__ out, const TapConvShape sh) {
    constexpr bool UPS = SRC == TapSrc::UP || SRC == TapSrc::UP_VEC, VEC = SRC == TapSrc::UP_VEC;
    const auto [base, gen] = aligned_smem();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // barriers: 0 weights, 1-2 a_full, 3-4 a_empty, 5-6 acc_full, 7-8 acc_empty; the TMEM base address after them
    const unsigned bar = base + TC_OFF_BAR;
    const unsigned b_w = bar, b_afull = bar + 8, b_aempty = bar + 24, b_accfull = bar + 40, b_accempty = bar + 56;

    if (tid == 0) {
        mbar_init(b_w, 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(b_afull + 8 * s, TC_PROD_THREADS);
            mbar_init(b_aempty + 8 * s, 1);
            mbar_init(b_accfull + 8 * s, 1);
            mbar_init(b_accempty + 8 * s, TC_EPI_WARPS * 32);
        }
        mbar_fence_init();
    }
    // zero both patches once (the chunks past cin and the pad pixels a tile never writes must be finite) and the bias pad
    for (unsigned i = tid; i < 2 * TC_A_BYTES / 16; i += TC_THREADS) sts128(base + TC_OFF_A + i * 16, 0.f, 0.f, 0.f, 0.f);
        if (tid < TC_N) reinterpret_cast<float*>(gen + TC_OFF_BIAS)[tid] = (bias != nullptr && tid < sh.cout) ? bias[tid] : 0.f;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const unsigned tmem = tmem_alloc<TC_TMEM_COLS>(bar + 96, warp);
    const TileWalker walk(sh.tiles_x, sh.tiles_y);

    if (warp < TC_EPI_WARPS) {
        // ===================== epilogue: TMEM lanes 32 * warp .. + 31 = tile pixels (row 4 * warp + lane / 8, column lane % 8)
        const float* sbias = reinterpret_cast<const float*>(gen + TC_OFF_BIAS);
        const int r = warp * 4 + (lane >> 3), c = lane & 7;
        const int64_t plane = (int64_t)sh.H * sh.W;
        const int tiles_y8 = (sh.H + 7) / 8, tiles_x8 = (sh.W + 7) / 8;
        int it = 0;
        for (TileIter ti = walk.first(); ti.tile < sh.ntiles; walk.advance(ti), ++it) {
            const int b = ti.b, Y0 = ti.ty * TC_TH, X0 = ti.tx * TC_TW;
            unsigned v[64];
            tc_take_acc(tmem + ((unsigned)(warp * 32) << 16), it, b_accfull, b_accempty, v);
            const int Y = Y0 + r, X = X0 + c;
            if (TILED_OUT) {
                // the 16 x 8 tile is two 8 x 8 blocks of the tile-major layout; a warp writes 32 consecutive floats per tap
                // (cout == 51 here).  Pad pixels of an existing block (ragged H / W) are written as zeros.
                if ((Y >> 3) < tiles_y8) {
                    float* p = out + (((int64_t)b * tiles_y8 + (Y >> 3)) * tiles_x8 + (X0 >> 3)) * (51 * 64) + (Y & 7) * 8 + c;
                    if (Y0 + TC_TH <= sh.H && X0 + TC_TW <= sh.W) {   // the whole tile is inside the image: no masks
#pragma unroll
                        for (int n4 = 0; n4 < 52; n4 += 4) {
                            const float4 b4 = *reinterpret_cast<const float4*>(sbias + n4);
                            p[(n4 + 0) * 64] = __uint_as_float(v[n4 + 0]) + b4.x;
                            p[(n4 + 1) * 64] = __uint_as_float(v[n4 + 1]) + b4.y;
                            p[(n4 + 2) * 64] = __uint_as_float(v[n4 + 2]) + b4.z;
                            if (n4 + 3 < 51) p[(n4 + 3) * 64] = __uint_as_float(v[n4 + 3]) + b4.w;
                        }
                    } else {
                        const bool ok = Y < sh.H && X < sh.W;
#pragma unroll
                        for (int n = 0; n < 51; ++n) p[n * 64] = ok ? __uint_as_float(v[n]) + sbias[n] : 0.f;
                    }
                }
            } else if (Y < sh.H && X < sh.W) {
                float* p = out + (int64_t)b * sh.cout * plane + (int64_t)Y * sh.W + X;
#pragma unroll
                for (int n = 0; n < TC_N; ++n)
                    if (n < sh.cout) p[(int64_t)n * plane] = __uint_as_float(v[n]) + sbias[n];
            }
        }
    } else if (warp == TC_EPI_WARPS) {
        // ===================== MMA issuer.  The whole warp walks the loop, so every descriptor is warp-uniform arithmetic in
        // uniform registers; one lane issues.  (Issued from inside an `if (lane == 0)` region the descriptors were
        // per-thread values moved to uniform registers one by one: ~110 cycles per MMA, 3.4x the tensor core's own time.)
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        if (lane == 0) {
            // weights: resident for the life of the CTA
            mbar_expect_tx(b_w, TC_W_BYTES);
            for (int t = 0; t < 9; ++t)
                bulk_load(base + t * TC_W_TAP_BYTES, reinterpret_cast<const char*>(wpacked) + (size_t)t * TC_W_TAP_BYTES, TC_W_TAP_BYTES, b_w);
            bulk_load(base + TC_W_ZERO_OFF, reinterpret_cast<const char*>(wpacked) + TC_W_ZERO_OFF, TC_N * 16, b_w);
        }
        __syncwarp();
        tc_wait(b_w, 0);
        constexpr unsigned idesc = tc_idesc_tf32(128, TC_N);
        // Descriptors differ only in their start-address field (units of 16 bytes, no carry out of the field: shared memory
        // addresses are < 2^18): per tap + (dy * 10 + dx) pixels for the patch, + 13 chunks for the weights; per K-step
        // + 2 chunks each.  The last K-step's second weight chunk is the zero chunk all taps share: its leading-byte
        // offset field is (zero chunk - chunk 12 of the tap) instead of one chunk.
        const uint64_t db0 = tc_desc(base, TC_N * 16, 128);
        const int k_steps = FULL ? TC_CHUNKS / 2 : sh.k_steps;
        int it = 0;
        for (int tile = blockIdx.x; tile < sh.ntiles; tile += gridDim.x, ++it) {   // (needs no coordinates)
            const int s = it & 1;
            const unsigned ph = (it >> 1) & 1;
            tc_wait(b_accempty + 8 * s, ph ^ 1);           // accumulator stage drained by the epilogue (passes at once the first time)
            tc_wait(b_afull + 8 * s, ph);                  // patch written and fenced by the producers
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t da0 = tc_desc(base + TC_OFF_A + s * TC_A_BYTES, TC_NPIX * 16, TC_PW * 16);
            const unsigned d_tmem = tmem_u + s * TC_N;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
                for (int ks = 0; ks < TC_CHUNKS / 2; ++ks) {
                    if (ks >= k_steps) break;
                    const uint64_t da = da0 + (uint64_t)((tap / 3) * TC_PW + (tap % 3) + ks * 2 * TC_NPIX);
                    uint64_t db = db0 + (uint64_t)((tap * TC_W_TAP_BYTES + ks * 2 * TC_N * 16) >> 4);
                    if (2 * ks + 1 >= TC_WCHUNKS)
                        db += (uint64_t)(((TC_W_ZERO_OFF - tap * TC_W_TAP_BYTES - ks * 2 * TC_N * 16) >> 4) - TC_N) << 16;
                    if (lane == 0) tc_mma(d_tmem, da, db, idesc, (tap | ks) != 0);
                }
            }
            __syncwarp();
            if (lane == 0) {
                tc_commit(b_aempty + 8 * s);               // patch stage may be overwritten
                tc_commit(b_accfull + 8 * s);              // accumulator complete
            }
        }
    } else {
        // ===================== producers: thread = (patch pixel, chunk parity); 180 of each 192 threads have a pixel
        const int ptid = tid - (TC_EPI_WARPS + 1) * 32;
        const int half = ptid >= TC_PIX_THREADS ? 1 : 0, pix = ptid - half * TC_PIX_THREADS;
        const int py = pix / TC_PW, px = pix % TC_PW;
        const bool has_pixel = pix < TC_NPIX;
        const int nchunks = (sh.cin + 3) >> 2;
        const int64_t src_plane = (int64_t)sh.h * sh.w;
        const unsigned win = base + TC_OFF_WIN;
        float* win_gen = reinterpret_cast<float*>(gen + TC_OFF_WIN);
        auto window_origin = [&](int Y0, int X0, int& sy0, int& sx0) {
            // PyTorch upsample_bilinear2d, align_corners = True: source index = scale * dst in float, cut to int
            sy0 = (int)(sh.ry * (float)max(Y0 - 1, 0));
            sx0 = (int)(sh.rx * (float)max(X0 - 1, 0)) & ~3;       // 16-byte aligned rows
        };
        // The window of tile i + 1 is fetched into registers while tile i's patch is computed (a whole tile of lookahead hides
        // the L2 / DRAM latency) and moves to shared memory once every producer is done reading the previous window.  A TMA
        // box per channel group was tried first: its 48-byte rows cost ~2 us per box and shared memory has no room for a
        // second window, so half of that latency stayed exposed (0.85 ms vs the register prefetch, see DESIGN 4.11).
        constexpr int ROW4 = TC_WIN_W / 4;                 // 16-byte pieces per window row: 3
        constexpr int NFILL = VEC ? (TC_MAXC * TC_WIN_H * ROW4 + TC_PROD_THREADS - 1) / TC_PROD_THREADS      // 5 x float4
                                   : (TC_MAXC * TC_WIN_CH + TC_PROD_THREADS - 1) / TC_PROD_THREADS;          // 18 x float
        float4 pre4[VEC ? NFILL : 1];
        float pre[VEC ? 1 : NFILL];
        // VEC: which 16-byte piece this thread fetches in round k does not depend on the tile: its channel offset (elements;
        // the host checks cin * h * w < 2^31), window row and column piece are computed once
        int f_choff[VEC ? NFILL : 1], f_wy[VEC ? NFILL : 1], f_c4[VEC ? NFILL : 1], f_dst[VEC ? NFILL : 1];
        if (VEC) {
#pragma unroll
            for (int k = 0; k < NFILL; ++k) {
                const int i = ptid + k * TC_PROD_THREADS;
                const int ch = i / (TC_WIN_H * ROW4), rem = i - ch * (TC_WIN_H * ROW4);
                f_wy[k] = rem / ROW4;
                f_c4[k] = 4 * (rem - f_wy[k] * ROW4);
                f_choff[k] = ch < sh.cin ? ch * (int)src_plane : -1;
                const int g = ch >= TC_WIN_GROUP_CH ? 1 : 0;
                f_dst[k] = ch < TC_MAXC ? (int)(g * TC_WIN_GROUP_PITCH + (ch - g * TC_WIN_GROUP_CH) * (TC_WIN_CH * 4) + rem * 16) : -1;
            }
        }
        auto load_window = [&](const TileIter& t) {
            int sy0, sx0;
            window_origin(t.ty * TC_TH, t.tx * TC_TW, sy0, sx0);
            const float* xb = x + (int64_t)t.b * sh.cin * src_plane;
#pragma unroll
            for (int k = 0; k < NFILL; ++k) {
                const int i = ptid + k * TC_PROD_THREADS;
                if (VEC) {
                    const int gy = min(sy0 + f_wy[k], sh.h - 1), gx = sx0 + f_c4[k];   // columns past the edge are never blended in
                    pre4[k] = (f_choff[k] >= 0 && gx < sh.w) ? __ldg(reinterpret_cast<const float4*>(xb + (f_choff[k] + gy * sh.w + gx)))
                                                             : make_float4(0.f, 0.f, 0.f, 0.f);
                } else {
                    const int ch = i / TC_WIN_CH, p = i - ch * TC_WIN_CH;
                    const int wy = p / TC_WIN_W, wx = p - wy * TC_WIN_W;
                    const int gy = min(sy0 + wy, sh.h - 1), gx = min(sx0 + wx, sh.w - 1);
                    pre[k] = ch < sh.cin ? __ldg(xb + (int64_t)ch * src_plane + (int64_t)gy * sh.w + gx) : 0.f;
                }
            }
        };
        auto store_window = [&]() {
#pragma unroll
            for (int k = 0; k < NFILL; ++k) {
                const int i = ptid + k * TC_PROD_THREADS;
                if (VEC) {
                    if (f_dst[k] >= 0) sts128(win + f_dst[k], pre4[k].x, pre4[k].y, pre4[k].z, pre4[k].w);
                } else {
                    const int ch = i / TC_WIN_CH, p = i - ch * TC_WIN_CH;
                    const int g = ch >= TC_WIN_GROUP_CH ? 1 : 0;
                    if (ch < TC_MAXC) win_gen[g * (TC_WIN_GROUP_PITCH / 4) + (ch - g * TC_WIN_GROUP_CH) * TC_WIN_CH + p] = pre[k];
                }
            }
        };
        TileIter ti = walk.first(), tn = ti;               // this tile and the next one of this CTA
        walk.advance(tn);
        if (UPS && ti.tile < sh.ntiles) load_window(ti);
        // per-thread constants of the blend: chunk parity folded into the base addresses, so every shared-memory offset
        // below is an immediate
        const unsigned half_win = half * 4 * (TC_WIN_CH * 4), half_dst = half * TC_NPIX * 16;
        int it = 0;
        for (; ti.tile < sh.ntiles; ti = tn, walk.advance(tn), ++it) {
            const int s = it & 1;
            const unsigned ph = (it >> 1) & 1;
            const int b = ti.b, Y0 = ti.ty * TC_TH, X0 = ti.tx * TC_TW;
            const int Y = Y0 - 1 + py, X = X0 - 1 + px;
            const bool inside = has_pixel && Y >= 0 && Y < sh.H && X >= 0 && X < sh.W;   // outside: the convolution's zero padding
            const unsigned a_dst = base + TC_OFF_A + s * TC_A_BYTES + pix * 16 + half_dst;
            const bool has_next = tn.tile < sh.ntiles;
            if (UPS) {
                int sy0, sx0;
                window_origin(Y0, X0, sy0, sx0);
                // neighbour = + 1 unless at the last row / column; weights from the fraction.  The four weights are multiplied
                // out first (ATen nests them); the difference is an fp32 rounding, far below the TF32 rounding that follows.
                const float h1r = sh.ry * (float)Y, w1r = sh.rx * (float)X;
                const int h1 = (int)h1r, w1 = (int)w1r;
                const int h1p = h1 < sh.h - 1 ? 1 : 0, w1p = w1 < sh.w - 1 ? 1 : 0;
                const float h1l = h1r - (float)h1, h0l = 1.f - h1l, w1l = w1r - (float)w1, w0l = 1.f - w1l;
                const float wa = h0l * w0l, wb = h0l * w1l, wc = h1l * w0l, wd = h1l * w1l;
                const int cell = min(max(h1 - sy0, 0), TC_WIN_H - 2) * TC_WIN_W + min(max(w1 - sx0, 0), TC_WIN_W - 2);
                const unsigned a00 = win + cell * 4 + half_win, a01 = a00 + w1p * 4, a10 = a00 + h1p * TC_WIN_W * 4, a11 = a10 + w1p * 4;
                asm volatile("bar.sync 2, %0;" ::"n"(TC_PROD_THREADS) : "memory");   // everyone is done reading the previous window
                store_window();
                asm volatile("bar.sync 2, %0;" ::"n"(TC_PROD_THREADS) : "memory");
                if (has_next) load_window(tn);
                tc_wait(b_aempty + 8 * s, ph ^ 1);         // the MMAs that read this patch stage two tiles ago are complete
#pragma unroll
                for (int g = 0; g < TC_WIN_GROUPS; ++g) {
                    if (has_pixel) {
                        // this thread's chunks of the group: 7 g + half + 2 k.  With 13 chunks (cin 49..52, FULL) that is
                        // k < 3, plus k = 3 for the even chunks of group 0; otherwise each chunk is checked against cin.
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int ck = g * (TC_CHUNKS / 2) + half + 2 * k;
                            const bool mine = FULL ? (k < 3 || (g == 0 && half == 0)) : (ck < (g + 1) * (TC_CHUNKS / 2) && ck < nchunks);
                            if (!mine) continue;
                            const unsigned dst = a_dst + (g * (TC_CHUNKS / 2) + 2 * k) * TC_NPIX * 16;
                            if (inside) {
                                float q[4];
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    const unsigned o = g * TC_WIN_GROUP_PITCH + (unsigned)(8 * k + j) * (TC_WIN_CH * 4);
                                    q[j] = to_tf32(wa * lds_f32(a00 + o) + wb * lds_f32(a01 + o) + wc * lds_f32(a10 + o) + wd * lds_f32(a11 + o));
                                }
                                sts128(dst, q[0], q[1], q[2], q[3]);
                            } else {
                                sts128(dst, 0.f, 0.f, 0.f, 0.f);
                            }
                        }
                    }
                }
            } else {
                const float* xb = x + (int64_t)b * sh.cin * src_plane;
                tc_wait(b_aempty + 8 * s, ph ^ 1);
                if (has_pixel) {
                    // the pixel's channels: tile-major (cin == 51, 13 chunks) at a stride of 64, NCHW at a stride of one plane
                    const int Yc = min(max(Y, 0), sh.H - 1), Xc = min(max(X, 0), sh.W - 1);
                    const float* xp = SRC == TapSrc::TILE_MAJOR
                        ? x + ((((int64_t)b * ((sh.H + 7) >> 3) + (Yc >> 3)) * ((sh.W + 7) >> 3) + (Xc >> 3)) * (51 * 64) + (Yc & 7) * 8 + (Xc & 7))
                        : xb + (int64_t)Yc * sh.W + Xc;
#pragma unroll 1
                    for (int ck0 = half; ck0 < nchunks; ck0 += 8) {    // chunks half, half + 2, ...: 16 independent loads in flight per thread
                        const unsigned dst0 = a_dst - half_dst;
                        float q[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int ch = (ck0 + 2 * (j >> 2)) * 4 + (j & 3);
                            q[j] = (inside && ch < sh.cin) ? __ldg(xp + (SRC == TapSrc::TILE_MAJOR ? ch * 64 : (int64_t)ch * src_plane)) : 0.f;
                        }
#pragma unroll
                        for (int c4 = 0; c4 < 4; ++c4)
                            if (ck0 + 2 * c4 < nchunks)
                                sts128(dst0 + (ck0 + 2 * c4) * TC_NPIX * 16, to_tf32(q[4 * c4]), to_tf32(q[4 * c4 + 1]), to_tf32(q[4 * c4 + 2]), to_tf32(q[4 * c4 + 3]));
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core's reads
            tc_arrive(b_afull + 8 * s);
        }
    }

    tmem_dealloc<TC_TMEM_COLS>(tmem, warp);
}

// Weights [cout][cin][3][3] -> [tap][chunk < CHUNKS][n = 64][4], zero padded, rounded to TF32; ZERO_CHUNK: followed by
// one zero chunk (the producer's, 13 chunks per tap, shared by all taps; the branch has 16 chunks and none).  ADJOINT:
// the image of W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx] instead, the convolution from cout to cin channels that the
// input gradient runs.
__host__ __device__ constexpr int packed_floats(int chunks, bool zero_chunk) { return (9 * chunks + (zero_chunk ? 1 : 0)) * TC_N * 4; }
static_assert(packed_floats(TC_WCHUNKS, true) == (int)(TC_W_BYTES / 4), "tap producer weight image");

template <bool ADJOINT, int CHUNKS, bool ZERO_CHUNK>
__global__ void conv3x3_pack_kernel(const float* __restrict__ w, float* __restrict__ packed, int cin, int cout) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= packed_floats(CHUNKS, ZERO_CHUNK)) return;
    if (ZERO_CHUNK && i >= 9 * CHUNKS * TC_N * 4) { packed[i] = 0.f; return; }
    const int j = i & 3, n = (i >> 2) % TC_N, ck = (i >> 2) / TC_N % CHUNKS, tap = (i >> 2) / TC_N / CHUNKS;
    const int ch = ck * 4 + j;                             // input channel of the packed convolution
    if (ADJOINT)                                           // W'[n][ch][tap] = W[ch][n][8 - tap]
        packed[i] = (n < cin && ch < cout) ? to_tf32(w[((int64_t)ch * cin + n) * 9 + (8 - tap)]) : 0.f;
    else
        packed[i] = (n < cout && ch < cin) ? to_tf32(w[((int64_t)n * cin + ch) * 9 + tap]) : 0.f;
}

// One persistent launch.  Templated on the kernel itself: every kernel needs its own PerDeviceOnce, or only the first
// would get its shared-memory size.
template <auto Kern, class... Args>
int launch_tc(unsigned smem, int threads, int ctas, cudaStream_t s, const Args&... args) {
    static PerDeviceOnce done;
    int dev = 0;
    cudaGetDevice(&dev);
    if (!done.test(dev)) {
        if (cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return (int)cudaGetLastError();
        done.set(dev);
    }
    Kern<<<ctas, threads, smem, s>>>(args...);
    count_launch();
    return finish_launch();
}

// The elementwise and reduction kernels: `blocks` blocks of 256 threads.
template <auto Kern, class... Args>
int launch256(int64_t blocks, cudaStream_t s, const Args&... args) {
    Kern<<<(unsigned)blocks, 256, 0, s>>>(args...);
    count_launch();
    return finish_launch();
}

template <TapSrc SRC>
int launch_tap_conv(bool tiled_out, bool full, const float* x, const float* wpacked, const float* bias, float* out,
                    const TapConvShape& sh, cudaStream_t s) {
    const int ctas = std::min(sh.ntiles, sm_count());
    if (tiled_out)
        return full ? launch_tc<tap_conv3x3_kernel<SRC, true, true>>(TC_SMEM, TC_THREADS, ctas, s, x, wpacked, bias, out, sh)
                    : launch_tc<tap_conv3x3_kernel<SRC, true, false>>(TC_SMEM, TC_THREADS, ctas, s, x, wpacked, bias, out, sh);
    return full ? launch_tc<tap_conv3x3_kernel<SRC, false, true>>(TC_SMEM, TC_THREADS, ctas, s, x, wpacked, bias, out, sh)
                : launch_tc<tap_conv3x3_kernel<SRC, false, false>>(TC_SMEM, TC_THREADS, ctas, s, x, wpacked, bias, out, sh);
}

// tap_conv3x3_kernel for (source layout, output layout, all 13 chunks).  A tile-major source is only the input
// gradient's: 51 channels (FULL), NCHW output.
int launch_tap_conv(TapSrc src, bool tiled_out, bool full, const float* x, const float* wpacked, const float* bias, float* out,
                    const TapConvShape& sh, cudaStream_t s) {
    switch (src) {
    case TapSrc::NCHW: return launch_tap_conv<TapSrc::NCHW>(tiled_out, full, x, wpacked, bias, out, sh, s);
    case TapSrc::UP: return launch_tap_conv<TapSrc::UP>(tiled_out, full, x, wpacked, bias, out, sh, s);
    case TapSrc::UP_VEC: return launch_tap_conv<TapSrc::UP_VEC>(tiled_out, full, x, wpacked, bias, out, sh, s);
    default: return launch_tc<tap_conv3x3_kernel<TapSrc::TILE_MAJOR, false, true>>(TC_SMEM, TC_THREADS, std::min(sh.ntiles, sm_count()),
                                                                                   s, x, wpacked, bias, out, sh);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Backward of y = conv3x3(up(x), W) + b (sstem_tap_conv3x3_backward).
//
// grad_x = up^T(conv3x3(gy, W')), W'[ci][co][ky][kx] = W[co][ci][2-ky][2-kx]: the convolution is tap_conv3x3_kernel on its
// no-upsample path (weights packed by the ADJOINT conv3x3_pack_kernel), up^T is the gather below.

// Weight with which output row (column) Y of the align_corners upsample reads source row i: ATen's float32 index and
// fraction, as the forward producer computes them.  At the last row the neighbour is the row itself (both weights land
// on it); with one source row the scale is 0 and every output row reads row 0.
__device__ __forceinline__ float up_adjoint_weight(int Y, int i, int n_in, int n_out, float r) {
    if (Y < 0 || Y >= n_out) return 0.f;
    const float fr = r * (float)Y;
    const int i0 = (int)fr, i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
    const float l1 = fr - (float)i0, l0 = 1.f - l1;
    return (i0 == i ? l0 : 0.f) + (i1 == i ? l1 : 0.f);
}

// grad_x[p][i][j] = sum_Y sum_X wy(Y, i) wx(X, j) gU[p][Y][X] as a gather (no atomics: deterministic).  The output rows that
// read source row i lie in [2i - 3, 2i + 4] (the scale (h - 1) / (2h - 1) is just below 1/2); weights of rows that do not
// read it are 0 and skip their loads.
__global__ void __launch_bounds__(256)
upsample2x_adjoint_kernel(const float* __restrict__ gU, float* __restrict__ gx, int64_t n, int h, int w, int H, int W,
                          float ry, float rx) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n) return;
    const int j = (int)(idx % w), i = (int)(idx / w % h);
    const float* g = gU + idx / ((int64_t)h * w) * ((int64_t)H * W);
    float wx[8];
#pragma unroll
    for (int d = 0; d < 8; ++d) wx[d] = up_adjoint_weight(2 * j - 3 + d, j, w, W, rx);
    float acc = 0.f;
#pragma unroll
    for (int dy = 0; dy < 8; ++dy) {
        const int Y = 2 * i - 3 + dy;
        const float wy = up_adjoint_weight(Y, i, h, H, ry);
        if (wy == 0.f) continue;
        float row = 0.f;
#pragma unroll
        for (int dx = 0; dx < 8; ++dx)
            if (wx[dx] != 0.f) row += wx[dx] * __ldg(g + (int64_t)Y * W + (2 * j - 3 + dx));
        acc += wy * row;
    }
    gx[idx] = acc;
}

// grad_weight / grad_bias.  Per output tile of 16 x 8 pixels and tap (dy, dx):
//     D_tap[co][ci] += sum_{pixels p} gy[co][p] * U[ci][p + (dy, dx)]            (U = up(x), zero padded by 1)
// as tcgen05.mma kind::tf32, M = 64 (co, padded), N = 56 (ci, padded), K = 8 = one row of the tile: 16 K-steps x 9 taps =
// 144 MMAs per tile, the nine accumulators (9 x 56 = 504 TMEM columns) resident for the whole tile loop.  Both operands
// are K-major, no swizzle (the encoding tapconv's forward and tools/microbench/umma_probe.cu pin down):
//   * A = gy of the tile: [tile row][K half][co group of 8][8 co][4 pixels], one K-step = one tile row (2 KB);
//   * B = the upsampled, TF32-rounded 18 x 10 patch, recomputed from x, as three copies shifted by dx = 0, 1, 2 columns:
//     [dx][patch row][K half][ci group of 8][8 ci][4 pixels].  Tap (dy, dx), K-step ky reads copy dx at patch row
//     ky + dy: a start-address shift of one 1792-byte row per dy.
// One stage: all 12 warps stage a tile, warp 0 issues its 144 MMAs, and the staging of the next tile waits for their
// completion (tcgen05.commit).  gy is summed per output channel on the way (grad_bias).  Each CTA writes one partial of
// both gradients at the end; sum_partials_kernel sums the partials over CTAs in a fixed order, so the result
// is run-to-run bit-identical.
constexpr int WG_THREADS = 384;
constexpr int WG_M = 64, WG_N = 56;
constexpr int WG_CO_PER_THREAD = 18;                       // output channels cgrp, cgrp + 3, ..., cgrp + 51 (cout <= 52)
constexpr unsigned WG_A_ROW = 2 * (WG_M / 8) * 128;        // 2048
constexpr unsigned WG_A_BYTES = TC_TH * WG_A_ROW;          // 32768
constexpr unsigned WG_B_ROW = 2 * (WG_N / 8) * 128;        // 1792
constexpr unsigned WG_B_COPY = TC_PH * WG_B_ROW;           // 32256
constexpr unsigned WG_OFF_B = WG_A_BYTES;
constexpr unsigned WG_OFF_BAR = WG_OFF_B + 3 * WG_B_COPY;  // 129536
constexpr unsigned WG_SMEM = WG_OFF_BAR + 16 + 128;
constexpr unsigned WG_TMEM_COLS = 512;
static_assert(9 * WG_N <= (int)WG_TMEM_COLS, "nine accumulators in tensor memory");
static_assert(WG_THREADS * WG_CO_PER_THREAD * 4 <= WG_OFF_BAR, "the bias reduction reuses the operand buffers");

// GY_TILED: gy is tile-major (cout == 51)
template <bool UPS, bool GY_TILED>
__global__ void __launch_bounds__(WG_THREADS, 1)
tap_conv3x3_wgrad_kernel(const float* __restrict__ gy, const float* __restrict__ x, float* __restrict__ part_w,
                         float* __restrict__ part_b, const TapConvShape sh) {
    const auto [base, gen] = aligned_smem();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned bar = base + WG_OFF_BAR;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    // padding rows / columns of both operands stay zero
    for (unsigned i = tid; i < WG_OFF_BAR / 16; i += WG_THREADS) sts128(base + i * 16, 0.f, 0.f, 0.f, 0.f);
    const unsigned tmem = tmem_alloc<WG_TMEM_COLS>(bar + 8, warp);

    // A staging: thread = (tile pixel, output-channel class); B staging: thread = (patch pixel, input-channel half)
    const int apx = tid & 127, acg = tid >> 7, ay = apx >> 3, ax = apx & 7;
    const unsigned a_dst = base + (unsigned)(ay * 2 + (ax >> 2)) * 8 * 128 + (ax & 3) * 4;
    const bool bitem = tid < 2 * TC_NPIX;
    const int bhalf = tid >= TC_NPIX ? 1 : 0, bpix = tid - bhalf * TC_NPIX, bpy = bpix / TC_PW, bpx = bpix % TC_PW;
    const int64_t plane = (int64_t)sh.H * sh.W, src_plane = (int64_t)sh.h * sh.w;
    const int tiles_y8 = (sh.H + 7) / 8, tiles_x8 = (sh.W + 7) / 8;
    float bacc[WG_CO_PER_THREAD];
#pragma unroll
    for (int k = 0; k < WG_CO_PER_THREAD; ++k) bacc[k] = 0.f;
    constexpr unsigned idesc = tc_idesc_tf32(WG_M, WG_N);

    int it = 0;
    for (int tile = blockIdx.x; tile < sh.ntiles; tile += gridDim.x, ++it) {
        const int r = tile / sh.tiles_x, tx = tile - r * sh.tiles_x, b = r / sh.tiles_y, ty = r - b * sh.tiles_y;
        const int Y0 = ty * TC_TH, X0 = tx * TC_TW;
        if (it > 0) {
            tc_wait(bar, (it - 1) & 1);                    // the MMAs of the previous tile have read the operands
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        {   // A: gy of the tile, and its per-channel sum
            const int Y = Y0 + ay, X = X0 + ax;
            const bool inside = Y < sh.H && X < sh.W;
            const float* g = GY_TILED ? gy + ((((int64_t)b * tiles_y8 + (Y >> 3)) * tiles_x8 + (X >> 3)) * (51 * 64) + (Y & 7) * 8 + (X & 7))
                                   : gy + (int64_t)b * sh.cout * plane + (int64_t)Y * sh.W + X;
            const int64_t cstride = GY_TILED ? 64 : plane;
#pragma unroll
            for (int k = 0; k < WG_CO_PER_THREAD; ++k) {
                const int co = acg + 3 * k;
                const float v = (inside && co < sh.cout) ? __ldg(g + co * cstride) : 0.f;
                bacc[k] += v;
                if (co < WG_M) asm volatile("st.shared.f32 [%0], %1;" ::"r"(a_dst + (co >> 3) * 128 + (co & 7) * 16), "f"(to_tf32(v)) : "memory");
            }
        }
        if (bitem) {   // B: the upsampled patch pixel, written into the (up to) three shifted copies that hold it
            const int Y = Y0 - 1 + bpy, X = X0 - 1 + bpx;
            const bool inside = Y >= 0 && Y < sh.H && X >= 0 && X < sh.W;
            int o00 = 0, o01 = 0, o10 = 0, o11 = 0;
            float wa = 0.f, wb = 0.f, wc = 0.f, wd = 0.f;
            if (UPS && inside) {
                const float h1r = sh.ry * (float)Y, w1r = sh.rx * (float)X;
                const int h1 = (int)h1r, w1 = (int)w1r;
                const int h1p = h1 < sh.h - 1 ? 1 : 0, w1p = w1 < sh.w - 1 ? 1 : 0;
                const float h1l = h1r - (float)h1, h0l = 1.f - h1l, w1l = w1r - (float)w1, w0l = 1.f - w1l;
                wa = h0l * w0l; wb = h0l * w1l; wc = h1l * w0l; wd = h1l * w1l;
                o00 = h1 * sh.w + w1; o01 = o00 + w1p; o10 = o00 + h1p * sh.w; o11 = o10 + w1p;
            } else if (inside) {
                o00 = Y * sh.w + X;
            }
            const float* xb = x + (int64_t)b * sh.cin * src_plane;
            const unsigned bdst = base + WG_OFF_B + bpy * WG_B_ROW;
#pragma unroll 4
            for (int k = 0; k < WG_N / 2; ++k) {
                const int ci = bhalf * (WG_N / 2) + k;
                float v = 0.f;
                if (inside && ci < sh.cin) {
                    const float* p = xb + ci * src_plane;
                    v = UPS ? wa * __ldg(p + o00) + wb * __ldg(p + o01) + wc * __ldg(p + o10) + wd * __ldg(p + o11) : __ldg(p + o00);
                }
                v = to_tf32(v);
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const int c = bpx - dx;
                    if (c >= 0 && c < TC_TW)
                        asm volatile("st.shared.f32 [%0], %1;" ::"r"(bdst + dx * WG_B_COPY + ((c >> 2) * (WG_N / 8) + (ci >> 3)) * 128 + (ci & 7) * 16 + (c & 3) * 4),
                                     "f"(v) : "memory");
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (warp == 0) {
            // the whole warp walks the loop (descriptors in uniform registers), one lane issues
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t da0 = tc_desc(base, WG_A_ROW / 2, 128);
            const uint64_t db0 = tc_desc(base + WG_OFF_B, WG_B_ROW / 2, 128);
#pragma unroll 1
            for (int tap = 0; tap < 9; ++tap) {
                const int dy = tap / 3, dx = tap % 3;
                const unsigned d_tmem = tmem + tap * WG_N;
#pragma unroll
                for (int ky = 0; ky < TC_TH; ++ky) {
                    const uint64_t da = da0 + (uint64_t)((ky * WG_A_ROW) >> 4);
                    const uint64_t db = db0 + (uint64_t)((dx * WG_B_COPY + (ky + dy) * WG_B_ROW) >> 4);
                    if (lane == 0) tc_mma(d_tmem, da, db, idesc, (it | ky) != 0);
                }
            }
            __syncwarp();
            if (lane == 0) tc_commit(bar);
            __syncwarp();
        }
    }
    if (it > 0) {
        tc_wait(bar, (it - 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    __syncthreads();

    const int nw = sh.cout * sh.cin * 9;
    if (warp < 4) {
        // M = 64: row m of D is TMEM lane 32 (m / 16) + m % 16 (tools/microbench/umma_probe.cu, mode m64), so warp q reads
        // rows 16 q .. 16 q + 15 in its lanes 0..15
        const int co = warp * 16 + lane;
        const bool mine = lane < 16 && co < sh.cout;
        float* pw = part_w + (int64_t)blockIdx.x * nw + (int64_t)co * sh.cin * 9;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
#pragma unroll 1
            for (int c8 = 0; c8 < WG_N; c8 += 8) {
                unsigned v[8];
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                             : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                             : "r"(tmem + ((unsigned)(warp * 32) << 16) + tap * WG_N + c8));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (mine) {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (c8 + j < sh.cin) pw[(c8 + j) * 9 + tap] = __uint_as_float(v[j]);
                }
            }
        }
    }
    // grad_bias partial: thread sums in shared memory (the operand buffers are free), then per channel in pixel order
    float* red = reinterpret_cast<float*>(gen);
#pragma unroll
    for (int k = 0; k < WG_CO_PER_THREAD; ++k) red[tid * WG_CO_PER_THREAD + k] = bacc[k];
    __syncthreads();
    if (tid < sh.cout) {
        const int cg = tid % 3, k = tid / 3;
        float sum = 0.f;
        for (int p = 0; p < 128; ++p) sum += red[(cg * 128 + p) * WG_CO_PER_THREAD + k];
        part_b[(int64_t)blockIdx.x * sh.cout + tid] = sum;
    }
    tmem_dealloc<WG_TMEM_COLS>(tmem, warp);
}

// sum of the partials of both weight-gradient kernels and of branch_grad_mask_kernel, in CTA / block order
// (deterministic); out[i] for i < n, NULL outputs skipped
__global__ void sum_partials_kernel(const float* __restrict__ part_w, const float* __restrict__ part_b,
                                    float* __restrict__ gw, float* __restrict__ gb, int nw, int nb, int parts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const float* src;
    float* dst;
    int n;
    if (i < nw) { src = part_w + i; dst = gw ? gw + i : nullptr; n = nw; }
    else if (i < nw + nb) { src = part_b + (i - nw); dst = gb ? gb + (i - nw) : nullptr; n = nb; }
    else return;
    if (!dst) return;
    float s = 0.f;
    for (int c = 0; c < parts; ++c) s += src[(int64_t)c * n];
    *dst = s;
}

// (h, w): the source; the output is (2h, 2w) with the upsample.  The callers have checked that the tile count fits.
TapConvShape tap_conv_shape(int64_t B, int cin, int cout, int64_t h, int64_t w, bool ups) {
    TapConvShape sh;
    sh.B = (int)B; sh.cin = cin; sh.cout = cout; sh.h = (int)h; sh.w = (int)w;
    sh.H = ups ? 2 * (int)h : (int)h;
    sh.W = ups ? 2 * (int)w : (int)w;
    sh.tiles_x = (sh.W + TC_TW - 1) / TC_TW;
    sh.tiles_y = (sh.H + TC_TH - 1) / TC_TH;
    sh.ntiles = (int)((int64_t)sh.tiles_x * sh.tiles_y * B);
    sh.k_steps = (cin + 7) / 8;
    sh.ry = sh.H > 1 ? (float)(sh.h - 1) / (float)(sh.H - 1) : 0.f;
    sh.rx = sh.W > 1 ? (float)(sh.w - 1) / (float)(sh.W - 1) : 0.f;
    return sh;
}

// Every pack entry point: conv3x3_pack_kernel for one weight image, within that entry point's channel limits.
template <bool ADJOINT, int CHUNKS, bool ZERO_CHUNK>
int pack_weights(const float* weight, float* packed, int cin, int cout, int max_cin, int max_cout, void* stream) {
    if (!weight || !packed) return SSTEM_E_NULL;
    if (cin <= 0 || cin > max_cin || cout <= 0 || cout > max_cout) return SSTEM_E_SHAPE;
    if (!aligned4(weight) || !aligned16(packed)) return SSTEM_E_ALIGN;
    DeviceGuard guard(packed);
    if (guard.err) return guard.err;
    return launch256<conv3x3_pack_kernel<ADJOINT, CHUNKS, ZERO_CHUNK>>((packed_floats(CHUNKS, ZERO_CHUNK) + 255) / 256,
                                                                       (cudaStream_t)stream, weight, packed, cin, cout);
}

// Image bounds of every entry point
bool image_fits(int64_t B, int64_t h, int64_t w) { return B > 0 && h > 0 && w > 0 && h <= (1 << 22) && w <= (1 << 22); }

// 16 x 8 output tiles of B images of H x W
int64_t tile_count(int64_t B, int64_t H, int64_t W) { return ((W + TC_TW - 1) / TC_TW) * ((H + TC_TH - 1) / TC_TH) * B; }

// ---------------------------------------------------------------------------------------------------------------------
// Tap branch convolutions (sstem_branch_conv3x3, DESIGN 4.11c): the three half-resolution layers in front of the
// producer, Conv2d(cin <= 64, cout <= 64, 3, 1, 1) -> ReLU, on the producer's operand encoding.  Activations between the
// layers are chunk-major, [B][C8/4][h][w][4] (C8 = channels rounded up to 8; padding channels 0), already rounded to TF32,
// so the patch needs no producer warps: one TMA box {40 floats = 10 pixels x 4 channels, 18 rows, 4 chunks} of that
// layout lands as [chunk][patch pixel][4], the canonical K-major operand of tap_conv3x3_kernel, and its out-of-image part
// is zero-filled, which is the convolution's zero padding.  Roles: 4 epilogue warps (TMEM -> + bias -> ReLU -> store), 1
// MMA warp (walks the loop uniformly, one lane issues), 1 warp whose lane 0 issues the bulk / TMA copies.
constexpr int BC_MAXC = 64;
constexpr int BC_CHUNKS = BC_MAXC / 4;                     // 16 weight chunks per tap
constexpr int BC_SLOT_CHUNKS = 4;                          // a ring slot holds a quarter of a 64-channel patch: 2 K-steps
constexpr int BC_SLOTS = 6;                                // 1.5 tiles of 64-channel patches in flight
constexpr unsigned BC_W_TAP_BYTES = BC_CHUNKS * TC_N * 16;                     // 16384
constexpr unsigned BC_W_BYTES = 9 * BC_W_TAP_BYTES;                            // 147456
constexpr unsigned BC_SLOT_BYTES = BC_SLOT_CHUNKS * TC_NPIX * 16;              // 11520
constexpr unsigned BC_OFF_A = BC_W_BYTES;
constexpr unsigned BC_OFF_BIAS = BC_OFF_A + BC_SLOTS * BC_SLOT_BYTES;          // 216576
constexpr unsigned BC_OFF_BAR = BC_OFF_BIAS + TC_N * 4;
constexpr unsigned BC_SMEM = BC_OFF_BAR + 256 + 128;       // + barriers and the TMEM address + alignment slack = 217 216
static_assert(BC_SMEM <= 232448, "shared memory budget");
static_assert(8 * (1 + 2 * BC_SLOTS + 4) + 4 <= 256, "barrier block");
static_assert(packed_floats(BC_CHUNKS, false) == (int)(BC_W_BYTES / 4), "branch weight image");
constexpr int BC_THREADS = (TC_EPI_WARPS + 2) * 32;        // 192

struct BranchConvShape {
    int h, w, cout;
    int tiles_x, tiles_y, ntiles;
    int in_chunks, out_chunks;                             // C8 / 4 of the input and of the output
    int k_steps;                                           // C8in / 8
    int slots_per_tile;                                    // ceil(k_steps / 2)
    int relu;
    int cin;
    int halves;                                            // weight gradient: CTAs per pair, 2 when cin > 32
};

// OUT_CHUNKED: the output is chunk-major and TF32-rounded (the next layer's input); else NCHW in full fp32
template <bool OUT_CHUNKED>
__global__ void __launch_bounds__(BC_THREADS, 1)
branch_conv3x3_kernel(const __grid_constant__ CUtensorMap map_x, const float* __restrict__ wpacked,
                      const float* __restrict__ bias, float* __restrict__ out, const BranchConvShape sh) {
    const auto [base, gen] = aligned_smem();
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // barriers: weights, slot full x 6, slot empty x 6, acc_full x 2, acc_empty x 2; the TMEM base address after them
    const unsigned bar = base + BC_OFF_BAR;
    const unsigned b_w = bar, b_full = bar + 8, b_empty = b_full + 8 * BC_SLOTS, b_accfull = b_empty + 8 * BC_SLOTS,
                   b_accempty = b_accfull + 16;
    if (tid == 0) {
        mbar_init(b_w, 1);
        for (int s = 0; s < BC_SLOTS; ++s) {
            mbar_init(b_full + 8 * s, 1);
            mbar_init(b_empty + 8 * s, 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(b_accfull + 8 * s, 1);
            mbar_init(b_accempty + 8 * s, TC_EPI_WARPS * 32);
        }
        mbar_fence_init();
    }
    if (tid < TC_N) reinterpret_cast<float*>(gen + BC_OFF_BIAS)[tid] = (bias != nullptr && tid < sh.cout) ? bias[tid] : 0.f;
    const unsigned tmem = tmem_alloc<TC_TMEM_COLS>(bar + 8 * (1 + 2 * BC_SLOTS + 4), warp);
    const TileWalker walk(sh.tiles_x, sh.tiles_y);

    if (warp < TC_EPI_WARPS) {
        // ===================== epilogue: TMEM lanes 32 * warp .. + 31 = tile pixels (row 4 * warp + lane / 8, column lane % 8)
        const float* sbias = reinterpret_cast<const float*>(gen + BC_OFF_BIAS);
        const int r = warp * 4 + (lane >> 3), c = lane & 7;
        const int64_t plane = (int64_t)sh.h * sh.w;
        int it = 0;
        for (TileIter ti = walk.first(); ti.tile < sh.ntiles; walk.advance(ti), ++it) {
            unsigned v[64];
            tc_take_acc(tmem + ((unsigned)(warp * 32) << 16), it, b_accfull, b_accempty, v);
            const int Y = ti.ty * TC_TH + r, X = ti.tx * TC_TW + c;
            if (Y >= sh.h || X >= sh.w) continue;
            // ReLU before rounding (rounding keeps the sign); `x < 0` keeps a NaN a NaN, as torch's ReLU does
            auto act = [&](int n) {
                const float y = __uint_as_float(v[n]) + sbias[n];
                return (sh.relu && y < 0.f) ? 0.f : y;
            };
            if (OUT_CHUNKED) {
                // chunk k of the pixel: 16 bytes; a warp row of 8 pixels writes 128 contiguous bytes per chunk.  Padding
                // channels come out 0: their weights and bias are 0.
                float4* p = reinterpret_cast<float4*>(out) + ((int64_t)ti.b * sh.out_chunks * sh.h + Y) * sh.w + X;
#pragma unroll
                for (int k = 0; k < BC_CHUNKS; ++k)
                    if (k < sh.out_chunks)
                        p[k * plane] = make_float4(to_tf32(act(4 * k)), to_tf32(act(4 * k + 1)), to_tf32(act(4 * k + 2)), to_tf32(act(4 * k + 3)));
            } else {
                float* p = out + (int64_t)ti.b * sh.cout * plane + (int64_t)Y * sh.w + X;
#pragma unroll
                for (int n = 0; n < TC_N; ++n)
                    if (n < sh.cout) p[(int64_t)n * plane] = act(n);
            }
        }
    } else if (warp == TC_EPI_WARPS) {
        // ===================== MMA issuer: the whole warp walks the loop (uniform descriptors), one lane issues
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        tc_wait(b_w, 0);
        constexpr unsigned idesc = tc_idesc_tf32(128, TC_N);
        constexpr int KS_SLOT = BC_SLOT_CHUNKS / 2;        // K-steps per slot
        // start-address fields only (units of 16 bytes): per tap + (dy * 10 + dx) pixels of the patch and + 16 chunks of
        // the weights, per K-step + 2 chunks of each
        const uint64_t db0 = tc_desc(base, TC_N * 16, 128);
        int slot = 0;
        unsigned sph = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < sh.ntiles; tile += gridDim.x, ++it) {
            const int as = it & 1;
            tc_wait(b_accempty + 8 * as, ((it >> 1) & 1) ^ 1);   // accumulator stage drained (passes at once the first time)
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const unsigned d_tmem = tmem_u + as * TC_N;
#pragma unroll 1
            for (int q = 0; q < sh.slots_per_tile; ++q) {
                tc_wait(b_full + 8 * slot, sph);           // the TMA box of this quarter patch has landed
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t da0 = tc_desc(base + BC_OFF_A + slot * BC_SLOT_BYTES, TC_NPIX * 16, TC_PW * 16);
                const uint64_t dbq = db0 + (uint64_t)(q * KS_SLOT * 2 * TC_N);
                const int ks_n = min(sh.k_steps - q * KS_SLOT, KS_SLOT);
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
                    for (int ks = 0; ks < KS_SLOT; ++ks) {
                        if (ks >= ks_n) break;
                        const uint64_t da = da0 + (uint64_t)((tap / 3) * TC_PW + (tap % 3) + ks * 2 * TC_NPIX);
                        const uint64_t db = dbq + (uint64_t)((tap * BC_W_TAP_BYTES + ks * 2 * TC_N * 16) >> 4);
                        if (lane == 0) tc_mma(d_tmem, da, db, idesc, (q | tap | ks) != 0);
                    }
                }
                __syncwarp();
                if (lane == 0) tc_commit(b_empty + 8 * slot);   // slot may be refilled once these MMAs have read it
                if (++slot == BC_SLOTS) { slot = 0; sph ^= 1; }
            }
            __syncwarp();
            if (lane == 0) tc_commit(b_accfull + 8 * as);  // accumulator complete
        }
    } else {
        // ===================== copies: the weights once, then a quarter patch per slot, running up to 6 slots ahead
        if (lane == 0) {
            tma_prefetch_desc(&map_x);
            mbar_expect_tx(b_w, BC_W_BYTES);
            for (int t = 0; t < 9; ++t)
                bulk_load(base + t * BC_W_TAP_BYTES, reinterpret_cast<const char*>(wpacked) + (size_t)t * BC_W_TAP_BYTES, BC_W_TAP_BYTES, b_w);
            int slot = 0;
            unsigned sph = 0;
            for (TileIter ti = walk.first(); ti.tile < sh.ntiles; walk.advance(ti)) {
                // box origin: one pixel up and left of the tile (zero-filled outside the image), chunk q of image b
                const int x0 = 4 * (ti.tx * TC_TW - 1), y0 = ti.ty * TC_TH - 1, c0 = ti.b * sh.in_chunks;
                for (int q = 0; q < sh.slots_per_tile; ++q) {
                    tc_wait(b_empty + 8 * slot, sph ^ 1);
                    mbar_expect_tx(b_full + 8 * slot, BC_SLOT_BYTES);
                    tma_load_3d(base + BC_OFF_A + slot * BC_SLOT_BYTES, &map_x, b_full + 8 * slot, x0, y0, c0 + q * BC_SLOT_CHUNKS);
                    if (++slot == BC_SLOTS) { slot = 0; sph ^= 1; }
                }
            }
        }
        __syncwarp();
    }

    tmem_dealloc<TC_TMEM_COLS>(tmem, warp);
}

// [B][c][h][w] -> chunk-major [B][chunks][h][w][4], rounded to TF32, channels past c = 0.  Thread = (image, chunk, pixel).
__global__ void __launch_bounds__(256)
nchw_to_chunked_kernel(const float* __restrict__ x, float* __restrict__ out, int64_t n, int c, int chunks, int64_t plane) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t p = i % plane, bk = i / plane;
    const int k = (int)(bk % chunks);
    const float* src = x + ((bk / chunks) * c + 4 * k) * plane + p;
    float q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = 4 * k + j < c ? to_tf32(__ldg(src + j * plane)) : 0.f;
    reinterpret_cast<float4*>(out)[i] = make_float4(q[0], q[1], q[2], q[3]);
}

// x [B][c][h][w] -> xc, its TF32-rounded chunk-major copy with `chunks` chunks per image
int to_chunked(const float* x, float* xc, int64_t B, int c, int chunks, int64_t plane, cudaStream_t s) {
    const int64_t n = B * chunks * plane;
    return launch256<nchw_to_chunked_kernel>((n + 255) / 256, s, x, xc, n, c, chunks, plane);
}

int launch_branch_conv(const float* xc, const float* wpacked, const float* bias, float* out, int64_t B, const BranchConvShape& sh,
                       bool out_chunked, cudaStream_t s) {
    // 3-D map over the chunk-major input: (chunk channel x column) merged into 160-byte box rows, rows, (image x chunk)
    CUtensorMap map;
    const int64_t dims[3] = {4 * (int64_t)sh.w, sh.h, B * sh.in_chunks};
    const int64_t strides[3] = {1, 4 * (int64_t)sh.w, 4 * (int64_t)sh.h * sh.w};
    const int box[3] = {4 * TC_PW, TC_PH, BC_SLOT_CHUNKS};
    if (!make_map_f32(&map, xc, 3, dims, strides, box)) return SSTEM_E_SHAPE;
    const int ctas = std::min(sh.ntiles, sm_count());
    return out_chunked ? launch_tc<branch_conv3x3_kernel<true>>(BC_SMEM, BC_THREADS, ctas, s, map, wpacked, bias, out, sh)
                       : launch_tc<branch_conv3x3_kernel<false>>(BC_SMEM, BC_THREADS, ctas, s, map, wpacked, bias, out, sh);
}

// ---------------------------------------------------------------------------------------------------------------------
// Backward of y = relu?(conv3x3(x, W) + b) (sstem_branch_conv3x3_backward, DESIGN 4.11d).
//
// g = (y <= 0) ? 0 : grad_out (grad_out without the ReLU), NCHW -> chunk-major [B][C8/4][h][w][4] rounded to TF32: the input
// of the adjoint convolution (grad_x = branch_conv3x3_kernel on W') and the A operand of the weight gradient.  The mask is
// torch's threshold_backward on the output: y == 0 gives 0, a NaN y passes the gradient.  Each block also writes the fp32 sums of the UNROUNDED g of its
// chunk's four channels (grad_bias, summed over blocks by sum_partials_kernel): per thread in pixel order, then
// a fixed shuffle tree, then the warps in order, so the result is bit-identical from run to run.  Block = (image b,
// chunk k, part bx of the plane), blockIdx.x = (b * chunks + k) * nbx + bx; bias partial p = b * nbx + bx.
template <bool Y_CHUNKED>
__global__ void __launch_bounds__(256)
branch_grad_mask_kernel(const float* __restrict__ gy, const float* __restrict__ y, float* __restrict__ gc,
                        float* __restrict__ part_b, int cout, int chunks, int nbx, int64_t plane) {
    const int bx = blockIdx.x % nbx, bk = blockIdx.x / nbx, k = bk % chunks, b = bk / chunks;
    const float* src = gy + ((int64_t)b * cout + 4 * k) * plane;
    const float* ysrc = Y_CHUNKED ? y + (int64_t)bk * plane * 4 : y + ((int64_t)b * cout + 4 * k) * plane;
    float4* dst = reinterpret_cast<float4*>(gc) + (int64_t)bk * plane;
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    for (int64_t p = (int64_t)bx * blockDim.x + threadIdx.x; p < plane; p += (int64_t)nbx * blockDim.x) {
        float yv[4] = {1.f, 1.f, 1.f, 1.f};                // no ReLU: every gradient passes
        if (y && Y_CHUNKED) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(ysrc) + p);
            yv[0] = t.x; yv[1] = t.y; yv[2] = t.z; yv[3] = t.w;
        }
        float q[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float v = 0.f;
            if (4 * k + j < cout) {
                v = __ldg(src + j * plane + p);
                if (y && !Y_CHUNKED) yv[j] = __ldg(ysrc + j * plane + p);
                if (yv[j] <= 0.f) v = 0.f;
            }
            s[j] += v;
            q[j] = to_tf32(v);
        }
        dst[p] = make_float4(q[0], q[1], q[2], q[3]);
    }
    __shared__ float red[8][4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
        if (lane == 0) red[warp][j] = s[j];
    }
    __syncthreads();
    if (threadIdx.x < 4 && 4 * k + (int)threadIdx.x < cout) {
        float t = 0.f;
        for (int q = 0; q < (int)(blockDim.x >> 5); ++q) t += red[q][threadIdx.x];
        part_b[((int64_t)b * nbx + bx) * cout + 4 * k + threadIdx.x] = t;
    }
}

// grad_weight.  Per 16 x 8 tile and tap (dy, dx):
//     D_tap[co][ci] += sum_{pixels p} g[co][p] * x[ci][p + (dy, dx)]               (x zero padded by 1)
// as tcgen05.mma kind::tf32, M = 64 (co, padded), N = 32 (ci), K = 8 = one tile row: 16 K-steps x 9 taps = 144 MMAs per
// tile.  Nine accumulators of N = 64 would need 576 TMEM columns, so a CTA owns one half of the input channels (32, nine
// accumulators = 288 columns, resident for the whole tile loop); CTAs 2j and 2j + 1 walk the same tiles for the two halves
// (one CTA per pair when cin <= 32) and write the two halves of partial j.
// Both operands are K-major, no swizzle (the encoding of the forward and of tap_conv3x3_wgrad_kernel), staged from the
// chunk-major activations, which are already TF32-rounded: a thread loads four or more pixels of one chunk (16 bytes
// each) and stores them transposed, one 16-byte row of four pixels per channel -- nothing is blended or rounded here:
//   * A = g of the tile: [tile row][K half][co group of 8][8 co][4 pixels], 2 KB per row;
//   * B = the 18 x 10 patch of x as three copies shifted by dx = 0, 1, 2 columns: [dx][patch row][K half][ci group of
//     8][8 ci][4 pixels], 1 KB per row.  Tap (dy, dx), K-step ky reads copy dx at patch row ky + dy.
// Two stages: the 8 staging warps load tile i + 1 into registers while the MMAs of tile i run, store it once the MMAs of
// tile i - 1 have released its stage (tcgen05.commit), and 1 warp issues.  At the end warps 0-3 write the CTA's partial.
constexpr int BW_STAGE_THREADS = 256;                      // thread = A item (tile row, co chunk) and B item (patch row, ci chunk)
constexpr int BW_THREADS = BW_STAGE_THREADS + 32;          // + the MMA warp = 288
constexpr int BW_M = 64, BW_N = 32;
constexpr unsigned BW_A_ROW = 2 * (BW_M / 8) * 128;        // 2048
constexpr unsigned BW_A_BYTES = TC_TH * BW_A_ROW;          // 32768
constexpr unsigned BW_B_ROW = 2 * (BW_N / 8) * 128;        // 1024
constexpr unsigned BW_B_COPY = TC_PH * BW_B_ROW;           // 18432
constexpr unsigned BW_STAGE = BW_A_BYTES + 3 * BW_B_COPY;  // 88064
constexpr unsigned BW_OFF_BAR = 2 * BW_STAGE;              // 176128
constexpr unsigned BW_SMEM = BW_OFF_BAR + 64 + 128;        // + barriers, TMEM address, alignment slack = 176 320
constexpr unsigned BW_TMEM_COLS = 512;                     // 288 used; an allocation is a power of 2
static_assert(BW_SMEM <= 232448, "shared memory budget");
static_assert(9 * BW_N <= (int)BW_TMEM_COLS, "nine accumulators in tensor memory");
static_assert(TC_TH * (BW_M / 4) == BW_STAGE_THREADS && TC_PH * (BW_N / 4) <= BW_STAGE_THREADS, "one A and one B item per thread");

// The callers check the limits first (see sstem_branch_conv3x3).
BranchConvShape branch_conv_shape(int64_t B, int cin, int cout, int64_t h, int64_t w, bool relu) {
    BranchConvShape sh;
    sh.h = (int)h; sh.w = (int)w; sh.cin = cin; sh.cout = cout;
    sh.tiles_x = (sh.w + TC_TW - 1) / TC_TW;
    sh.tiles_y = (sh.h + TC_TH - 1) / TC_TH;
    sh.in_chunks = (cin + 7) / 8 * 2;
    sh.out_chunks = (cout + 7) / 8 * 2;
    sh.k_steps = sh.in_chunks / 2;
    sh.slots_per_tile = (sh.in_chunks + BC_SLOT_CHUNKS - 1) / BC_SLOT_CHUNKS;
    sh.relu = relu ? 1 : 0;
    sh.ntiles = (int)tile_count(B, h, w);
    sh.halves = cin > BW_N ? 2 : 1;
    return sh;
}

// sh: the shape of the forward convolution (in_chunks: x, out_chunks: g)
__global__ void __launch_bounds__(BW_THREADS, 1)
branch_conv3x3_wgrad_kernel(const float* __restrict__ g, const float* __restrict__ x, float* __restrict__ part_w,
                            const BranchConvShape sh) {
    const unsigned base = aligned_smem().addr;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // barriers: full x 2, empty x 2, done; the TMEM base address after them
    const unsigned bar = base + BW_OFF_BAR;
    const unsigned b_full = bar, b_empty = bar + 16, b_done = bar + 32;
    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(b_full + 8 * s, BW_STAGE_THREADS);
            mbar_init(b_empty + 8 * s, 1);
        }
        mbar_init(b_done, 1);
        mbar_fence_init();
    }
    // channels past cout / cin are never written and stay zero
    for (unsigned i = tid; i < BW_OFF_BAR / 16; i += BW_THREADS) sts128(base + i * 16, 0.f, 0.f, 0.f, 0.f);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const unsigned tmem = tmem_alloc<BW_TMEM_COLS>(bar + 40, warp);
    const int half = blockIdx.x % sh.halves, pair = blockIdx.x / sh.halves, npairs = gridDim.x / sh.halves;

    if (warp < BW_STAGE_THREADS / 32) {
        // ===================== staging
        const int ay = tid >> 4, ak = tid & 15;            // A: tile row, g chunk (co 4 ak .. 4 ak + 3)
        const int by = tid >> 3, bk = tid & 7;             // B: patch row, x chunk 8 half + bk (ci 32 half + 4 bk ..)
        const bool a_item = ak < sh.out_chunks, b_item = by < TC_PH && 8 * half + bk < sh.in_chunks;
        const float4* g4 = reinterpret_cast<const float4*>(g);
        const float4* x4 = reinterpret_cast<const float4*>(x);
        const unsigned a_off = ay * BW_A_ROW + ak * 64, b_off = BW_A_BYTES + by * BW_B_ROW + bk * 64;
        // 4 pixels x 4 channels -> one 16-byte row of 4 pixels per channel (rows of a core matrix are 16 bytes apart)
        auto store_t = [](unsigned dst, const float4& p0, const float4& p1, const float4& p2, const float4& p3) {
            sts128(dst, p0.x, p1.x, p2.x, p3.x);
            sts128(dst + 16, p0.y, p1.y, p2.y, p3.y);
            sts128(dst + 32, p0.z, p1.z, p2.z, p3.z);
            sts128(dst + 48, p0.w, p1.w, p2.w, p3.w);
        };
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
        int it = 0;
        for (int tile = pair; tile < sh.ntiles; tile += npairs, ++it) {
            const int s = it & 1;
            const int r = tile / sh.tiles_x, tx = tile - r * sh.tiles_x, b = r / sh.tiles_y, ty = r - b * sh.tiles_y;
            const int Y0 = ty * TC_TH, X0 = tx * TC_TW;
            float4 av[8], bv[TC_PW];
            if (a_item) {
                const int Y = Y0 + ay;
                const float4* p = g4 + ((int64_t)(b * sh.out_chunks + ak) * sh.h + min(Y, sh.h - 1)) * sh.w + X0;
#pragma unroll
                for (int j = 0; j < 8; ++j) av[j] = (Y < sh.h && X0 + j < sh.w) ? __ldg(p + j) : zero;
            }
            if (b_item) {
                const int Y = Y0 - 1 + by;
                const bool row_in = Y >= 0 && Y < sh.h;
                const float4* p = x4 + ((int64_t)(b * sh.in_chunks + 8 * half + bk) * sh.h + min(max(Y, 0), sh.h - 1)) * sh.w;
#pragma unroll
                for (int c = 0; c < TC_PW; ++c) {
                    const int X = X0 - 1 + c;
                    bv[c] = (row_in && X >= 0 && X < sh.w) ? __ldg(p + X) : zero;
                }
            }
            tc_wait(b_empty + 8 * s, ((it >> 1) & 1) ^ 1);   // the MMAs of tile it - 2 have read this stage
            const unsigned st = base + s * BW_STAGE;
            if (a_item) {
                store_t(st + a_off, av[0], av[1], av[2], av[3]);
                store_t(st + a_off + BW_A_ROW / 2, av[4], av[5], av[6], av[7]);
            }
            if (b_item) {
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    store_t(st + b_off + dx * BW_B_COPY, bv[dx], bv[dx + 1], bv[dx + 2], bv[dx + 3]);
                    store_t(st + b_off + dx * BW_B_COPY + BW_B_ROW / 2, bv[dx + 4], bv[dx + 5], bv[dx + 6], bv[dx + 7]);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
            tc_arrive(b_full + 8 * s);
        }
    } else {
        // ===================== MMA issuer: the whole warp walks the loop (uniform descriptors), one lane issues
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
        constexpr unsigned idesc = tc_idesc_tf32(BW_M, BW_N);
        int it = 0;
        for (int tile = pair; tile < sh.ntiles; tile += npairs, ++it) {
            const int s = it & 1;
            tc_wait(b_full + 8 * s, (it >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t da0 = tc_desc(base + s * BW_STAGE, BW_A_ROW / 2, 128);
            const uint64_t db0 = tc_desc(base + s * BW_STAGE + BW_A_BYTES, BW_B_ROW / 2, 128);
#pragma unroll 1
            for (int tap = 0; tap < 9; ++tap) {
                const int dy = tap / 3, dx = tap % 3;
                const unsigned d_tmem = tmem_u + tap * BW_N;
#pragma unroll
                for (int ky = 0; ky < TC_TH; ++ky) {
                    const uint64_t da = da0 + (uint64_t)((ky * BW_A_ROW) >> 4);
                    const uint64_t db = db0 + (uint64_t)((dx * BW_B_COPY + (ky + dy) * BW_B_ROW) >> 4);
                    if (lane == 0) tc_mma(d_tmem, da, db, idesc, (it | ky) != 0);
                }
            }
            __syncwarp();
            if (lane == 0) tc_commit(b_empty + 8 * s);     // the stage may be refilled once these MMAs have read it
            __syncwarp();
        }
        if (lane == 0) tc_commit(b_done);                  // every accumulator complete
        __syncwarp();
    }

    if (warp < 4) {
        // M = 64: row m of D is TMEM lane 32 (m / 16) + m % 16 (as in tap_conv3x3_wgrad_kernel), so warp q reads co
        // 16 q .. 16 q + 15 in its lanes 0..15
        tc_wait(b_done, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int co = warp * 16 + lane, nci = min(sh.cin - half * BW_N, BW_N);
        float* pw = part_w + (int64_t)pair * (sh.cout * sh.cin * 9) + ((int64_t)co * sh.cin + half * BW_N) * 9;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
            unsigned v[32];
            tc_ld32(tmem + ((unsigned)(warp * 32) << 16) + tap * BW_N, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (lane < 16 && co < sh.cout) {
#pragma unroll
                for (int c = 0; c < BW_N; ++c)
                    if (c < nci) pw[c * 9 + tap] = __uint_as_float(v[c]);
            }
        }
    }
    tmem_dealloc<BW_TMEM_COLS>(tmem, warp);
}

}  // namespace

}  // namespace sstem

using namespace sstem;

extern "C" int64_t sstem_tap_conv3x3_packed_elems(void) { return (int64_t)TC_W_BYTES / 4; }

extern "C" int sstem_tap_conv3x3_pack_weights(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream) {
    return pack_weights<false, TC_WCHUNKS, true>(weight, packed, cin, cout, TC_MAXC, TC_N, stream);
}

extern "C" int sstem_tap_conv3x3(const float* x, const float* packed_weight, const float* bias, float* out,
                                 int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream) {
    if (!x || !packed_weight || !out) return SSTEM_E_NULL;
    if (flags & ~(SSTEM_TAPCONV_UPSAMPLE2X | SSTEM_TAPCONV_TILED)) return SSTEM_E_FLAG;
    const bool ups = flags & SSTEM_TAPCONV_UPSAMPLE2X, tiled = flags & SSTEM_TAPCONV_TILED;
    if (!image_fits(B, h, w)) return SSTEM_E_SHAPE;
    if (cin <= 0 || cin > TC_MAXC || cout <= 0 || cout > TC_N) return SSTEM_E_SHAPE;
    if (tiled && cout != 51) return SSTEM_E_SHAPE;         // the tile-major layout is the 51-tap consumer's
    if (!aligned4(x) || !aligned16(packed_weight) || !aligned4(out) || (bias && !aligned4(bias))) return SSTEM_E_ALIGN;
    DeviceGuard guard(out);
    if (guard.err) return guard.err;
    const TapConvShape sh = tap_conv_shape(B, cin, cout, h, w, ups);
    if (tile_count(B, sh.H, sh.W) > INT32_MAX / 2 || (int64_t)cin * h * w > INT32_MAX) return SSTEM_E_SHAPE;
    const TapSrc src = !ups ? TapSrc::NCHW : (w % 4 == 0 && aligned16(x)) ? TapSrc::UP_VEC : TapSrc::UP;
    const bool full = cin > 48;                            // all 13 channel chunks exist: the common (51-channel) case, no per-chunk checks
    return launch_tap_conv(src, tiled, full, x, packed_weight, bias, out, sh, (cudaStream_t)stream);
}

extern "C" int sstem_tap_conv3x3_pack_weights_adjoint(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream) {
    return pack_weights<true, TC_WCHUNKS, true>(weight, packed, cin, cout, TC_MAXC, TC_MAXC, stream);
}

extern "C" int sstem_tap_conv3x3_backward(const float* grad_out, const float* x, const float* packed_adjoint,
                                          float* grad_x, float* grad_weight, float* grad_bias,
                                          int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream) {
    if (!grad_out || !x || (grad_x && !packed_adjoint)) return SSTEM_E_NULL;
    if (flags & ~(SSTEM_TAPCONV_UPSAMPLE2X | SSTEM_TAPCONV_TILED)) return SSTEM_E_FLAG;
    const bool ups = flags & SSTEM_TAPCONV_UPSAMPLE2X, tiled = flags & SSTEM_TAPCONV_TILED;
    if (!image_fits(B, h, w)) return SSTEM_E_SHAPE;
    if (cin <= 0 || cin > TC_MAXC || cout <= 0 || cout > TC_MAXC) return SSTEM_E_SHAPE;
    if (tiled && cout != 51) return SSTEM_E_SHAPE;
    if (!aligned4(grad_out) || !aligned4(x) || (packed_adjoint && !aligned16(packed_adjoint)) || (grad_x && !aligned4(grad_x)) ||
        (grad_weight && !aligned4(grad_weight)) || (grad_bias && !aligned4(grad_bias)))
        return SSTEM_E_ALIGN;
    const int64_t H = ups ? 2 * h : h, W = ups ? 2 * w : w;
    if (tile_count(B, H, W) > INT32_MAX / 2 || (int64_t)cout * H * W > INT32_MAX || (int64_t)cin * H * W > INT32_MAX) return SSTEM_E_SHAPE;
    if (!grad_x && !grad_weight && !grad_bias) return 0;
    DeviceGuard guard(grad_out);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    const TapConvShape sh = tap_conv_shape(B, cin, cout, h, w, ups);

    if (grad_x) {
        // gU = conv3x3(gy, W'), cout -> cin channels at full resolution; with the upsample into a workspace, then up^T
        const TapConvShape sd = tap_conv_shape(B, cout, cin, H, W, false);
        float* gU = grad_x;
        if (ups && workspace_alloc(reinterpret_cast<void**>(&gU), (size_t)(B * cin * H * W) * sizeof(float), s)) return cudaErrorMemoryAllocation;
        int e = launch_tap_conv(tiled ? TapSrc::TILE_MAJOR : TapSrc::NCHW, false, cout > 48, grad_out, packed_adjoint, nullptr, gU, sd, s);
        if (!e && ups) {
            const int64_t n = B * cin * h * w;
            e = launch256<upsample2x_adjoint_kernel>((n + 255) / 256, s, gU, grad_x, n, (int)h, (int)w, (int)H, (int)W, sh.ry, sh.rx);
        }
        if (ups) cudaFreeAsync(gU, s);
        if (e) return e;
    }
    if (grad_weight || grad_bias) {
        const int ctas = std::min(sh.ntiles, sm_count());
        const int nw = cout * cin * 9;
        float* part = nullptr;
        if (workspace_alloc(reinterpret_cast<void**>(&part), (size_t)ctas * (nw + cout) * sizeof(float), s)) return cudaErrorMemoryAllocation;
        float* part_b = part + (size_t)ctas * nw;
        int e = ups ? (tiled ? launch_tc<tap_conv3x3_wgrad_kernel<true, true>>(WG_SMEM, WG_THREADS, ctas, s, grad_out, x, part, part_b, sh)
                             : launch_tc<tap_conv3x3_wgrad_kernel<true, false>>(WG_SMEM, WG_THREADS, ctas, s, grad_out, x, part, part_b, sh))
                    : (tiled ? launch_tc<tap_conv3x3_wgrad_kernel<false, true>>(WG_SMEM, WG_THREADS, ctas, s, grad_out, x, part, part_b, sh)
                             : launch_tc<tap_conv3x3_wgrad_kernel<false, false>>(WG_SMEM, WG_THREADS, ctas, s, grad_out, x, part, part_b, sh));
        if (!e) e = launch256<sum_partials_kernel>((nw + cout + 255) / 256, s, part, part_b, grad_weight, grad_bias, nw, cout, ctas);
        cudaFreeAsync(part, s);
        if (e) return e;
    }
    return 0;
}

extern "C" int64_t sstem_branch_conv3x3_packed_elems(void) { return (int64_t)BC_W_BYTES / 4; }

extern "C" int sstem_branch_conv3x3_pack_weights(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream) {
    return pack_weights<false, BC_CHUNKS, false>(weight, packed, cin, cout, BC_MAXC, TC_N, stream);
}

extern "C" int sstem_branch_conv3x3_pack_weights_adjoint(const float* weight, float* packed, int32_t cin, int32_t cout, void* stream) {
    return pack_weights<true, BC_CHUNKS, false>(weight, packed, cin, cout, BC_MAXC, TC_N, stream);
}

extern "C" int64_t sstem_chunked_elems(int64_t B, int64_t c, int64_t h, int64_t w) {
    if (B <= 0 || c <= 0 || h <= 0 || w <= 0) return 0;
    return B * ((c + 7) / 8 * 8) * h * w;
}

extern "C" int sstem_branch_conv3x3(const float* x, const float* packed_weight, const float* bias, float* out,
                                    int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream) {
    if (!x || !packed_weight || !out) return SSTEM_E_NULL;
    if (flags & ~(SSTEM_BRANCH_RELU | SSTEM_BRANCH_IN_CHUNKED | SSTEM_BRANCH_OUT_CHUNKED)) return SSTEM_E_FLAG;
    const bool in_chunked = flags & SSTEM_BRANCH_IN_CHUNKED, out_chunked = flags & SSTEM_BRANCH_OUT_CHUNKED;
    if (!image_fits(B, h, w)) return SSTEM_E_SHAPE;
    if (cin <= 0 || cin > BC_MAXC || cout <= 0 || cout > TC_N) return SSTEM_E_SHAPE;
    // tile indices and the TMA chunk coordinate are 32-bit
    if (tile_count(B, h, w) > INT32_MAX / 2 || B * ((cin + 7) / 8 * 2) > INT32_MAX / 2) return SSTEM_E_SHAPE;
    const BranchConvShape sh = branch_conv_shape(B, cin, cout, h, w, flags & SSTEM_BRANCH_RELU);
    if (!(in_chunked ? aligned16(x) : aligned4(x)) || !aligned16(packed_weight) || !(out_chunked ? aligned16(out) : aligned4(out)) ||
        (bias && !aligned4(bias)))
        return SSTEM_E_ALIGN;
    DeviceGuard guard(out);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    const float* xc = x;
    float* ws = nullptr;
    if (!in_chunked) {   // NCHW input: a TF32-rounded chunk-major copy in a stream-ordered workspace
        if (workspace_alloc(reinterpret_cast<void**>(&ws), (size_t)(B * sh.in_chunks * h * w) * 16, s)) return cudaErrorMemoryAllocation;
        xc = ws;
    }
    int e = in_chunked ? 0 : to_chunked(x, ws, B, cin, sh.in_chunks, h * w, s);
    if (!e) e = launch_branch_conv(xc, packed_weight, bias, out, B, sh, out_chunked, s);
    if (ws) cudaFreeAsync(ws, s);
    return e;
}

extern "C" int sstem_branch_conv3x3_backward(const float* grad_out, const float* y, const float* x, const float* packed_adjoint,
                                             float* grad_x, float* grad_weight, float* grad_bias,
                                             int64_t B, int32_t cin, int32_t cout, int64_t h, int64_t w, uint32_t flags, void* stream) {
    const bool relu = flags & SSTEM_BRANCH_RELU, in_chunked = flags & SSTEM_BRANCH_IN_CHUNKED, out_chunked = flags & SSTEM_BRANCH_OUT_CHUNKED;
    if (!grad_out || !x || (relu && !y) || (grad_x && !packed_adjoint)) return SSTEM_E_NULL;
    if (flags & ~(SSTEM_BRANCH_RELU | SSTEM_BRANCH_IN_CHUNKED | SSTEM_BRANCH_OUT_CHUNKED)) return SSTEM_E_FLAG;
    if (!image_fits(B, h, w)) return SSTEM_E_SHAPE;
    if (cin <= 0 || cin > BC_MAXC || cout <= 0 || cout > BC_MAXC) return SSTEM_E_SHAPE;
    // tile indices, the TMA chunk coordinate of the adjoint convolution and the mask kernel's block index are 32-bit
    if (tile_count(B, h, w) > INT32_MAX / 2 || B * ((cout + 7) / 8 * 2) * 64 > INT32_MAX / 2) return SSTEM_E_SHAPE;
    if (!aligned4(grad_out) || (y && !(out_chunked ? aligned16(y) : aligned4(y))) || !(in_chunked ? aligned16(x) : aligned4(x)) ||
        (packed_adjoint && !aligned16(packed_adjoint)) || (grad_x && !aligned4(grad_x)) || (grad_weight && !aligned4(grad_weight)) ||
        (grad_bias && !aligned4(grad_bias)))
        return SSTEM_E_ALIGN;
    if (!grad_x && !grad_weight && !grad_bias) return 0;
    DeviceGuard guard(grad_out);
    if (guard.err) return guard.err;
    cudaStream_t s = (cudaStream_t)stream;
    const BranchConvShape sh = branch_conv_shape(B, cin, cout, h, w, false);
    const int64_t plane = h * w;
    const bool wgrad = grad_weight != nullptr;
    const int pairs = std::min(sh.ntiles, std::max(sm_count() / sh.halves, 1));
    const int nw = cout * cin * 9;
    // about 64 bias partials per channel whatever the batch: (64 / B) blocks per image and chunk
    const int nbx = (int)std::max<int64_t>(64 / B, 1);
    // one stream-ordered workspace: g chunk-major | bias partials | x chunk-major (NCHW x, weight gradient) | weight partials
    const size_t g_floats = (size_t)(B * sh.out_chunks * plane) * 4, pb_floats = (size_t)(B * nbx * cout);
    const size_t xc_floats = (wgrad && !in_chunked) ? (size_t)(B * sh.in_chunks * plane) * 4 : 0, pw_floats = wgrad ? (size_t)pairs * nw : 0;
    const size_t off_pb = (g_floats + 3) / 4 * 4, off_xc = off_pb + (pb_floats + 3) / 4 * 4, off_pw = off_xc + xc_floats;
    float* ws = nullptr;
    if (workspace_alloc(reinterpret_cast<void**>(&ws), (off_pw + pw_floats) * sizeof(float), s)) return cudaErrorMemoryAllocation;
    float *gc = ws, *part_b = ws + off_pb, *xc = ws + off_xc, *part_w = ws + off_pw;
    const float* ym = relu ? y : nullptr;
    const int64_t mask_blocks = B * sh.out_chunks * nbx;
    int e = out_chunked ? launch256<branch_grad_mask_kernel<true>>(mask_blocks, s, grad_out, ym, gc, part_b, cout, sh.out_chunks, nbx, plane)
                        : launch256<branch_grad_mask_kernel<false>>(mask_blocks, s, grad_out, ym, gc, part_b, cout, sh.out_chunks, nbx, plane);
    if (!e && grad_bias)
        e = launch256<sum_partials_kernel>((cout + 255) / 256, s, nullptr, part_b, nullptr, grad_bias, 0, cout, (int)(B * nbx));
    if (!e && grad_x)   // the adjoint convolution, cout -> cin channels, from g: no bias, no ReLU, NCHW out
        e = launch_branch_conv(gc, packed_adjoint, nullptr, grad_x, B, branch_conv_shape(B, cout, cin, h, w, false), false, s);
    if (!e && wgrad) {
        if (!in_chunked) e = to_chunked(x, xc, B, cin, sh.in_chunks, plane, s);   // as the forward does
        if (!e) e = launch_tc<branch_conv3x3_wgrad_kernel>(BW_SMEM, BW_THREADS, pairs * sh.halves, s, gc, in_chunked ? x : xc, part_w, sh);
        if (!e) e = launch256<sum_partials_kernel>((nw + 255) / 256, s, part_w, nullptr, grad_weight, nullptr, nw, 0, pairs);
    }
    cudaFreeAsync(ws, s);
    return e;
}
