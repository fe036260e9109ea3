// Probe: tcgen05.mma kind::tf32 with SWIZZLE_NONE K-major shared-memory descriptors whose start address is a shifted
// view into a [chunk][pixel][4 channels] patch -- the layout the tap-producer convolution (csrc/tapconv.cu) relies on.
// One CTA, D[128 x 64] = A[128 x 16] * B[64 x 16]^T, two K = 8 steps.  The descriptor strides, the shift and the
// roles of the two stride fields come from argv, so one binary answers every encoding question:
//   umma_probe <lbo_bytes> <sbo_bytes> <shift_pixels> [swap]
// Two more questions, asked by the weight gradient of the tap producer (M = 64 output channels, N = 56 input channels):
//   umma_probe m64                    M = 64, N = 56, both operands K-major: which TMEM lane holds which row of D
//   umma_probe mnb <lbo> <sbo> <shift> M = 64, N = 56, B MN-major (transpose-B bit) read from a [chunk][pixel][4] patch
//                                     at a shifted start, two K-steps of one 10-pixel patch row each
// Each prints one JSON line: the TMEM lane each row of D was found in, and the largest error against the CPU product.
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o umma_probe umma_probe.cu
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>

constexpr int PW = 10, NPIX = 180, NCHUNK = 4, M = 128, N = 64, K = 16;
constexpr int A_BYTES = NCHUNK * NPIX * 16, B_BYTES = NCHUNK * N * 16;

__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((addr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;                                // descriptor version (Blackwell)
    return d;                                              // base offset 0, layout type 0 = no swizzle
}

__global__ void __launch_bounds__(128, 1)
probe_kernel(const float* a_img, const float* b_img, float* out, int* status, uint32_t lbo_a, uint32_t sbo_a,
             uint32_t lbo_b, uint32_t sbo_b, int shift) {
    extern __shared__ __align__(1024) unsigned char smem[];
    float* sa = reinterpret_cast<float*>(smem);
    float* sb = reinterpret_cast<float*>(smem + A_BYTES);
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < A_BYTES / 4; i += 128) sa[i] = a_img[i];
    for (int i = tid; i < B_BYTES / 4; i += 128) sb[i] = b_img[i];
    const uint32_t bar_addr = (uint32_t)__cvta_generic_to_shared(&bar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_addr));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 64;" ::"r"((uint32_t)__cvta_generic_to_shared(&tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_slot;
    if (tid == 0) {
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
        const uint32_t a0 = (uint32_t)__cvta_generic_to_shared(sa) + (uint32_t)shift * 16u;
        const uint32_t b0 = (uint32_t)__cvta_generic_to_shared(sb);
        for (int ks = 0; ks < K / 8; ++ks) {
            const uint64_t da = make_desc(a0 + ks * 2 * NPIX * 16, lbo_a, sbo_a);
            const uint64_t db = make_desc(b0 + ks * 2 * N * 16, lbo_b, sbo_b);
            const uint32_t acc = ks > 0;
            asm volatile(
                "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_addr) : "memory");
    }
    // bounded wait: a wrong encoding must not hang the box
    const long long t0 = clock64();
    bool ok = false;
    while (!ok) {
        uint32_t p;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(p) : "r"(bar_addr) : "memory");
        ok = p != 0;
        if (!ok && clock64() - t0 > 2000000000ll) break;
    }
    if (!ok) { if (tid == 0) *status = 1; }
    else {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        uint32_t v[64];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16) + h * 32;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                : "=r"(v[h*32+0]), "=r"(v[h*32+1]), "=r"(v[h*32+2]), "=r"(v[h*32+3]), "=r"(v[h*32+4]), "=r"(v[h*32+5]),
                  "=r"(v[h*32+6]), "=r"(v[h*32+7]), "=r"(v[h*32+8]), "=r"(v[h*32+9]), "=r"(v[h*32+10]), "=r"(v[h*32+11]),
                  "=r"(v[h*32+12]), "=r"(v[h*32+13]), "=r"(v[h*32+14]), "=r"(v[h*32+15]), "=r"(v[h*32+16]), "=r"(v[h*32+17]),
                  "=r"(v[h*32+18]), "=r"(v[h*32+19]), "=r"(v[h*32+20]), "=r"(v[h*32+21]), "=r"(v[h*32+22]), "=r"(v[h*32+23]),
                  "=r"(v[h*32+24]), "=r"(v[h*32+25]), "=r"(v[h*32+26]), "=r"(v[h*32+27]), "=r"(v[h*32+28]), "=r"(v[h*32+29]),
                  "=r"(v[h*32+30]), "=r"(v[h*32+31])
                : "r"(ta));
        }
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 64; ++j) out[tid * 64 + j] = __uint_as_float(v[j]);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 64;" ::"r"(tmem));
}

// Generic one-CTA probe: `img` (A and B images, byte offsets a_off / b_off) to shared memory, `ksteps` MMAs with the given
// descriptor fields and per-K-step start increments, then all 128 TMEM lanes x 64 columns to out[lane][col].
__global__ void __launch_bounds__(128, 1)
probe2_kernel(const float* img, int img_floats, float* out, int* status, uint32_t a_off, uint32_t b_off,
              uint32_t lbo_a, uint32_t sbo_a, uint32_t lbo_b, uint32_t sbo_b, uint32_t a_step, uint32_t b_step, int ksteps,
              uint32_t idesc) {
    extern __shared__ __align__(1024) unsigned char smem[];
    float* s = reinterpret_cast<float*>(smem);
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < img_floats; i += 128) s[i] = img[i];
    const uint32_t bar_addr = (uint32_t)__cvta_generic_to_shared(&bar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_addr));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 64;" ::"r"((uint32_t)__cvta_generic_to_shared(&tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_slot;
    if (tid == 0) {
        const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(s);
        for (int ks = 0; ks < ksteps; ++ks) {
            const uint64_t da = make_desc(s0 + a_off + ks * a_step, lbo_a, sbo_a);
            const uint64_t db = make_desc(s0 + b_off + ks * b_step, lbo_b, sbo_b);
            asm volatile(
                "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"((uint32_t)(ks > 0)) : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_addr) : "memory");
    }
    const long long t0 = clock64();
    bool ok = false;
    while (!ok) {
        uint32_t p;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(p) : "r"(bar_addr) : "memory");
        ok = p != 0;
        if (!ok && clock64() - t0 > 2000000000ll) break;
    }
    if (!ok) { if (tid == 0) *status = 1; }
    else {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        uint32_t v[64];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16) + h * 32;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                : "=r"(v[h*32+0]), "=r"(v[h*32+1]), "=r"(v[h*32+2]), "=r"(v[h*32+3]), "=r"(v[h*32+4]), "=r"(v[h*32+5]),
                  "=r"(v[h*32+6]), "=r"(v[h*32+7]), "=r"(v[h*32+8]), "=r"(v[h*32+9]), "=r"(v[h*32+10]), "=r"(v[h*32+11]),
                  "=r"(v[h*32+12]), "=r"(v[h*32+13]), "=r"(v[h*32+14]), "=r"(v[h*32+15]), "=r"(v[h*32+16]), "=r"(v[h*32+17]),
                  "=r"(v[h*32+18]), "=r"(v[h*32+19]), "=r"(v[h*32+20]), "=r"(v[h*32+21]), "=r"(v[h*32+22]), "=r"(v[h*32+23]),
                  "=r"(v[h*32+24]), "=r"(v[h*32+25]), "=r"(v[h*32+26]), "=r"(v[h*32+27]), "=r"(v[h*32+28]), "=r"(v[h*32+29]),
                  "=r"(v[h*32+30]), "=r"(v[h*32+31])
                : "r"(ta));
        }
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 64; ++j) out[tid * 64 + j] = __uint_as_float(v[j]);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 64;" ::"r"(tmem));
}

static float tf32(float x) { uint32_t u; memcpy(&u, &x, 4); u &= 0xffffe000u; memcpy(&x, &u, 4); return x; }

// M = 64, N = 56, K = 16 (two K-steps).  A is K-major: [k-step][k half][row group of 8][8 rows][4].  B is K-major like A
// (m64) or MN-major from a [chunk of 4 columns][180 patch pixels][4] patch, K-step ks = patch row ks from `shift` (mnb).
static int probe_m64(bool mnb, uint32_t lbo_b, uint32_t sbo_b, int shift) {
    constexpr int M2 = 64, N2 = 56, K2 = 16;
    const uint32_t a_floats = 2 * 2 * 8 * 32, b_floats = mnb ? 14 * NPIX * 4 : 2 * 2 * 7 * 32;
    std::vector<float> img(a_floats + b_floats), out(128 * 64, -1.f);
    srand(11);
    for (auto& x : img) x = (float)(rand() % 2001 - 1000) / 500.f;
    auto A = [&](int m, int k) { return img[(((k / 8) * 2 + (k % 8) / 4) * 8 + m / 8) * 32 + (m % 8) * 4 + k % 4]; };
    auto Bv = [&](int n, int k) {
        return mnb ? img[a_floats + ((n / 4) * NPIX + shift + (k / 8) * PW + k % 8) * 4 + n % 4]
                   : img[a_floats + (((k / 8) * 2 + (k % 8) / 4) * 7 + n / 8) * 32 + (n % 8) * 4 + k % 4];
    };
    if (!mnb) { lbo_b = 7 * 128; sbo_b = 128; }
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((mnb ? 1u : 0u) << 16) | ((uint32_t)(N2 >> 3) << 17) |
                           ((uint32_t)(M2 >> 4) << 24);
    float *dimg, *dout; int* dst;
    cudaMalloc(&dimg, img.size() * 4); cudaMalloc(&dout, out.size() * 4); cudaMalloc(&dst, 4);
    cudaMemcpy(dimg, img.data(), img.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dout, out.data(), out.size() * 4, cudaMemcpyHostToDevice);
    cudaMemset(dst, 0, 4);
    const int smem = (int)(img.size() * 4) + 96 * 1024;   // slack: a misread stride field stays inside shared memory
    cudaFuncSetAttribute(probe2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    probe2_kernel<<<1, 128, smem>>>(dimg, (int)img.size(), dout, dst, 0, a_floats * 4, 8 * 128, 128, lbo_b, sbo_b, 2048,
                                    mnb ? PW * 16 : 2 * 7 * 128, K2 / 8, idesc);
    cudaError_t e = cudaDeviceSynchronize();
    int st = 0;
    if (e == cudaSuccess) { cudaMemcpy(out.data(), dout, out.size() * 4, cudaMemcpyDeviceToHost); cudaMemcpy(&st, dst, 4, cudaMemcpyDeviceToHost); }
    // for each row of D: the lane whose 56 columns match it best
    double maxerr = 0, maxref = 0;
    printf("{\"mode\": \"%s\", \"lbo_b\": %u, \"sbo_b\": %u, \"shift\": %d, \"cuda\": \"%s\", \"timeout\": %d, \"row_lane\": [",
           mnb ? "mnb" : "m64", lbo_b, sbo_b, shift, cudaGetErrorString(e), st);
    for (int m = 0; m < M2; ++m) {
        double ref[N2];
        for (int n = 0; n < N2; ++n) {
            ref[n] = 0;
            for (int k = 0; k < K2; ++k) ref[n] += (double)tf32(A(m, k)) * (double)tf32(Bv(n, k));
            maxref = fmax(maxref, fabs(ref[n]));
        }
        int best = -1; double best_err = 1e30;
        for (int lane = 0; lane < 128; ++lane) {
            double err = 0;
            for (int n = 0; n < N2; ++n) err = fmax(err, fabs(ref[n] - out[lane * 64 + n]));
            if (err < best_err) { best_err = err; best = lane; }
        }
        maxerr = fmax(maxerr, best_err);
        printf("%s%d", m ? ", " : "", best);
    }
    printf("], \"max_err\": %.3e, \"max_ref\": %.3e}\n", maxerr, maxref);
    return 0;
}

int main(int argc, char** argv) {
    if (argc > 1 && !strcmp(argv[1], "m64")) return probe_m64(false, 0, 0, 0);
    if (argc > 1 && !strcmp(argv[1], "mnb"))
        return probe_m64(true, argc > 2 ? atoi(argv[2]) : NPIX * 16, argc > 3 ? atoi(argv[3]) : 128, argc > 4 ? atoi(argv[4]) : 0);
    uint32_t lbo = argc > 1 ? atoi(argv[1]) : NPIX * 16, sbo = argc > 2 ? atoi(argv[2]) : PW * 16;
    int shift = argc > 3 ? atoi(argv[3]) : 0;
    const bool swap = argc > 4 && atoi(argv[4]);
    std::vector<float> a(A_BYTES / 4), b(B_BYTES / 4), out(M * N, -1.f);
    srand(7);
    for (auto& x : a) x = (float)(rand() % 2001 - 1000) / 500.f;
    for (auto& x : b) x = (float)(rand() % 2001 - 1000) / 500.f;
    float *da, *db, *dout; int* dst;
    cudaMalloc(&da, A_BYTES); cudaMalloc(&db, B_BYTES); cudaMalloc(&dout, M * N * 4); cudaMalloc(&dst, 4);
    cudaMemcpy(da, a.data(), A_BYTES, cudaMemcpyHostToDevice); cudaMemcpy(db, b.data(), B_BYTES, cudaMemcpyHostToDevice);
    cudaMemset(dst, 0, 4); cudaMemcpy(dout, out.data(), M * N * 4, cudaMemcpyHostToDevice);
    uint32_t lbo_b = N * 16, sbo_b = 128;
    uint32_t la = lbo, sa_ = sbo, lb = lbo_b, sb_ = sbo_b;
    if (swap) { la = sbo; sa_ = lbo; lb = sbo_b; sb_ = lbo_b; }
    cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, A_BYTES + B_BYTES);
    probe_kernel<<<1, 128, A_BYTES + B_BYTES>>>(da, db, dout, dst, la, sa_, lb, sb_, shift);
    cudaError_t e = cudaDeviceSynchronize();
    int st = 0;
    if (e == cudaSuccess) { cudaMemcpy(out.data(), dout, M * N * 4, cudaMemcpyDeviceToHost); cudaMemcpy(&st, dst, 4, cudaMemcpyDeviceToHost); }
    double maxerr = 0, maxref = 0;
    for (int m = 0; m < M; ++m)
        for (int n = 0; n < N; ++n) {
            double r = 0;
            const int pix = (m / 8) * PW + (m % 8) + shift;
            for (int k = 0; k < K; ++k)
                r += (double)tf32(a[((k / 4) * NPIX + pix) * 4 + k % 4]) * (double)tf32(b[((k / 4) * N + n) * 4 + k % 4]);
            maxerr = fmax(maxerr, fabs(r - out[m * N + n]));
            maxref = fmax(maxref, fabs(r));
        }
    printf("{\"lbo\": %u, \"sbo\": %u, \"shift\": %d, \"swap\": %d, \"cuda\": \"%s\", \"timeout\": %d, \"max_err\": %.3e, \"max_ref\": %.3e}\n",
           lbo, sbo, shift, (int)swap, cudaGetErrorString(e), st, maxerr, maxref);
    return 0;
}
