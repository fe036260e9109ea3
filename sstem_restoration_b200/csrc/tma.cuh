// TMA (cp.async.bulk.tensor), bulk-copy, mbarrier and shared-memory load helpers shared by the warp, sepconv and
// tap-producer kernels, and the host-side tensor-map encoder (driver entry point resolved through the runtime: no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sstem {

// Shared-space (unsigned) addresses are the primary form; the pointer forms convert and forward.
__device__ __forceinline__ void mbar_init(unsigned bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {   // unbounded: spins until the phase completes
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) { mbar_init((unsigned)__cvta_generic_to_shared(bar), count); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) { mbar_expect_tx((unsigned)__cvta_generic_to_shared(bar), bytes); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) { mbar_wait((unsigned)__cvta_generic_to_shared(bar), parity); }
// 1-D bulk copy global -> shared (16-byte aligned, size a multiple of 16), completion on an mbarrier
__device__ __forceinline__ void bulk_load(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ float lds_f32(unsigned addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(map), "r"((unsigned)__cvta_generic_to_shared(bar)),
          "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(map), "r"((unsigned)__cvta_generic_to_shared(bar)),
          "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {      // C++11 static init: thread-safe
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            return reinterpret_cast<EncodeTiledFn>(p);
        cudaGetLastError();
        return nullptr;
    }();
    return fn;
}

// N-D fp32 tensor map: dims[i] elements, strides in ELEMENTS for dims 1..n-1 (dim 0 is dense), box[i] elements.
// Out-of-bounds parts of a box are zero-filled.  false: the shape breaks a tensor-map rule (16-byte strides / base).
inline bool make_map_f32(CUtensorMap* m, const float* base, int n, const int64_t* dims, const int64_t* strides, const int* box) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn || n < 1 || n > 5) return false;
    if (reinterpret_cast<uintptr_t>(base) & 15u) return false;
    cuuint64_t d[5], st[4];
    cuuint32_t b[5], es[5];
    for (int i = 0; i < n; ++i) {
        if (dims[i] <= 0 || box[i] <= 0 || box[i] > 256) return false;
        d[i] = (cuuint64_t)dims[i];
        b[i] = (cuuint32_t)box[i];
        es[i] = 1;
        if (i > 0) {
            st[i - 1] = (cuuint64_t)strides[i] * 4;
            if (st[i - 1] & 15u) return false;
        }
    }
    if (((int64_t)box[0] * 4) & 15) return false;
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)n, const_cast<float*>(base), d, st, b, es,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace sstem
