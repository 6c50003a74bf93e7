// gemm_common.cuh -- PTX wrappers shared by the leaf-GEMM kernels (mbarrier) and the driver entry
// point for tensor-map encoding.
#pragma once
#include "matrix.cuh"
#include <cuda.h>   // CUtensorMap types only; the encoder is fetched through cudaGetDriverEntryPoint

namespace hbsm_b200 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}


struct GemmMeta { int ctile; int flags; };   // flags: 1 = first chunk of a C tile, 2 = last chunk, 4 = no more work

// fp32 leaf GEMM on the 5th-generation tensor cores (gemm_f32.cu) for leaves of 32, 64, 128 and 256.  Leaves of 32 and 64 run
// the kernels over 2 x 2 groups of C tiles, which are built from ckeys and task_k (C's Morton keys and the k of every product);
// single_tile runs the single-C-tile kernels there instead (the parity hook of hbsm_set_gemm_variant(3)).
void launch_gemm_f32_tc(const Matrix& A, bool tA, const Matrix& B, bool tB, const uint2* ab, const uint64_t* begin,
                        uint32_t n_ctiles, const uint32_t* tile_list, unsigned* counter, float* Ct, const uint64_t* ckeys,
                        const uint32_t* task_k, size_t n_products, bool single_tile);

}  // namespace hbsm_b200
