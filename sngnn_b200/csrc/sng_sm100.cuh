// tcgen05 / TMA primitives shared by the tensor-core kernels, K1 (sng_simknn.cu), the N x N producer (sng_gemm.cu) and the
// similarity histogram (sng_simhist.cu): mbarriers with the bounded wait, tcgen05 fences and TMEM loads, the cta_group::1
// TMA load / MMA / commit, the descriptors of a K-major FP16 MMA and the TMA map of its operands.  Forms that only one
// kernel uses (cta_group::2, cluster, multicast) stay in that kernel's file.
#pragma once
#include "sng_common.cuh"
#include <cuda.h>        // CUtensorMap + enums only; cuTensorMapEncodeTiled is resolved at run time

namespace sng {

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    return done != 0;
}
// Bounded wait: a protocol bug must trap (error returned to the caller) instead of hanging the GPU.
static __device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
    uint32_t done, polls = 0;
    unsigned long long t0 = 0;
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) return;
        if (++polls > 4096u) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ull) __trap();     // 4 s
        }
    }
}
// hot-loop form: one inline try (it suspends in hardware for a while), the bounded polling loop stays out of line
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (!mbar_try(bar, parity)) mbar_wait_slow(bar, parity);
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// cta_group::1 forms: TMA tile load into this CTA's shared memory, one kind::f16 MMA into TMEM, and the commit that arrives
// on an mbarrier when every MMA issued before it has retired
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// K-major, 128-byte-swizzled shared-memory matrix descriptor (sm_100 "version 1"):
// rows are 128 B apart, 8-row groups 1024 B apart (SBO); LBO unused for swizzled K-major.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor of an M x N MMA: A, B = FP16 (0), D = FP32 (1 at bit 4), both K-major, N/8 at [17,23),
// M/16 at [24,29)
constexpr uint32_t f16_idesc(int m, int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24); }

// TMA map of an FP16 row-major matrix of `rows` rows, `ld` elements apart, read as `k` columns: box = 64 (K) x 128 (rows),
// 128-byte swizzle, zero fill (columns beyond k and rows beyond `rows` read as zero).  `row_stride` > 1 maps every
// row_stride-th row of the matrix.
inline int make_tma_map_f16(CUtensorMap* map, const uint16_t* ptr, int64_t rows, int64_t k, int64_t ld, int64_t row_stride) {
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeTiledFn enc = nullptr;
    if (!enc) {
        void* fp = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            enc = reinterpret_cast<EncodeTiledFn>(fp);
        else
            cudaGetLastError();
    }
    if (!enc) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return SNG_ERR_CUDA; }
    cuuint64_t gdim[2] = {(cuuint64_t)k, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)ld * 2 * (cuuint64_t)row_stride};
    cuuint32_t box[2] = {64u, 128u};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<uint16_t*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld k=%lld ld=%lld row_stride=%lld)", (int)r, (long long)rows,
                  (long long)k, (long long)ld, (long long)row_stride);
        return SNG_ERR_CUDA;
    }
    return SNG_OK;
}

}  // namespace sng
