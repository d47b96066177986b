// Dense NT contraction on the 5th-generation tensor cores for the Sim-GFA metrics that RETURN an N x N matrix
// (R: SimGFAToolbox/dense.py:138-149 `norm.mm(norm.t())`, R: SimGFAToolbox/sparse.py:8-14 M^T M of the column-normalised
// adjacency):  out[i, j] = row_scale[i] * col_scale[j] * sum_k A[i, k] B[j, k],  A / B FP16 row-major, FP32 accumulation in
// TMEM, FP32 output.
//   * dense features: the caller passes A = [hi | hi | lo], B = [hi | lo | hi] with x-hat = hi + lo split into two FP16
//     halves, so the single FP16 contraction over K' = 3K equals the FP32 product to ~2^-22 (the dropped lo.lo term);
//   * adjacency-as-features: A = B = the 0/1 (small-integer) adjacency columns, EXACT in FP16 with FP32 accumulation, i.e.
//     exact common-neighbour counts; the cosine is that count times 1/(|a_i| |a_j|) applied by the epilogue scales.
// One CTA per 128 x 128 output tile: warp 0 = TMA producer (two K blocks of 64 in flight), warp 1 = MMA issuer
// (tcgen05.mma.cta_group::1, M = 128, N = 128, accumulator = 128 TMEM columns), warps 2-5 = epilogue (tcgen05.ld, one
// output row per thread).  Unlike the kNN builder this kernel materialises its output -- it exists for the functions
// whose contract is the matrix itself.
#include "sng_sm100.cuh"
#include <cuda_fp16.h>

namespace sng {
namespace gemm {

constexpr int TM = 128, TN = 128, TK = 64;
constexpr int kStages = 3;
constexpr int kTile = 128 * TK * 2;          // 16 KiB: 128 rows x 64 FP16
constexpr int kThreads = 192;
static_assert(TK == 64 && TM == 128 && TN == 128, "make_tma_map_f16 loads 64 (K) x 128 (rows) boxes");

constexpr uint32_t kIdesc = f16_idesc(TM, TN);

struct Params {
    int m, n, kblocks, accumulate;         // accumulate != 0: out += result (K segments of a long contraction, see the host entry)
    const float* row_scale; const float* col_scale;
    float* out; int64_t ldo;
};

__global__ void __launch_bounds__(kThreads) gemm_nt_f16_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                                                              const Params p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t a_off = 0, b_off = kStages * kTile, bar_off = 2 * kStages * kTile;
    const uint32_t bar_full = base + bar_off, bar_empty = bar_full + 8 * kStages, bar_acc = bar_empty + 8 * kStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + bar_off + 8 * (2 * kStages + 1));
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    } else if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int kb = 0; kb < p.kblocks; ++kb) {
                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                mbar_expect_tx(bar_full + 8 * stage, 2u * kTile);
                tma_load_2d(base + a_off + (uint32_t)stage * kTile, &map_a, bar_full + 8 * stage, kb * TK, m0);
                tma_load_2d(base + b_off + (uint32_t)stage * kTile, &map_b, bar_full + 8 * stage, kb * TK, n0);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int kb = 0; kb < p.kblocks; ++kb) {
                mbar_wait(bar_full + 8 * stage, phase);
                tc_fence_after();
                const uint64_t adesc = make_smem_desc(base + a_off + (uint32_t)stage * kTile);
                const uint64_t bdesc = make_smem_desc(base + b_off + (uint32_t)stage * kTile);
#pragma unroll
                for (int ks = 0; ks < TK / 16; ++ks)               // one K step = 16 elements = 32 bytes = 2 descriptor units
                    umma_f16(tmem, adesc + (uint64_t)(ks * 2), bdesc + (uint64_t)(ks * 2), kIdesc, (kb | ks) != 0 ? 1u : 0u);
                umma_commit(bar_empty + 8 * stage);                // frees the stage when the MMAs that read it retire
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
            umma_commit(bar_acc);                                  // accumulator complete
        }
    } else {
        // epilogue: thread = one output row (TMEM lane = 32 * (warp % 4) + lane)
        const int quarter = warp & 3;
        const int r = quarter * 32 + lane;
        const int row = m0 + r;
        mbar_wait(bar_acc, 0);
        tc_fence_after();
        const float rs = (p.row_scale && row < p.m) ? __ldg(p.row_scale + row) : 1.0f;
        const bool vec = (p.ldo % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
#pragma unroll 1
        for (int c = 0; c < TN / 32; ++c) {
            uint32_t v[32];
            tmem_ld32(tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c * 32), v);
            tmem_ld_wait();
            if (row < p.m) {
                const int col0 = n0 + c * 32;
                float* o = p.out + (int64_t)row * p.ldo + col0;
                if (vec && col0 + 32 <= p.n) {
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        float4 w;
                        w.x = __uint_as_float(v[i]) * rs; w.y = __uint_as_float(v[i + 1]) * rs;
                        w.z = __uint_as_float(v[i + 2]) * rs; w.w = __uint_as_float(v[i + 3]) * rs;
                        if (p.col_scale) {
                            const float4 cs = ldg4(p.col_scale + col0 + i);
                            w.x *= cs.x; w.y *= cs.y; w.z *= cs.z; w.w *= cs.w;
                        }
                        if (p.accumulate) { const float4 prev = *reinterpret_cast<const float4*>(o + i); w.x += prev.x; w.y += prev.y; w.z += prev.z; w.w += prev.w; }
                        *reinterpret_cast<float4*>(o + i) = w;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (col0 + i < p.n) o[i] = __uint_as_float(v[i]) * rs * (p.col_scale ? __ldg(p.col_scale + col0 + i) : 1.0f) + (p.accumulate ? o[i] : 0.f);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem) : "memory");
    }
}

}  // namespace gemm
}  // namespace sng

using namespace sng;

extern "C" int sng_gemm_nt_f16(const uint16_t* a, int64_t lda, const uint16_t* b, int64_t ldb, int64_t m, int64_t n, int64_t k,
                               const float* row_scale, const float* col_scale, float* out, int64_t ldo, void* stream) {
    SNG_REQUIRE(a && b && out && m > 0 && n > 0 && k > 0 && m < (1ll << 31) && n < (1ll << 31) && k < (1ll << 30), "sng_gemm_nt_f16: bad sizes");
    SNG_REQUIRE(lda >= k && ldb >= k && lda % 8 == 0 && ldb % 8 == 0 && ldo >= n, "sng_gemm_nt_f16: lda / ldb must be multiples of 8 and >= k, ldo >= n");
    SNG_REQUIRE(((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0, "sng_gemm_nt_f16: operands must be 16-byte aligned");
    SNG_REQUIRE((m + gemm::TM - 1) / gemm::TM < 65536, "sng_gemm_nt_f16: m too large for one launch");
    const size_t smem = 1024 + 2 * gemm::kStages * gemm::kTile + 8 * (2 * gemm::kStages + 1) + 16;
    cudaError_t e = cudaFuncSetAttribute(gemm::gemm_nt_f16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("sng_gemm_nt_f16: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return SNG_ERR_CUDA; }
    dim3 grid((unsigned)((n + gemm::TN - 1) / gemm::TN), (unsigned)((m + gemm::TM - 1) / gemm::TM));
    // The tensor cores add into their FP32 accumulators with truncation: ~2.5e-9 of the accumulated magnitude per product.  A
    // long contraction is therefore cut into K segments of 1024 whose results are added in the epilogue with IEEE FP32 adds
    // (out += segment), which keeps unit-row products within ~5e-6 whatever K is.
    const int64_t kseg = 1024;
    for (int64_t k0 = 0; k0 < k; k0 += kseg) {
        const int64_t kk = k - k0 < kseg ? k - k0 : kseg;
        CUtensorMap ma, mb;
        if (int rc = make_tma_map_f16(&ma, a + k0, m, kk, lda, 1)) return rc;
        if (int rc = make_tma_map_f16(&mb, b + k0, n, kk, ldb, 1)) return rc;
        gemm::Params p;
        p.m = (int)m; p.n = (int)n; p.kblocks = (int)((kk + gemm::TK - 1) / gemm::TK); p.accumulate = k0 > 0;
        p.row_scale = row_scale; p.col_scale = col_scale; p.out = out; p.ldo = ldo;
        gemm::gemm_nt_f16_kernel<<<grid, gemm::kThreads, smem, (cudaStream_t)stream>>>(ma, mb, p);
    }
    return check_launch("sng_gemm_nt_f16");
}

// ------------------------------------------------------------------------------------------ sparse columns
// Cosine between COLUMNS of a sparse matrix at given column pairs, by merging the two sorted row-index lists (CSC with sorted,
// duplicate-free indices): s[e] = inv_norm[a] inv_norm[b] sum_k M[k, a] M[k, b].  This is the adjacency-as-features cosine
// of R: SimGFAToolbox/sparse.py:8-14 evaluated only where the edge metrics need it (:44-119), without densifying anything.
namespace sng {
__global__ void __launch_bounds__(256) sparse_col_cos_kernel(const int* __restrict__ indptr, const int* __restrict__ indices, const float* __restrict__ data,
                                                            const float* __restrict__ inv_norm, const int* __restrict__ a, const int* __restrict__ b,
                                                            int64_t ne, float* __restrict__ s) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < ne; e += (int64_t)gridDim.x * blockDim.x) {
        const int ca = __ldg(a + e), cb = __ldg(b + e);
        int i = __ldg(indptr + ca), j = __ldg(indptr + cb);
        const int ie = __ldg(indptr + ca + 1), je = __ldg(indptr + cb + 1);
        double acc = 0.0;
        while (i < ie && j < je) {
            const int ri = __ldg(indices + i), rj = __ldg(indices + j);
            if (ri == rj) { acc += (double)__ldg(data + i) * (double)__ldg(data + j); ++i; ++j; }
            else if (ri < rj) ++i;
            else ++j;
        }
        s[e] = (float)(acc * (double)__ldg(inv_norm + ca) * (double)__ldg(inv_norm + cb));
    }
}
}  // namespace sng

extern "C" int sng_sparse_col_cos(const int32_t* indptr, const int32_t* indices, const float* data, const float* inv_norm, const int32_t* a,
                                  const int32_t* b, int64_t num_pairs, float* s, void* stream) {
    SNG_REQUIRE(indptr && indices && data && inv_norm && a && b && s && num_pairs >= 0, "sng_sparse_col_cos: bad arguments");
    if (num_pairs == 0) return SNG_OK;
    sng::sparse_col_cos_kernel<<<grid_capped(num_pairs, 256, 8), 256, 0, (cudaStream_t)stream>>>(indptr, indices, data, inv_norm, a, b, num_pairs, s);
    return check_launch("sng_sparse_col_cos");
}
