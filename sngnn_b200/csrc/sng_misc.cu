// Small data-format kernels either side of the hot path: kNN lists -> CSR, the unfused SNGNN++ backward, segmented means.
#include "sng_common.cuh"
#include <cub/device/device_scan.cuh>

namespace sng {

__global__ void __launch_bounds__(256) clamp_counts_kernel(const int* __restrict__ cnt, int64_t nq, int k, int* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= nq; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = i < nq ? min(max(__ldg(cnt + i), 0), k) : 0;
}

// one thread per list slot: slot (r, t) with t < cnt[r] lands at rowptr[r] + t (rank order is kept)
__global__ void __launch_bounds__(256) knn_compact_kernel(const int* __restrict__ rowptr, const int* __restrict__ idx, const float* __restrict__ sim,
                                                         int64_t nq, int k, int* __restrict__ col, float* __restrict__ val) {
    const int64_t total = nq * k;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / k;
        const int t = (int)(e - r * k);
        const int b = __ldg(rowptr + r);
        if (t < __ldg(rowptr + r + 1) - b) {
            col[b + t] = __ldg(idx + e);
            if (val) val[b + t] = __ldg(sim + e);
        }
    }
}

// g0 = beta g, g1 = (1 - beta) g
__global__ void __launch_bounds__(256) beta_split_kernel(const float* __restrict__ g, const float* __restrict__ beta_p, int64_t n4,
                                                        float* __restrict__ g0, float* __restrict__ g1) {
    const float beta = __ldg(beta_p);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = ldg4(g + 4 * i);
        reinterpret_cast<float4*>(g0)[i] = scale4(v, beta);
        reinterpret_cast<float4*>(g1)[i] = scale4(v, 1.0f - beta);
    }
}

__global__ void __launch_bounds__(256) segment_accum_kernel(const float* __restrict__ val, const int* __restrict__ seg, int64_t ne, int n_seg,
                                                           double* __restrict__ sums, int* __restrict__ counts) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < ne; e += (int64_t)gridDim.x * blockDim.x) {
        const int s = __ldg(seg + e);
        if (s >= 0 && s < n_seg) { atomicAdd(sums + s, (double)__ldg(val + e)); atomicAdd(counts + s, 1); }
    }
}

__global__ void __launch_bounds__(256) segment_finish_kernel(const double* __restrict__ sums, const int* __restrict__ counts, int n_seg,
                                                            float* __restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_seg; i += gridDim.x * blockDim.x)
        out[i] = (float)(sums[i] / (double)max(counts[i], 1));
}

}  // namespace sng

using namespace sng;

extern "C" size_t sng_knn_to_csr_workspace_bytes(int64_t nq) {
    if (nq < 0 || nq >= (1ll << 31) - 1) return 0;
    size_t t = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, t, (const int*)nullptr, (int*)nullptr, (int)(nq + 1));
    return t + (size_t)(nq + 1) * 4 + 512;
}

extern "C" int sng_knn_to_csr(const int32_t* idx, const float* sim, const int32_t* cnt, int64_t nq, int top_k, int32_t* rowptr, int32_t* col,
                              float* val, void* workspace, size_t workspace_bytes, void* stream) {
    SNG_REQUIRE(idx && cnt && rowptr && col && workspace && nq >= 0 && top_k >= 1 && nq * (int64_t)top_k < (1ll << 31), "sng_knn_to_csr: bad arguments");
    SNG_REQUIRE(!val || sim, "sng_knn_to_csr: val needs sim");
    if (workspace_bytes < sng_knn_to_csr_workspace_bytes(nq)) { set_error("sng_knn_to_csr: workspace too small"); return SNG_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    int* clamped = reinterpret_cast<int*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    void* temp = reinterpret_cast<uint8_t*>(clamped) + (((size_t)(nq + 1) * 4 + 255) & ~(size_t)255);
    size_t temp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, (const int*)nullptr, (int*)nullptr, (int)(nq + 1));
    clamp_counts_kernel<<<grid_capped(nq + 1, 256, 8), 256, 0, st>>>(cnt, nq, top_k, clamped);
    if (cub::DeviceScan::ExclusiveSum(temp, temp_bytes, clamped, rowptr, (int)(nq + 1), st) != cudaSuccess) return check_launch("sng_knn_to_csr scan");
    if (nq > 0) knn_compact_kernel<<<grid_capped(nq * top_k, 256, 8), 256, 0, st>>>(rowptr, idx, sim, nq, top_k, col, val);
    return check_launch("sng_knn_to_csr");
}

extern "C" int sng_pp_fuse_bwd(const float* out0, const float* out1, const float* g, const float* beta, int64_t n, int64_t c, int64_t ld,
                               const int32_t* rowptr_in, const int32_t* col_in_shift, float* dbeta, float* partials, float* g0, float* dout1,
                               float* dwt, void* stream) {
    SNG_REQUIRE(out0 && out1 && g && beta && rowptr_in && col_in_shift && dbeta && partials && g0 && dout1 && dwt, "sng_pp_fuse_bwd: null pointer");
    SNG_REQUIRE(n >= 0 && c > 0 && c % 4 == 0 && ld == c, "sng_pp_fuse_bwd: rows must be contiguous with a multiple of 4 channels");
    if (n == 0) return SNG_OK;
    if (int rc = sng_pp_beta_grad(out0, out1, g, n * c, dbeta, partials, stream)) return rc;
    beta_split_kernel<<<grid_capped(n * c / 4, 256, 8), 256, 0, (cudaStream_t)stream>>>(g, beta, n * c / 4, g0, dout1);
    if (int rc = check_launch("sng_pp_fuse_bwd split")) return rc;
    return sng_spmm_fwd(g0, n, c, c, rowptr_in, col_in_shift, nullptr, nullptr, nullptr, dwt, c, stream);   // dL/dW^T = A^T g0
}

extern "C" int sng_segment_mean(const float* val, const int32_t* seg, int64_t num, int64_t n_seg, float* out, void* workspace,
                                size_t workspace_bytes, void* stream) {
    SNG_REQUIRE(val && seg && out && workspace && num >= 0 && n_seg > 0 && n_seg < (1ll << 31), "sng_segment_mean: bad arguments");
    SNG_REQUIRE(workspace_bytes >= (size_t)n_seg * 12 + 256, "sng_segment_mean: workspace needs 12 bytes per segment + 256");
    cudaStream_t st = (cudaStream_t)stream;
    double* sums = reinterpret_cast<double*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    int* counts = reinterpret_cast<int*>(sums + n_seg);
    if (cudaMemsetAsync(sums, 0, (size_t)n_seg * 12, st) != cudaSuccess) return check_launch("sng_segment_mean memset");
    if (num > 0) segment_accum_kernel<<<grid_capped(num, 256, 8), 256, 0, st>>>(val, seg, num, (int)n_seg, sums, counts);
    segment_finish_kernel<<<grid_capped(n_seg, 256, 8), 256, 0, st>>>(sums, counts, (int)n_seg, out);
    return check_launch("sng_segment_mean");
}

// ------------------------------------------------------------------------------------------ lin + bias + 1/norm (SURVEY.md §8(f) 2)
// h = x W^T + b with the output width zero-padded to cp, and inv_norm[i] = 1 / max(||h_i||, 1e-12), in one pass over x
// (R: models/models.py:121-122 `x = self.lin(x); norm = F.normalize(x)`; the library GEMM + separate norm pass it replaces
// reads h twice more).  FP32 FMA on the CUDA cores: at the shapes of this path (F x C <= 24 K weights) the layer is
// bound by reading x, not by arithmetic.  Block = 256 threads; a thread owns 4 rows x 4 channels; x is staged TRANSPOSED
// in K chunks of 32 (one 128-bit shared load = the 4 rows of a thread), W^T chunks beside it.
namespace sng {
constexpr int kLinKC = 32;

__device__ __forceinline__ void cp_async4(float* dst, const float* src, bool ok) {       // 4-byte async copy; !ok writes a zero
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "r"(ok ? 4 : 0) : "memory");
}

__device__ __forceinline__ void cp_async16z(float* dst, const float* src, bool ok) {     // 16-byte async copy; !ok writes zeros
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "r"(ok ? 16 : 0) : "memory");
}

template <int CG>                                   // CG = cp / 4 channel groups per row (power of two <= 32)
__global__ void __launch_bounds__(256) lin_norm_kernel(const float* __restrict__ x, int64_t n, int f, int64_t ldx, const float* __restrict__ w, int c,
                                                      int64_t ldw, const float* __restrict__ bias, float* __restrict__ h, float* __restrict__ inv) {
    constexpr int KC = CG <= 2 ? 16 : kLinKC;       // K chunk (narrow outputs have 512 / 1024 rows per tile: a shorter chunk keeps the tile in shared memory)
    constexpr int RG = 256 / CG;                    // row groups per block
    constexpr int R = RG * 4;                       // rows per block tile
    constexpr int RS = R;                           // row stride of the transposed x tile; groups of 4 rows are XOR-swizzled by kk & 7
    constexpr int cp = CG * 4;
    constexpr int XB = KC * RS, WB = KC * cp;
    extern __shared__ float sm[];
    float* xs = sm;                                 // 2 x [KC][RS]   (x chunk, transposed: 4-byte cp.async, two chunks in flight)
    float* ws = sm + 2 * XB;                        // 2 x [KC][cp]
    const int cg = threadIdx.x % CG, rg = threadIdx.x / CG;
    const int nkc = (f + KC - 1) / KC;
    const int64_t ntiles = (n + R - 1) / R;
    const int64_t my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t total = my_tiles * nkc;           // flattened (row tile, K chunk) sequence of this block

    auto stage = [&](int64_t it) {                  // chunk `it` -> buffer it & 1 (an empty group beyond the end keeps the counting uniform)
        if (it < total) {
            const int64_t r0 = (blockIdx.x + (it / nkc) * gridDim.x) * R;
            const int k0 = (int)(it % nkc) * KC;
            float* xb = xs + (it & 1) * XB;
            float* wb = ws + (it & 1) * WB;
            // a warp copies 4 rows x 8 consecutive k (32-byte segments of global memory) and stores them transposed: row group
            // (4 rows = one 128-bit read of the compute loop) XOR (k & 7) makes the 32 stores of a warp hit 32 different banks
#pragma unroll 4
            for (int t = threadIdx.x; t < R * KC; t += 256) {
                const int l = t & 31, s = t >> 5;
                const int kk = (s % (KC / 8)) * 8 + (l & 7), rr = (s / (KC / 8)) * 4 + (l >> 3);
                const int64_t row = r0 + rr;
                if (k0 + kk < f)                                                  // columns beyond f are never read by the compute loop
                    cp_async4(xb + kk * RS + ((((rr >> 2) ^ (kk & 7))) << 2) + (rr & 3), row < n ? x + row * ldx + k0 + kk : x, row < n);
            }
            for (int t = threadIdx.x; t < cp * KC; t += 256) {
                const int cc = t / KC, kk = t % KC;
                if (k0 + kk < f) cp_async4(wb + kk * cp + cc, cc < c ? w + (int64_t)cc * ldw + k0 + kk : w, cc < c);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) {
        b4.x = cg * 4 + 0 < c ? __ldg(bias + cg * 4 + 0) : 0.f; b4.y = cg * 4 + 1 < c ? __ldg(bias + cg * 4 + 1) : 0.f;
        b4.z = cg * 4 + 2 < c ? __ldg(bias + cg * 4 + 2) : 0.f; b4.w = cg * 4 + 3 < c ? __ldg(bias + cg * 4 + 3) : 0.f;
    }
    float acc[4][4];
    stage(0);
    for (int64_t it = 0; it < total; ++it) {
        stage(it + 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        const int kc = (int)(it % nkc);
        if (kc == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        }
        const float* xb = xs + (it & 1) * XB;
        const float* wb = ws + (it & 1) * WB;
        const int kmax = min(KC, f - kc * KC);                                    // the K tail is not padded with zero work
#pragma unroll 8
        for (int kk = 0; kk < kmax; ++kk) {
            const float4 xv = *reinterpret_cast<const float4*>(xb + kk * RS + ((rg ^ (kk & 7)) << 2));
            const float4 wv = *reinterpret_cast<const float4*>(wb + kk * cp + cg * 4);
            const float xr[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                acc[i][0] = fmaf(xr[i], wv.x, acc[i][0]); acc[i][1] = fmaf(xr[i], wv.y, acc[i][1]);
                acc[i][2] = fmaf(xr[i], wv.z, acc[i][2]); acc[i][3] = fmaf(xr[i], wv.w, acc[i][3]);
            }
        }
        if (kc == nkc - 1) {
            const int64_t r0 = (blockIdx.x + (it / nkc) * gridDim.x) * R;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int64_t row = r0 + rg * 4 + i;
                const float4 o = make_float4(acc[i][0] + b4.x, acc[i][1] + b4.y, acc[i][2] + b4.z, acc[i][3] + b4.w);   // padding channels stay 0
                float ss = dot4(o, o);
                ss = group_sum<CG>(ss);                                            // the CG threads of a row are consecutive lanes
                if (row < n) {
                    *reinterpret_cast<float4*>(h + row * cp + cg * 4) = o;
                    if (inv && cg == 0) inv[row] = inv_norm_of(ss);
                }
            }
        }
        __syncthreads();                                                           // the buffer is refilled by the next stage()
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}
}  // namespace sng

// ------------------------------------------------------------------------------------------ lin backward: dW = g^T x, db = sum g
// The weight gradient of `x = self.lin(x)` (R: models/models.py:121): dW [c, f] = sum_n g[n, :]^T x[n, :], db [c] = sum_n g[n, :].
// A reduction over N (10^6) rows with a tiny output: the library GEMM runs it as one skinny split-K kernel at 10-20 % of the
// bandwidth this takes (0.86 ms at the pokec shape, c = 32, f = 65, where reading g and x once costs 0.1 ms).  Here every CTA
// streams a contiguous range of rows through shared memory (cp.async, two tiles in flight).  A thread owns 4 channels
// (consecutive) x 4 columns (ft, ft + FT, ft + 2 FT, ft + 3 FT: consecutive lanes read consecutive words, so the tile needs no
// 16-byte row alignment) of the output in registers; RG row groups of FT x CT threads split the rows of a tile and are
// summed in shared memory at the end; the CTA writes one partial [c4, 4 FT], and a second kernel adds the partials of all
// row chunks in a fixed order: deterministic, no float atomics.
// FLAT staging (x contiguous, ldx == f): a tile of 32 rows is one contiguous, 16-byte aligned block of memory whatever f is
// (32 f floats), so it is copied with 16-byte cp.async in the layout it has (row stride f) -- a few instructions per tile where
// element-wise 4-byte copies of rows that start at odd addresses (f = 65) cost more than the arithmetic.
namespace sng {
constexpr int kLbRows = 32;                         // rows per shared-memory tile (small tiles: 6-8 CTAs per SM hide the barriers)
constexpr int kLbMaxF = 128;                        // widest x this kernel takes (one slab of 4 x 32 columns)

struct LinBwdPlan { int ft, ct, rg, threads, nchunk; bool flat; size_t smem; };

template <int RG, bool FLAT>
__global__ void lin_bwd_partial_kernel(const float* __restrict__ g, int64_t ldg, const float* __restrict__ x, int64_t ldx, int64_t n, int f, int c,
                                       int FT, int CT, int64_t rows_per_chunk, float* __restrict__ part, float* __restrict__ part_b) {
    const int fslab = FT * 4, cslab = CT * 4;
    const int XS = FLAT ? f : fslab, GS = cslab + 4;
    const int xtile = FLAT ? ((kLbRows * f + 3) & ~3) + 4 * FT : kLbRows * XS;      // FLAT: columns >= f of the last row read (unused) words behind the tile
    extern __shared__ __align__(16) float lsm[];
    float* xs = lsm;                                // 2 x xtile
    float* gs = lsm + 2 * xtile;                    // 2 x [kLbRows][GS]
    const int tpg = FT * CT;                        // threads per row group
    const int t = threadIdx.x;
    const bool active = t < tpg * RG;
    const int rgi = t / tpg, tt = t % tpg, ft = tt % FT, ct = tt / FT;
    const int64_t r_beg = (int64_t)blockIdx.x * rows_per_chunk, r_end = min(n, r_beg + rows_per_chunk);
    const int ntile = r_beg < r_end ? (int)((r_end - r_beg + kLbRows - 1) / kLbRows) : 0;
    const int c4u = (c + 3) & ~3;
    const bool g16 = (ldg & 3) == 0 && ldg >= c4u && ((uintptr_t)g & 15) == 0;

    auto stage = [&](int it) {
        if (it < ntile) {
            const int64_t r0 = r_beg + (int64_t)it * kLbRows;
            float* xb = xs + (it & 1) * xtile;
            float* gb = gs + (it & 1) * kLbRows * GS;
            const int warp = t >> 5, lane = t & 31, nwarp = blockDim.x >> 5;
            if (FLAT) {
                // floats [r0 f, min(r0 + 32, r_end) f) of x: 16-byte chunks, the last one possibly partial (zero filled)
                const float* src = x + r0 * (int64_t)f;
                const int64_t valid = (min(r0 + kLbRows, r_end) - r0) * (int64_t)f;   // floats
                for (int q = t; q * 4 < kLbRows * f; q += blockDim.x) {
                    const int64_t left = valid - (int64_t)q * 4;
                    const int bytes = left >= 4 ? 16 : (left > 0 ? (int)left * 4 : 0);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(xb + q * 4)),
                                 "l"(bytes ? src + q * 4 : x), "r"(bytes) : "memory");
                }
            } else {
                for (int rr = warp; rr < kLbRows; rr += nwarp) {                    // warp per tile row, lanes across the columns
                    const bool rok = r0 + rr < r_end;
                    const float* xr = x + (r0 + rr) * ldx;
                    for (int ff = lane; ff < fslab; ff += 32) {
                        const bool ok = rok && ff < f;
                        cp_async4(xb + rr * XS + ff, ok ? xr + ff : x, ok);
                    }
                }
            }
            for (int rr = warp; rr < kLbRows; rr += nwarp) {
                const bool rok = r0 + rr < r_end;
                const float* gr = g + (r0 + rr) * ldg;
                if (g16) {
                    for (int q = lane; q < CT; q += 32) {
                        const bool ok = rok && q * 4 < c4u;
                        cp_async16z(gb + rr * GS + q * 4, ok ? gr + q * 4 : g, ok);
                    }
                } else {
                    for (int cc = lane; cc < cslab; cc += 32) {
                        const bool ok = rok && cc < c;
                        cp_async4(gb + rr * GS + cc, ok ? gr + cc : g, ok);
                    }
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    float acc[4][4], accb[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { accb[i] = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f; }
    stage(0);
    for (int it = 0; it < ntile; ++it) {
        stage(it + 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        if (active) {
            const float* xb = xs + (it & 1) * xtile + ft;
            const float* gb = gs + (it & 1) * kLbRows * GS + ct * 4;
#pragma unroll
            for (int u = 0; u < kLbRows / RG; ++u) {                               // rows beyond r_end: g was staged as zeros
                const int rr = rgi + u * RG;
                const float4 gv = *reinterpret_cast<const float4*>(gb + rr * GS);
                const float* xr = xb + rr * XS;
                const float x0 = xr[0], x1 = xr[FT], x2 = xr[2 * FT], x3 = xr[3 * FT];
                const float gr[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    acc[i][0] = fmaf(gr[i], x0, acc[i][0]); acc[i][1] = fmaf(gr[i], x1, acc[i][1]);
                    acc[i][2] = fmaf(gr[i], x2, acc[i][2]); acc[i][3] = fmaf(gr[i], x3, acc[i][3]);
                }
            }
        }
        if (t < 32) {                                                              // db: warp 0 sums the columns of the g tile (lane = channel)
            const float* gb = gs + (it & 1) * kLbRows * GS;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int ch = t + 32 * k;
                if (ch < cslab) {
#pragma unroll 8
                    for (int rr = 0; rr < kLbRows; ++rr) accb[k] += gb[rr * GS + ch];
                }
            }
        }
        __syncthreads();
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    if (t < 32) {
#pragma unroll
        for (int k = 0; k < 4; ++k) if (t + 32 * k < cslab) part_b[(size_t)blockIdx.x * cslab + t + 32 * k] = accb[k];
    }
    // sum over the row groups in a fixed order, through shared memory (the tiles are dead): red[rg][tt][16]
    float* red = lsm;
    if (active) {
        float* o = red + ((size_t)rgi * tpg + tt) * 16;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) o[i * 4 + j] = acc[i][j];
    }
    __syncthreads();
    for (int i = t; i < tpg * 16; i += blockDim.x) {
        const int tt2 = i >> 4, e = i & 15;
        float sum = 0.f;
#pragma unroll
        for (int r = 0; r < RG; ++r) sum += red[((size_t)r * tpg + tt2) * 16 + e];
        const int ft2 = tt2 % FT, ct2 = tt2 / FT;
        part[((size_t)blockIdx.x * cslab + ct2 * 4 + (e >> 2)) * fslab + ft2 + (e & 3) * FT] = sum;
    }
}

// one warp per output element: lanes stride over the row chunks, then a fixed shuffle tree (deterministic).  A thread per
// output walking ~1000 partials serially took longer than the streaming pass itself.
__global__ void __launch_bounds__(256) lin_bwd_finish_kernel(const float* __restrict__ part, const float* __restrict__ part_b, int nchunk, int cslab, int fslab,
                                                            int c, int f, float* __restrict__ dw, int64_t lddw, float* __restrict__ db) {
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int fe = db ? f + 1 : f;
    if (i >= c * fe) return;
    const int cc = i / fe, ff = i % fe;
    const float* p0 = ff < f ? part + (size_t)cc * fslab + ff : part_b + cc;
    const size_t stride = ff < f ? (size_t)cslab * fslab : (size_t)cslab;
    float s = 0.f;
    for (int k = lane; k < nchunk; k += 32) s += __ldg(p0 + (size_t)k * stride);
    s = group_sum<32>(s);
    if (lane == 0) {
        if (ff < f) dw[(int64_t)cc * lddw + ff] = s;
        else db[cc] = s;
    }
}

template <int RG, bool FLAT>
static void lin_bwd_launch(const LinBwdPlan& p, int* occ, bool launch, const float* g, int64_t ldg, const float* x, int64_t ldx, int64_t n, int f, int c,
                           int64_t rows_per_chunk, float* part, float* part_b, cudaStream_t st) {
    cudaFuncSetAttribute(lin_bwd_partial_kernel<RG, FLAT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
    if (occ && (cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, lin_bwd_partial_kernel<RG, FLAT>, p.threads, p.smem) != cudaSuccess || *occ < 1)) {
        cudaGetLastError(); *occ = 1;
    }
    if (launch)
        lin_bwd_partial_kernel<RG, FLAT><<<(unsigned)p.nchunk, p.threads, p.smem, st>>>(g, ldg, x, ldx, n, f, c, p.ft, p.ct, rows_per_chunk, part, part_b);
}
#define SNG_LB_DISPATCH(p, ...)                                                                  \
    switch ((p).rg) {                                                                            \
        case 1: if ((p).flat) lin_bwd_launch<1, true>(__VA_ARGS__); else lin_bwd_launch<1, false>(__VA_ARGS__); break;    \
        case 2: if ((p).flat) lin_bwd_launch<2, true>(__VA_ARGS__); else lin_bwd_launch<2, false>(__VA_ARGS__); break;    \
        case 4: if ((p).flat) lin_bwd_launch<4, true>(__VA_ARGS__); else lin_bwd_launch<4, false>(__VA_ARGS__); break;    \
        case 8: if ((p).flat) lin_bwd_launch<8, true>(__VA_ARGS__); else lin_bwd_launch<8, false>(__VA_ARGS__); break;    \
        case 16: if ((p).flat) lin_bwd_launch<16, true>(__VA_ARGS__); else lin_bwd_launch<16, false>(__VA_ARGS__); break; \
        default: if ((p).flat) lin_bwd_launch<32, true>(__VA_ARGS__); else lin_bwd_launch<32, false>(__VA_ARGS__); break; \
    }

static LinBwdPlan lin_bwd_plan(int64_t n, int64_t f, int64_t c, bool flat) {
    LinBwdPlan p;
    p.flat = flat;
    p.ft = (int)((f + 3) / 4);                                                     // <= 32
    p.ct = (int)((c + 3) / 4);                                                     // <= 32
    int rg = 1;
    while (rg < 32 && p.ft * p.ct * rg * 2 <= 256) rg *= 2;                        // power of two: the row loop is unrolled at compile time
    p.rg = rg;
    p.threads = (p.ft * p.ct * p.rg + 31) / 32 * 32;
    if (p.threads > 1024) p.threads = 1024;
    const size_t xtile = flat ? (size_t)((kLbRows * f + 3) & ~(int64_t)3) + 4 * p.ft : (size_t)kLbRows * p.ft * 4;
    const size_t tiles = (2 * xtile + (size_t)2 * kLbRows * (p.ct * 4 + 4)) * sizeof(float);
    const size_t red = (size_t)p.ft * p.ct * p.rg * 16 * sizeof(float);
    p.smem = tiles > red ? tiles : red;
    int occ = 1;
    SNG_LB_DISPATCH(p, p, &occ, false, nullptr, 0, nullptr, 0, 0, 0, 0, 0, nullptr, nullptr, nullptr)
    p.nchunk = grid_capped(n, 4 * kLbRows, occ);                                    // one resident wave, at least 4 tiles per CTA
    return p;
}
}  // namespace sng

// one row group must fit 256 threads (f x c <= 4096 outputs): beyond that the SIMT FMA rate, not memory, bounds the kernel and the
// library GEMM is as fast (measured at f = c = 128)
extern "C" int sng_lin_bwd_supported(int64_t f, int64_t c) { return f > 0 && c > 0 && f <= sng::kLbMaxF && c <= 128 && ((f + 3) / 4) * ((c + 3) / 4) <= 256 ? 1 : 0; }

extern "C" size_t sng_lin_bwd_workspace_bytes(int64_t n, int64_t f, int64_t c) {
    if (n <= 0 || !sng_lin_bwd_supported(f, c)) return 256;
    // chunk count bound that does not depend on the staging mode: one resident wave is at most 32 CTAs per SM
    const size_t f4 = (size_t)(f + 3) / 4 * 4, c4 = (size_t)(c + 3) / 4 * 4;
    return (size_t)sng::sm_count() * 32 * c4 * (f4 + 1) * sizeof(float) + 256;
}

extern "C" int sng_lin_bwd(const float* g, int64_t ldg, const float* x, int64_t ldx, int64_t n, int64_t f, int64_t c, float* dw, int64_t lddw,
                           float* db, void* workspace, size_t workspace_bytes, void* stream) {
    SNG_REQUIRE(dw && n >= 0 && f > 0 && c > 0 && ldg >= c && ldx >= f && lddw >= f, "sng_lin_bwd: bad arguments");
    SNG_REQUIRE(sng_lin_bwd_supported(f, c), "sng_lin_bwd: unsupported shape (f=%lld c=%lld): f <= 128, c <= 128", (long long)f, (long long)c);
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        for (int64_t r = 0; r < c; ++r) if (cudaMemsetAsync(dw + r * lddw, 0, (size_t)f * sizeof(float), st) != cudaSuccess) return check_launch("sng_lin_bwd memset");
        if (db && cudaMemsetAsync(db, 0, (size_t)c * sizeof(float), st) != cudaSuccess) return check_launch("sng_lin_bwd memset");
        return SNG_OK;
    }
    SNG_REQUIRE(g && x, "sng_lin_bwd: null input");
    SNG_REQUIRE(workspace && workspace_bytes >= sng_lin_bwd_workspace_bytes(n, f, c), "sng_lin_bwd: workspace too small (%zu < %zu)",
                workspace_bytes, sng_lin_bwd_workspace_bytes(n, f, c));
    const bool flat = ldx == f && ((uintptr_t)x & 15) == 0;
    const LinBwdPlan p = lin_bwd_plan(n, f, c, flat);
    const int cslab = p.ct * 4, fslab = p.ft * 4;
    float* part = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    float* part_b = part + (size_t)p.nchunk * cslab * fslab;
    const int64_t rows_per_chunk = ((n + p.nchunk - 1) / p.nchunk + kLbRows - 1) / kLbRows * kLbRows;
    SNG_LB_DISPATCH(p, p, nullptr, true, g, ldg, x, ldx, n, (int)f, (int)c, rows_per_chunk, part, part_b, st)
    const int64_t outs = c * (f + (db ? 1 : 0));
    lin_bwd_finish_kernel<<<(unsigned)((outs + 7) / 8), 256, 0, st>>>(part, part_b, p.nchunk, cslab, fslab, (int)c, (int)f, dw, lddw, db);
    return check_launch("sng_lin_bwd");
}

extern "C" int sng_lin_norm_supported(int64_t f, int64_t c) {
    if (f <= 0 || c <= 0) return 0;
    const int64_t cp = (c + 3) / 4 * 4;
    return (cp == 4 || cp == 8 || cp == 16 || cp == 32 || cp == 64 || cp == 128) && f * cp <= 24576 ? 1 : 0;
}

extern "C" int sng_lin_norm_fwd(const float* x, int64_t n, int64_t f, int64_t ldx, const float* w, int64_t c, int64_t ldw, const float* bias,
                                float* h, float* inv_norm, void* stream) {
    SNG_REQUIRE(x && w && h && n >= 0 && f > 0 && c > 0 && ldx >= f && ldw >= f, "sng_lin_norm_fwd: bad arguments");
    SNG_REQUIRE(sng_lin_norm_supported(f, c), "sng_lin_norm_fwd: unsupported shape (f=%lld c=%lld): padded c must be a power of two in [4,128], f*c_padded <= 24576",
                (long long)f, (long long)c);
    if (n == 0) return SNG_OK;
    const int cgn = (int)((c + 3) / 4);
    cudaStream_t st = (cudaStream_t)stream;
#define SNG_LIN_LAUNCH(CGV)                                                                                                      \
    {                                                                                                                            \
        constexpr int R = (256 / CGV) * 4;                                                                                       \
        const size_t smem = (size_t)2 * (CGV <= 2 ? 16 : kLinKC) * (R + CGV * 4) * sizeof(float);                                                  \
        cudaFuncSetAttribute(lin_norm_kernel<CGV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                      \
        lin_norm_kernel<CGV><<<grid_resident(lin_norm_kernel<CGV>, n, R, smem), 256, smem, st>>>(x, n, (int)f, ldx, w, (int)c, ldw, bias, h, inv_norm); \
    }
    switch (cgn) {
        case 1: SNG_LIN_LAUNCH(1) break;
        case 2: SNG_LIN_LAUNCH(2) break;
        case 3: case 4: SNG_LIN_LAUNCH(4) break;
        case 5: case 6: case 7: case 8: SNG_LIN_LAUNCH(8) break;
        default:
            if (cgn <= 16) SNG_LIN_LAUNCH(16) else SNG_LIN_LAUNCH(32)
            break;
    }
#undef SNG_LIN_LAUNCH
    return check_launch("sng_lin_norm_fwd");
}
