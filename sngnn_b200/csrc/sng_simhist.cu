// Histogram of all node-pair cosine similarities (the distribution behind R: SimGFAToolbox/plot.py
// plot_similarity_distribution, whose values R: SimGFAToolbox/dense.py:144-149 gets from the N x N matrix) without the
// N x N matrix: a tcgen05 contraction whose epilogue bins the scores in shared memory.
//
// Scores: A = [hi | hi | lo], B = [hi | lo | hi] of the FP16 split x-hat = hi + lo (as sng_gemm_nt_f16), contracted over
// K' = 3d: the FP32 product to ~2^-22.  The tensor cores truncate while they accumulate, so K' is cut into segments of
// 1024 whose accumulators the epilogue adds with IEEE FP32 adds.
//
// Symmetric schedule: T = ceil(N / 128) row tiles; one CTA per row tile I scores the tile pairs (I, (I + s) mod T) for
// s = 0 .. floor(T / 2), the pair at s = T / 2 (T even) only when I < T / 2.  Every unordered tile pair is scored exactly
// once, every row tile does the same work, so a contiguous range of row tiles is a balanced shard.  Every counted score
// stands for two ordered pairs (i, j) and (j, i): off-diagonal tiles count all their valid scores, the diagonal tile counts
// i < j, rows >= N (TMA zero fill) are never counted, and the result is the histogram of the N (N - 1) off-diagonal values.
//
// Counting: unsigned 32-bit shared-memory sub-histograms (H copies, epilogue thread t uses copy t mod H, so lanes of a warp
// that hit the same bin mostly hit different copies), flushed as 2 x count with 64-bit integer atomics into `counts` at
// the end and every kFlushTiles tiles (no copy can pass 2^30 in between).  Integer adds only: the counts are the same bits
// whatever the run, the tile split or the world size.
//
// Warps: 0 = TMA producer (A block of the row tile resident in shared memory when K' <= 384, else streamed with B through
// the ring), 1 = MMA issuer (M = N = 128, two TMEM accumulator stages of 128 columns), 2-9 = epilogue (tcgen05.ld; warp w
// reads TMEM lanes 32 (w mod 4) .. + 32, i.e. one row per thread, and columns 64 ((w - 2) / 4) .. + 64).
#include "sng_sm100.cuh"
#include <math.h>

namespace sng {
namespace simhist {

constexpr int TM = 128, TK = 64;
constexpr int kTile = 128 * TK * 2;              // 16 KiB: 128 rows x 64 FP16
constexpr int kStages = 4;
constexpr int kAcc = 2;                          // TMEM accumulator stages
constexpr int kEpiWarps = 8, kEpiThreads = 32 * kEpiWarps;
constexpr int kThreads = 64 + kEpiThreads;
constexpr int kMaxResidentKb = 6;                // resident A block <= 96 KiB (K' <= 384, d <= 128)
constexpr int kSegKb = 16;                       // K segment = 1024 = 16 K blocks
constexpr int kHistBytes = 64 * 1024;            // shared memory of the sub-histograms
constexpr int kFlushTiles = 1 << 16;             // per tile a copy gains <= 64 x 256 = 2^14 counts -> <= 2^30 between flushes
constexpr uint32_t kIdesc = f16_idesc(TM, 128);
static_assert(kEpiWarps == 8, "two epilogue warps per TMEM lane quarter, 64 columns each");
static_assert(SNG_SIMHIST_MAX_BINS * 4 * 2 <= kHistBytes, "at least two sub-histograms must fit at the largest bin count");

struct Params {
    int n, t, tile_lo, kblocks, nseg, resident;
    float lo, hi, scale;                         // bin = floor((s - lo) * scale), scale = bins / (hi - lo)
    int bins, stride, copies;                    // sub-histogram c lives at hist + c * stride (stride odd: copies spread over banks)
    unsigned long long* counts;
};

__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }

// adds 2 x (sum of the copies) of every bin into counts and clears the copies; epilogue threads only
__device__ __forceinline__ void flush(uint32_t* hist, const Params& p, int et) {
    epi_sync();
    for (int b = et; b < p.bins; b += kEpiThreads) {
        unsigned long long s = 0;
        for (int c = 0; c < p.copies; ++c) { s += hist[c * p.stride + b]; hist[c * p.stride + b] = 0; }
        if (s) atomicAdd(p.counts + b, 2ull * s);
    }
    epi_sync();
}

__global__ void __launch_bounds__(kThreads, 1) simhist_f16_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                                                                  const Params p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t stage_bytes = p.resident ? kTile : 2 * kTile;        // [A |] B of one K block
    const uint32_t ring_off = p.resident ? (uint32_t)p.kblocks * kTile : 0u;
    const uint32_t bar_off = ring_off + kStages * stage_bytes;
    const uint32_t bar_full = base + bar_off, bar_empty = bar_full + 8 * kStages, bar_accf = bar_empty + 8 * kStages,
                   bar_acce = bar_accf + 8 * kAcc, bar_a = bar_acce + 8 * kAcc;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + bar_off + 8 * (2 * kStages + 2 * kAcc + 1));
    uint32_t* hist = reinterpret_cast<uint32_t*>(smem + bar_off + 8 * (2 * kStages + 2 * kAcc + 2));

    const int I = p.tile_lo + blockIdx.x;
    const int ntiles = p.t / 2 + ((p.t & 1) || I < p.t / 2 ? 1 : 0);     // s = 0 .. ntiles - 1

    for (int i = threadIdx.x; i < p.copies * p.stride; i += kThreads) hist[i] = 0;
    if (warp == 0 && lane == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int s = 0; s < kAcc; ++s) { mbar_init(bar_accf + 8 * s, 1); mbar_init(bar_acce + 8 * s, kEpiWarps); }
        mbar_init(bar_a, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    } else if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(128 * kAcc) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            if (p.resident) {
                mbar_expect_tx(bar_a, (uint32_t)p.kblocks * kTile);
                for (int kb = 0; kb < p.kblocks; ++kb) tma_load_2d(base + (uint32_t)kb * kTile, &map_a, bar_a, kb * TK, I * TM);
            }
            int stage = 0; uint32_t phase = 0;
            for (int s = 0; s < ntiles; ++s) {
                int J = I + s; if (J >= p.t) J -= p.t;
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    const uint32_t dst = base + ring_off + (uint32_t)stage * stage_bytes;
                    mbar_expect_tx(bar_full + 8 * stage, stage_bytes);
                    if (!p.resident) tma_load_2d(dst + kTile, &map_a, bar_full + 8 * stage, kb * TK, I * TM);
                    tma_load_2d(dst, &map_b, bar_full + 8 * stage, kb * TK, J * TM);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            if (p.resident) { mbar_wait(bar_a, 0); tc_fence_after(); }
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t aphase = 0;
            for (int s = 0; s < ntiles; ++s) {
                for (int seg = 0; seg < p.nseg; ++seg) {
                    mbar_wait(bar_acce + 8 * acc, aphase ^ 1);
                    tc_fence_after();
                    const uint32_t d = tmem + (uint32_t)(acc * 128);
                    const int kb0 = seg * kSegKb, kb1 = min(p.kblocks, kb0 + kSegKb);
                    for (int kb = kb0; kb < kb1; ++kb) {
                        mbar_wait(bar_full + 8 * stage, phase);
                        tc_fence_after();
                        const uint32_t st = base + ring_off + (uint32_t)stage * stage_bytes;
                        const uint64_t adesc = make_smem_desc(p.resident ? base + (uint32_t)kb * kTile : st + kTile);
                        const uint64_t bdesc = make_smem_desc(st);
#pragma unroll
                        for (int ks = 0; ks < TK / 16; ++ks)           // one K step = 16 elements = 32 bytes = 2 descriptor units
                            umma_f16(d, adesc + (uint64_t)(ks * 2), bdesc + (uint64_t)(ks * 2), kIdesc, (kb > kb0 || ks > 0) ? 1u : 0u);
                        umma_commit(bar_empty + 8 * stage);            // frees the stage when the MMAs that read it retire
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(bar_accf + 8 * acc);                   // segment accumulator complete
                    if (++acc == kAcc) { acc = 0; aphase ^= 1; }
                }
            }
        }
    } else {
        const int et = threadIdx.x - 64;
        const int quarter = warp & 3, half = (warp - 2) >> 2;
        const int r = quarter * 32 + lane;
        const int row = I * TM + r;
        uint32_t* my = hist + (et % p.copies) * p.stride;
        const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 64);
        int acc = 0; uint32_t aphase = 0;
        int since_flush = 0;
#pragma unroll 1
        for (int s = 0; s < ntiles; ++s) {
            int J = I + s; if (J >= p.t) J -= p.t;
            float v[64];
#pragma unroll 1
            for (int seg = 0; seg < p.nseg; ++seg) {
                mbar_wait(bar_accf + 8 * acc, aphase);
                tc_fence_after();
                uint32_t u0[32], u1[32];
                tmem_ld32(taddr + (uint32_t)(acc * 128), u0);
                tmem_ld32(taddr + (uint32_t)(acc * 128 + 32), u1);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_acce + 8 * acc);       // the accumulator is in registers: MMA may reuse it
                if (++acc == kAcc) { acc = 0; aphase ^= 1; }
                if (seg == 0) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) { v[i] = __uint_as_float(u0[i]); v[32 + i] = __uint_as_float(u1[i]); }
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) { v[i] += __uint_as_float(u0[i]); v[32 + i] += __uint_as_float(u1[i]); }
                }
            }
            // columns c of this thread's row that count: c0 <= c < c1 (diagonal tile: j > i only; columns and rows < N)
            const int c0 = (s == 0 ? r + 1 : 0) - half * 64;
            const int c1 = (row < p.n ? min(TM, p.n - J * TM) : 0) - half * 64;
#pragma unroll
            for (int i = 0; i < 64; ++i) {
                const float x = fminf(fmaxf(v[i], -1.0f), 1.0f);        // the exact cosine never leaves [-1, 1]
                const int b = min(max(__float2int_rd((x - p.lo) * p.scale), 0), p.bins - 1);
                if (i >= c0 && i < c1 && x >= p.lo && x <= p.hi) atomicAdd(my + b, 1u);
            }
            if (++since_flush == kFlushTiles) { flush(hist, p, et); since_flush = 0; }
        }
        flush(hist, p, et);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(128 * kAcc) : "memory");
    }
}

}  // namespace simhist
}  // namespace sng

using namespace sng;

extern "C" int sng_simhist_f16(const uint16_t* a, int64_t lda, const uint16_t* b, int64_t ldb, int64_t n, int64_t k, int64_t tile_lo,
                               int64_t tile_hi, float lo, float hi, int bins, uint64_t* counts, void* stream) {
    SNG_REQUIRE(a && b && counts && n > 0 && n < (1ll << 31) && k > 0 && k < (1ll << 30), "sng_simhist_f16: bad sizes (0 < n < 2^31, 0 < k < 2^30)");
    SNG_REQUIRE(lda >= k && ldb >= k && lda % 8 == 0 && ldb % 8 == 0, "sng_simhist_f16: lda / ldb must be multiples of 8 and >= k");
    SNG_REQUIRE(((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0, "sng_simhist_f16: operands must be 16-byte aligned");
    SNG_REQUIRE(bins >= 1 && bins <= SNG_SIMHIST_MAX_BINS, "sng_simhist_f16: bins = %d outside [1, %d]", bins, SNG_SIMHIST_MAX_BINS);
    SNG_REQUIRE(isfinite(lo) && isfinite(hi) && lo < hi && isfinite(hi - lo), "sng_simhist_f16: the range must be finite with lo < hi (got %g, %g)", (double)lo, (double)hi);
    const int64_t t = (n + simhist::TM - 1) / simhist::TM;
    SNG_REQUIRE(0 <= tile_lo && tile_lo <= tile_hi && tile_hi <= t, "sng_simhist_f16: tile range [%lld, %lld) outside [0, %lld)",
                (long long)tile_lo, (long long)tile_hi, (long long)t);
    if (tile_lo == tile_hi) return SNG_OK;

    simhist::Params p;
    p.n = (int)n; p.t = (int)t; p.tile_lo = (int)tile_lo;
    p.kblocks = (int)((k + simhist::TK - 1) / simhist::TK);
    p.nseg = (p.kblocks + simhist::kSegKb - 1) / simhist::kSegKb;
    p.resident = p.kblocks <= simhist::kMaxResidentKb;
    p.lo = lo; p.hi = hi; p.scale = (float)bins / (hi - lo);
    p.bins = bins; p.stride = bins | 1;
    p.copies = simhist::kEpiThreads;
    while (p.copies > 1 && (int64_t)p.copies * p.stride * 4 > simhist::kHistBytes) p.copies >>= 1;
    p.counts = reinterpret_cast<unsigned long long*>(counts);

    CUtensorMap ma, mb;
    if (int rc = make_tma_map_f16(&ma, a, n, k, lda, 1)) return rc;
    if (int rc = make_tma_map_f16(&mb, b, n, k, ldb, 1)) return rc;
    const size_t stage_bytes = p.resident ? simhist::kTile : 2 * simhist::kTile;
    const size_t smem = 1024 + (p.resident ? (size_t)p.kblocks * simhist::kTile : 0) + simhist::kStages * stage_bytes +
                        8 * (2 * simhist::kStages + 2 * simhist::kAcc + 2) + (size_t)p.copies * p.stride * 4;
    cudaError_t e = cudaFuncSetAttribute(simhist::simhist_f16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("sng_simhist_f16: cudaFuncSetAttribute(%zu bytes): %s", smem, cudaGetErrorString(e)); return SNG_ERR_CUDA; }
    simhist::simhist_f16_kernel<<<(unsigned)(tile_hi - tile_lo), simhist::kThreads, smem, (cudaStream_t)stream>>>(ma, mb, p);
    return check_launch("sng_simhist_f16");
}
