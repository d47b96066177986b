// K1: all-pairs similarity-kNN builder for sm_100a -- tcgen05.mma + TMEM accumulators + TMA operand
// staging, with the threshold / top-k selection fused into the epilogue so the N x N similarity matrix
// never exists in HBM.
//
// Replaces (as "the reference selection rule on the complete graph", SURVEY.md §0) the k-round
// scatter_max selection of R: models/models.py:145-156 and the blocked X X^T of
// R: SimGFAToolbox/dense.py:17-27.
//
// One build = seed pass -> main pass -> FP32 rescore + proof -> retry pass -> exact scan (see sng_simknn_build at the bottom).
// Seed, main and retry pass are the same kernel.  A CTA pair (cluster of 2, cta_group::2) owns 256 query rows and sweeps
// the database in 256-column tiles; one CTA per SM, 4 + 4*EW warps:
//   warp 0      TMA producer: A (the CTA's 128 query rows, all of K) once; its half of every B tile through an S-stage ring
//   warps 1-2   MMA issuers (leader CTA): tcgen05.mma.cta_group::2, FP16 in, FP32 accumulators in TMEM.  Small K (EW = 4):
//               two N = 128 halves per tile into four 128-column stages, two issuers; else one N = 256 MMA chain, two stages
//   warp 3      list warp: drains the hit queue into the per-row candidate lists (shared memory), owns the row thresholds
//   warps 4..   epilogue: thread = one query row (TMEM lane); tcgen05.ld 32 columns at a time, 3-input-max tree against the
//               row's pruning threshold; a chunk that beats it is handed to the list warp as 11 column-triple maxima
// Why it looks like this (issue-bound, not tensor-bound, at small K) is measured in DESIGN.md §5 / profiles/README.md.
//
// Operands are FP16 (not BF16): unit-norm rows live in [-1,1] where FP16 has 3 more mantissa bits, so the
// worst-case score error is 2^-10 instead of 2^-8 and the candidate margin needed for exact indices is 4x
// smaller; kind::f16 runs FP16 and BF16 at the same rate.
#include "sng_sm100.cuh"
#include <cuda_fp16.h>
#include <math_constants.h>
#include <stdlib.h>

namespace sng {
namespace knn {

constexpr int BM = 128;                 // query rows per CTA = TMEM lanes (a CTA pair owns 256 rows)
constexpr int BN = 256;                 // database columns per pair tile = UMMA N
constexpr int BK = 64;                  // K elements per smem tile row = 128 bytes = one swizzle span
constexpr int kTileBytes = 128 * BK * 2;// 16 KiB: one K block of 128 rows (A block, or this CTA's half of a B tile)
static_assert(BK == 64 && BM == 128, "make_tma_map_f16 loads 64 (K) x 128 (rows) boxes");
constexpr int kUmmaK = 16;
constexpr int kNonEpiThreads = 128;
constexpr int kMaxStages = 10;
constexpr int kMaxD = 4096;             // feature width limit (d > ~640 streams the query block, see Stage1Params::stream_a)
constexpr int kMaxCandTotal = 192;      // lists per row * cand <= this; stage 2 expands every candidate into 3 columns
constexpr uint32_t kPeerMask = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address -> leader CTA
constexpr int kQueue = 256;             // hit queue entries per CTA (power of two; the plan may shrink it); one entry = 64 bytes
constexpr int kSeedGroups = 16;         // disjoint column groups of the seed sample: (tile parity) x (32-column chunk of the tile)
// Candidate scores are kept in shared memory as 16-bit bins (6 bytes per slot with the 32-bit column id instead of 8): at
// d = 512 the resident A block leaves ~60 KB for the lists, and the 25 % saved is what lets top_k = 50 keep a 22-slot margin
// (with 8 slots almost no row of a dense cluster can be proven and everything falls to the exact scan).  A bin is 3.1e-5
// wide; every use below takes the bin's UPPER edge (+ half a bin for float rounding), so thresholds stay valid bounds.
constexpr float kQScale = 32512.0f, kQOff = 1.0078125f, kQBin = 1.0f / 32512.0f;
__device__ __forceinline__ unsigned short q_of(float v) {
    const int q = __float2int_rd((v + kQOff) * kQScale);
    return (unsigned short)min(max(q, 0), 65535);
}
__device__ __forceinline__ float q_upper(unsigned q) { return ((float)q + 1.5f) * kQBin - kQOff; }

// ------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(p));
    return p != 0;
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
    asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tmbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
                 ::"r"(bar), "r"(cta) : "memory");
}
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t addr, uint32_t cta) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(addr), "r"(cta));
    return ra;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load issued by either CTA of the pair into its OWN shared memory; the bytes are credited to the LEADER's barrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar_leader, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_leader), "r"(c0), "r"(c1) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T over the CTA pair: M = 256 (128 rows per CTA), N = 256 (128 B rows per CTA), K = 16
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive (once all previously issued MMAs have retired) on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ float max3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
constexpr uint32_t kIdesc = f16_idesc(256, BN);            // M = 256 spans the pair

struct Stage1Params {
    int nq, n, q_offset;          // query rows in this call, database rows, global id of query row 0
    int kblocks, ksteps_last;     // K tiling: kblocks tiles of 64, the last one has ksteps_last MMA steps of 16
    int stages;                   // B ring depth (K blocks)
    int stream_a;                 // 1 = the query block does not stay resident (large d): every ring stage holds an A K block AND a B K block
    int cand;                     // candidate slots per row list (L)
    int qcap;                     // hit queue entries (power of two)
    int nsplit, tiles_total;      // 256-column tiles are split across gridDim.y cluster columns
    float thr_lo;                 // approximate scores <= thr_lo can never be selected
    int remove_self;
    float* cand_val;              // [nq, nsplit, cand]
    int* cand_idx;                // [nq, nsplit, cand]   (-1 = empty)
    float* cand_min;              // [nq, nsplit]  largest threshold the row's list pruned with, -inf if it never left thr_lo
    // threshold seeding (see "Seeding" below): the seed pass writes seed_out, the main pass reads seeds
    const float* seeds;           // [nq, kSeedGroups] group maxima over a 1/seed_stride column sample, or nullptr
    float* seed_out;              // SEED kernel only
    int seed_q, seed_stride;      // row threshold = seed_q-th largest group maximum; sample = every seed_stride-th column
    int issuers;                  // MMA-issuing warps (1 or 2).  Placed here, the padding keeps the block at 136 bytes: at 128,
                                  // ptxas (CUDA 12.9) schedules and register-allocates every instance differently
    const int* nq_dev;            // retry pass: number of query rows actually present (device), or nullptr
    const int* row_ids;           // retry pass: global row id (minus q_offset) of query row r, or nullptr (= r)
    int* phase;                   // [nsplit] sweep phase shared by all CTAs of a column split (see "Phase alignment"), or nullptr
};

// MMA issue loop of the SPLIT (four 128-column accumulator stages) mode for issuer W of NI, kblocks <= 2.  W / NI are compile
// time so that every address, descriptor and ring index below is provably warp-uniform and stays in uniform registers: on a
// busy SM the issuer's dependent instruction chain, not the tensor pipe, sets the tile period (per-tile clock stamps).
template <int W, int NI>
__device__ __forceinline__ void issue_split(const Stage1Params& p, uint32_t base, uint32_t a_off, uint32_t b_off, uint32_t bar_full, uint32_t bar_empty,
                                            uint32_t bar_tfull, uint32_t bar_tempty, int t_beg, int t_end, bool issuer) {
    constexpr uint32_t kIdescHalf = f16_idesc(256, 128);
    const uint64_t adesc0 = make_smem_desc(base + a_off);
    const uint64_t bdesc0 = make_smem_desc(base + b_off);
    const int kb2 = p.kblocks == 2;                          // second K block present
    const int ks0 = kb2 ? 4 : p.ksteps_last;                 // K steps of block 0
    const int ks1 = kb2 ? p.ksteps_last : 0;                 // K steps of block 1
    const int nst = p.stages, step = NI * p.kblocks;
    int st0 = (W * p.kblocks) % nst;                         // ring slot of this tile's K block 0
    uint32_t ph0 = (uint32_t)((W * p.kblocks) / nst) & 1u;
    for (int tt = W; tt < t_end - t_beg; tt += NI) {
        const int st1 = st0 + 1;                             // same ring lap: stages % kblocks == 0
        const uint32_t acc_phase = (uint32_t)(tt >> 1) & 1u;
        const int acc0 = 2 * (tt & 1);
        const uint64_t b0 = bdesc0 + (uint64_t)(st0 * (kTileBytes >> 4)), b1 = bdesc0 + (uint64_t)(st1 * (kTileBytes >> 4));
        mbar_wait(bar_full + 8 * st0, ph0);                  // every K block of the tile landed (one barrier per tile)
        mbar_wait(bar_tempty + 8 * (tt & 1), acc_phase ^ 1); // both accumulator halves of this tile parity drained
        tc_fence_after();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t tmem_d = (uint32_t)((acc0 + h) * 128);
            const uint64_t hb = (uint64_t)(h * (kTileBytes >> 5));                       // + 64 rows x 128 B
            if (issuer) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                    if (ks < ks0) umma_f16_pair(tmem_d, adesc0 + (uint64_t)(ks * 2), b0 + hb + (uint64_t)(ks * 2), kIdescHalf, ks != 0 ? 1u : 0u);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                    if (ks < ks1) umma_f16_pair(tmem_d, adesc0 + (uint64_t)((kTileBytes >> 4) + ks * 2), b1 + hb + (uint64_t)(ks * 2), kIdescHalf, 1u);
                if (h == 1) umma_commit_pair(bar_empty + 8 * st0);                       // both halves read: free the tile's B slots
                umma_commit_pair(bar_tfull + 8 * (acc0 + h));
            }
            __syncwarp();
        }
        st0 += step;
        while (st0 >= nst) { st0 -= nst; ph0 ^= 1u; }
    }
}

// EW = epilogue warps per TMEM lane quarter; every epilogue thread owns one query row x (256/EW) columns of each tile; the
// EW threads of a row share the row's pruning threshold and (through the hit queue and the list warp) its candidate list.
//
// Seeding.  A list that starts from thr_lo inserts ~L ln(n/L) times, and every insert is a slow, divergent detour off the
// max-tree fast path (ncu, pokec shape: 3/4 of all warp instructions).  So the build first runs this kernel in SEED mode
// over every seed_stride-th database row: the epilogue is a branch-free running maximum per (row, column group), 16 groups
// per row.  The main pass starts each row at tau = the seed_q-th largest group maximum: at least seed_q sampled columns
// score >= tau, so >= top_k columns of the full set do unless >= seed_q of the row's true top_k fell into the 1/stride
// sample (probability chosen < 2e-5 on the host).  As with every pruning threshold here, a bad tau costs time, never
// correctness: tau is reported through cand_min and stage 2 sends unproven rows to the exact scan.
template <int EW, bool SEED>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kNonEpiThreads + 128 * EW, 1)
simknn_stage1_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_db, const Stage1Params p) {
    constexpr int CPT = BN / EW;                                  // columns per thread per tile
    // SPLIT (EW == 4, i.e. small K): a 256-column tile is computed as two N = 128 halves into FOUR 128-column accumulator
    // stages.  With only two stages, the hand-back of a stage (tcgen05.commit -> epilogue loads -> remote arrive -> issuer)
    // sits on the critical path of every tile and any late epilogue warp stalls the tensor pipe; with four, each issuer owns
    // two stages and a stage is not needed again for a whole tile period after it was drained.
    constexpr bool SPLIT = (EW == 4);
    // retry pass: the grid is sized for the maximum, the number of rows lives on the device; idle pairs leave together
    const int nq_eff = p.nq_dev ? min(__ldg(p.nq_dev), p.nq) : p.nq;
    if ((int)(blockIdx.x >> 1) * 2 * BM >= nq_eff) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();                      // 0 = leader (issues the MMAs)
    const uint32_t a_off = 0;
    // resident A: all K blocks of the CTA's 128 query rows, then the B ring.  Streamed A (d too large for that, p.stream_a):
    // no resident block; a ring stage is 32 KiB = the A K block followed by the B K block, both reloaded for every tile
    // (the query block of a CTA is 128 x d FP16 -- 0.6 MB at d = 2,325 --, it stays in L2 between tiles)
    const uint32_t b_off = a_off + (p.stream_a ? 0u : (uint32_t)p.kblocks * kTileBytes);
    const uint32_t stage_bytes = p.stream_a ? 2u * kTileBytes : (uint32_t)kTileBytes;
    // per-ROW candidate lists (slot-major: slot s of row r at [s * BM + r]), their bookkeeping, and the hit queue
    const uint32_t list_off = b_off + (uint32_t)p.stages * stage_bytes;
    const uint32_t thr_off = list_off + (uint32_t)p.cand * BM * 6u;
    const uint32_t q_off = (thr_off + BM * 12u + 15u) & ~15u;         // row_thr, list_cnt, list_minpos; then the 16-byte aligned queue
    const uint32_t qcap = (uint32_t)p.qcap;
    const uint32_t bar_off = q_off + qcap * 68u + 16u;             // entries (64 B), flags (4 B) + {q_head, q_tail, done}
    int* list_idx = reinterpret_cast<int*>(smem + list_off);
    unsigned short* list_val = reinterpret_cast<unsigned short*>(smem + list_off + (size_t)p.cand * BM * 4);     // 16-bit score bins
    volatile float* row_thr = reinterpret_cast<volatile float*>(smem + thr_off);
    int* list_cnt = reinterpret_cast<int*>(smem + thr_off + BM * 4);
    int* list_minpos = reinterpret_cast<int*>(smem + thr_off + BM * 8);
    float4* q_ent = reinterpret_cast<float4*>(smem + q_off);         // entry e = q_ent[4e .. 4e+3]: 11 triple maxima, col0, row
    volatile int* q_flag = reinterpret_cast<volatile int*>(smem + q_off + qcap * 64);
    unsigned* q_head = reinterpret_cast<unsigned*>(smem + q_off + qcap * 68);
    volatile unsigned* q_tail = reinterpret_cast<volatile unsigned*>(smem + q_off + qcap * 68 + 4);
    unsigned* q_done = reinterpret_cast<unsigned*>(smem + q_off + qcap * 68 + 8);
    const uint32_t bar_full = base + bar_off;                       // [kMaxStages]  leader only: B K-block landed in both CTAs
    const uint32_t bar_empty = bar_full + 8 * kMaxStages;           // [kMaxStages]  per CTA: MMAs that read the stage retired
    const uint32_t bar_a = bar_empty + 8 * kMaxStages;              // [1]           leader only: both A blocks landed
    const uint32_t bar_tfull = bar_a + 8;                           // [4]           per CTA: accumulator stage complete
    const uint32_t bar_tempty = bar_tfull + 32;                     // [4]           leader only: both CTAs drained the stage
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + bar_off + 8 * (2 * kMaxStages + 9));

    const int row0 = (int)blockIdx.x * BM;                          // blockIdx.x = 2 * pair + rank
    const int t_beg = (int)(((long long)p.tiles_total * blockIdx.y) / p.nsplit);
    const int t_end = (int)(((long long)p.tiles_total * (blockIdx.y + 1)) / p.nsplit);
    const int T = t_end - t_beg;
    // Phase alignment.  Every CTA sweeps all T tiles of its column split, but the database (261 MB FP16 at pokec scale) does
    // not fit in L2 and CTAs of later waves start at arbitrary times: with every sweep starting at tile 0 the resident CTAs
    // drift to random phases, the working set becomes the whole matrix and DRAM serves a third of the B traffic (ncu: 652 GB
    // per build).  So a CTA starts its sweep at the tile the others are currently working on (a global counter the producers
    // keep current) and wraps around: all resident CTAs stream the same few tiles and B is read from DRAM once per wave.
    uint32_t* t0_slot = tmem_slot + 1;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(bar_full + 8 * s, 2); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_a, 2);
        // SPLIT: four 128-column accumulator stages handed back in PAIRS (tempty[tile parity], all 16 warps of both CTAs);
        // else two 256-column stages, 4*EW warps per CTA each
        for (int s = 0; s < 4; ++s) { mbar_init(bar_tfull + 8 * s, 1); mbar_init(bar_tempty + 8 * s, SPLIT ? 32 : 2 * 4 * EW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    } else if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else if (warp == 3) {
        for (int i = lane; i < BM; i += 32) {
            float tau = p.thr_lo;
            const int grow = row0 + i;
            if (!SEED && grow >= nq_eff) tau = CUDART_INF_F;         // rows beyond the query matrix (TMA zero fill / stale retry slots) never hit
            if (!SEED && p.seeds != nullptr && grow < nq_eff) {
                const int srow = p.row_ids ? __ldg(p.row_ids + grow) : grow;     // retry pass: the seeds belong to the original row
                float g[kSeedGroups];
#pragma unroll
                for (int j = 0; j < kSeedGroups / 4; ++j) {
                    const float4 t4 = __ldg(reinterpret_cast<const float4*>(p.seeds + (size_t)srow * kSeedGroups) + j);
                    g[4 * j] = t4.x; g[4 * j + 1] = t4.y; g[4 * j + 2] = t4.z; g[4 * j + 3] = t4.w;
                }
                const int self = p.q_offset + srow;                  // the row itself may sit in the sample: drop its group
                if (p.remove_self && self % p.seed_stride == 0) {
                    const int cs = self / p.seed_stride, sg = ((cs >> 8) & 1) * 8 + ((cs & 255) >> 5);
#pragma unroll
                    for (int j = 0; j < kSeedGroups; ++j) if (j == sg) g[j] = -CUDART_INF_F;
                }
                float cur = CUDART_INF_F;
                for (int r = 0; r < p.seed_q; ++r) {                 // seed_q-th largest by repeated removal of the maximum
                    float mx = -CUDART_INF_F;
#pragma unroll
                    for (int j = 0; j < kSeedGroups; ++j) mx = fmaxf(mx, g[j]);
                    bool gone = false;
#pragma unroll
                    for (int j = 0; j < kSeedGroups; ++j) if (!gone && g[j] == mx) { g[j] = -CUDART_INF_F; gone = true; }
                    cur = mx;
                }
                tau = fmaxf(tau, cur);
            }
            row_thr[i] = tau;
            list_cnt[i] = 0;
            list_minpos[i] = 0;
        }
        for (int i = lane; i < (int)qcap; i += 32) q_flag[i] = 0;
        if (lane == 0) { *q_head = 0u; *q_tail = 0u; *q_done = 0u; }
        if (lane == 0 && rank == 0) {                                 // the pair's common starting tile, written to both CTAs
            const uint32_t t0 = (p.phase != nullptr && T > 0) ? (uint32_t)(*reinterpret_cast<volatile int*>(p.phase + blockIdx.y)) % (uint32_t)T : 0u;
            *t0_slot = t0;                                            // the peer reads it from here after the cluster barrier
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    if (*tmem_slot != 0u) __trap();            // the CTA owns the SM, so all 512 columns start at 0; addresses below assume it
    int t_start;                               // first tile of this pair's sweep (leader's shared memory, read over DSMEM)
    asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %1, 0;\n\tld.shared::cluster.u32 %0, [ra];\n\t}"
                 : "=r"(t_start) : "r"(smem_u32(t0_slot)) : "memory");
    t_start += t_beg;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (both CTAs, whole warp, one lane issues)
        const bool issuer = elect_one();
        const uint32_t bar_a_leader = bar_a & kPeerMask;
        if (issuer && !p.stream_a) {
            for (int kb = 0; kb < p.kblocks; ++kb)
                tma_load_2d_pair(base + a_off + (uint32_t)kb * kTileBytes, &map_q, bar_a_leader, kb * BK, row0);
            if (rank == 0) mbar_expect_tx(bar_a, 2u * (uint32_t)p.kblocks * kTileBytes);
            else mbar_arrive_cluster(bar_a, 0);
        }
        int stage = 0; uint32_t phase = 0;
        for (int tt = 0, t = t_start; tt < T; ++tt, t = (t + 1 == t_end) ? t_beg : t + 1) {
            if (p.phase != nullptr && rank == 0 && (tt & 63) == 0 && issuer) p.phase[blockIdx.y] = t - t_beg;   // where this sweep is
            const int brow = t * BN + (int)rank * 128;              // this CTA stages its half of the tile's database rows
            if constexpr (SPLIT) {
                // all K blocks of a tile share the barriers of the tile's first ring slot (stages % kblocks == 0): the issuers
                // pay one wait and one commit per tile instead of one per K block
                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                if (issuer) {
                    for (int kb = 0; kb < p.kblocks; ++kb)
                        tma_load_2d_pair(base + b_off + (uint32_t)(stage + kb) * kTileBytes, &map_db, (bar_full + 8 * stage) & kPeerMask, kb * BK, brow);
                    if (rank == 0) mbar_expect_tx(bar_full + 8 * stage, 2u * (uint32_t)p.kblocks * kTileBytes);
                    else mbar_arrive_cluster(bar_full + 8 * stage, 0);
                }
                stage += p.kblocks;
                if (stage >= p.stages) { stage = 0; phase ^= 1; }
            } else {
            for (int kb = 0; kb < p.kblocks; ++kb) {
                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                if (issuer) {
                    const uint32_t sdst = base + b_off + (uint32_t)stage * stage_bytes;
                    if (p.stream_a) tma_load_2d_pair(sdst, &map_q, (bar_full + 8 * stage) & kPeerMask, kb * BK, row0);
                    tma_load_2d_pair(sdst + (p.stream_a ? (uint32_t)kTileBytes : 0u), &map_db, (bar_full + 8 * stage) & kPeerMask, kb * BK, brow);
                    if (rank == 0) mbar_expect_tx(bar_full + 8 * stage, 2u * stage_bytes);
                    else mbar_arrive_cluster(bar_full + 8 * stage, 0);
                }
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            }
        }
    } else if (warp == 1 || warp == 2) {
        // ------------------------------------------------------------------ MMA issuers (leader CTA; whole warp runs the loop, one lane issues)
        // The chain "accumulator free -> B landed -> issue -> commit" costs one thread ~1300 cycles per tile (mbarrier
        // try_wait ~90 each even when complete, plus issue / commit latencies; measured with per-tile clock stamps), twice the
        // 640 cycles the tensor pipe needs for a K = 80 tile.  So TWO warps issue, each owning every other tile and one
        // of the two accumulator stages; their chains overlap and the pipe stays fed.  (tcgen05.commit tracks the MMAs
        // of the executing thread only, and each accumulator is only ever written by one of the two threads.)
        const int w = warp - 1;
        if (rank == 0 && w < p.issuers) {
            const bool issuer = elect_one();
            if (!p.stream_a) mbar_wait(bar_a, 0);
            tc_fence_after();
            const uint64_t adesc0 = make_smem_desc(base + a_off);
            const uint64_t bdesc0 = make_smem_desc(base + b_off);
            int stage = 0; uint32_t phase = 0;
            auto advance = [&](int steps) { for (int i = 0; i < steps; ++i) if (++stage == p.stages) { stage = 0; phase ^= 1; } };
            advance(w * p.kblocks);
            if constexpr (SPLIT) {
                if (p.issuers == 1) issue_split<0, 1>(p, base, a_off, b_off, bar_full, bar_empty, bar_tfull, bar_tempty, t_beg, t_end, issuer);
                else if (warp == 1) issue_split<0, 2>(p, base, a_off, b_off, bar_full, bar_empty, bar_tfull, bar_tempty, t_beg, t_end, issuer);
                else issue_split<1, 2>(p, base, a_off, b_off, bar_full, bar_empty, bar_tfull, bar_tempty, t_beg, t_end, issuer);
            } else {
            for (int tt = w; tt < T; tt += p.issuers) {
                const int acc = tt & 1;
                const uint32_t acc_phase = (uint32_t)(tt >> 1) & 1u;
                mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = (uint32_t)(acc * BN);
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    const int ksteps = (kb == p.kblocks - 1) ? p.ksteps_last : (BK / kUmmaK);
                    // descriptors count 16-byte units: one 16 KiB tile = 1024 units, one K step (32 B) = 2 units
                    const uint64_t adesc = p.stream_a ? bdesc0 + (uint64_t)(stage * 2 * (kTileBytes >> 4)) : adesc0 + (uint64_t)(kb * (kTileBytes >> 4));
                    const uint64_t bdesc = p.stream_a ? adesc + (uint64_t)(kTileBytes >> 4) : bdesc0 + (uint64_t)(stage * (kTileBytes >> 4));
                    if (issuer) {
                        for (int ks = 0; ks < ksteps; ++ks)
                            umma_f16_pair(tmem_d, adesc + (uint64_t)(ks * 2), bdesc + (uint64_t)(ks * 2), kIdesc, (kb | ks) != 0 ? 1u : 0u);
                        umma_commit_pair(bar_empty + 8 * stage);        // frees this B stage in both CTAs when the MMAs retire
                        if (kb == p.kblocks - 1) umma_commit_pair(bar_tfull + 8 * acc);   // accumulator of tile t complete (both CTAs)
                    }
                    __syncwarp();
                    advance(1);
                }
                advance((p.issuers - 1) * p.kblocks);                   // the other issuer's tile
            }
            }
        }
    } else if (warp == 3) {
        // ------------------------------------------------------------------ list warp: drains the hit queue into the per-row lists
        // The epilogue warps only FILTER: a lane whose 32-score chunk beats the row threshold dumps the chunk's 11 column-triple
        // maxima (already in registers from the max tree) into a shared-memory queue -- ~25 instructions -- and moves on.
        // This warp owns the candidate lists, at column-TRIPLE granularity (stage 2 rescoring expands a triple into its 3
        // columns).  Everything data dependent and slow happens here, off the warps whose pace gates the tensor pipe: an
        // accumulator stage is reusable only once ALL 32 epilogue warps of the pair have drained it, and on a busy SM a
        // dependent chain of ~150 instructions (the former in-line insert) costs ~1900 cycles, three tile periods.
        if (!SEED) {
            const int L = p.cand;
            unsigned tail = 0;
            while (true) {
                const unsigned s = (tail + lane) & (qcap - 1);
                const unsigned ready = __ballot_sync(0xffffffffu, q_flag[s] != 0);
                const int nr = ready == 0xffffffffu ? 32 : __ffs(~ready) - 1;       // leading published entries
                if (nr == 0) {
                    const unsigned done = *reinterpret_cast<volatile unsigned*>(q_done);
                    const unsigned head = *reinterpret_cast<volatile unsigned*>(q_head);
                    if (done == (unsigned)(4 * EW) && head == tail) break;
                    __nanosleep(200);
                    continue;
                }
                __threadfence_block();
                const bool mine = lane < nr;
                // Usually one or two of an entry's 11 triples beat the row threshold (bit i of `mleft`, computed here, lane =
                // entry).  Round j applies the j-th such triple of EVERY entry of the batch at once: the insert
                // below -- a divergent detour with a 32-slot minimum scan when the list is full -- runs once per round for up to
                // 32 values, not once per triple index per batch (11 x), which made this warp the pacer of the whole CTA on small
                // databases, where hits are dense (arxiv shape: 38 % of all warp-chunks hit).
                int row = 0, col0 = 0; unsigned mleft = 0u;
                const float* qf = reinterpret_cast<const float*>(q_ent + 4 * s);
                if (mine) {
                    col0 = __float_as_int(qf[11]); row = __float_as_int(qf[12]);
                    const float thr0 = row_thr[row];
#pragma unroll
                    for (int i = 0; i < 11; ++i) mleft |= (qf[i] > thr0 ? 1u : 0u) << i;
                }
                while (__any_sync(0xffffffffu, mleft != 0u)) {
                    const bool has = mleft != 0u;
                    const int i = has ? __ffs(mleft) - 1 : 0;
                    mleft &= mleft - 1u;                                             // (0 stays 0)
                    const float val = has ? qf[i] : 0.f;
                    const int rowk = has ? row : -1 - lane;                          // distinct sentinel rows for idle lanes
                    unsigned pending = __ballot_sync(0xffffffffu, has);
                    while (pending) {                                               // values of one row are applied one at a time
                        const unsigned same = __match_any_sync(0xffffffffu, rowk) & pending;
                        const bool go = has && ((pending >> lane) & 1u) && (__ffs(same) - 1 == lane);
                        if (go) {
                            const float thr = row_thr[row];
                            if (val > thr) {
                                int c = list_cnt[row], slot;
                                if (c < L) { slot = c; list_cnt[row] = ++c; }
                                else slot = list_minpos[row];
                                list_val[slot * BM + row] = q_of(val);
                                list_idx[slot * BM + row] = col0 + 3 * i;
                                if (c == L) {                                        // full: the minimum's bin becomes the row's threshold
                                    unsigned mn = list_val[row]; int mp = 0;
#pragma unroll 4
                                    for (int s2 = 1; s2 < L; ++s2) { const unsigned y = list_val[s2 * BM + row]; if (y < mn) { mn = y; mp = s2; } }
                                    list_minpos[row] = mp;
                                    const float tn = q_upper(mn);                    // nothing in the minimum's bin can be told from it
                                    if (tn > thr) row_thr[row] = tn;
                                }
                            }
                        }
                        __syncwarp();
                        pending &= ~__ballot_sync(0xffffffffu, go);
                    }
                }
                if (mine) q_flag[s] = 0;
                __threadfence_block();
                __syncwarp();
                tail += (unsigned)nr;
                if (lane == 0) *q_tail = tail;
            }
            // all epilogue warps are done and the queue is empty: emit the lists and the drop bounds
            __threadfence_block();
            const int lists = p.nsplit;
            for (int i = lane; i < BM * L; i += 32) {
                const int r = i / L, sl = i - r * L, grow = row0 + r;
                if (grow < nq_eff) {
                    const size_t o = ((size_t)grow * lists + blockIdx.y) * L + sl;
                    const bool ok = sl < list_cnt[r];
                    p.cand_val[o] = ok ? q_upper(list_val[sl * BM + r]) : -CUDART_INF_F;    // upper bound of the triple's maximum
                    p.cand_idx[o] = ok ? list_idx[sl * BM + r] : -1;
                }
            }
            for (int r = lane; r < BM; r += 32) {
                const int grow = row0 + r;
                // bound on everything dropped for this row: the final threshold (seed, evictions and filtered columns included)
                if (grow < nq_eff) p.cand_min[(size_t)grow * lists + blockIdx.y] = row_thr[r] > p.thr_lo ? row_thr[r] : -CUDART_INF_F;
            }
        }
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue: thread = one query row x CPT columns per tile
        constexpr int CT = CPT / 32;                               // 32-column chunks per thread per tile
        const int quarter = warp & 3, slice = (warp - 4) >> 2;
        const int r = quarter * 32 + lane;                        // row within the CTA == TMEM lane
        const int grow = row0 + r;
        const int self_col = p.remove_self ? p.q_offset + ((p.row_ids && grow < nq_eff) ? __ldg(p.row_ids + grow) : grow) : -1;
        const int n = p.n;
        float thr_cur = p.thr_lo;                                  // the row's pruning threshold as last read from shared memory
        float gmax[2 * CT];                                        // SEED: running maxima of this thread's column groups
#pragma unroll
        for (int i = 0; i < 2 * CT; ++i) gmax[i] = -CUDART_INF_F;

        // Pruning thresholds are heuristics: ANY threshold is safe because the row reports the largest threshold anything
        // was pruned with (cand_min) and stage 2 only accepts a row whose k-th exact score clears it.
        // `ci` = chunk index within the thread's tile slice (compile time after unrolling), `odd` = tile parity.
        auto process = [&](uint32_t (&v)[32], int col0, int ci, bool odd) {
            float m[11];
            auto tree = [&]() {
#pragma unroll
                for (int i = 0; i < 10; ++i) m[i] = max3(__uint_as_float(v[3 * i]), __uint_as_float(v[3 * i + 1]), __uint_as_float(v[3 * i + 2]));
                m[10] = fmaxf(__uint_as_float(v[30]), __uint_as_float(v[31]));
                const float m0 = max3(m[0], m[1], m[2]), m1 = max3(m[3], m[4], m[5]), m2 = max3(m[6], m[7], m[8]);
                return max3(max3(m0, m1, m2), m[9], m[10]);
            };
            float mx = tree();
            if (SEED) {
                if (col0 + 32 > n) {                                 // last tile: zero-filled columns beyond n must not count
                    mx = -CUDART_INF_F;
#pragma unroll
                    for (int i = 0; i < 32; ++i) if (col0 + i < n) mx = fmaxf(mx, __uint_as_float(v[i]));
                }
                gmax[ci] = fmaxf(gmax[ci], odd ? -CUDART_INF_F : mx);
                gmax[CT + ci] = fmaxf(gmax[CT + ci], odd ? mx : -CUDART_INF_F);
                return;
            }
            if (__any_sync(0xffffffffu, mx > thr_cur)) {           // rare slow path
                if ((unsigned)(self_col - col0) < 32u || col0 + 32 > n) {
                    // the chunk holds the row's own column, or columns beyond n (zero filled): once per row / last tile only
#pragma unroll
                    for (int i = 0; i < 32; ++i) if (col0 + i == self_col || col0 + i >= n) v[i] = 0xff800000u;
                    mx = tree();
                }
                if (mx > thr_cur) {                                  // hit lanes only: dump the triple maxima for the list warp
                    const unsigned at = atomicAdd(q_head, 1u);
                    while ((int)(at - *q_tail) >= (int)qcap) __nanosleep(20);           // queue full: wait for the list warp
                    const unsigned s = at & (qcap - 1);
                    q_ent[4 * s] = make_float4(m[0], m[1], m[2], m[3]);
                    q_ent[4 * s + 1] = make_float4(m[4], m[5], m[6], m[7]);
                    q_ent[4 * s + 2] = make_float4(m[8], m[9], m[10], __int_as_float(col0));
                    q_ent[4 * s + 3] = make_float4(__int_as_float(r), 0.f, 0.f, 0.f);
                    __threadfence_block();
                    q_flag[s] = 1;                                                   // publishes the entry
                }
                __syncwarp();
                thr_cur = fmaxf(thr_cur, row_thr[r]);                // the list warp may already have raised it
            }
        };

        uint32_t va[32], vb[32];
        // columns of the tile this thread owns: [tile_col, tile_col + CPT) -- SPLIT: 64 columns of half h = slice & 1, taken from
        // CTA (slice >> 1)'s staged rows, i.e. accumulator columns [64 (slice >> 1), +64) of stage 2 * (tile parity) + h
        const int tile_col = SPLIT ? 128 * (slice >> 1) + 64 * (slice & 1) : slice * CPT;
        // loop-invariant addresses, pinned in registers (the per-tile loop is issue-bound; left alone the compiler re-derives
        // them from threadIdx every tile to save registers): TMEM address / accumulator-full barrier of the EVEN tiles, the
        // leader's hand-back barrier; odd tiles are a constant away
        uint32_t taddr_e = ((uint32_t)(quarter * 32) << 16) + (uint32_t)(SPLIT ? (slice & 1) * 128 + (slice >> 1) * 64 : slice * CPT);
        uint32_t bar_tf_e = bar_tfull + 8u * (SPLIT ? (uint32_t)(slice & 1) : 0u);
        uint32_t bar_te_e = mapa_cluster(bar_tempty, 0);
        for (int tt = 0, t = t_start; tt < T; ++tt, t = (t + 1 == t_end) ? t_beg : t + 1) {
            asm volatile("" : "+r"(taddr_e), "+r"(bar_tf_e), "+r"(bar_te_e));
            const uint32_t par = (uint32_t)tt & 1u;
            const uint32_t acc_phase = (uint32_t)(tt >> 1) & 1u;
            mbar_wait(bar_tf_e + par * (SPLIT ? 16u : 8u), acc_phase);
            tc_fence_after();
            if (!SEED) thr_cur = fmaxf(thr_cur, row_thr[r]);
            const uint32_t taddr = taddr_e + par * (uint32_t)(SPLIT ? 256 : BN);
            const int col0 = t * BN + tile_col;
            const bool odd = (t & 1) != 0;
            if (CPT == 64) {
                // both loads in flight at once; the accumulator stage goes back to the MMA warp before any processing
                tmem_ld32(taddr, va);
                tmem_ld32(taddr + 32, vb);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_remote(bar_te_e + 8u * par);
                process(va, col0, 0, odd);
                process(vb, col0 + 32, CT > 1 ? 1 : 0, odd);
            } else {
                tmem_ld32(taddr, va);
#pragma unroll
                for (int c = 0; c < CT; c += 2) {
                    tmem_ld_wait();
                    tmem_ld32(taddr + (c + 1) * 32, vb);
                    process(va, col0 + c * 32, c, odd);
                    tmem_ld_wait();
                    if (c + 2 < CT) tmem_ld32(taddr + (c + 2) * 32, va);
                    else {
                        // every load of this accumulator stage has landed: hand the stage back to the leader's MMA warp
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_remote(bar_te_e + 8u * par);
                    }
                    process(vb, col0 + (c + 1) * 32, c + 1, odd);
                }
            }
        }
        if (SEED) {
            if (grow < nq_eff) {
                // group id of sample column cs = ((cs >> 8) & 1) * 8 + ((cs & 255) >> 5)  (tile parity, chunk of the tile)
#pragma unroll
                for (int i = 0; i < 2 * CT; ++i)
                    p.seed_out[(size_t)grow * kSeedGroups + (i / CT) * 8 + (tile_col >> 5) + (i % CT)] = gmax[i];
            }
        } else {
            __syncwarp();
            __threadfence_block();
            if (lane == 0) atomicAdd(q_done, 1u);                    // this warp will push nothing more
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                        // neither CTA may exit (or free TMEM) while the other can still signal / write it
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(0u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------ exact FP32 score
// ONE definition of the "exact" cosine used by stage 2 and stage 3: sequential fmaf over c = 0..d-1 of the
// FP32 unit rows (d padded to a multiple of 4 with zeros, which leaves the value unchanged).
__device__ __forceinline__ float dot_seq(const float* __restrict__ a, const float* __restrict__ b, int d4) {
    float s = 0.f;
    for (int k = 0; k < d4; ++k) {
        const float4 x = ldg4(a + 4 * k), y = ldg4(b + 4 * k);
        s = fmaf(x.x, y.x, s); s = fmaf(x.y, y.y, s); s = fmaf(x.z, y.z, s); s = fmaf(x.w, y.w, s);
    }
    return s;
}
__device__ __forceinline__ bool better(float sa, int ia, float sb, int ib) { return sa > sb || (sa == sb && ia < ib); }

// Stage 2: one warp per query row.  Every candidate is a column triple {c, c+1, c+2} (two columns when c % 32 == 30, the
// last triple of a 32-column chunk).  Rescore all their columns exactly, order them by (score desc, index asc), apply
// thr / top_k, and prove that no dropped column could belong to the answer.
__global__ void __launch_bounds__(256) simknn_rescore_kernel(
    const float* __restrict__ xq, const float* __restrict__ xall, int64_t ld32, int d4, int nq, int n, int q_offset, int remove_self, int m_total,
    int nsplit, int top_k, float thr, float eps, const float* __restrict__ cand_val, const int* __restrict__ cand_idx,
    const float* __restrict__ cand_min,
    int* __restrict__ idx_out, float* __restrict__ sim_out, int* __restrict__ cnt_out, int* __restrict__ fb_rows, int* __restrict__ n_fallback,
    const int* __restrict__ nq_dev, const int* __restrict__ row_map) {
    extern __shared__ float sm2[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m3 = 3 * m_total;
    float* sc = sm2 + (size_t)warp * 2 * m3;
    int* id = reinterpret_cast<int*>(sc + m3);
    if (nq_dev) nq = min(nq, __ldg(nq_dev));
    // retry pass: candidate lists are indexed by f, everything else by the row f stands for
    for (int f = blockIdx.x * 8 + warp; f < nq; f += gridDim.x * 8) {
        const int row = row_map ? __ldg(row_map + f) : f;
        const float* a = xq + (int64_t)row * ld32;
        const int self_col = remove_self ? q_offset + row : -1;
        // An all-zero query row (F.normalize maps a zero feature row to zero) scores exactly 0 against every column: its list is
        // the lowest top_k column ids (minus itself) when 0 >= thr, else empty -- by the rule itself, no scan.  (No tensor-core
        // list can prove such a row: every score ties; it used to cost an exact scan of all n columns.)
        {
            bool nz = false;
            for (int k4 = lane; k4 < d4; k4 += 32) { const float4 v = ldg4(a + 4 * k4); nz = nz || v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f; }
            if (!__any_sync(0xffffffffu, nz)) {
                const int avail = n - ((self_col >= 0 && self_col < n) ? 1 : 0);
                const int cnt0 = 0.0f >= thr ? min(top_k, avail) : 0;
                for (int t = lane; t < top_k; t += 32) {
                    const int j = (self_col >= 0 && t >= self_col) ? t + 1 : t;
                    idx_out[(size_t)row * top_k + t] = t < cnt0 ? j : -1;
                    sim_out[(size_t)row * top_k + t] = 0.f;
                }
                if (lane == 0) cnt_out[row] = cnt0;
                __syncwarp();
                continue;
            }
        }
        // Triples that cannot matter are not rescored.  Let t_k be the top_k-th largest triple maximum (FP16 scores).  The
        // top_k largest triples each hold a column whose exact score is >= t_k - eps, so the top_k-th best exact score is
        // too; every column of a triple whose maximum is < t_k - 2 eps scores < t_k - eps exactly: strictly below the cut.
        for (int m = lane; m < m_total; m += 32)
            sc[m] = __ldg(cand_idx + (size_t)f * m_total + m) >= 0 ? __ldg(cand_val + (size_t)f * m_total + m) : -CUDART_INF_F;
        __syncwarp();
        float tk = CUDART_INF_F; int ntrip = 0;
        for (int m0 = 0; m0 < m_total; m0 += 32) {                    // fixed trip counts: rank of every maximum by counting
            const int m = m0 + lane;
            const float v = m < m_total ? sc[m] : -CUDART_INF_F;
            int above = 0;
            for (int o = 0; o < m_total; ++o) above += sc[o] > v ? 1 : 0;
            if (v > -CUDART_INF_F && above < top_k) tk = fminf(tk, v);
            ntrip += __popc(__ballot_sync(0xffffffffu, v > -CUDART_INF_F));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tk = fminf(tk, __shfl_xor_sync(0xffffffffu, tk, o));
        const float cutoff = ntrip >= top_k ? tk - 2.0f * eps - 2.0f * kQBin : -CUDART_INF_F;   // the maxima are 16-bit bin upper edges
        __syncwarp();
        int nvalid = 0;
        for (int m0 = 0; m0 < m3; m0 += 32) {
            const int m = m0 + lane;
            int j = -1; float s = -CUDART_INF_F;
            if (m < m3) {
                const int base = __ldg(cand_idx + (size_t)f * m_total + m / 3), e = m % 3;
                if (base >= 0 && __ldg(cand_val + (size_t)f * m_total + m / 3) >= cutoff && (e < 2 || (base & 31) != 30) && base + e < n &&
                    base + e != self_col) {
                    j = base + e;
                    s = dot_seq(a, xall + (int64_t)j * ld32, d4);
                }
                sc[m] = s; id[m] = j;
            }
            nvalid += __popc(__ballot_sync(0xffffffffu, j >= 0 && s >= thr));
        }
        __syncwarp();
        const int cnt = min(nvalid, top_k);
        float kth = thr;                                            // cut value: k-th exact score, or thr if fewer than k qualify
        for (int m0 = 0; m0 < m3; m0 += 32) {
            const int m = m0 + lane;
            int rank = 0x7fffffff; float s = 0.f; int j = -1;
            if (m < m3) {
                s = sc[m]; j = id[m];
                if (j >= 0 && s >= thr) {
                    rank = 0;
                    for (int o = 0; o < m3; ++o) rank += (id[o] >= 0 && better(sc[o], id[o], s, j)) ? 1 : 0;
                }
            }
            if (rank < top_k) {
                idx_out[(size_t)row * top_k + rank] = j;
                sim_out[(size_t)row * top_k + rank] = s;
            }
            const unsigned hit = __ballot_sync(0xffffffffu, rank == top_k - 1);
            if (hit) kth = __shfl_sync(0xffffffffu, s, __ffs(hit) - 1);
        }
        for (int t = cnt + lane; t < top_k; t += 32) { idx_out[(size_t)row * top_k + t] = -1; sim_out[(size_t)row * top_k + t] = 0.f; }
        float bound = -CUDART_INF_F;                                 // best exact score any DROPPED column may have
        for (int s0 = lane; s0 < nsplit; s0 += 32) bound = fmaxf(bound, __ldg(cand_min + (size_t)f * nsplit + s0) + eps);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) bound = fmaxf(bound, __shfl_xor_sync(0xffffffffu, bound, o));
        if (lane == 0) {
            cnt_out[row] = cnt;
            if (!(kth > bound)) fb_rows[atomicAdd(n_fallback, 1)] = row;
        }
        __syncwarp();
    }
}

// Retry pass, step 1: compact the FP16 rows of the first kRetryRows flagged query rows into one matrix (the TMA operand of
// the second tensor-core pass); flagged rows beyond that go straight to the exact-scan list.
// Capacity of the retry pass (flagged rows beyond it go to the exact scan): every query row of small calls, a quarter of a
// million for large ones.  It used to be 16 K: inputs whose rows sit closer together than the FP16 scoring error (dense
// clusters at large d with a large top_k) flag most rows, and the exact scan re-reads the whole database per row.
constexpr int kRetryRowsMin = 16384, kRetryRowsMax = 262144;
static int retry_rows(int64_t nq) {
    int64_t c = (nq + 255) / 256 * 256;
    if (c < kRetryRowsMin) c = kRetryRowsMin;
    if (c > kRetryRowsMax) c = kRetryRowsMax;
    return (int)c;
}
constexpr int kRetryRounds = 48;           // the retry pass runs in rounds of retry_rows(nq) flagged rows (fixed buffers, counts on the device)
// round_cnt[r] = flagged rows of round r; flagged rows beyond the last round go straight to the exact-scan list
__global__ void __launch_bounds__(256) simknn_retry_rounds_kernel(const int* __restrict__ fb_rows, const int* __restrict__ n_fb, int cap, int rounds,
                                                                 int* __restrict__ round_cnt, int* __restrict__ fb2_rows, int* __restrict__ n_fb2) {
    const int nfb = *n_fb;
    for (int r = threadIdx.x; r < rounds; r += blockDim.x) round_cnt[r] = max(0, min(cap, nfb - r * cap));
    for (long long f = (long long)rounds * cap + threadIdx.x; f < nfb; f += blockDim.x) fb2_rows[atomicAdd(n_fb2, 1)] = fb_rows[f];
}
__global__ void __launch_bounds__(256) simknn_retry_gather_kernel(const uint16_t* __restrict__ xq, int64_t ldb, const int* __restrict__ fb_rows,
                                                                 const int* __restrict__ n_round, uint16_t* __restrict__ xq_retry) {
    const int nr = *n_round;
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * 8 + (threadIdx.x >> 5), nw = gridDim.x * 8;
    const int64_t vec = ldb / 8;                                             // 16-byte chunks per row (ldb % 8 == 0)
    for (int f = w; f < nr; f += nw) {
        const uint4* src = reinterpret_cast<const uint4*>(xq + (int64_t)fb_rows[f] * ldb);
        uint4* dst = reinterpret_cast<uint4*>(xq_retry + (int64_t)f * ldb);
        for (int64_t i = lane; i < vec; i += 32) dst[i] = src[i];
    }
}

// Stage 3 (parallel form): work item = (flagged row f, chunk of kChunk columns).  Scan: exact scores of the chunk in
// shared memory, then top_k rounds of block argmax under (score desc, index asc) -> partial[f][chunk][top_k].
// Merge: one block per flagged row reduces its n_chunks * top_k partial entries the same way.  Exact, tie-correct,
// and parallel over columns, so a handful of flagged rows costs microseconds instead of a serial N-long scan.
constexpr int kChunk = 8192;
constexpr int kFbWaveRows = 4096;       // flagged rows handled per (scan, merge) wave
constexpr int kFbWaves = 4;             // rows beyond kFbWaves * kFbWaveRows go to the serial kernel below

struct Pick { float s; int i; };
__device__ __forceinline__ Pick block_argmax(float bs, int bi, float* red_s, int* red_i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float os = __shfl_xor_sync(0xffffffffu, bs, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(os, oi, bs, bi)) { bs = os; bi = oi; }
    }
    if ((threadIdx.x & 31) == 0) { red_s[threadIdx.x >> 5] = bs; red_i[threadIdx.x >> 5] = bi; }
    __syncthreads();
    bs = red_s[0]; bi = red_i[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) if (better(red_s[w], red_i[w], bs, bi)) { bs = red_s[w]; bi = red_i[w]; }
    __syncthreads();
    return Pick{bs, bi};
}

__global__ void __launch_bounds__(256) simknn_fb_scan_kernel(
    const float* __restrict__ xq, const float* __restrict__ xall, int64_t ld32, int d4, int n, int q_offset, int top_k, float thr,
    int remove_self, const int* __restrict__ fb_rows, const int* __restrict__ n_fallback, int wave, int n_chunks,
    float* __restrict__ part_s, int* __restrict__ part_i) {
    __shared__ float sc[kChunk];
    __shared__ float red_s[8];
    __shared__ int red_i[8];
    const int f_lo = wave * kFbWaveRows;
    const int f_hi = min(*n_fallback, f_lo + kFbWaveRows);
    const long long items = (long long)max(f_hi - f_lo, 0) * n_chunks;
    for (long long it = blockIdx.x; it < items; it += gridDim.x) {
        const int fl = (int)(it / n_chunks), ch = (int)(it % n_chunks);
        const int row = fb_rows[f_lo + fl];
        const float* a = xq + (int64_t)row * ld32;
        const int self_col = remove_self ? q_offset + row : -1;
        const int c0 = ch * kChunk, cn = min(kChunk, n - c0);
        for (int j = threadIdx.x; j < cn; j += blockDim.x)
            sc[j] = (c0 + j == self_col) ? -CUDART_INF_F : dot_seq(a, xall + (int64_t)(c0 + j) * ld32, d4);
        __syncthreads();
        float prev_s = CUDART_INF_F; int prev_i = -1;
        const size_t o = ((size_t)fl * n_chunks + ch) * top_k;
        for (int t = 0; t < top_k; ++t) {
            float bs = -CUDART_INF_F; int bi = 0x7fffffff;
            for (int j = threadIdx.x; j < cn; j += blockDim.x) {
                const float s = sc[j];
                const int gi = c0 + j;
                const bool after = s < prev_s || (s == prev_s && gi > prev_i);
                if (after && s >= thr && better(s, gi, bs, bi)) { bs = s; bi = gi; }
            }
            const Pick pk = block_argmax(bs, bi, red_s, red_i);
            prev_s = pk.s; prev_i = pk.i;
            if (threadIdx.x == 0) { part_s[o + t] = pk.s; part_i[o + t] = pk.i == 0x7fffffff ? -1 : pk.i; }
            if (pk.i == 0x7fffffff) {                                  // chunk exhausted: pad the remaining slots
                for (int u = t + 1 + threadIdx.x; u < top_k; u += blockDim.x) { part_s[o + u] = -CUDART_INF_F; part_i[o + u] = -1; }
                break;
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) simknn_fb_merge_kernel(
    const int* __restrict__ fb_rows, const int* __restrict__ n_fallback, int wave, int n_chunks, int top_k,
    const float* __restrict__ part_s, const int* __restrict__ part_i, int* __restrict__ idx_out, float* __restrict__ sim_out,
    int* __restrict__ cnt_out) {
    __shared__ float red_s[8];
    __shared__ int red_i[8];
    const int f_lo = wave * kFbWaveRows;
    const int f_hi = min(*n_fallback, f_lo + kFbWaveRows);
    const int m = n_chunks * top_k;
    for (int fl = blockIdx.x; fl < f_hi - f_lo; fl += gridDim.x) {
        const int row = fb_rows[f_lo + fl];
        const float* ps = part_s + (size_t)fl * m;
        const int* pi = part_i + (size_t)fl * m;
        float prev_s = CUDART_INF_F; int prev_i = -1; int cnt = 0;
        for (int t = 0; t < top_k; ++t) {
            float bs = -CUDART_INF_F; int bi = 0x7fffffff;
            for (int j = threadIdx.x; j < m; j += blockDim.x) {
                const int gi = pi[j];
                if (gi < 0) continue;
                const float s = ps[j];
                const bool after = s < prev_s || (s == prev_s && gi > prev_i);
                if (after && better(s, gi, bs, bi)) { bs = s; bi = gi; }
            }
            const Pick pk = block_argmax(bs, bi, red_s, red_i);
            if (pk.i == 0x7fffffff) break;
            prev_s = pk.s; prev_i = pk.i;
            if (threadIdx.x == 0) { idx_out[(size_t)row * top_k + t] = pk.i; sim_out[(size_t)row * top_k + t] = pk.s; }
            ++cnt;
        }
        if (threadIdx.x == 0) {
            for (int t = cnt; t < top_k; ++t) { idx_out[(size_t)row * top_k + t] = -1; sim_out[(size_t)row * top_k + t] = 0.f; }
            cnt_out[row] = cnt;
        }
        __syncthreads();
    }
}

// Stage 3 (throughput form) for flagged rows beyond the parallel waves: one block streams all chunks of one row and keeps
// the running top_k (sorted by (score desc, index asc)) in shared memory.  Chunks arrive in increasing column order, so a
// chunk whose best score does not strictly beat the current k-th entry cannot change the answer and is skipped.
__global__ void __launch_bounds__(256) simknn_fb_stream_kernel(
    const float* __restrict__ xq, const float* __restrict__ xall, int64_t ld32, int d4, int n, int q_offset, int top_k, float thr,
    int remove_self, const int* __restrict__ fb_rows, const int* __restrict__ n_fallback, int f_start,
    int* __restrict__ idx_out, float* __restrict__ sim_out, int* __restrict__ cnt_out) {
    __shared__ float sc[kChunk];
    __shared__ float red_s[8];
    __shared__ int red_i[8];
    __shared__ float best_s[SNG_KNN_MAX_TOPK];
    __shared__ int best_i[SNG_KNN_MAX_TOPK];
    __shared__ int best_n;
    const int nfb = *n_fallback;
    for (int f = f_start + blockIdx.x; f < nfb; f += gridDim.x) {
        const int row = fb_rows[f];
        const float* a = xq + (int64_t)row * ld32;
        const int self_col = remove_self ? q_offset + row : -1;
        if (threadIdx.x == 0) best_n = 0;
        __syncthreads();
        for (int c0 = 0; c0 < n; c0 += kChunk) {
            const int cn = min(kChunk, n - c0);
            for (int j = threadIdx.x; j < cn; j += blockDim.x)
                sc[j] = (c0 + j == self_col) ? -CUDART_INF_F : dot_seq(a, xall + (int64_t)(c0 + j) * ld32, d4);
            __syncthreads();
            float prev_s = CUDART_INF_F; int prev_i = -1;
            for (int t = 0; t < top_k; ++t) {
                const int bn = best_n;
                const float kth = bn == top_k ? best_s[top_k - 1] : -CUDART_INF_F;
                float bs = -CUDART_INF_F; int bi = 0x7fffffff;
                for (int j = threadIdx.x; j < cn; j += blockDim.x) {
                    const float sv = sc[j];
                    const int gi = c0 + j;
                    const bool after = sv < prev_s || (sv == prev_s && gi > prev_i);
                    if (after && sv >= thr && sv > kth && better(sv, gi, bs, bi)) { bs = sv; bi = gi; }
                }
                const Pick pk = block_argmax(bs, bi, red_s, red_i);
                if (pk.i == 0x7fffffff) break;                          // nothing left in this chunk that beats the k-th entry
                prev_s = pk.s; prev_i = pk.i;
                if (threadIdx.x == 0) {                                   // sorted insert (new columns lose ties: larger index)
                    int pos = bn < top_k ? bn : top_k - 1;
                    while (pos > 0 && best_s[pos - 1] < pk.s) { best_s[pos] = best_s[pos - 1]; best_i[pos] = best_i[pos - 1]; --pos; }
                    best_s[pos] = pk.s; best_i[pos] = pk.i;
                    if (bn < top_k) best_n = bn + 1;
                }
                __syncthreads();
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            const int bn = best_n;
            for (int t = 0; t < top_k; ++t) {
                idx_out[(size_t)row * top_k + t] = t < bn ? best_i[t] : -1;
                sim_out[(size_t)row * top_k + t] = t < bn ? best_s[t] : 0.f;
            }
            cnt_out[row] = bn;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------ host side
struct Plan {
    int ew, stages, cand, qcap, nsplit, kblocks, ksteps_last, tiles, stream_a;
    int seed_stride, seed_q;      // 0 = no seed pass
    size_t smem;
    int lists() const { return nsplit; }          // one candidate list per (row, column split)
};

// Smallest q with P(Binomial(top_k, 1/stride) >= q) <= tol: the chance that q of a row's true top_k landed in the sample.
static int seed_quantile(int top_k, int stride, double tol) {
    const double pr = 1.0 / stride;
    double pmf = 1.0;
    for (int i = 0; i < top_k; ++i) pmf *= 1.0 - pr;          // P(X = 0)
    double tail = 1.0 - pmf;                                   // P(X >= 1)
    for (int q = 1; q <= top_k; ++q) {
        if (tail <= tol) return q;
        pmf *= (double)(top_k - q + 1) / q * pr / (1.0 - pr);  // P(X = q)
        tail -= pmf;
    }
    return top_k + 1;
}

static size_t smem_bytes(int ew, int kblocks, int stages, int cand, int qcap, bool stream_a = false) {
    (void)ew;
    return 1024 + (stream_a ? (size_t)stages * 2 * kTileBytes : (size_t)kblocks * kTileBytes + (size_t)stages * kTileBytes) + (size_t)cand * BM * 6 + BM * 12 +
           16 + (size_t)qcap * 68 + 16 + 8 * (2 * kMaxStages + 9) + 16;
}

// The overrides the tests use to reach the seeded and no-retry builds (SNG_KNN_CAND, SNG_KNN_SEED_S, SNG_KNN_SEED_Q,
// SNG_KNN_NORETRY) are OFF unless switched on with sng_set_debug_env(1): the product call path reads no environment (one
// static flag is tested instead) and keeps no other global state besides the cached SM count and driver entry point.
static int g_debug_env = 0;
static int env_int(const char* name, int lo, int hi) {
    if (!g_debug_env) return 0;
    const char* e = getenv(name);
    if (!e) return 0;
    const int v = atoi(e);
    return (v >= lo && v <= hi) ? v : 0;
}
static bool env_flag(const char* name) { return g_debug_env && getenv(name) != nullptr; }

// Candidate slots per row list.  The list keeps the row's best `cand` FP16 scores; stage 2 proves a row only if its k-th
// exact score clears the list's drop bound by the FP16 error, so cand - top_k is the number of near-cut columns a row may
// have before it has to go to the exact scan.
static int cand_for(int top_k, int margin) {
    const int o = env_int("SNG_KNN_CAND", top_k, 128);
    if (o) return o;
    return (top_k + margin + 1) / 2 * 2;
}

// top_k > 0: derive cand from top_k;  top_k == 0: use the explicit `cand` (stage-1 test entry point)
static int make_plan(Plan* pl, int64_t nq, int64_t n, int64_t d, int top_k, int cand, int force_ew) {
    const size_t kMaxSmem = 227 * 1024;
    const int d16 = (int)((d + 15) / 16 * 16);
    pl->kblocks = (d16 + BK - 1) / BK;
    pl->ksteps_last = (d16 - (pl->kblocks - 1) * BK) / kUmmaK;
    pl->tiles = (int)((n + BN - 1) / BN);
    pl->ew = 0;
    pl->stream_a = 0;
    // small K: the epilogue (TMEM reads) paces the kernel -> 16 epilogue warps; large K: the MMAs do -> fewer, deeper B ring
    const int ew_pref = d16 <= 128 ? 4 : (d16 <= 320 ? 2 : 1);
    if (force_ew == 4 && pl->kblocks > 2) force_ew = 2;        // EW = 4 is the split-N mode, built for at most two K blocks
    // Preference: a B ring of >= 3 stages first (pass 0), then the widest candidate margin, then the full hit queue.  Large
    // d (A alone is 128 KB at d = 512) or large top_k trade the margin away: the retry pass catches the rows that costs.
    static const int kMargins[] = {22, 14, 8, 4};
    for (int pass = 0; pass < 2 && !pl->ew; ++pass) {
        for (int ew = force_ew ? force_ew : ew_pref; ew >= 1 && !pl->ew; ew >>= 1) {
            // pass 0 wants BOTH a 3-stage ring and a margin of >= 14 slots; pass 1 gives up the third stage before the margin (a
            // row that cannot be proven costs an exact scan, a shallower ring a few per cent of the main pass)
            for (int mi = 0; mi < (top_k > 0 ? (pass ? 4 : 2) : 1) && !pl->ew; ++mi) {
                const int c = top_k > 0 ? cand_for(top_k, kMargins[mi]) : cand;
                if (c > kMaxCandTotal) continue;
                for (int qc = kQueue; qc >= 64 && !pl->ew; qc /= 4) {
                    const int want = pl->kblocks * 4 < kMaxStages ? (pl->kblocks * 4 > 4 ? pl->kblocks * 4 : 4) : kMaxStages;
                    for (int st = want; st >= (pass ? 2 : 3); --st) {
                        if (ew == 4 && st % pl->kblocks != 0) continue;      // split mode: a tile's K blocks share one ring lap
                        const size_t sz = smem_bytes(ew, pl->kblocks, st, c, qc);
                        if (sz <= kMaxSmem) { pl->ew = ew; pl->stages = st; pl->smem = sz; pl->cand = c; pl->qcap = qc; break; }
                    }
                }
            }
            if (force_ew) break;
        }
    }
    if (!pl->ew && force_ew != 4) {
        // the query block cannot stay resident (d > ~640): stream it through the ring with B, K block by K block.  One epilogue
        // warp per lane quarter (the MMAs of a large-K tile take far longer than its epilogue), the deepest ring that fits.
        static const int kMarginsS[] = {22, 14, 8, 4};
        for (int mi = 0; mi < (top_k > 0 ? 4 : 1) && !pl->ew; ++mi) {
            const int c = top_k > 0 ? cand_for(top_k, kMarginsS[mi]) : cand;
            if (c > kMaxCandTotal) continue;
            for (int qc = kQueue; qc >= 64 && !pl->ew; qc /= 4)
                for (int st = 5; st >= 2; --st) {
                    const size_t sz = smem_bytes(1, pl->kblocks, st, c, qc, true);
                    if (sz <= kMaxSmem) { pl->ew = 1; pl->stages = st; pl->smem = sz; pl->cand = c; pl->qcap = qc; pl->stream_a = 1; break; }
                }
        }
    }
    if (!pl->ew) { set_error("simknn: d=%lld top_k=%d does not fit in shared memory", (long long)d, top_k); return SNG_ERR_UNSUPPORTED; }
    // the pair kernel allocates all 512 TMEM columns: a CTA must own its SM, so never request less than half the shared memory
    if (pl->smem <= kMaxSmem / 2) pl->smem = kMaxSmem / 2 + 1024;
    const int64_t ctas = 2 * ((nq + 2 * BM - 1) / (2 * BM));
    int ns = (int)((3ll * sm_count() + ctas - 1) / ctas);
    if (ns > 8) ns = 8;
    if (ns > pl->tiles) ns = pl->tiles;
    while (ns > 1 && ns * pl->cand > kMaxCandTotal) --ns;
    if (ns < 1) ns = 1;
    pl->nsplit = ns;
    // threshold seeding: only for full builds (top_k known) that sweep many tiles with one list set per row
    pl->seed_stride = pl->seed_q = 0;
    // (the seed pass is never column-split: with ns splits it costs ns / stride of the main pass.  It still pays at every ns --
    // a rank's share of a sharded build of a small database gets 3 splits, and measured there (arxiv shape, 1/8 of the rows)
    // the unseeded lists cost 9.4 ms against 2.3 ms seeded: without a threshold every list starts with its warm-up inserts.)
    const bool forced = env_int("SNG_KNN_SEED_S", 2, 256) != 0;
    if (top_k > 0) {
        if (forced) {
            const int stride = env_int("SNG_KNN_SEED_S", 2, 256);
            int q = env_int("SNG_KNN_SEED_Q", 1, kSeedGroups - 2);
            if (!q) q = seed_quantile(top_k, stride, 2e-5);
            if (pl->tiles / stride >= 8 && q <= kSeedGroups - 4) { pl->seed_stride = stride; pl->seed_q = q; }
        } else {
            // sample 1/32 (1/16) of the columns when there are plenty, more of them for small databases; a large top_k needs a
            // sparser sample for the quantile to stay inside the 16 groups
            // (pokec shape, 6,379 tiles: stride 16 / 24 / 32 / 48 / 64 -> 397.1 / 392.5 / 389.1 / 389.7 / 390.5 ms per build: the
            // seed pass costs 1/stride of a sweep, a looser threshold a few more inserts)
            for (int stride = pl->tiles >= 2048 ? 32 : (pl->tiles >= 512 ? 16 : (pl->tiles / 32 > 4 ? pl->tiles / 32 : 4)); stride <= 64 && !pl->seed_stride; stride *= 2) {
                const int q = seed_quantile(top_k, stride, 2e-5);
                if (pl->tiles / stride >= 8 && q <= kSeedGroups - 4) { pl->seed_stride = stride; pl->seed_q = q; }
            }
        }
    }
    return SNG_OK;
}

template <int EW, bool SEED>
static cudaError_t launch_ew(dim3 grid, size_t smem, cudaStream_t st, const CUtensorMap& mq, const CUtensorMap& mdb, const Stage1Params& p) {
    cudaError_t e = cudaFuncSetAttribute(simknn_stage1_kernel<EW, SEED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    simknn_stage1_kernel<EW, SEED><<<grid, kNonEpiThreads + 128 * EW, smem, st>>>(mq, mdb, p);
    return cudaSuccess;
}

// seeds != nullptr && seed_out == nullptr: main pass starting from the seeded thresholds;  seed_out != nullptr: SEED pass.
static int launch_stage1(const Plan& pl, const uint16_t* xq, const uint16_t* xall, int64_t ldb, int64_t nq, int64_t q_offset, int64_t n,
                         float thr_lo, int remove_self, float* cand_val, int* cand_idx, float* cand_min, const float* seeds,
                         float* seed_out, int* phase, cudaStream_t st, const int* nq_dev = nullptr, const int* row_ids = nullptr) {
    const bool seed_pass = seed_out != nullptr;
    const int64_t n_db = seed_pass ? (n + pl.seed_stride - 1) / pl.seed_stride : n;
    CUtensorMap mq, mdb;
    if (int rc = make_tma_map_f16(&mq, xq, nq, ldb, ldb, 1)) return rc;
    if (int rc = make_tma_map_f16(&mdb, xall, n_db, ldb, ldb, seed_pass ? pl.seed_stride : 1)) return rc;   // seed pass: the column sample
    Stage1Params p;
    p.nq = (int)nq; p.n = (int)n_db; p.q_offset = (int)q_offset;
    p.kblocks = pl.kblocks; p.ksteps_last = pl.ksteps_last; p.stages = pl.stages; p.stream_a = pl.stream_a; p.cand = seed_pass ? 0 : pl.cand; p.qcap = pl.qcap;
    p.nsplit = seed_pass ? 1 : pl.nsplit; p.tiles_total = (int)((n_db + BN - 1) / BN); p.thr_lo = thr_lo; p.remove_self = remove_self;
    p.issuers = pl.stream_a ? 1 : (pl.kblocks <= 3 ? 2 : 1);
    p.cand_val = cand_val; p.cand_idx = cand_idx; p.cand_min = cand_min;
    p.phase = seed_pass ? nullptr : phase;
    p.nq_dev = nq_dev; p.row_ids = row_ids;
    p.seeds = seed_pass ? nullptr : seeds; p.seed_out = seed_out; p.seed_q = pl.seed_q; p.seed_stride = pl.seed_stride > 0 ? pl.seed_stride : 1;
    dim3 grid((unsigned)(2 * ((nq + 2 * BM - 1) / (2 * BM))), (unsigned)p.nsplit);        // x: CTA pairs (cluster of 2), y: column splits
    cudaError_t e;
    if (seed_pass) e = pl.ew == 4 ? launch_ew<4, true>(grid, pl.smem, st, mq, mdb, p)
                     : pl.ew == 2 ? launch_ew<2, true>(grid, pl.smem, st, mq, mdb, p)
                                  : launch_ew<1, true>(grid, pl.smem, st, mq, mdb, p);
    else e = pl.ew == 4 ? launch_ew<4, false>(grid, pl.smem, st, mq, mdb, p)
           : pl.ew == 2 ? launch_ew<2, false>(grid, pl.smem, st, mq, mdb, p)
                        : launch_ew<1, false>(grid, pl.smem, st, mq, mdb, p);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("simknn stage 1: cudaFuncSetAttribute(%zu B smem): %s", pl.smem, cudaGetErrorString(e)); return SNG_ERR_CUDA; }
    return check_launch(seed_pass ? "simknn seed pass" : "simknn stage 1");
}

static int check_common(const char* fn, const void* xq, const void* xall, int64_t ldb, int64_t nq, int64_t q_offset, int64_t n, int64_t d) {
    if (!xq || !xall) { set_error("%s: null operand", fn); return SNG_ERR_ARG; }
    if (nq <= 0 || n <= 0 || d <= 0 || q_offset < 0 || n >= (1ll << 31) || nq >= (1ll << 31)) { set_error("%s: bad nq/n/d/q_offset", fn); return SNG_ERR_ARG; }
    if (ldb % 8 != 0 || ldb < (d + 15) / 16 * 16) { set_error("%s: ldb=%lld must be a multiple of 8 and >= d rounded up to 16", fn, (long long)ldb); return SNG_ERR_ARG; }
    if (((uintptr_t)xq | (uintptr_t)xall) & 15) { set_error("%s: FP16 operands must be 16-byte aligned", fn); return SNG_ERR_ARG; }
    if (d > kMaxD) { set_error("%s: d=%lld > %d not supported", fn, (long long)d, kMaxD); return SNG_ERR_UNSUPPORTED; }
    return SNG_OK;
}

// worst-case |fp16-tensor-core score - exact FP32 score| for unit rows: 2 * 2^-11 (operand rounding) + accumulation slack
// The accumulation slack grows with the contraction length (the tensor cores add into their FP32 accumulators with truncation):
// 1.2e-4 covers K <= 640, longer contractions scale it.
constexpr float kScoreEps = 0.0009765625f + 1.2e-4f;
static float score_eps(int64_t d) { return 0.0009765625f + 1.2e-4f * (d > 640 ? (float)d / 640.0f : 1.0f); }
static int64_t retry_ld(int64_t d) { return (d + 15) / 16 * 16 + 64; }   // widest ldb (FP16 row pitch) the build accepts: the retry query matrix is sized for it

}  // namespace knn
}  // namespace sng

using namespace sng;
using namespace sng::knn;

static size_t align256(size_t x) { return (x + 255) / 256 * 256; }

extern "C" int sng_set_debug_env(int enabled) { const int was = sng::knn::g_debug_env; sng::knn::g_debug_env = enabled ? 1 : 0; return was; }

extern "C" size_t sng_simknn_workspace_bytes(int64_t nq, int64_t n, int64_t d, int top_k) {
    if (nq <= 0 || n <= 0 || d <= 0 || top_k <= 0 || top_k > SNG_KNN_MAX_TOPK) return 0;
    Plan pl;
    if (make_plan(&pl, nq, n, d, top_k, 0, 0)) return 0;
    const size_t slots = (size_t)nq * pl.lists() * pl.cand;
    const size_t part = (size_t)kFbWaveRows * ((n + kChunk - 1) / kChunk) * top_k;
    return align256(slots * 4) * 2 + align256((size_t)nq * pl.lists() * 4) + align256((size_t)nq * 4) + 2 * align256(part * 4) +
           align256((size_t)nq * kSeedGroups * 4) + 256 +
           align256((size_t)retry_rows(nq) * retry_ld(d) * 2) + 2 * align256((size_t)retry_rows(nq) * kMaxCandTotal * 4) + align256((size_t)retry_rows(nq) * 8 * 4) +
           align256((size_t)nq * 4) + 256 + 1024;
}

// The launch plan sng_simknn_build uses for this shape: out[0..7] = epilogue warps per lane quarter, candidate slots per list,
// column splits, seed stride (0 = no seed pass), seed quantile, B ring stages, K blocks, lists per row.
extern "C" int sng_simknn_plan(int64_t nq, int64_t n, int64_t d, int top_k, int32_t* out8) {
    SNG_REQUIRE(out8 && nq > 0 && n > 0 && d > 0 && top_k >= 1 && top_k <= SNG_KNN_MAX_TOPK, "sng_simknn_plan: bad arguments");
    Plan pl;
    if (int rc = make_plan(&pl, nq, n, d, top_k, 0, 0)) return rc;
    out8[0] = pl.ew; out8[1] = pl.cand; out8[2] = pl.nsplit; out8[3] = pl.seed_stride; out8[4] = pl.seed_q; out8[5] = pl.stages;
    out8[6] = pl.kblocks; out8[7] = pl.lists();
    return SNG_OK;
}

// Seed pass only (profiling / tests): seeds_out [nq, 16] = per-row maxima of the 16 column groups of the stride-sample.
extern "C" int sng_simknn_seed(const uint16_t* xq, const uint16_t* xall, int64_t ldb, int64_t nq, int64_t n, int64_t d, int seed_stride,
                               int force_ew, float* seeds_out, void* stream) {
    if (int rc = check_common("sng_simknn_seed", xq, xall, ldb, nq, 0, n, d)) return rc;
    SNG_REQUIRE(seeds_out && seed_stride >= 1 && seed_stride <= 256, "sng_simknn_seed: bad seed_stride / output");
    SNG_REQUIRE(force_ew == 0 || force_ew == 1 || force_ew == 2 || force_ew == 4, "sng_simknn_seed: force_ew must be 0, 1, 2 or 4");
    Plan pl;
    if (int rc = make_plan(&pl, nq, n, d, 0, 8, force_ew)) return rc;
    pl.seed_stride = seed_stride; pl.seed_q = 1;
    return launch_stage1(pl, xq, xall, ldb, nq, 0, n, -3.0e38f, 0, nullptr, nullptr, nullptr, nullptr, seeds_out, nullptr, (cudaStream_t)stream);
}

extern "C" int sng_simknn_stage1(const uint16_t* xq, const uint16_t* xall, int64_t ldb, int64_t nq, int64_t q_offset, int64_t n, int64_t d,
                                 int cand, float thr_lo, int remove_self, int32_t* cand_idx, float* cand_val, float* cand_min,
                                 int force_ew, int force_nsplit, int* lists_out, const float* seeds, int seed_q, int seed_stride,
                                 int32_t* sweep_phase, void* stream) {
    if (int rc = check_common("sng_simknn_stage1", xq, xall, ldb, nq, q_offset, n, d)) return rc;
    SNG_REQUIRE(cand >= 8 && cand <= 128 && cand_idx && cand_val && cand_min, "sng_simknn_stage1: bad cand / outputs");
    SNG_REQUIRE(force_ew == 0 || force_ew == 1 || force_ew == 2 || force_ew == 4, "sng_simknn_stage1: force_ew must be 0, 1, 2 or 4");
    Plan pl;
    if (int rc = make_plan(&pl, nq, n, d, 0, cand, force_ew)) return rc;
    if (force_nsplit > 0) pl.nsplit = force_nsplit < pl.tiles ? force_nsplit : pl.tiles;
    SNG_REQUIRE(pl.lists() * cand <= kMaxCandTotal, "sng_simknn_stage1: nsplit*ew*cand = %d exceeds %d", pl.lists() * cand, kMaxCandTotal);
    if (lists_out) *lists_out = pl.lists();
    SNG_REQUIRE(!seeds || (seed_q >= 1 && seed_q <= kSeedGroups - 2 && seed_stride >= 1),
                "sng_simknn_stage1: seeds need 1 <= seed_q <= %d, seed_stride >= 1", kSeedGroups - 2);
    pl.seed_q = seeds ? seed_q : 0; pl.seed_stride = seeds ? seed_stride : 0;
    return launch_stage1(pl, xq, xall, ldb, nq, q_offset, n, thr_lo, remove_self, cand_val, cand_idx, cand_min, seeds, nullptr, sweep_phase, (cudaStream_t)stream);
}

extern "C" int sng_simknn_build(const uint16_t* xq, const uint16_t* xall, int64_t ldb, const float* xq32, const float* xall32, int64_t ld32,
                                int64_t nq, int64_t q_offset, int64_t n, int64_t d, int top_k, float thr, int remove_self,
                                int32_t* idx, float* sim, int32_t* cnt, int32_t* n_fallback, int32_t* n_retry, void* workspace,
                                size_t workspace_bytes, void* stream) {
    if (int rc = check_common("sng_simknn_build", xq, xall, ldb, nq, q_offset, n, d)) return rc;
    SNG_REQUIRE(xq32 && xall32 && ld32 % 4 == 0 && ld32 >= d, "sng_simknn_build: FP32 rows must be padded to a multiple of 4 floats (ld32=%lld)", (long long)ld32);
    SNG_REQUIRE(top_k >= 1 && top_k <= SNG_KNN_MAX_TOPK, "sng_simknn_build: top_k=%d out of [1,%d]", top_k, SNG_KNN_MAX_TOPK);
    SNG_REQUIRE(idx && sim && cnt && n_fallback && workspace, "sng_simknn_build: null output / workspace");
    SNG_REQUIRE(ldb <= retry_ld(d), "sng_simknn_build: ldb=%lld > %lld (rows padded far beyond d)", (long long)ldb, (long long)retry_ld(d));
    const float eps = score_eps(d);
    if (workspace_bytes < sng_simknn_workspace_bytes(nq, n, d, top_k)) { set_error("sng_simknn_build: workspace too small (%zu < %zu)", workspace_bytes, sng_simknn_workspace_bytes(nq, n, d, top_k)); return SNG_ERR_WORKSPACE; }
    Plan pl;
    if (int rc = make_plan(&pl, nq, n, d, top_k, 0, 0)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int m_total = pl.lists() * pl.cand;
    uint8_t* w = reinterpret_cast<uint8_t*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    float* cand_val = reinterpret_cast<float*>(w); w += align256((size_t)nq * m_total * 4);
    int* cand_idx = reinterpret_cast<int*>(w); w += align256((size_t)nq * m_total * 4);
    float* cand_min = reinterpret_cast<float*>(w); w += align256((size_t)nq * pl.lists() * 4);
    int* fb_rows = reinterpret_cast<int*>(w); w += align256((size_t)nq * 4);
    const int n_chunks = (int)((n + kChunk - 1) / kChunk);
    const size_t part = (size_t)kFbWaveRows * n_chunks * top_k;
    float* part_s = reinterpret_cast<float*>(w); w += align256(part * 4);
    int* part_i = reinterpret_cast<int*>(w); w += align256(part * 4);
    float* seeds = reinterpret_cast<float*>(w); w += align256((size_t)nq * kSeedGroups * 4);
    int* phase = reinterpret_cast<int*>(w); w += 256;
    // retry pass buffers
    const int kRetryRows = retry_rows(nq);
    uint16_t* xq_retry = reinterpret_cast<uint16_t*>(w); w += align256((size_t)kRetryRows * retry_ld(d) * 2);
    float* rcand_val = reinterpret_cast<float*>(w); w += align256((size_t)kRetryRows * kMaxCandTotal * 4);
    int* rcand_idx = reinterpret_cast<int*>(w); w += align256((size_t)kRetryRows * kMaxCandTotal * 4);
    float* rcand_min = reinterpret_cast<float*>(w); w += align256((size_t)kRetryRows * 8 * 4);
    int* fb2_rows = reinterpret_cast<int*>(w); w += align256((size_t)nq * 4);
    int* n_fb1 = reinterpret_cast<int*>(w);                          // rows stage 2 could not prove (device counter)
    // retry plan (decided up front: it determines where stage 2 files the rows it cannot prove): the longest list that fits
    Plan pr;
    bool retry = false;
    if (!env_flag("SNG_KNN_NORETRY")) {
        const int want = top_k + 32 <= 64 ? 64 : (top_k + 32 <= 96 ? 96 : 128);
        for (int rcand = want; rcand >= top_k + 8 && !retry; rcand -= 16) {
            if (make_plan(&pr, kRetryRows, n, d, 0, rcand, pl.ew) != SNG_OK || pr.ew != pl.ew) continue;
            pr.seed_stride = pr.seed_q = 0;
            pr.nsplit = kMaxCandTotal / rcand < pr.tiles ? kMaxCandTotal / rcand : pr.tiles;
            if (pr.nsplit < 1) pr.nsplit = 1;
            // The retry pass is a handful of CTA pairs sweeping all n columns, so its latency is one pair's sweep.  The same total
            // list capacity per row (splits x slots <= 192) cut into the maximum of 8 column splits with shorter lists sweeps 8/3
            // as fast; a list still keeps top_k + 14 triples of ITS column range.
            if (pr.tiles >= 64) {
                const int rc8 = ((top_k + 14 > kMaxCandTotal / 8 ? top_k + 14 : kMaxCandTotal / 8) + 1) / 2 * 2;
                Plan p8;
                if (rc8 < rcand && 8 * rc8 <= kMaxCandTotal && make_plan(&p8, kRetryRows, n, d, 0, rc8, pl.ew) == SNG_OK && p8.ew == pl.ew) {
                    pr = p8; pr.seed_stride = pr.seed_q = 0; pr.nsplit = 8;
                }
            }
            retry = true;
        }
    }
    if (cudaMemsetAsync(phase, 0, 8 * sizeof(int), st) != cudaSuccess) return check_launch("sng_simknn_build memset");
    if (cudaMemsetAsync(n_fb1, 0, sizeof(int), st) != cudaSuccess) return check_launch("sng_simknn_build memset");
    if (cudaMemsetAsync(n_fallback, 0, sizeof(int), st) != cudaSuccess) return check_launch("sng_simknn_build memset");
    // approximate scores below thr - eps can never reach thr exactly
    const float thr_lo = thr - 1.01f * eps;
    if (pl.seed_stride > 0)
        if (int rc = launch_stage1(pl, xq, xall, ldb, nq, q_offset, n, thr_lo, remove_self, nullptr, nullptr, nullptr, nullptr, seeds, nullptr, st)) return rc;
    if (int rc = launch_stage1(pl, xq, xall, ldb, nq, q_offset, n, thr_lo, remove_self, cand_val, cand_idx, cand_min,
                               pl.seed_stride > 0 ? seeds : nullptr, nullptr, phase, st)) return rc;
    const int d4 = (int)((d + 3) / 4);
    // stage 2 flags the rows it cannot prove: into the retry list when there is a retry pass, else straight into the scan list
    int* flag_rows = retry ? fb_rows : fb2_rows;
    int* flag_cnt = retry ? n_fb1 : n_fallback;
    {
        simknn_rescore_kernel<<<grid_capped(nq, 8, 8), 256, (size_t)8 * 2 * 3 * m_total * 4, st>>>(
            xq32, xall32, ld32, d4, (int)nq, (int)n, (int)q_offset, remove_self, m_total, pl.lists(), top_k, thr, eps, cand_val, cand_idx, cand_min,
            idx, sim, cnt, flag_rows, flag_cnt, nullptr, nullptr);
        if (int rc = check_launch("simknn stage 2")) return rc;
    }
    if (retry) {
        // Retry pass: the (few) unproven rows -- a seed threshold that hid a neighbour, or more near-cut columns than the list
        // has slots -- go through the tensor cores once more as their own small query matrix, unseeded, with long lists and
        // the column range split over many CTAs; only rows that fail this proof too reach the exact FP32 scan.
        // seeded like the main pass but from a much lower quantile (10th..12th of the 16 group maxima instead of the 6th): it
        // cannot hide a neighbour (that would take top_k of top_k in a 1/stride sample) and spares the lists the warm-up
        if (pl.seed_stride > 0) { pr.seed_stride = pl.seed_stride; pr.seed_q = pl.seed_q + 4 < kSeedGroups - 4 ? pl.seed_q + 4 : kSeedGroups - 4; }
        // How many rows were flagged decides how many launches follow and how large they are, and a launch sized for the worst
        // case costs its CTAs' scheduling even when they leave at once (16 K idle CTAs of this kernel: 0.9 ms).  So the call
        // reads the 4-byte count back -- its one host synchronisation -- and sizes the rounds exactly: none at all for an input
        // whose rows were all proven, rounds of kRetryRows rows through the same buffers otherwise.  On a capturing stream
        // (no synchronisation allowed) one round of at most 16 K rows is launched with the count on the device; the rest
        // of the flagged rows then go to the exact scan.
        cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cap_status) != cudaSuccess) { cudaGetLastError(); cap_status = cudaStreamCaptureStatusNone; }
        const bool capturing = cap_status != cudaStreamCaptureStatusNone;
        int flagged = 0, rounds = 1, cap = kRetryRows;
        if (capturing) {
            cap = kRetryRowsMin < kRetryRows ? kRetryRowsMin : kRetryRows;
        } else {
            if (cudaMemcpyAsync(&flagged, n_fb1, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
                return check_launch("sng_simknn_build flagged-row count");
            rounds = (flagged + cap - 1) / cap;
            if (rounds > kRetryRounds) rounds = kRetryRounds;
        }
        int* round_cnt = phase + 16;                                  // (the 256-byte phase block: ints 0..7 = sweep phases)
        if (rounds > 0) simknn_retry_rounds_kernel<<<1, 256, 0, st>>>(fb_rows, n_fb1, cap, rounds, round_cnt, fb2_rows, n_fallback);
        const int mr = pr.lists() * pr.cand;
        for (int r = 0; r < rounds; ++r) {
            const int* rows_r = fb_rows + (size_t)r * cap;
            // rows of this round: exact on the host unless capturing (then the grid covers `cap` rows and the device count trims it)
            const int n_r = capturing ? cap : (flagged - r * cap < cap ? flagged - r * cap : cap);
            const int n_launch = (n_r + 2 * BM - 1) / (2 * BM) * (2 * BM);
            simknn_retry_gather_kernel<<<sm_count() * 2, 256, 0, st>>>(xq, ldb, rows_r, round_cnt + r, xq_retry);
            if (int rc = launch_stage1(pr, xq_retry, xall, ldb, n_launch, q_offset, n, thr_lo, remove_self, rcand_val, rcand_idx, rcand_min,
                                       pl.seed_stride > 0 ? seeds : nullptr, nullptr, nullptr, st, round_cnt + r, rows_r)) return rc;
            const int rblocks = (n_launch + 7) / 8 < 4096 ? (n_launch + 7) / 8 : 4096;
            simknn_rescore_kernel<<<rblocks, 256, (size_t)8 * 2 * 3 * mr * 4, st>>>(
                xq32, xall32, ld32, d4, n_launch, (int)n, (int)q_offset, remove_self, mr, pr.lists(), top_k, thr, eps, rcand_val, rcand_idx, rcand_min,
                idx, sim, cnt, fb2_rows, n_fallback, round_cnt + r, rows_r);
        }
        if (int rc = check_launch("simknn retry pass")) return rc;
    }
    if (n_retry) {
        if (cudaMemcpyAsync(n_retry, retry ? n_fb1 : n_fallback, sizeof(int), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            return check_launch("sng_simknn_build n_retry");
    }
    const int fb_grid = sm_count() * 4;                          // one resident wave: the flagged-row count is on the device
    for (int wave = 0; wave < kFbWaves; ++wave) {
        simknn_fb_scan_kernel<<<fb_grid, 256, 0, st>>>(xq32, xall32, ld32, d4, (int)n, (int)q_offset, top_k, thr, remove_self, fb2_rows, n_fallback,
                                                      wave, n_chunks, part_s, part_i);
        simknn_fb_merge_kernel<<<fb_grid, 256, 0, st>>>(fb2_rows, n_fallback, wave, n_chunks, top_k, part_s, part_i, idx, sim, cnt);
    }
    simknn_fb_stream_kernel<<<fb_grid, 256, 0, st>>>(xq32, xall32, ld32, d4, (int)n, (int)q_offset, top_k, thr, remove_self, fb2_rows,
                                                    n_fallback, kFbWaves * kFbWaveRows, idx, sim, cnt);
    return check_launch("simknn stage 3");
}
