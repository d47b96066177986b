// Edge-restricted similarity / selection / aggregation kernels (K0, K2, K2b, K3, K4, SDDMM).
//
// All of these are HBM/L2-gather bound (SURVEY.md §8(d)): one warp owns one target row; a group of
// G = C/4 lanes owns one in-edge at a time and fetches its source row with ONE 128-bit load per lane, so
// a warp step touches 32/G full rows (coalesced 16..512-byte segments).  Wider rows (C > 128, up to SNG_MAX_CHANNELS) take the
// whole warp, G/32 loads per lane (RowShape).  Scores, selection and the weighted reduction never leave registers / shared
// memory; nothing of size E is written.
//
// Reference call sites replaced: R: models/models.py:121-137,139-158 (++), :233-263 (+), :322-334 (base).
#include "sng_common.cuh"
#include <cuda_fp16.h>
#include <math_constants.h>
#include <stdlib.h>
#include <type_traits>

namespace sng {

constexpr int kWarpsPerBlock = 8;
constexpr int kThreads = kWarpsPerBlock * 32;

// Row layout of the lane-group kernels for G float4 slots per row (4 G channels).  G <= 32: a group of L = G lanes owns a row,
// one slot per lane, EPW = 32 / G rows per warp step.  G > 32 (wide rows, up to SNG_MAX_CHANNELS): the warp owns the row and
// lane l holds the V = G / 32 slots l, l + 32, ... (channels 4 (32 v + l) .. + 3), so each load instruction of the warp is one
// contiguous 512-byte segment of the row.
template <int G> struct RowShape {
    static constexpr int L = G < 32 ? G : 32;
    static constexpr int V = G / L;
    static constexpr int EPW = 32 / L;
};
// first channel of slot v of the lane with group index q
__device__ __forceinline__ int slot_c4(int q, int v) { return 4 * (q + 32 * v); }
template <int V> __device__ __forceinline__ float dotv(const float4 (&a)[V], const float4 (&b)[V]) {
    float d = dot4(a[0], b[0]);
#pragma unroll
    for (int v = 1; v < V; ++v) d += dot4(a[v], b[v]);
    return d;
}

// rows in flight per lane group: four (one 16-byte load each) for G <= 32; wide rows keep the same four loads per lane
template <int G> struct Unroll { static constexpr int value = G > 32 ? 128 / G : (G >= 4) ? 4 : G; };

// ------------------------------------------------------------------------------------------ K0
__global__ void __launch_bounds__(kThreads) rownorm_kernel(const float* __restrict__ x, int64_t n, int d, int64_t ldx,
                                                          float* __restrict__ xf, int ldf, __half* __restrict__ xh, int ldh,
                                                          float* __restrict__ inv) {
    const int lane = threadIdx.x & 31;
    int64_t row = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const int64_t stride = (int64_t)gridDim.x * kWarpsPerBlock;
    const int kmax = max(xf ? ldf : 0, xh ? ldh : 0);
    for (; row < n; row += stride) {
        const float* xr = x + row * ldx;
        float ss = 0.f;
        for (int k = lane; k < d; k += 32) { float v = __ldg(xr + k); ss = fmaf(v, v, ss); }
        ss = group_sum<32>(ss);
        const float r = fmaxf(sqrtf(ss), kNormEps);
        if (inv && lane == 0) inv[row] = 1.0f / r;
        for (int k = lane; k < kmax; k += 32) {
            const float v = k < d ? __ldg(xr + k) / r : 0.f;     // true division, as F.normalize does; zero padding beyond d
            if (xf && k < ldf) xf[row * ldf + k] = v;
            if (xh && k < ldh) xh[row * ldh + k] = __float2half_rn(v);
        }
    }
}

// inv_r[i] = 1 / max(||h_i||, 1e-12).  The edge kernels gather this scalar per edge (the array is L2 resident) instead of
// recomputing every source row's norm from its gathered features.  Row layout RowShape<G>, four rows in flight per group.
template <int G>
__global__ void __launch_bounds__(kThreads) row_inv_norm_kernel(const float* __restrict__ h, int64_t n, int c, int64_t ld, float* __restrict__ inv) {
    using S = RowShape<G>;
    constexpr int RPW = S::EPW;                                        // rows per warp step
    const int lane = threadIdx.x & 31, q = lane % S::L, grp = lane / S::L;
    const bool ch_ok = q * 4 < c;
    const int64_t nw = (int64_t)gridDim.x * kWarpsPerBlock;
    for (int64_t r0 = ((int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5)) * RPW * 4; r0 < n; r0 += nw * RPW * 4) {
        float ss[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t row = r0 + u * RPW + grp;
            ss[u] = 0.f;
            if (row < n && ch_ok) {
                const float4 v = ldg4(h + row * ld + q * 4);
                ss[u] = dot4(v, v);
#pragma unroll
                for (int s = 1; s < S::V; ++s) {
                    if (slot_c4(q, s) < c) { const float4 w = ldg4(h + row * ld + slot_c4(q, s)); ss[u] += dot4(w, w); }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float t = group_sum<S::L>(ss[u]);
            const int64_t row = r0 + u * RPW + grp;
            if (q == 0 && row < n) inv[row] = inv_norm_of(t);
        }
    }
}

// ------------------------------------------------------------------------------------------ K2 forward (+ fused K4 epilogue)
// One launch family computes, for every target row i with in-edge list P_i (CSR by target, position order):
//   s_e = <n_i, n_j>, S_i = first min(top_k, |P_i|) edges under (s desc, position asc) with s >= thr,
//   out_1[i] = sum_{e in S_i} s_e h_j / max(|P_i|, 1)                                  (R: models/models.py:139-158, 244-263, 331-334)
// or, with DSEL (denominator='selected', top_k > 0), out_1[i] = sum_{e in S_i} s_e h_j / max(|S_i|, 1): every variant
// applies sel_factor(|S_i|) where it knows the final count, and writes that factor to inv_denom[i] (training) for the backward.
// DSEL is a template flag: read at run time, it changed the registers or spills of 31 candidates-mode instances.
// and, when `wt` is given (SNGNN++ on a graph whose in-lists equal its out-lists), in the SAME pass over the edges
//   out_0[i] = sum_{e in P_i} Wt[j] + b_w,  out[i] = beta out_0 + (1 - beta) out_1 (+ bias)   (R: models/models.py:124-136)
// Rows are dispatched by in-degree (tables built once per graph, sngnn_b200/graph.py):
//   C <= 32:  deg <= 32   edge_fwd_staged_kernel<.., CHUNK = false>: warp per row, the in-list staged in shared memory, one pass
//             deg  > 32   the row is cut into <= 32-edge chunks; edge_fwd_staged_kernel<.., CHUNK = true> scores each chunk like a
//                         short row (so a hub is spread over many warps), edge_fwd_merge_kernel merges the chunk candidates
//   C  > 32 or no tables: edge_fwd_long_kernel (warp per row, 32-edge chunks, running top-k in shared memory) on every row,
//                         edge_fwd_hub_kernel (block per row) for the listed rows with deg > 1024
struct EdgeFwdArgs {
    const float* h; const float* inv_r;
    int n, row_offset, c, ldh;
    const int* rowptr; const int* col; const int* tpos;
    const int* rows; int n_rows;             // long / hub kernels: explicit list of (local) row ids, or nullptr = all n rows
    // rows with more than 32 in-edges, cut into <= 32-edge chunks that the staged kernel scores like short rows (CHUNK mode);
    // edge_fwd_merge_kernel then merges the per-chunk candidates of every long row
    const int4* chunk_tab; int n_chunks;     // (first edge position, edges, local row id, 0) per chunk
    const int* lrows; const int* lrow_ptr; int n_lrows;      // long rows (ascending) and their chunk ranges [lrow_ptr[i], lrow_ptr[i+1])
    float* tmp_s; int* tmp_p; int* tmp_cnt; float* tmp_acc; float* tmp_a0;   // per-chunk candidates [n_chunks, min(top_k,32)], partial sums [n_chunks, 4G]
    int skip_deg;                            // long kernel over all rows: rows with more in-edges are left to the hub kernel (0 = none)
    int top_k; float thr;
    float* inv_denom;                        // DSEL instances: the factor applied per row [n], or nullptr
    float* out; int ldo;
    int* sel_src; float* sel_w; int* sel_q; int* sel_cnt;      // saved for backward; all nullptr in inference
    const float* wt; int ldw; const float* b_w; const float* beta; const float* bias; float* diff;   // fused SNGNN++ epilogue
    int slots;                               // staged kernel: row slots per warp (>= 33, fused >= 65: any single item fits)
};

constexpr unsigned kFull = 0xffffffffu;
__device__ __forceinline__ void add4(float4& a, const float4& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
// order-preserving integer image of a float; 0 is reserved for "not a candidate"
__device__ __forceinline__ unsigned okey(float s) { const unsigned ub = __float_as_uint(s); return (ub & 0x80000000u) ? ~ub : (ub | 0x80000000u); }
__device__ __forceinline__ bool better_sp(float sa, int pa, float sb, int pb) { return sa > sb || (sa == sb && pa < pb); }

template <int G>
__device__ __forceinline__ void cross_group_sum4(float4& a) {
    a.x = cross_group_sum<G>(a.x); a.y = cross_group_sum<G>(a.y); a.z = cross_group_sum<G>(a.z); a.w = cross_group_sum<G>(a.w);
}

// denominator='selected': the per-row factor 1 / max(|S_i|, 1); the forward writes the same float to inv_denom for the backward
__device__ __forceinline__ float sel_factor(int cnt) { return 1.0f / (float)max(cnt, 1); }

// den = the row's in-degree (PyG aggr='mean': every candidate, selected or not) or, with DSEL, its selected count
template <bool FUSE>
__device__ __forceinline__ void write_row(const EdgeFwdArgs& a, int row, int c4, const float4& acc, const float4& a0, int den, float beta,
                                          const float4& bw, const float4& bb) {
    const float invd = 1.0f / (float)max(den, 1);
    const float4 o1 = scale4(acc, invd);
    const int64_t o = (int64_t)row * a.ldo + c4;
    if (FUSE) {
        const float4 o0 = make_float4(a0.x + bw.x, a0.y + bw.y, a0.z + bw.z, a0.w + bw.w);
        float4 r;
        r.x = beta * o0.x + (1.f - beta) * o1.x + bb.x; r.y = beta * o0.y + (1.f - beta) * o1.y + bb.y;
        r.z = beta * o0.z + (1.f - beta) * o1.z + bb.z; r.w = beta * o0.w + (1.f - beta) * o1.w + bb.w;
        *reinterpret_cast<float4*>(a.out + o) = r;
        if (a.diff) *reinterpret_cast<float4*>(a.diff + o) = make_float4(o0.x - o1.x, o0.y - o1.y, o0.z - o1.z, o0.w - o1.w);   // d out / d beta
    } else {
        *reinterpret_cast<float4*>(a.out + o) = o1;
    }
}

// ---- short rows (and the <= 32-edge chunks of long rows): the staged kernel ------------------------------------------------
// Built around shared-memory row staging so that the gathers of the NEXT row are in flight while the current row is scored
// (the floor of gathering random 128-byte rows on this part is ~10 TB/s, scripts/micro/gather_bw.cu; what a row-at-a-time
// kernel pays is the chain rowptr -> source ids -> rows, once per row): a warp copies the <= 32 source rows of a target row (and the Wt rows of the
// fused epilogue, and the target row itself) into its private stage with cp.async (LDGSTS, 16 bytes per lane, 32/G rows per
// instruction, no registers held by loads in flight), two stages per warp.  Row metadata runs three rows ahead (rowptr),
// source ids two rows ahead, gathers one row ahead, so no global load is consumed in the iteration that issued it.
// Scoring is lane = edge: every lane reads its own staged row with 128-bit shared loads against the staged target row --
// no shuffles, no butterfly (row slots are padded by one 16-byte chunk, which makes both this lane-per-row pattern and
// the lane-per-channel pattern below bank-conflict free without any address swizzle).  Selection is top_k rounds of a
// one-instruction warp max; the round's winner is known warp-wide, so the same round adds score x staged row to the
// output (lane = channel) -- rows that are not selected are never touched again, and the output row leaves as one
// coalesced store.  This kernel is bound by instruction issue, not by memory (ncu: profiles/): every phase is written to
// keep the per-row instruction count down.
constexpr int kStWarps = 4;
// resident CTAs per SM the staged kernels are compiled for (register caps): they are latency / issue bound with few warps
constexpr int kStMinBlocks = 8;
__device__ __forceinline__ void cp_async16(uint32_t dst, const float* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
// bytes of a staged row slot: the row padded by one 16-byte chunk (G > 1), so that slot strides are odd multiples of 16 B
template <int G> constexpr int staged_row_bytes() { return G == 1 ? 16 : 16 * G + 16; }

template <int G, bool FUSE, bool SELECT_ALL, bool CHUNK, bool DSEL = false>
__global__ void __launch_bounds__(kStWarps * 32, kStMinBlocks) edge_fwd_staged_kernel(const EdgeFwdArgs a) {
    constexpr int C = 4 * G;                    // channels of a padded row
    constexpr int RB = staged_row_bytes<G>();
    constexpr int EPW = 32 / G;                 // rows copied per cp.async instruction
    // Compact staging: an item takes deg source rows, the target row (slot deg) and, fused, deg Wt rows behind it from the
    // warp's pool of `slots` row slots; two items are alive at a time (A = being scored, B = in flight).  B goes behind A
    // when it fits there, else in front of A when it fits there, else it is staged after A is done (that item loses its
    // prefetch).  A fixed two-stage layout reserves 2 x 33 (65) slots per warp where an average row needs 20 (39): the pool
    // is what lets 28-32 warps share an SM instead of 20 (12), and this kernel is latency / issue bound.
    extern __shared__ __align__(128) unsigned char smraw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slots = a.slots;
    const uint32_t sbase = smem_u32(smraw) + (uint32_t)(warp * slots * RB);
    const int q = lane % G, grp = lane / G;     // copy role: chunk q of the row of edge st * EPW + grp
    const bool cq_ok = q * 4 < a.c;
    const int nch = (a.c + 3) >> 2;             // 16-byte chunks per row that hold data
    const int ch = lane % C;                    // accumulation role: channel ch (lanes >= C duplicate lanes < C)
    const bool ch_ok = ch < a.c;
    const char* hq = reinterpret_cast<const char*>(a.h + q * 4);
    const char* wq = FUSE ? reinterpret_cast<const char*>(a.wt + q * 4) : nullptr;
    const int64_t ldhb = (int64_t)a.ldh * 4, ldwb = (int64_t)a.ldw * 4;
    const int egrp = cq_ok ? grp : 64;                          // lanes of a chunk beyond the channel count never copy
    const uint32_t cp_off = (uint32_t)(grp * RB + q * 16);      // this lane's copy destination inside a step's EPW slots
    const uint32_t ch_off = (uint32_t)(ch * 4);
    float beta = 0.f, bw = 0.f, bb = 0.f;
    if (FUSE) { beta = __ldg(a.beta); if (ch_ok) { bw = __ldg(a.b_w + ch); if (a.bias) bb = __ldg(a.bias + ch); } }
    const bool train = !CHUNK && !SELECT_ALL && a.sel_cnt != nullptr;
    const bool want_q = train && a.sel_q != nullptr;
    const int stride = gridDim.x * kStWarps;
    const int row0 = blockIdx.x * kStWarps + warp;
    const int n_items = CHUNK ? a.n_chunks : a.n;               // CHUNK: work item = one <= 32-edge chunk of a long row
    const int kk = min(a.top_k, 32);

    // deg < 0: no such item; rows with more than 32 in-edges are left to the chunk pass ("active" = 0 <= deg <= 32).
    // trow = the item's target row (local id): the row itself, or the long row a chunk belongs to
    auto load_rp = [&](int item, int& beg, int& deg, int& trow) {
        beg = 0; deg = -1; trow = item;
        if (item < n_items) {
            if (CHUNK) { const int4 t = __ldg(a.chunk_tab + item); beg = t.x; deg = t.y; trow = t.z; }
            else { beg = __ldg(a.rowptr + item); deg = __ldg(a.rowptr + item + 1) - beg; }
        }
    };
    auto load_col = [&](int beg, int deg) { return ((unsigned)deg <= 32u && lane < deg) ? __ldg(a.col + beg + lane) : 0; };
    auto copy_steps = [&](uint32_t dst, uint32_t woff, int deg, int jl, auto lo, auto hi) {   // steps [lo, hi): per-lane predicates only, no branches
#pragma unroll
        for (int st = decltype(lo)::value; st < decltype(hi)::value; ++st) {
            const int j = __shfl_sync(kFull, jl, st * EPW + grp);
            if (st * EPW + egrp < deg) {
                cp_async16(dst + (uint32_t)(st * EPW * RB), reinterpret_cast<const float*>(hq + j * ldhb));
                if (FUSE) cp_async16(dst + woff + (uint32_t)(st * EPW * RB), reinterpret_cast<const float*>(wq + j * ldwb));
            }
        }
    };
    auto issue = [&](uint32_t st0, int row, int deg, int jl) {                           // gathers of one item -> one cp.async group (row = target row)
        if ((unsigned)deg <= 32u) {
            const uint32_t dst = st0 + cp_off;
            const uint32_t woff = (uint32_t)((deg + 1) * RB);                            // Wt rows behind the target row
            constexpr int H = G > 1 ? G / 2 : 1;
            copy_steps(dst, woff, deg, jl, std::integral_constant<int, 0>{}, std::integral_constant<int, H>{});
            if (G > 1 && deg > 16) copy_steps(dst, woff, deg, jl, std::integral_constant<int, H>{}, std::integral_constant<int, G>{});
            if (lane < nch) cp_async16(st0 + (uint32_t)(deg * RB) + (uint32_t)lane * 16u, a.h + (int64_t)(a.row_offset + row) * a.ldh + lane * 4);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto need_of = [&](int deg) { return (unsigned)deg <= 32u ? (FUSE ? 2 * deg + 1 : deg + 1) : 0; };
    auto place = [&](int bA, int nA, int nB) { return bA + nA + nB <= slots ? bA + nA : (nB <= bA ? 0 : -1); };

    // pipeline registers: item A = being computed, B = gathers in flight, C = source ids in flight, D = rowptr in flight
    int begA, degA, trA, begB, degB, trB, begC, degC, trC, begD, degD, trD;
    load_rp(row0, begA, degA, trA);
    load_rp(row0 + stride, begB, degB, trB);
    load_rp(row0 + 2 * stride, begC, degC, trC);
    int jlA = load_col(begA, degA), jlB = load_col(begB, degB);
    issue(sbase, trA, degA, jlA);
    int bA = 0, nA = need_of(degA);
    float irlA = 0.f, iriA = 0.f; int tqA = 0;
    if ((unsigned)degA <= 32u) {
        irlA = lane < degA ? __ldg(a.inv_r + jlA) : 0.f;
        iriA = __ldg(a.inv_r + a.row_offset + trA);
        if (want_q && lane < degA) tqA = __ldg(a.tpos + begA + lane);
    }
    for (int row = row0; row < n_items; row += stride) {
        // ---- look ahead: rowptr of item + 3 strides, source ids of item + 2, gathers (+ scalars) of item + 1
        load_rp(row + 3 * stride, begD, degD, trD);
        const int jlC = load_col(begC, degC);
        const int nB = need_of(degB);
        int bB = place(bA, nA, nB);
        const bool ahead = bB >= 0;                                                      // warp-uniform
        if (ahead) issue(sbase + (uint32_t)(bB * RB), trB, degB, jlB);
        const uint32_t stA = sbase + (uint32_t)(bA * RB);
        float irlB = 0.f, iriB = 0.f; int tqB = 0;
        if ((unsigned)degB <= 32u) {
            irlB = lane < degB ? __ldg(a.inv_r + jlB) : 0.f;
            iriB = __ldg(a.inv_r + a.row_offset + trB);
            if (want_q && lane < degB) tqB = __ldg(a.tpos + begB + lane);
        }
        if (ahead) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        // ---- row A
        if (degA <= 32) {                                                                // (degA >= 0 here)
            const int deg = degA;
            const bool has = lane < deg;
            // lane = edge: its own row slot; lanes without an edge read the target row's slot (inside the item, value unused)
            const uint32_t tgt = stA + (uint32_t)(deg * RB), own = stA + (uint32_t)(min(lane, deg) * RB);
            const uint32_t WOFF = (uint32_t)((deg + 1) * RB);
            float d = 0.f;
#pragma unroll
            for (int i = 0; i < G; ++i) {
                if (i < nch) {                                                           // warp-uniform
                    const float4 o4 = lds128(own + 16u * i), t4 = lds128(tgt + 16u * i);
                    d = fmaf(o4.x, t4.x, fmaf(o4.y, t4.y, fmaf(o4.z, t4.z, fmaf(o4.w, t4.w, d))));
                }
            }
            const float my_s = (d * iriA) * irlA + 0.0f;                                 // + 0: -0 becomes +0, equal scores get equal keys
            const uint32_t rd = stA + ch_off;                                            // lane = channel: word ch of a row slot
            float acc = 0.f, a0 = 0.f;
            int cnt = 0, myrank = -1;
            if (SELECT_ALL) {
                const float wsel = has ? my_s : 0.f;
#pragma unroll 4
                for (int e = 0; e < deg; ++e) acc = fmaf(__shfl_sync(kFull, wsel, e), lds32(rd + (uint32_t)(e * RB)), acc);
            } else {
                const bool cand = has && my_s >= a.thr;
                unsigned key = cand ? okey(my_s) : 0u;
                const int rounds = min(a.top_k, __popc(__ballot_sync(kFull, cand)));       // every round finds a candidate: no emptiness test inside
#pragma unroll 2
                for (; cnt < rounds; ++cnt) {
                    const unsigned mx = __reduce_max_sync(kFull, key);
                    const int w = __ffs(__ballot_sync(kFull, key == mx)) - 1;            // lowest lane = lowest edge position wins ties
                    if (!CHUNK) acc = fmaf(__shfl_sync(kFull, my_s, w), lds32(rd + (uint32_t)(w * RB)), acc);
                    if (lane == w) { key = 0u; myrank = cnt; }
                }
            }
            if (FUSE) {
#pragma unroll 4
                for (int e = 0; e < deg; ++e) a0 += lds32(rd + WOFF + (uint32_t)(e * RB));
            }
            if (CHUNK) {
                // a chunk only reports: its <= top_k candidates (score, edge position) in rank order and its partial sums
                if (!SELECT_ALL) {
                    if (myrank >= 0) { a.tmp_s[(int64_t)row * kk + myrank] = my_s; a.tmp_p[(int64_t)row * kk + myrank] = begA + lane; }
                    if (lane == 0) a.tmp_cnt[row] = cnt;
                }
                if (lane < C) {
                    if (SELECT_ALL) a.tmp_acc[(int64_t)row * C + ch] = acc;
                    if (FUSE) a.tmp_a0[(int64_t)row * C + ch] = a0;
                }
            } else {
                if (lane < C && ch_ok) {
                    // PyG aggr='mean': the full in-degree; denominator='selected': the selected count
                    const float o1 = DSEL ? acc * sel_factor(cnt) : __fdividef(acc, (float)max(deg, 1));
                    const int64_t o = (int64_t)row * a.ldo + ch;
                    if (FUSE) {
                        const float o0 = a0 + bw;
                        a.out[o] = beta * o0 + (1.f - beta) * o1 + bb;
                        if (a.diff) a.diff[o] = o0 - o1;
                    } else {
                        a.out[o] = o1;
                    }
                }
                if (train) {
                    const int64_t lo = (int64_t)row * a.top_k;
                    if (myrank >= 0) {
                        a.sel_src[lo + myrank] = jlA; a.sel_w[lo + myrank] = my_s;
                        if (want_q) a.sel_q[lo + myrank] = tqA;
                    }
                    for (int t = cnt + lane; t < a.top_k; t += 32) {                     // -1 padding behind the list
                        a.sel_src[lo + t] = -1; a.sel_w[lo + t] = 0.f;
                        if (want_q) a.sel_q[lo + t] = 0;
                    }
                    if (lane == 0) a.sel_cnt[row] = cnt;
                }
                if (DSEL && lane == 0 && a.inv_denom) a.inv_denom[row] = sel_factor(cnt);
            }
        }
        __syncwarp();                                                                    // A's slots are free from here
        if (!ahead) { bB = 0; issue(sbase, trB, degB, jlB); }                            // B did not fit next to A: staged now, waited for in full next iteration
        begA = begB; degA = degB; trA = trB; jlA = jlB; irlA = irlB; iriA = iriB; tqA = tqB; bA = bB; nA = nB;
        begB = begC; degB = degC; trB = trC; jlB = jlC;
        begC = begD; degC = degD; trC = trD;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// ---- narrow rows (C <= 4: a row is one float4), rows with <= 32 in-edges ---------------------------------------------------
// With 16-byte rows nothing is bound by bytes: the staged kernel spends ~400 warp instructions per row on copy issue,
// shared-memory row slots and lane = channel loops in which 4 of 32 lanes do useful work (1.3 ms per forward at the pokec
// shape for a layer whose rows total 26 MB).  Here lane = edge and the whole row lives in registers: each lane loads its
// source id, its source row (one LDG.128), 1/norm and (fused) its Wt row one item ahead of their use -- registers are the
// stage --, scores it against the target row, the top_k rounds run on the keys, and the weighted rows are summed ACROSS
// lanes with a recursive-halving reduction (K values over 32 lanes in ~4K instructions instead of 10 K).
// After lane_reduce_scatter<K> lane l holds the warp total of value index (l >> (5 - log2 K)) -- bit 4 of the lane is the
// most significant index bit.
template <int K>
__device__ __forceinline__ float lane_reduce_scatter(float (&v)[K], int lane) {
#pragma unroll
    for (int n = K; n > 1; n >>= 1) {
        const int m = 16 * n / K;                                                    // compile time after unrolling: 16, 8, ...
        const bool hi = (lane & m) != 0;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
            const float send = hi ? v[i] : v[i + n / 2];
            const float keep = hi ? v[i + n / 2] : v[i];
            v[i] = keep + __shfl_xor_sync(kFull, send, m);
        }
    }
    float r = v[0];
#pragma unroll
    for (int m = 16 / K; m > 0; m >>= 1) r += __shfl_xor_sync(kFull, r, m);
    return r;
}

struct NarrowGather { float4 hj, wj, hi; float irl, iri; int tq; };

template <bool FUSE, bool SELECT_ALL, bool DSEL = false>
__global__ void __launch_bounds__(kThreads) edge_fwd_narrow_kernel(const EdgeFwdArgs a) {
    constexpr int K = FUSE ? 8 : 4;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int stride = gridDim.x * kWarpsPerBlock;
    const int row0 = blockIdx.x * kWarpsPerBlock + warp;
    const bool train = !SELECT_ALL && a.sel_cnt != nullptr;
    const bool want_q = train && a.sel_q != nullptr;
    // the lane that holds (and writes) channel wc of out_1 after the reduction; fused: the Wt total of the channel sits in lane ^ 16
    const int wc = FUSE ? (lane >> 2) & 3 : (lane >> 3) & 3;
    const bool writer = (FUSE ? (lane & 0x13) == 0 : (lane & 7) == 0) && wc < a.c;
    float beta = 0.f, bw = 0.f, bb = 0.f;
    if (FUSE) { beta = __ldg(a.beta); if (wc < a.c) { bw = __ldg(a.b_w + wc); if (a.bias) bb = __ldg(a.bias + wc); } }
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);

    auto load_rp = [&](int row, int& beg, int& deg) {
        beg = 0; deg = -1;
        if (row < a.n) { beg = __ldg(a.rowptr + row); deg = __ldg(a.rowptr + row + 1) - beg; }
    };
    auto load_col = [&](int beg, int deg) { return ((unsigned)deg <= 32u && lane < deg) ? __ldg(a.col + beg + lane) : -1; };
    auto gather = [&](int row, int beg, int deg, int j, NarrowGather& g) {
        g.hj = z4; g.wj = z4; g.hi = z4; g.irl = 0.f; g.iri = 0.f; g.tq = 0;
        if ((unsigned)deg <= 32u) {
            g.hi = ldg4(a.h + (int64_t)(a.row_offset + row) * a.ldh);
            g.iri = __ldg(a.inv_r + a.row_offset + row);
            if (j >= 0) {
                g.hj = ldg4(a.h + (int64_t)j * a.ldh);
                g.irl = __ldg(a.inv_r + j);
                if (FUSE) g.wj = ldg4(a.wt + (int64_t)j * a.ldw);
                if (want_q) g.tq = __ldg(a.tpos + beg + lane);
            }
        }
    };

    // pipeline registers: A = being computed, B = gathers in flight, C = source ids in flight, D = rowptr in flight
    int begA, degA, begB, degB, begC, degC, begD, degD;
    load_rp(row0, begA, degA);
    load_rp(row0 + stride, begB, degB);
    load_rp(row0 + 2 * stride, begC, degC);
    int jA = load_col(begA, degA), jB = load_col(begB, degB);
    NarrowGather gA, gB;
    gather(row0, begA, degA, jA, gA);
    for (int row = row0; row < a.n; row += stride) {
        load_rp(row + 3 * stride, begD, degD);
        const int jC = load_col(begC, degC);
        gather(row + stride, begB, degB, jB, gB);
        if ((unsigned)degA <= 32u) {
            const int deg = degA;
            const bool has = lane < deg;
            // same operation order as the staged kernel (and its chunk pass): the scores are bit-identical to theirs
            const float d = fmaf(gA.hj.x, gA.hi.x, fmaf(gA.hj.y, gA.hi.y, fmaf(gA.hj.z, gA.hi.z, fmaf(gA.hj.w, gA.hi.w, 0.f))));
            const float my_s = (d * gA.iri) * gA.irl + 0.0f;
            int cnt = 0, myrank = -1;
            float wgt;
            if (SELECT_ALL) {
                wgt = has ? my_s : 0.f;
            } else {
                const bool cand = has && my_s >= a.thr;
                unsigned key = cand ? okey(my_s) : 0u;
                const int ncand = __popc(__ballot_sync(kFull, cand));
                const int rounds = min(a.top_k, ncand);
                if (!train && ncand <= a.top_k) {                                    // inference: every candidate is selected, no order needed
                    myrank = cand ? 0 : -1; cnt = ncand;
                } else {
#pragma unroll 2
                    for (; cnt < rounds; ++cnt) {
                        const unsigned mx = __reduce_max_sync(kFull, key);
                        const int w = __ffs(__ballot_sync(kFull, key == mx)) - 1;    // lowest lane = lowest edge position wins ties
                        if (lane == w) { key = 0u; myrank = cnt; }
                    }
                }
                wgt = myrank >= 0 ? my_s : 0.f;
            }
            float v[K];
            v[0] = wgt * gA.hj.x; v[1] = wgt * gA.hj.y; v[2] = wgt * gA.hj.z; v[3] = wgt * gA.hj.w;
            if (FUSE) { v[4] = gA.wj.x; v[5] = gA.wj.y; v[6] = gA.wj.z; v[7] = gA.wj.w; }       // zero for lanes without an edge
            const float tot = lane_reduce_scatter<K>(v, lane);
            const float a0 = FUSE ? __shfl_xor_sync(kFull, tot, 16) : 0.f;
            if (writer) {
                // PyG aggr='mean': the full in-degree; denominator='selected': the selected count
                const float o1 = DSEL ? tot * sel_factor(cnt) : __fdividef(tot, (float)max(deg, 1));
                const int64_t o = (int64_t)row * a.ldo + wc;
                if (FUSE) {
                    const float o0 = a0 + bw;
                    a.out[o] = beta * o0 + (1.f - beta) * o1 + bb;
                    if (a.diff) a.diff[o] = o0 - o1;
                } else {
                    a.out[o] = o1;
                }
            }
            if (train) {
                const int64_t lo = (int64_t)row * a.top_k;
                if (myrank >= 0) {
                    a.sel_src[lo + myrank] = jA; a.sel_w[lo + myrank] = my_s;
                    if (want_q) a.sel_q[lo + myrank] = gA.tq;
                }
                for (int t = cnt + lane; t < a.top_k; t += 32) {                     // -1 padding behind the list
                    a.sel_src[lo + t] = -1; a.sel_w[lo + t] = 0.f;
                    if (want_q) a.sel_q[lo + t] = 0;
                }
                if (lane == 0) a.sel_cnt[row] = cnt;
            }
            if (DSEL && lane == 0 && a.inv_denom) a.inv_denom[row] = sel_factor(cnt);
        }
        begA = begB; degA = degB; jA = jB; gA = gB;
        begB = begC; degB = degC; jB = jC;
        begC = begD; degC = degD;
    }
}

// Sorted (score desc, position asc) candidate list of one warp, in shared memory.
struct TopList {
    float* s;
    int* p;
    int cnt;
    float kth;   // score of the last entry once the list is full, else -inf
    // a warp scans its chunks in increasing position order, so a newcomer loses every tie: entries with score >= sc stay in front
    __device__ __forceinline__ void insert(float sc, int pos, int top_k, int lane) {
        int at = 0;
        for (int t0 = 0; t0 < cnt; t0 += 32) {
            const int t = t0 + lane;
            at += __popc(__ballot_sync(kFull, t < cnt && s[t] >= sc));
        }
        const int ncnt = min(cnt + 1, top_k);
        // shift [at, ncnt-1) one slot down; top_k <= 64 => two slots per lane
        float a0 = 0.f, a1 = 0.f; int b0 = 0, b1 = 0;
        const int t0 = lane, t1 = lane + 32;
        const bool m0 = t0 > at && t0 < ncnt, m1 = t1 > at && t1 < ncnt;
        if (m0) { a0 = s[t0 - 1]; b0 = p[t0 - 1]; }
        if (m1) { a1 = s[t1 - 1]; b1 = p[t1 - 1]; }
        __syncwarp();
        if (m0) { s[t0] = a0; p[t0] = b0; }
        if (m1) { s[t1] = a1; p[t1] = b1; }
        if (lane == 0 && at < top_k) { s[at] = sc; p[at] = pos; }
        __syncwarp();
        cnt = ncnt;
        kth = (cnt == top_k) ? s[top_k - 1] : -CUDART_INF_F;
    }
};

// One warp scans the 32-edge chunks first, first + step, ... of a row: lane e owns edge e of the chunk (source id, 1/norm,
// score); a group of RowShape<G>::L lanes fetches one source row per step.  SELECT_ALL accumulates the weighted rows on the
// fly, the selection variant only maintains the warp's top-k list (winners are re-gathered afterwards: they were loaded
// moments ago).  hb / wb / ni / ch_ok / acc / a0 hold one entry per float4 slot of the lane (RowShape<G>::V).
template <int G, bool FUSE, bool SELECT_ALL>
__device__ __forceinline__ void scan_row(const EdgeFwdArgs& a, const float* const (&hb)[RowShape<G>::V], const float* const (&wb)[RowShape<G>::V],
                                         int grow, int end, int first, int step, const float4 (&ni)[RowShape<G>::V],
                                         const bool (&ch_ok)[RowShape<G>::V], int lane, TopList& L, float4 (&acc)[RowShape<G>::V],
                                         float4 (&a0)[RowShape<G>::V]) {
    using S = RowShape<G>;
    constexpr int EPW = S::EPW, V = S::V;
    constexpr int U = (G <= 8) ? G : 8 / V;     // steps whose loads are issued together (eight 16-byte loads per lane from G = 8 on)
    const int grp = lane / S::L;
    for (int base = first; base < end; base += step) {
        const int nchunk = min(32, end - base);
        const bool has = lane < nchunk;
        const int jl = has ? __ldg(a.col + base + lane) : grow;                          // missing edges read the target row itself
        const float irl = __ldg(a.inv_r + jl);
        float my_d = 0.f;                                                               // <n_i, h_j> of edge base + lane
        for (int st = 0; st < nchunk; st += EPW * U) {
            float4 v[U][V];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = st + u * EPW + grp;
                const int j = __shfl_sync(kFull, jl, e & 31);
#pragma unroll
                for (int s = 0; s < V; ++s) v[u][s] = ldg4(hb[s] + (int64_t)j * a.ldh);
                if (FUSE && e < nchunk) {
#pragma unroll
                    for (int s = 0; s < V; ++s) add4(a0[s], ldg4(wb[s] + (int64_t)j * a.ldw));
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const float d = group_sum<S::L>(dotv<V>(ni, v[u]));
                if (SELECT_ALL) {
                    const int e = st + u * EPW + grp;
                    const float w = __shfl_sync(kFull, irl, e & 31);
#pragma unroll
                    for (int s = 0; s < V; ++s)
                        if (e < nchunk && ch_ok[s]) fma4(acc[s], d * w + 0.0f, v[u][s]);
                } else {
                    const float t = __shfl_sync(kFull, d, (lane % EPW) * S::L);          // hand (step, group) to the edge's lane
                    if (lane / EPW == st / EPW + u) my_d = t;
                }
            }
        }
        if (!SELECT_ALL) {
            const float my_s = my_d * irl + 0.0f;
            const bool valid = has && my_s >= a.thr;
            if (L.cnt == 0) {
                // empty list: top_k rounds of a one-instruction warp max; the lowest lane among the maxima = lowest edge position
                unsigned key = valid ? okey(my_s) : 0u;
                int t = 0;
                for (; t < a.top_k; ++t) {
                    const unsigned mx = __reduce_max_sync(kFull, key);
                    if (mx == 0u) break;
                    const int w = __ffs(__ballot_sync(kFull, key == mx)) - 1;
                    if (lane == w) { L.s[t] = my_s; L.p[t] = base + lane; key = 0u; }
                }
                __syncwarp();
                L.cnt = t;
                L.kth = (t == a.top_k) ? L.s[a.top_k - 1] : -CUDART_INF_F;
            } else {
                unsigned m = __ballot_sync(kFull, valid && (L.cnt < a.top_k || my_s > L.kth));
                while (m) {                                                             // ascending lane == ascending edge position
                    const int l = __ffs(m) - 1;
                    m &= m - 1;
                    const float sg = __shfl_sync(kFull, my_s, l);
                    if (L.cnt < a.top_k || sg > L.kth) L.insert(sg, base + l, a.top_k, lane);
                }
            }
        }
    }
}

// weighted sum of the <= top_k winners of a finished list (source ids re-read through their positions) + the saved lists
template <int G, bool DSEL>
__device__ __forceinline__ void finish_list(const EdgeFwdArgs& a, const float* const (&hb)[RowShape<G>::V], int row, const float* ls,
                                            const int* lp, int cnt, int lane, float4 (&acc)[RowShape<G>::V]) {
    using S = RowShape<G>;
    constexpr int EPW = S::EPW;
    const int grp = lane / S::L;
    for (int st = 0; st < cnt; st += EPW) {
        const int t = min(st + grp, cnt - 1);                                            // clamp: the duplicate gets weight 0
        const float w = st + grp < cnt ? ls[t] : 0.f;
        const int64_t o = (int64_t)__ldg(a.col + lp[t]) * a.ldh;
#pragma unroll
        for (int s = 0; s < S::V; ++s) fma4(acc[s], w, ldg4(hb[s] + o));
    }
    if (a.sel_cnt) {
        const int64_t lo = (int64_t)row * a.top_k;
        for (int t = lane; t < a.top_k; t += 32) {
            const bool ok = t < cnt;
            const int p = ok ? lp[t] : 0;
            a.sel_src[lo + t] = ok ? __ldg(a.col + p) : -1;
            a.sel_w[lo + t] = ok ? ls[t] : 0.f;
            if (a.sel_q) a.sel_q[lo + t] = (ok && a.tpos) ? __ldg(a.tpos + p) : 0;
        }
        if (lane == 0) a.sel_cnt[row] = cnt;
    }
    if (DSEL && lane == 0 && a.inv_denom) a.inv_denom[row] = sel_factor(cnt);
}

template <int G, bool FUSE, bool SELECT_ALL, bool DSEL = false>
__global__ void __launch_bounds__(kThreads) edge_fwd_long_kernel(const EdgeFwdArgs a) {
    using S = RowShape<G>;
    constexpr int V = S::V;
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    bool ch_ok[V];
    const float* hb[V];
    const float* wb[V];
    float beta = 0.f;
    float4 bw[V], bb[V];
    if (FUSE) beta = __ldg(a.beta);
#pragma unroll
    for (int s = 0; s < V; ++s) {
        ch_ok[s] = slot_c4(q, s) < a.c;
        const int c4 = ch_ok[s] ? slot_c4(q, s) : 0;
        hb[s] = a.h + c4;
        wb[s] = FUSE ? a.wt + c4 : nullptr;
        bw[s] = z4; bb[s] = z4;
        if (FUSE && ch_ok[s]) { bw[s] = ldg4(a.b_w + c4); if (a.bias) bb[s] = ldg4(a.bias + c4); }
    }
    TopList L;
    L.s = smem + (size_t)warp * 2 * max(a.top_k, 1);
    L.p = reinterpret_cast<int*>(L.s + max(a.top_k, 1));
    const int total = a.rows ? a.n_rows : a.n;
    for (int ri = blockIdx.x * kWarpsPerBlock + warp; ri < total; ri += gridDim.x * kWarpsPerBlock) {
        const int row = a.rows ? __ldg(a.rows + ri) : ri;
        const int grow = a.row_offset + row;
        const int beg = __ldg(a.rowptr + row), end = __ldg(a.rowptr + row + 1);
        if (a.skip_deg && end - beg > a.skip_deg) continue;
        float4 ni[V], acc[V], a0[V];
#pragma unroll
        for (int s = 0; s < V; ++s) {
            ni[s] = scale4(ldg4(hb[s] + (int64_t)grow * a.ldh), __ldg(a.inv_r + grow));
            if (!ch_ok[s]) ni[s] = z4;
            acc[s] = z4; a0[s] = z4;
        }
        L.cnt = 0; L.kth = -CUDART_INF_F;
        scan_row<G, FUSE, SELECT_ALL>(a, hb, wb, grow, end, beg, 32, ni, ch_ok, lane, L, acc, a0);
        if (!SELECT_ALL) { finish_list<G, DSEL>(a, hb, row, L.s, L.p, L.cnt, lane, acc); __syncwarp(); }
        const int den = DSEL ? L.cnt : end - beg;
#pragma unroll
        for (int s = 0; s < V; ++s) {
            cross_group_sum4<G>(acc[s]);
            if (FUSE) cross_group_sum4<G>(a0[s]);
            if (grp == 0 && ch_ok[s]) write_row<FUSE>(a, row, slot_c4(q, s), acc[s], a0[s], den, beta, bw[s], bb[s]);
        }
    }
}

// Long rows under the staged kernel (C <= 32): warp per long row.  Merges the per-chunk candidate lists (each in rank order,
// chunks in position order) into the row's top-k, sums the per-chunk partial sums, gathers the winners' rows (lane =
// channel) and writes the row exactly like the staged kernel does for a short row.
// top_k <= 16: a register tournament -- lanes [0, nw) hold the winners so far in rank order, the following lanes take the
// candidates of as many further chunks as fit, and top_k rounds of a warp max pick the new winners; lane order equals edge
// position order, so the lowest lane among equal scores is the reference's tie-break.  Larger top_k: sorted insertion into
// a shared-memory list (a newcomer loses every tie).
template <int G, bool FUSE, bool SELECT_ALL, bool DSEL = false>
__global__ void __launch_bounds__(kThreads) edge_fwd_merge_kernel(const EdgeFwdArgs a) {
    constexpr int C = 4 * G;
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ch = lane % C;
    const bool ch_ok = ch < a.c;
    const int k1 = max(a.top_k, 1), kk = max(min(a.top_k, 32), 1);
    const bool tournament = a.top_k + kk <= 32;
    float beta = 0.f, bw = 0.f, bb = 0.f;
    if (FUSE) { beta = __ldg(a.beta); if (ch_ok) { bw = __ldg(a.b_w + ch); if (a.bias) bb = __ldg(a.bias + ch); } }
    TopList L;
    L.s = smem + (size_t)warp * 2 * k1;
    L.p = reinterpret_cast<int*>(L.s + k1);
    for (int li = blockIdx.x * kWarpsPerBlock + warp; li < a.n_lrows; li += gridDim.x * kWarpsPerBlock) {
        const int row = __ldg(a.lrows + li);
        const int c0 = __ldg(a.lrow_ptr + li), c1 = __ldg(a.lrow_ptr + li + 1);
        const int deg = __ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row);
        float acc = 0.f, a0 = 0.f;
        int nsel = 0;                                                        // the row's final selected count
        if (SELECT_ALL || FUSE) {
#pragma unroll 4
            for (int ci = c0; ci < c1; ++ci) {
                if (SELECT_ALL) acc += __ldg(a.tmp_acc + (int64_t)ci * C + ch);
                if (FUSE) a0 += __ldg(a.tmp_a0 + (int64_t)ci * C + ch);
            }
        }
        if (!SELECT_ALL) {
            float ws = 0.f; int wp = 0, nw = 0;                              // winner of rank `lane` (lane < nw): score, edge position
            if (tournament) {
                for (int ci = c0; ci < c1;) {
                    const int nslots = (32 - nw) / kk;                       // chunks that fit behind the current winners
                    const int m = (lane - nw) / kk, t = (lane - nw) - m * kk;
                    const bool slot_ok = lane >= nw && m < nslots && ci + m < c1;
                    const int64_t o = (int64_t)(ci + (slot_ok ? m : 0)) * kk + (slot_ok ? t : 0);
                    const int n_c = slot_ok ? __ldg(a.tmp_cnt + ci + m) : 0;
                    const float sc = __ldg(a.tmp_s + o);                     // unconditional: [n_chunks, kk] is always in bounds
                    const int pc = __ldg(a.tmp_p + o);
                    const bool cand = slot_ok && t < n_c;
                    const bool valid = cand || lane < nw;
                    const float s = cand ? sc : ws;
                    const int p = cand ? pc : wp;
                    unsigned key = valid ? okey(s) : 0u;
                    const int rounds = min(a.top_k, __popc(__ballot_sync(kFull, valid)));
                    float ns = 0.f; int np = 0;
                    for (int r = 0; r < rounds; ++r) {
                        const unsigned mx = __reduce_max_sync(kFull, key);
                        const int w = __ffs(__ballot_sync(kFull, key == mx)) - 1;
                        const float ts = __shfl_sync(kFull, s, w);
                        const int tp = __shfl_sync(kFull, p, w);
                        if (lane == r) { ns = ts; np = tp; }
                        if (lane == w) key = 0u;
                    }
                    ws = ns; wp = np; nw = rounds;
                    ci += nslots;
                }
            } else {
                L.cnt = 0; L.kth = -CUDART_INF_F;
                for (int ci = c0; ci < c1; ++ci) {
                    const int n_c = __ldg(a.tmp_cnt + ci);
                    const float s = lane < n_c ? __ldg(a.tmp_s + (int64_t)ci * kk + lane) : 0.f;
                    const int p = lane < n_c ? __ldg(a.tmp_p + (int64_t)ci * kk + lane) : 0;
                    for (int t = 0; t < n_c; ++t) {                          // descending scores: the first one that cannot enter ends the chunk
                        const float sg = __shfl_sync(kFull, s, t);
                        if (!(L.cnt < a.top_k || sg > L.kth)) break;
                        L.insert(sg, __shfl_sync(kFull, p, t), a.top_k, lane);
                    }
                }
                nw = L.cnt;
            }
            // two winners per lane when top_k > 32 (list path only): ranks lane and lane + 32
            float ws1 = 0.f; int wp1 = 0;
            if (!tournament) {
                ws = lane < nw ? L.s[lane] : 0.f; wp = lane < nw ? L.p[lane] : 0;
                ws1 = lane + 32 < nw ? L.s[lane + 32] : 0.f; wp1 = lane + 32 < nw ? L.p[lane + 32] : 0;
                __syncwarp();
            }
            const int j0 = lane < nw ? __ldg(a.col + wp) : -1;
            const int j1 = lane + 32 < nw ? __ldg(a.col + wp1) : -1;
            for (int t0 = 0; t0 < nw; t0 += 4) {                             // the winners' rows four at a time, lane = channel
                float v[4], w[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int t = t0 + u;
                    const int j = t < 32 ? __shfl_sync(kFull, j0, t & 31) : __shfl_sync(kFull, j1, t & 31);
                    w[u] = t < 32 ? __shfl_sync(kFull, ws, t & 31) : __shfl_sync(kFull, ws1, t & 31);
                    v[u] = (t < nw && ch_ok) ? __ldg(a.h + (int64_t)j * a.ldh + ch) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) acc = fmaf(t0 + u < nw ? w[u] : 0.f, v[u], acc);
            }
            if (a.sel_cnt) {
                const int64_t lo = (int64_t)row * a.top_k;
                if (lane < a.top_k) {
                    a.sel_src[lo + lane] = j0; a.sel_w[lo + lane] = ws;
                    if (a.sel_q) a.sel_q[lo + lane] = (lane < nw && a.tpos) ? __ldg(a.tpos + wp) : 0;
                }
                if (lane + 32 < a.top_k) {
                    a.sel_src[lo + lane + 32] = j1; a.sel_w[lo + lane + 32] = ws1;
                    if (a.sel_q) a.sel_q[lo + lane + 32] = (lane + 32 < nw && a.tpos) ? __ldg(a.tpos + wp1) : 0;
                }
                if (lane == 0) a.sel_cnt[row] = nw;
            }
            nsel = nw;
        }
        if (DSEL && lane == 0 && a.inv_denom) a.inv_denom[row] = sel_factor(nsel);
        if (lane < C && ch_ok) {
            const float o1 = DSEL ? acc * sel_factor(nsel) : __fdividef(acc, (float)max(deg, 1));
            const int64_t o = (int64_t)row * a.ldo + ch;
            if (FUSE) {
                const float o0 = a0 + bw;
                a.out[o] = beta * o0 + (1.f - beta) * o1 + bb;
                if (a.diff) a.diff[o] = o0 - o1;
            } else {
                a.out[o] = o1;
            }
        }
    }
}

// Hub rows (in-degree > 1024): one block per row.  Warp w scans chunks w, w + 8, ... with its own top-k list; the 8 lists
// are merged by ranking their <= 8 top_k entries against each other (positions are unique, so (score, position) is a
// strict order and the ranks are the final ranks); warp 0 then finishes the row exactly like the long-row kernel.
template <int G, bool FUSE, bool SELECT_ALL, bool DSEL = false>
__global__ void __launch_bounds__(kThreads) edge_fwd_hub_kernel(const EdgeFwdArgs a) {
    using S = RowShape<G>;
    constexpr int V = S::V;
    constexpr int PW = 128 * V;                 // channels of a partial-sum row: a warp's 32 lanes x V slots x 4
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int k1 = max(a.top_k, 1);
    bool ch_ok[V];
    const float* hb[V];
    const float* wb[V];
    float beta = 0.f;
    float4 bw[V], bb[V];
    if (FUSE) beta = __ldg(a.beta);
#pragma unroll
    for (int s = 0; s < V; ++s) {
        ch_ok[s] = slot_c4(q, s) < a.c;
        const int c4 = ch_ok[s] ? slot_c4(q, s) : 0;
        hb[s] = a.h + c4;
        wb[s] = FUSE ? a.wt + c4 : nullptr;
        bw[s] = z4; bb[s] = z4;
        if (FUSE && ch_ok[s]) { bw[s] = ldg4(a.b_w + c4); if (a.bias) bb[s] = ldg4(a.bias + c4); }
    }
    // shared memory: the warps' partial sums (acc, a0: PW channels each; first, so they stay 16-byte aligned), 8 warp lists,
    // the final list, the list lengths
    float* part = smem;
    float* lists = smem + (size_t)kWarpsPerBlock * 2 * PW;
    float* fin_s = lists + (size_t)kWarpsPerBlock * 2 * k1;
    int* fin_p = reinterpret_cast<int*>(fin_s + k1);
    int* wcnt = fin_p + k1;
    TopList L;
    L.s = lists + (size_t)warp * 2 * k1;
    L.p = reinterpret_cast<int*>(L.s + k1);
    for (int ri = blockIdx.x; ri < a.n_rows; ri += gridDim.x) {
        const int row = __ldg(a.rows + ri);
        const int grow = a.row_offset + row;
        const int beg = __ldg(a.rowptr + row), end = __ldg(a.rowptr + row + 1);
        float4 ni[V], acc[V], a0[V];
#pragma unroll
        for (int s = 0; s < V; ++s) {
            ni[s] = scale4(ldg4(hb[s] + (int64_t)grow * a.ldh), __ldg(a.inv_r + grow));
            if (!ch_ok[s]) ni[s] = z4;
            acc[s] = z4; a0[s] = z4;
        }
        L.cnt = 0; L.kth = -CUDART_INF_F;
        scan_row<G, FUSE, SELECT_ALL>(a, hb, wb, grow, end, beg + 32 * warp, 32 * kWarpsPerBlock, ni, ch_ok, lane, L, acc, a0);
#pragma unroll
        for (int s = 0; s < V; ++s) {
            cross_group_sum4<G>(acc[s]);
            cross_group_sum4<G>(a0[s]);
        }
        if (grp == 0) {
#pragma unroll
            for (int s = 0; s < V; ++s) {
                *reinterpret_cast<float4*>(part + (size_t)(warp * 2) * PW + slot_c4(q, s)) = acc[s];
                *reinterpret_cast<float4*>(part + (size_t)(warp * 2 + 1) * PW + slot_c4(q, s)) = a0[s];
            }
        }
        if (lane == 0) wcnt[warp] = L.cnt;
        __syncthreads();
        int cnt = 0;
        if (!SELECT_ALL) {
            int total = 0;
            for (int w = 0; w < kWarpsPerBlock; ++w) total += wcnt[w];
            cnt = min(total, a.top_k);
            for (int m = threadIdx.x; m < kWarpsPerBlock * k1; m += kThreads) {
                const int w = m / k1, i = m - w * k1;
                if (i >= wcnt[w]) continue;
                const float s = lists[(size_t)w * 2 * k1 + i];
                const int p = reinterpret_cast<int*>(lists + (size_t)w * 2 * k1 + k1)[i];
                int rank = 0;
                for (int w2 = 0; w2 < kWarpsPerBlock; ++w2) {
                    const float* s2 = lists + (size_t)w2 * 2 * k1;
                    const int* p2 = reinterpret_cast<const int*>(s2 + k1);
                    for (int i2 = 0; i2 < wcnt[w2]; ++i2) rank += better_sp(s2[i2], p2[i2], s, p) ? 1 : 0;
                }
                if (rank < a.top_k) { fin_s[rank] = s; fin_p[rank] = p; }
            }
            __syncthreads();
        }
        if (warp == 0) {
            float4 sacc[V], sa0[V];
#pragma unroll
            for (int s = 0; s < V; ++s) {
                sacc[s] = z4; sa0[s] = z4;
                if (grp == 0) {
                    for (int w = 0; w < kWarpsPerBlock; ++w) {
                        if (SELECT_ALL) add4(sacc[s], *reinterpret_cast<const float4*>(part + (size_t)(w * 2) * PW + slot_c4(q, s)));
                        if (FUSE) add4(sa0[s], *reinterpret_cast<const float4*>(part + (size_t)(w * 2 + 1) * PW + slot_c4(q, s)));
                    }
                }
            }
            if (!SELECT_ALL) {
                finish_list<G, DSEL>(a, hb, row, fin_s, fin_p, cnt, lane, sacc);
#pragma unroll
                for (int s = 0; s < V; ++s) cross_group_sum4<G>(sacc[s]);
            }
#pragma unroll
            for (int s = 0; s < V; ++s)
                if (grp == 0 && ch_ok[s]) write_row<FUSE>(a, row, slot_c4(q, s), sacc[s], sa0[s], DSEL ? cnt : end - beg, beta, bw[s], bb[s]);
        }
        __syncthreads();
    }
}

// list-only aggregation (all-pairs mode)
template <int G>
__global__ void __launch_bounds__(kThreads) list_agg_fwd_kernel(
    const float* __restrict__ h, int n_rows, int c, int64_t ldh, int list_k, const int* __restrict__ sel_src,
    const float* __restrict__ sel_w, const int* __restrict__ sel_cnt, const float* __restrict__ inv_denom,
    float* __restrict__ out, int64_t ldo) {
    using S = RowShape<G>;
    constexpr int EPW = S::EPW, V = S::V;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L, c4 = q * 4;
    const bool ch_ok = c4 < c;
    for (int row = blockIdx.x * kWarpsPerBlock + warp; row < n_rows; row += gridDim.x * kWarpsPerBlock) {
        const int cnt = min(__ldg(sel_cnt + row), list_k);
        float4 acc[V];
#pragma unroll
        for (int s = 0; s < V; ++s) acc[s] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int st = 0; st < cnt; st += EPW) {
            const int t = st + grp;
            if (t < cnt && ch_ok) {                                  // ch_ok = slot 0 holds data; a lane's later slots may not
                const int j = __ldg(sel_src + (int64_t)row * list_k + t);
                const float w = __ldg(sel_w + (int64_t)row * list_k + t);
#pragma unroll
                for (int s = 0; s < V; ++s)
                    if (s == 0 || slot_c4(q, s) < c) fma4(acc[s], w, ldg4(h + (int64_t)j * ldh + slot_c4(q, s)));
            }
        }
#pragma unroll
        for (int s = 0; s < V; ++s) {
            acc[s].x = cross_group_sum<G>(acc[s].x); acc[s].y = cross_group_sum<G>(acc[s].y);
            acc[s].z = cross_group_sum<G>(acc[s].z); acc[s].w = cross_group_sum<G>(acc[s].w);
            if (grp == 0 && slot_c4(q, s) < c)
                *reinterpret_cast<float4*>(out + (int64_t)row * ldo + slot_c4(q, s)) = scale4(acc[s], inv_denom ? __ldg(inv_denom + row) : 1.f);
        }
    }
}

// ------------------------------------------------------------------------------------------ K2b backward
template <int G, bool SELECT_ALL>
__global__ void __launch_bounds__(kThreads) edge_agg_bwd_scatter_kernel(
    const float* __restrict__ h, const float* __restrict__ inv_r, const float* __restrict__ g, int n, int row_offset, int c, int64_t ld, const int* __restrict__ rowptr,
    const int* __restrict__ col, int top_k, const int* __restrict__ sel_src, const float* __restrict__ sel_w,
    const int* __restrict__ sel_cnt, const float* __restrict__ inv_denom, float* __restrict__ dval, float* __restrict__ dnrm) {
    using S = RowShape<G>;
    constexpr int EPW = S::EPW, V = S::V;
    constexpr int U = Unroll<G>::value;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    bool ok[V];                                                  // slot holds data; ok[s] implies ok[0]
    int c4[V];
#pragma unroll
    for (int s = 0; s < V; ++s) { c4[s] = slot_c4(q, s); ok[s] = c4[s] < c; }
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int row = blockIdx.x * kWarpsPerBlock + warp; row < n; row += gridDim.x * kWarpsPerBlock) {
        int beg, cnt;
        float invd;
        if (SELECT_ALL) {
            beg = __ldg(rowptr + row);
            cnt = __ldg(rowptr + row + 1) - beg;
            invd = 1.0f / (float)max(cnt, 1);
        } else {
            beg = 0;
            cnt = __ldg(sel_cnt + row);
            invd = __ldg(inv_denom + row);
        }
        if (cnt == 0) continue;
        const int grow = row_offset + row;                       // h / inv_r / dval / dnrm hold all nodes, g and the lists are shard-local
        float4 ni[V], gs[V], dni[V];
#pragma unroll
        for (int s = 0; s < V; ++s) {
            const float4 hi = ok[s] ? ldg4(h + (int64_t)grow * ld + c4[s]) : z4;
            ni[s] = scale4(hi, __ldg(inv_r + grow));
            gs[s] = ok[s] ? scale4(ldg4(g + (int64_t)row * ld + c4[s]), invd) : z4;    // g_i / deg_i
            dni[s] = z4;
        }
        for (int st = 0; st < cnt; st += EPW * U) {
            float4 v[U][V]; int j[U]; float w[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int t = st + u * EPW + grp;
                j[u] = -1; w[u] = 0.f;
                if (t < cnt) {
                    if (SELECT_ALL) j[u] = __ldg(col + beg + t);
                    else { j[u] = __ldg(sel_src + (int64_t)row * top_k + t); w[u] = __ldg(sel_w + (int64_t)row * top_k + t); }
                }
#pragma unroll
                for (int s = 0; s < V; ++s) v[u][s] = (j[u] >= 0 && ok[s]) ? ldg4(h + (int64_t)j[u] * ld + c4[s]) : z4;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (st + u * EPW >= cnt) break;
                const float inv_rj = j[u] >= 0 ? __ldg(inv_r + j[u]) : 0.f;
                const float sc = SELECT_ALL ? group_sum<S::L>(dotv<V>(ni, v[u])) * inv_rj + 0.0f : w[u];
                const float ds = group_sum<S::L>(dotv<V>(v[u], gs));           // dL/ds_e = (h_j . g_i)/deg_i
                if (j[u] >= 0 && ok[0]) {
#pragma unroll
                    for (int s = 0; s < V; ++s) {
                        if (s > 0 && !ok[s]) continue;
                        atomicAdd(reinterpret_cast<float4*>(dval + (int64_t)j[u] * ld + c4[s]), scale4(gs[s], sc));
                        atomicAdd(reinterpret_cast<float4*>(dnrm + (int64_t)j[u] * ld + c4[s]), scale4(ni[s], ds));
                        fma4(dni[s], ds * inv_rj, v[u][s]);                    // ds * n_j
                    }
                }
            }
        }
#pragma unroll
        for (int s = 0; s < V; ++s) {
            dni[s].x = cross_group_sum<G>(dni[s].x); dni[s].y = cross_group_sum<G>(dni[s].y);
            dni[s].z = cross_group_sum<G>(dni[s].z); dni[s].w = cross_group_sum<G>(dni[s].w);
            if (grp == 0 && ok[s]) atomicAdd(reinterpret_cast<float4*>(dnrm + (int64_t)grow * ld + c4[s]), dni[s]);
        }
    }
}

// pass 2: dh = dval + (dnrm - n (n . dnrm)) / r      (one lane-group per row)
template <int G>
__global__ void __launch_bounds__(kThreads) norm_bwd_finish_kernel(const float* __restrict__ h, const float* __restrict__ inv_rv, int n, int c, int64_t ld,
                                                                  const float* __restrict__ dval, const float* __restrict__ dnrm,
                                                                  float* __restrict__ dh) {
    using S = RowShape<G>;
    constexpr int RPW = S::EPW, V = S::V;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    int c4[V];
    bool ch_ok[V];
#pragma unroll
    for (int s = 0; s < V; ++s) { c4[s] = slot_c4(q, s); ch_ok[s] = c4[s] < c; }
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r0 = (blockIdx.x * kWarpsPerBlock + warp) * RPW; r0 < n; r0 += gridDim.x * kWarpsPerBlock * RPW) {
        const int row = r0 + grp;
        bool ok[V];
        float4 hi[V], ni[V], dn[V];
#pragma unroll
        for (int s = 0; s < V; ++s) ok[s] = row < n && ch_ok[s];
#pragma unroll
        for (int s = 0; s < V; ++s) hi[s] = ok[s] ? ldg4(h + (int64_t)row * ld + c4[s]) : z4;
        const float inv_r = row < n ? __ldg(inv_rv + row) : 0.f;
#pragma unroll
        for (int s = 0; s < V; ++s) ni[s] = scale4(hi[s], inv_r);
#pragma unroll
        for (int s = 0; s < V; ++s) dn[s] = ok[s] ? ldg4(dnrm + (int64_t)row * ld + c4[s]) : z4;
        const float proj = group_sum<S::L>(dotv<V>(ni, dn));
#pragma unroll
        for (int s = 0; s < V; ++s) {
            if (ok[s]) {
                const float4 dv = ldg4(dval + (int64_t)row * ld + c4[s]);
                float4 o;
                o.x = dv.x + (dn[s].x - ni[s].x * proj) * inv_r; o.y = dv.y + (dn[s].y - ni[s].y * proj) * inv_r;
                o.z = dv.z + (dn[s].z - ni[s].z * proj) * inv_r; o.w = dv.w + (dn[s].w - ni[s].w * proj) * inv_r;
                *reinterpret_cast<float4*>(dh + (int64_t)row * ld + c4[s]) = o;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------ K2b backward, deterministic (two gather passes)
// Closed form of SURVEY.md §3.4 without float atomics.  For a selected edge e = (j -> i), g1 = gscale * g (gscale = 1 - beta
// under the fused SNGNN++ epilogue, else 1), deg_i = max(|P_i|, 1):
//   dval_j += (s_e / deg_i) g1_i          ds_e = (h_j . g1_i) / deg_i          dn_i += ds_e n_j          dn_j += ds_e n_i
//   dh = dval + (dn - n (n . dn)) / r
// Pass T (by target, over the saved selection lists or the whole CSR): ds_e, the target side dn_i -> dnT, and the two
//   per-edge coefficients A_e = s_e gscale / deg_i, B_e = ds_e / r_i written at the edge's position in the BY-SOURCE
//   arrays (tpos, built once by sng_graph_prepare).
// Pass S (by source, over the out-edges): dval_j = sum A_e g_i, dn_j = dnT_j + sum B_e h_i, then the normalisation
//   backward, all in registers; under the fused epilogue the same walk also sums beta g_i over ALL out-edges = dL/dWt_j.
// Every sum runs in a fixed order: the result is bit-reproducible.
// Row shards: the call owns target rows [row_offset, row_offset + n) of h (all n_total rows); g, the lists, the CSR by
// target, dnT and the by-source CSR (the shard's in-edges only, targets as local ids) are shard-local.  Pass S still runs
// every source row j of n_total and writes dh_j = this shard's contribution; dnT_j exists only for the rows it owns.
// Neighbour lists (sng_list_bwd): the saved lists are fixed-width kNN lists, inv_denom[i] replaces 1 / deg_i (the pass-T
// kernels then never read rowptr), and the by-source CSR is their transpose (sng_list_transpose, src_shift 0).
// Edges under denominator='selected' (sng_edge_bwd_denom): the same inv_denom, the factor the forward applied per row.  Selection
// carries no gradient, so it is a per-row constant and the closed form holds with 1 / deg_i replaced by it.
struct EdgeBwdArgs {
    const float* h; const float* inv_r; const float* g;
    int n_total, n, row_offset, c, ld, ldg;
    const int* rowptr; const int* col; const int* tpos;
    int top_k; const int* sel_src; const float* sel_w; const int* sel_q; const int* sel_cnt;
    const float* inv_denom;                  // NULL: 1 / max(deg_i, 1) from rowptr (edges); else per target row (lists, 'selected')
    const float* beta; const float* diff; int lddiff; float* dbeta_part;
    float2* coef; float* dnT;
    const int* rowptr_out; const int* col_out; int shift;
    float* dh; float* dwt; int lddw;
    // staged source pass: source rows with more than 32 out-edges are cut into <= 32-edge chunks (tables over the by-source
    // CSR, built like the forward's), each chunk writes partial sums, edge_bwd_source_merge_kernel adds them and finishes
    const int4* chunk_tab; int n_chunks; const int* lrows; const int* lrow_ptr; int n_lrows;
    float* tmp_part;                         // [n_chunks, 3, 4G]
    int slots;                               // staged source pass: row slots per warp (>= 64: any single item fits)
};

// source row j is one of the call's target rows: pass T wrote its target-side dn at dnT[j - row_offset]
__device__ __forceinline__ bool owns_row(const EdgeBwdArgs& a, int j) { return (unsigned)(j - a.row_offset) < (unsigned)a.n; }

// LIST: the saved lists come with a.inv_denom -- neighbour lists, or edges under denominator='selected' (a template flag: a
// runtime branch costs the edge instances at C = 32 / 64 an 8-byte spill)
template <int G, bool SELECT_ALL, bool LIST = false>
__global__ void __launch_bounds__(kThreads) edge_bwd_target_kernel(const EdgeBwdArgs a) {
    using S = RowShape<G>;
    constexpr int EPW = S::EPW, V = S::V;
    constexpr int U = Unroll<G>::value;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    bool ok[V];                                                              // slot holds data; ok[s] implies ok[0]
    int c4[V];
#pragma unroll
    for (int s = 0; s < V; ++s) { c4[s] = slot_c4(q, s); ok[s] = c4[s] < a.c; }
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float gscale = a.beta ? 1.0f - __ldg(a.beta) : 1.0f;
    float bpart = 0.f;
    for (int row = blockIdx.x * kWarpsPerBlock + warp; row < a.n; row += gridDim.x * kWarpsPerBlock) {
        const int grow = a.row_offset + row;
        int beg = 0, cnt;
        float invd;
        if (SELECT_ALL) { beg = __ldg(a.rowptr + row); cnt = __ldg(a.rowptr + row + 1) - beg; invd = 1.0f / (float)max(cnt, 1); }
        else {
            cnt = __ldg(a.sel_cnt + row);
            invd = LIST ? __ldg(a.inv_denom + row) : 1.0f / (float)max(__ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row), 1);
        }
        const float iri = __ldg(a.inv_r + grow);
        float4 graw[V], gs[V], ni[V], dni[V];
#pragma unroll
        for (int s = 0; s < V; ++s) {
            graw[s] = ok[s] ? ldg4(a.g + (int64_t)row * a.ldg + c4[s]) : z4;
            gs[s] = scale4(graw[s], invd * gscale);                           // g1_i / deg_i
            ni[s] = ok[s] ? scale4(ldg4(a.h + (int64_t)grow * a.ld + c4[s]), iri) : z4;
        }
        if (a.diff && grp == 0 && ok[0]) {                                   // dL/dbeta
            float b = dot4(ldg4(a.diff + (int64_t)row * a.lddiff + c4[0]), graw[0]);
#pragma unroll
            for (int s = 1; s < V; ++s)
                if (ok[s]) b += dot4(ldg4(a.diff + (int64_t)row * a.lddiff + c4[s]), graw[s]);
            bpart += b;
        }
#pragma unroll
        for (int s = 0; s < V; ++s) dni[s] = z4;
        for (int st = 0; st < cnt; st += EPW * U) {
            float4 v[U][V]; int j[U], qp[U]; float w[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int t = st + u * EPW + grp;
                j[u] = -1; w[u] = 0.f; qp[u] = 0;
                if (t < cnt) {
                    if (SELECT_ALL) { j[u] = __ldg(a.col + beg + t); qp[u] = __ldg(a.tpos + beg + t); }
                    else {
                        const int64_t o = (int64_t)row * a.top_k + t;
                        j[u] = __ldg(a.sel_src + o); w[u] = __ldg(a.sel_w + o); qp[u] = __ldg(a.sel_q + o);
                    }
                }
#pragma unroll
                for (int s = 0; s < V; ++s) v[u][s] = (j[u] >= 0 && ok[s]) ? ldg4(a.h + (int64_t)j[u] * a.ld + c4[s]) : z4;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (st + u * EPW >= cnt) break;                              // warp-uniform
                const float irj = j[u] >= 0 ? __ldg(a.inv_r + j[u]) : 0.f;
                const float ds = group_sum<S::L>(dotv<V>(v[u], gs));         // dL/ds_e
                const float sc = SELECT_ALL ? group_sum<S::L>(dotv<V>(ni, v[u])) * irj + 0.0f : w[u];
                if (j[u] >= 0) {
#pragma unroll
                    for (int s = 0; s < V; ++s) fma4(dni[s], ds * irj, v[u][s]);   // ds_e n_j
                    if (q == 0) a.coef[qp[u]] = make_float2(sc * invd * gscale, ds * iri);
                }
            }
        }
#pragma unroll
        for (int s = 0; s < V; ++s) {
            cross_group_sum4<G>(dni[s]);
            if (grp == 0 && ok[s]) *reinterpret_cast<float4*>(a.dnT + (int64_t)row * a.ld + c4[s]) = dni[s];
        }
    }
    if (a.dbeta_part) {                                                      // fixed-order block sum -> one partial per block
        bpart = group_sum<32>(bpart);
        __shared__ float red[kWarpsPerBlock];
        if (lane == 0) red[warp] = bpart;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int w = 0; w < kWarpsPerBlock; ++w) t += red[w];
            a.dbeta_part[blockIdx.x] = t;
        }
    }
}

template <int G, bool FUSE>
__global__ void __launch_bounds__(kThreads) edge_bwd_source_kernel(const EdgeBwdArgs a) {
    using S = RowShape<G>;
    constexpr int EPW = S::EPW, V = S::V;
    constexpr int U = Unroll<G>::value;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    bool ok[V];                                                              // slot holds data; ok[s] implies ok[0]
    int c4[V];
#pragma unroll
    for (int s = 0; s < V; ++s) { c4[s] = slot_c4(q, s); ok[s] = c4[s] < a.c; }
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float beta = FUSE ? __ldg(a.beta) : 0.f;
    const float* ht = a.h + (int64_t)a.row_offset * a.ld;                  // h rows of the call's targets (col_out: local ids)
    for (int j = blockIdx.x * kWarpsPerBlock + warp; j < a.n_total; j += gridDim.x * kWarpsPerBlock) {
        const int jr = j - a.shift;                                          // rows of the by-source CSR are shifted source ids
        int beg = 0, end = 0;
        if (jr >= 0) { beg = __ldg(a.rowptr_out + jr); end = __ldg(a.rowptr_out + jr + 1); }
        float4 dval[V], dnj[V], dw[V];
#pragma unroll
        for (int s = 0; s < V; ++s) { dval[s] = z4; dnj[s] = z4; dw[s] = z4; }
        for (int base = beg; base < end; base += 32) {
            const int nchunk = min(32, end - base);
            const int il = lane < nchunk ? __ldg(a.col_out + base + lane) : 0;
            const float2 cf = lane < nchunk ? __ldg(a.coef + base + lane) : make_float2(0.f, 0.f);
            for (int st = 0; st < nchunk; st += EPW * U) {
                float4 gv[U][V], hv[U][V]; float ca[U], cb[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int e = st + u * EPW + grp;
                    const int i = __shfl_sync(kFull, il, e & 31);
                    ca[u] = __shfl_sync(kFull, cf.x, e & 31);
                    cb[u] = __shfl_sync(kFull, cf.y, e & 31);
                    const bool on = e < nchunk && ok[0];
                    const bool sel = on && (ca[u] != 0.f || cb[u] != 0.f);   // an unselected edge has both coefficients 0
                    if (!on) { ca[u] = 0.f; cb[u] = 0.f; }
#pragma unroll
                    for (int s = 0; s < V; ++s) {
                        const bool sok = s == 0 || ok[s];
                        gv[u][s] = ((FUSE ? on : sel) && sok) ? ldg4(a.g + (int64_t)i * a.ldg + c4[s]) : z4;
                        hv[u][s] = (sel && sok) ? ldg4(ht + (int64_t)i * a.ld + c4[s]) : z4;
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
#pragma unroll
                    for (int s = 0; s < V; ++s) {
                        fma4(dval[s], ca[u], gv[u][s]);
                        fma4(dnj[s], cb[u], hv[u][s]);
                        if (FUSE) add4(dw[s], gv[u][s]);
                    }
                }
            }
        }
        const float irj = __ldg(a.inv_r + j);
        const bool own = owns_row(a, j);
        float4 nj[V], dn[V];
#pragma unroll
        for (int s = 0; s < V; ++s) {
            cross_group_sum4<G>(dval[s]);
            cross_group_sum4<G>(dnj[s]);
            if (FUSE) cross_group_sum4<G>(dw[s]);
            nj[s] = ok[s] ? scale4(ldg4(a.h + (int64_t)j * a.ld + c4[s]), irj) : z4;
            dn[s] = (own && ok[s]) ? ldg4(a.dnT + (int64_t)(j - a.row_offset) * a.ld + c4[s]) : z4;
            add4(dn[s], dnj[s]);
        }
        const float proj = group_sum<S::L>(dotv<V>(nj, dn));
#pragma unroll
        for (int s = 0; s < V; ++s) {
            if (grp == 0 && ok[s]) {
                float4 o;
                o.x = dval[s].x + (dn[s].x - nj[s].x * proj) * irj; o.y = dval[s].y + (dn[s].y - nj[s].y * proj) * irj;
                o.z = dval[s].z + (dn[s].z - nj[s].z * proj) * irj; o.w = dval[s].w + (dn[s].w - nj[s].w * proj) * irj;
                *reinterpret_cast<float4*>(a.dh + (int64_t)j * a.ld + c4[s]) = o;
                if (FUSE) *reinterpret_cast<float4*>(a.dwt + (int64_t)j * a.lddw + c4[s]) = scale4(dw[s], beta);
            }
        }
    }
}

// ---- staged forms of the two passes (C <= 32, top_k <= 32), same pipeline as edge_fwd_staged_kernel: the rows an item needs
// are copied into the warp's stage with cp.async one item ahead, metadata runs two / three items ahead.
// Pass T, item = target row: stage = its <= top_k selected source rows (lane = edge for ds_e = <h_j, g_i>, lane = channel for
// dn_i = sum ds_e n_j), plus h_i and g_i.
template <int G>
__global__ void __launch_bounds__(kStWarps * 32, kStMinBlocks) edge_bwd_target_staged_kernel(const EdgeBwdArgs a) {
    constexpr int C = 4 * G;
    constexpr int RB = staged_row_bytes<G>();
    constexpr int EPW = 32 / G;
    // a stage holds only what a row can need: min(top_k, 32) selected source rows, then h_i and g_i.  (Sized for 32 rows, the
    // stages cost 9.8 KB per warp at C = 32 and 20 warps fit an SM; at top_k = 10 they cost 3.4 KB and registers set the limit.)
    const uint32_t KS = (uint32_t)min(a.top_k, 32);
    const uint32_t SB = (KS + 2u) * RB;
    const uint32_t HI = KS * RB, GI = HI + RB;  // byte offsets of h_i and g_i inside a stage
    extern __shared__ __align__(128) unsigned char smraw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t sbase = smem_u32(smraw) + (uint32_t)warp * 2u * SB;
    const int q = lane % G, grp = lane / G;
    const bool cq_ok = q * 4 < a.c;
    const int nch = (a.c + 3) >> 2;
    const int ch = lane % C;
    const bool ch_ok = ch < a.c;
    const char* hq = reinterpret_cast<const char*>(a.h + q * 4);
    const int64_t ldhb = (int64_t)a.ld * 4;
    const int egrp = cq_ok ? grp : 64;
    const uint32_t cp_off = (uint32_t)(grp * RB + q * 16), own_off = (uint32_t)(min(lane, (int)KS - 1) * RB), ch_off = (uint32_t)(ch * 4);
    const float gscale = a.beta ? 1.0f - __ldg(a.beta) : 1.0f;
    const int stride = gridDim.x * kStWarps;
    const int row0 = blockIdx.x * kStWarps + warp;
    float bpart = 0.f;

    auto load_meta = [&](int row, int& cnt, float& invd) {                            // invd = 1 / deg_i
        cnt = -1; invd = 1.f;
        if (row < a.n) {
            cnt = __ldg(a.sel_cnt + row);
            invd = a.inv_denom ? __ldg(a.inv_denom + row) : __fdividef(1.0f, (float)max(__ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row), 1));
        }
    };
    auto load_list = [&](int row, int cnt, int& j, float& w, int& qp) {
        j = 0; w = 0.f; qp = 0;
        if (lane < cnt) { const int64_t o = (int64_t)row * a.top_k + lane; j = __ldg(a.sel_src + o); w = __ldg(a.sel_w + o); qp = __ldg(a.sel_q + o); }
    };
    auto issue = [&](uint32_t st0, int row, int cnt, int jl) {
        if (cnt >= 0) {
            const uint32_t dst = st0 + cp_off;
#pragma unroll
            for (int st = 0; st < G; ++st) {
                if (st * EPW < cnt) {                                                    // warp-uniform
                    const int j = __shfl_sync(kFull, jl, st * EPW + grp);
                    if (st * EPW + egrp < cnt) cp_async16(dst + (uint32_t)(st * EPW * RB), reinterpret_cast<const float*>(hq + j * ldhb));
                }
            }
            if (lane < nch) {
                cp_async16(st0 + HI + (uint32_t)lane * 16u, a.h + (int64_t)(a.row_offset + row) * a.ld + lane * 4);
                cp_async16(st0 + GI + (uint32_t)lane * 16u, a.g + (int64_t)row * a.ldg + lane * 4);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    int cntA, cntB, cntC, cntD; float idA, idB, idC, idD;
    load_meta(row0, cntA, idA);
    load_meta(row0 + stride, cntB, idB);
    load_meta(row0 + 2 * stride, cntC, idC);
    int jA, qA, jB, qB; float wA, wB;
    load_list(row0, cntA, jA, wA, qA);
    load_list(row0 + stride, cntB, jB, wB, qB);
    issue(sbase, row0, cntA, jA);
    float irjA = lane < cntA ? __ldg(a.inv_r + jA) : 0.f;
    float iriA = cntA >= 0 ? __ldg(a.inv_r + a.row_offset + row0) : 0.f;
    float dfA = (a.diff && cntA >= 0 && ch_ok) ? __ldg(a.diff + (int64_t)row0 * a.lddiff + ch) : 0.f;
    uint32_t stA = sbase, stB = sbase + SB;
    for (int row = row0; row < a.n; row += stride) {
        load_meta(row + 3 * stride, cntD, idD);
        int jC, qC; float wC;
        load_list(row + 2 * stride, cntC, jC, wC, qC);
        issue(stB, row + stride, cntB, jB);
        const float irjB = lane < cntB ? __ldg(a.inv_r + jB) : 0.f;
        const float iriB = cntB >= 0 ? __ldg(a.inv_r + a.row_offset + row + stride) : 0.f;
        const float dfB = (a.diff && cntB >= 0 && ch_ok) ? __ldg(a.diff + (int64_t)(row + stride) * a.lddiff + ch) : 0.f;
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncwarp();
        {
            const int cnt = cntA;
            const float invd = idA * gscale;                                             // g1_i / deg_i = g_i * invd
            const uint32_t own = stA + own_off, gt = stA + GI;
            float d = 0.f;
#pragma unroll
            for (int i = 0; i < G; ++i) {
                if (i < nch) {
                    const float4 o4 = lds128(own + 16u * i), g4 = lds128(gt + 16u * i);
                    d = fmaf(o4.x, g4.x, fmaf(o4.y, g4.y, fmaf(o4.z, g4.z, fmaf(o4.w, g4.w, d))));
                }
            }
            const float ds = d * invd;                                                   // dL/ds_e (lane = selected edge)
            if (lane < cnt) a.coef[qA] = make_float2(wA * invd, ds * iriA);
            const float wdn = lane < cnt ? ds * irjA : 0.f;                              // ds_e / r_j: dn_i += wdn h_j
            const uint32_t rd = stA + ch_off;
            float dni = 0.f;
#pragma unroll 2
            for (int t = 0; t < cnt; ++t) dni = fmaf(__shfl_sync(kFull, wdn, t), lds32(rd + (uint32_t)(t * RB)), dni);
            if (lane < C && ch_ok) {
                a.dnT[(int64_t)row * a.ld + ch] = dni;
                if (a.diff) bpart = fmaf(dfA, lds32(rd + GI), bpart);                    // dL/dbeta: diff . g (raw g)
            }
        }
        __syncwarp();
        cntA = cntB; idA = idB; jA = jB; wA = wB; qA = qB; irjA = irjB; iriA = iriB; dfA = dfB;
        cntB = cntC; idB = idC; jB = jC; wB = wC; qB = qC;
        cntC = cntD; idC = idD;
        const uint32_t t = stA; stA = stB; stB = t;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    if (a.dbeta_part) {                                                                  // fixed-order block sum -> one partial per block
        bpart = group_sum<32>(bpart);
        __shared__ float red[kStWarps];
        if (lane == 0) red[warp] = bpart;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int w = 0; w < kStWarps; ++w) t += red[w];
            a.dbeta_part[blockIdx.x] = t;
        }
    }
}

// Pass S, item = source row (or a <= 32-edge chunk of one, CHUNK): stage = g_i of its out-edges (all of them under the fused
// epilogue, else only the selected ones) and h_i of the selected ones; the sums are lane = channel.
// Staging is COMPACT: an item takes exactly the row slots it needs (FUSE: deg + nsel, else 2 nsel; on average 26 / 14 of the
// 64 a fixed layout reserves) from the warp's slot pool.  Two items are alive at a time (A = being summed, B = in flight):
// B goes behind A when it fits there, else to the front of the pool when it fits before A, and otherwise waits until A
// is done (that item loses its prefetch, nothing else).  The pool is `slots` rows (launcher: 64 -> 8 KB per warp at C = 32,
// 24+ warps per SM where the fixed two-stage layout allowed 12).
template <int G, bool FUSE, bool CHUNK>
__global__ void __launch_bounds__(kStWarps * 32, kStMinBlocks) edge_bwd_source_staged_kernel(const EdgeBwdArgs a) {
    constexpr int C = 4 * G;
    constexpr int RB = 16 * G;                  // no lane-per-row reads here: no padding needed
    constexpr int EPW = 32 / G;
    extern __shared__ __align__(128) unsigned char smraw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slots = a.slots;
    const uint32_t sbase = smem_u32(smraw) + (uint32_t)(warp * slots * RB);
    const int q = lane % G, grp = lane / G;
    const bool cq_ok = q * 4 < a.c;
    const int ch = lane % C;
    const bool ch_ok = ch < a.c;
    const char* hq = reinterpret_cast<const char*>(a.h + (int64_t)a.row_offset * a.ld + q * 4);   // targets' h rows (local ids)
    const char* gq = reinterpret_cast<const char*>(a.g + q * 4);
    const int64_t ldhb = (int64_t)a.ld * 4, ldgb = (int64_t)a.ldg * 4;
    const int egrp = cq_ok ? grp : 64;
    const uint32_t cp_off = (uint32_t)(q * 16), ch_off = (uint32_t)(ch * 4);
    const unsigned lt_grp = (1u << grp) - 1u;   // edges below this lane's edge inside a copy step
    const float beta = FUSE ? __ldg(a.beta) : 0.f;
    const int stride = gridDim.x * kStWarps;
    const int row0 = blockIdx.x * kStWarps + warp;
    const int n_items = CHUNK ? a.n_chunks : a.n_total;

    auto load_rp = [&](int item, int& beg, int& deg) {
        beg = 0; deg = -1;
        if (item < n_items) {
            if (CHUNK) { const int4 t = __ldg(a.chunk_tab + item); beg = t.x; deg = t.y; }
            else {
                const int jr = item - a.shift;                               // rows of the by-source CSR are shifted source ids
                deg = 0;
                if (jr >= 0) { beg = __ldg(a.rowptr_out + jr); deg = __ldg(a.rowptr_out + jr + 1) - beg; }
            }
        }
    };
    auto load_edges = [&](int beg, int deg, int& il, float2& cf) {
        il = 0; cf = make_float2(0.f, 0.f);
        if ((unsigned)deg <= 32u && lane < deg) { il = __ldg(a.col_out + beg + lane); cf = __ldg(a.coef + beg + lane); }
    };
    auto need_of = [&](int deg, unsigned selm) { return (unsigned)deg <= 32u ? (FUSE ? deg : __popc(selm)) + __popc(selm) : 0; };
    // g rows at slots [0, ng) of the item (FUSE: slot = edge, else slot = rank among the selected), h rows of the selected behind them
    auto issue = [&](uint32_t st0, int deg, int il, unsigned selm) {
        if ((unsigned)deg <= 32u) {
            const uint32_t dst = st0 + cp_off;
            const uint32_t hoff = (uint32_t)((FUSE ? deg : __popc(selm)) * RB);
#pragma unroll
            for (int st = 0; st < G; ++st) {
                if (st * EPW < deg) {                                                    // warp-uniform
                    const int i = __shfl_sync(kFull, il, st * EPW + grp);
                    const int e = st * EPW + egrp;
                    const bool sel = e < 32 && ((selm >> e) & 1u);
                    const uint32_t rk = (uint32_t)(__popc(selm & ((1u << (st * EPW)) - 1u)) + __popc((selm >> (st * EPW)) & lt_grp));   // selected edges before e
                    const uint32_t gs = FUSE ? (uint32_t)(st * EPW + grp) : rk;
                    if (FUSE ? e < deg : sel) cp_async16(dst + gs * RB, reinterpret_cast<const float*>(gq + i * ldgb));
                    if (sel) cp_async16(dst + hoff + rk * RB, reinterpret_cast<const float*>(hq + i * ldhb));
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // where item B may be staged while item A (slots [bA, bA + nA)) is alive: behind A, in front of A, or nowhere (-1)
    auto place = [&](int bA, int nA, int nB) { return bA + nA + nB <= slots ? bA + nA : (nB <= bA ? 0 : -1); };

    int begA, degA, begB, degB, begC, degC, begD, degD;
    load_rp(row0, begA, degA);
    load_rp(row0 + stride, begB, degB);
    load_rp(row0 + 2 * stride, begC, degC);
    int ilA, ilB; float2 cfA, cfB;
    load_edges(begA, degA, ilA, cfA);
    load_edges(begB, degB, ilB, cfB);
    unsigned smA = __ballot_sync(kFull, cfA.x != 0.f || cfA.y != 0.f);                   // an unselected edge has both coefficients 0
    int bA = 0, nA = need_of(degA, smA);
    issue(sbase, degA, ilA, smA);
    // finish operands of row A (non-chunk items): h_j, dnT_j, 1/r_j -- lane = channel, requested one item ahead like the rows
    float hjA = 0.f, dnA = 0.f, irA = 0.f;
    if (!CHUNK && degA >= 0 && degA <= 32) {
        irA = __ldg(a.inv_r + row0);
        if (ch_ok) {
            hjA = __ldg(a.h + (int64_t)row0 * a.ld + ch);
            if (owns_row(a, row0)) dnA = __ldg(a.dnT + (int64_t)(row0 - a.row_offset) * a.ld + ch);
        }
    }
    for (int row = row0; row < n_items; row += stride) {
        load_rp(row + 3 * stride, begD, degD);
        int ilC; float2 cfC;
        load_edges(begC, degC, ilC, cfC);
        const unsigned smB = __ballot_sync(kFull, cfB.x != 0.f || cfB.y != 0.f);
        const int nB = need_of(degB, smB);
        int bB = place(bA, nA, nB);
        const bool ahead = bB >= 0;                                                      // warp-uniform
        if (ahead) issue(sbase + (uint32_t)(bB * RB), degB, ilB, smB);
        float hjB = 0.f, dnB = 0.f, irB = 0.f;
        if (!CHUNK && degB >= 0 && degB <= 32) {
            irB = __ldg(a.inv_r + row + stride);
            if (ch_ok) {
                hjB = __ldg(a.h + (int64_t)(row + stride) * a.ld + ch);
                if (owns_row(a, row + stride)) dnB = __ldg(a.dnT + (int64_t)(row + stride - a.row_offset) * a.ld + ch);
            }
        }
        if (ahead) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        if (degA <= 32) {                                                                // (degA >= 0 here; longer rows go through the chunk pass)
            const uint32_t rd = sbase + (uint32_t)(bA * RB) + ch_off;
            const uint32_t rh = rd + (uint32_t)((FUSE ? degA : __popc(smA)) * RB);
            float dval = 0.f, dnj = 0.f, dw = 0.f;
            if (FUSE) {
                uint32_t hs = rh;
                for (int e = 0; e < degA; ++e) {
                    const float gv = lds32(rd + (uint32_t)(e * RB));
                    dw += gv;
                    if ((smA >> e) & 1u) {                                               // warp-uniform
                        dval = fmaf(__shfl_sync(kFull, cfA.x, e), gv, dval);
                        dnj = fmaf(__shfl_sync(kFull, cfA.y, e), lds32(hs), dnj);
                        hs += RB;
                    }
                }
            } else {
                uint32_t gs = rd, hs = rh;
                for (unsigned m = smA; m; m &= m - 1u) {                                 // selected edges only, ascending position
                    const int e = __ffs(m) - 1;
                    dval = fmaf(__shfl_sync(kFull, cfA.x, e), lds32(gs), dval);
                    dnj = fmaf(__shfl_sync(kFull, cfA.y, e), lds32(hs), dnj);
                    gs += RB; hs += RB;
                }
            }
            if (CHUNK) {
                if (lane < C) {
                    float* o = a.tmp_part + (int64_t)row * 3 * C + ch;
                    o[0] = dval; o[C] = dnj; o[2 * C] = dw;
                }
            } else {
                // dh_j = dval + (dn - n_j (n_j . dn)) / r_j with dn = the target-side part (dnT) + the source-side part
                const float nj = hjA * irA;
                const float dn = dnA + dnj;
                float proj = (lane < C && ch_ok) ? nj * dn : 0.f;
                proj = group_sum<32>(proj);
                if (lane < C && ch_ok) {
                    a.dh[(int64_t)row * a.ld + ch] = dval + (dn - nj * proj) * irA;
                    if (FUSE) a.dwt[(int64_t)row * a.lddw + ch] = dw * beta;
                }
            }
        }
        __syncwarp();                                                                    // A's slots are free from here
        if (!ahead) { bB = 0; issue(sbase, degB, ilB, smB); }                            // B did not fit next to A: staged now, waited for in full next iteration
        begA = begB; degA = degB; ilA = ilB; cfA = cfB; smA = smB; hjA = hjB; dnA = dnB; irA = irB; bA = bB; nA = nB;
        begB = begC; degB = degC; ilB = ilC; cfB = cfC;
        begC = begD; degC = degD;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// ---- narrow rows (C <= 4) of the two passes: lane = edge, rows in registers, cross-lane sums by recursive halving (see
// edge_fwd_narrow_kernel).  Pass T covers every row (a saved list has <= top_k <= 32 entries); pass S the source rows with
// <= 32 out-edges (longer ones go through the staged chunk pass + merge).
__global__ void __launch_bounds__(kThreads) edge_bwd_target_narrow_kernel(const EdgeBwdArgs a) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int stride = gridDim.x * kWarpsPerBlock;
    const int row0 = blockIdx.x * kWarpsPerBlock + warp;
    const float gscale = a.beta ? 1.0f - __ldg(a.beta) : 1.0f;
    const int wc = (lane >> 3) & 3;                                                  // lane_reduce_scatter<4>: lane 8 c holds channel c
    const bool writer = (lane & 7) == 0 && wc < a.c;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float bpart = 0.f;
    struct Gt { float4 hj, hi, gi; float irj, iri, df, gc; };
    auto load_meta = [&](int row, int& cnt, float& invd) {                            // invd = 1 / deg_i
        cnt = -1; invd = 1.f;
        if (row < a.n) {
            cnt = __ldg(a.sel_cnt + row);
            invd = a.inv_denom ? __ldg(a.inv_denom + row) : __fdividef(1.0f, (float)max(__ldg(a.rowptr + row + 1) - __ldg(a.rowptr + row), 1));
        }
    };
    auto load_list = [&](int row, int cnt, int& j, float& w, int& qp) {
        j = -1; w = 0.f; qp = 0;
        if (lane < cnt) { const int64_t o = (int64_t)row * a.top_k + lane; j = __ldg(a.sel_src + o); w = __ldg(a.sel_w + o); qp = __ldg(a.sel_q + o); }
    };
    auto gather = [&](int row, int cnt, int j, Gt& g) {
        g.hj = z4; g.hi = z4; g.gi = z4; g.irj = 0.f; g.iri = 0.f; g.df = 0.f; g.gc = 0.f;
        if (cnt >= 0) {
            g.gi = ldg4(a.g + (int64_t)row * a.ldg);
            g.iri = __ldg(a.inv_r + a.row_offset + row);
            if (j >= 0) { g.hj = ldg4(a.h + (int64_t)j * a.ld); g.irj = __ldg(a.inv_r + j); }
            if (a.diff && writer) { g.df = __ldg(a.diff + (int64_t)row * a.lddiff + wc); g.gc = __ldg(a.g + (int64_t)row * a.ldg + wc); }
        }
    };
    int cntA, cntB, cntC, cntD; float idA, idB, idC, idD;
    load_meta(row0, cntA, idA);
    load_meta(row0 + stride, cntB, idB);
    load_meta(row0 + 2 * stride, cntC, idC);
    int jA, qA, jB, qB; float wA, wB;
    load_list(row0, cntA, jA, wA, qA);
    load_list(row0 + stride, cntB, jB, wB, qB);
    Gt gA, gB;
    gather(row0, cntA, jA, gA);
    for (int row = row0; row < a.n; row += stride) {
        load_meta(row + 3 * stride, cntD, idD);
        int jC, qC; float wC;
        load_list(row + 2 * stride, cntC, jC, wC, qC);
        gather(row + stride, cntB, jB, gB);
        {
            const float invd = idA * gscale;                                             // g1_i / deg_i = g_i * invd
            const float d = fmaf(gA.hj.x, gA.gi.x, fmaf(gA.hj.y, gA.gi.y, fmaf(gA.hj.z, gA.gi.z, fmaf(gA.hj.w, gA.gi.w, 0.f))));
            const float ds = d * invd;                                                   // dL/ds_e (lane = selected edge)
            if (lane < cntA) a.coef[qA] = make_float2(wA * invd, ds * gA.iri);
            const float wdn = lane < cntA ? ds * gA.irj : 0.f;                           // ds_e / r_j: dn_i += wdn h_j
            float v[4] = {wdn * gA.hj.x, wdn * gA.hj.y, wdn * gA.hj.z, wdn * gA.hj.w};
            const float tot = lane_reduce_scatter<4>(v, lane);
            if (writer) {
                a.dnT[(int64_t)row * a.ld + wc] = tot;
                bpart = fmaf(gA.df, gA.gc, bpart);                                       // dL/dbeta: diff . g (raw g); df = 0 without diff
            }
        }
        cntA = cntB; idA = idB; jA = jB; wA = wB; qA = qB; gA = gB;
        cntB = cntC; idB = idC; jB = jC; wB = wC; qB = qC;
        cntC = cntD; idC = idD;
    }
    if (a.dbeta_part) {                                                                  // fixed-order block sum -> one partial per block
        bpart = group_sum<32>(bpart);
        __shared__ float red[kWarpsPerBlock];
        if (lane == 0) red[warp] = bpart;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int w = 0; w < kWarpsPerBlock; ++w) t += red[w];
            a.dbeta_part[blockIdx.x] = t;
        }
    }
}

// (5 blocks per SM: the row-shard operands would otherwise push it to 55-62 registers and 4 blocks; at 48 it does not spill)
template <bool FUSE>
__global__ void __launch_bounds__(kThreads, 5) edge_bwd_source_narrow_kernel(const EdgeBwdArgs a) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int stride = gridDim.x * kWarpsPerBlock;
    const int row0 = blockIdx.x * kWarpsPerBlock + warp;
    const float beta = FUSE ? __ldg(a.beta) : 0.f;
    // after lane_reduce_scatter<8> of (dval, dn_source): lanes with bit 4 clear hold dval[c], lanes with bit 4 set dn_source[c],
    // c = bits 3:2.  The lanes 16 + 4 c finish channel c; after lane_reduce_scatter<4> of dw lane 8 c holds channel c.
    const int fc = (lane >> 2) & 3;
    const bool fin = (lane & 0x13) == 0x10;
    const bool fin_ok = fin && fc < a.c;
    const int wc = (lane >> 3) & 3;
    const bool wwriter = (lane & 7) == 0 && wc < a.c;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* ht = a.h + (int64_t)a.row_offset * a.ld;                  // h rows of the call's targets (col_out: local ids)
    struct Gs { float4 gv, hv; float hj, dn, ir; };
    auto load_rp = [&](int item, int& beg, int& deg) {
        beg = 0; deg = -1;
        if (item < a.n_total) {
            const int jr = item - a.shift;                                   // rows of the by-source CSR are shifted source ids
            deg = 0;
            if (jr >= 0) { beg = __ldg(a.rowptr_out + jr); deg = __ldg(a.rowptr_out + jr + 1) - beg; }
        }
    };
    auto load_edges = [&](int beg, int deg, int& il, float2& cf) {
        il = -1; cf = make_float2(0.f, 0.f);
        if ((unsigned)deg <= 32u && lane < deg) { il = __ldg(a.col_out + beg + lane); cf = __ldg(a.coef + beg + lane); }
    };
    auto gather = [&](int item, int deg, int il, const float2& cf, Gs& g) {
        g.gv = z4; g.hv = z4; g.hj = 0.f; g.dn = 0.f; g.ir = 0.f;
        if ((unsigned)deg <= 32u) {
            const bool sel = cf.x != 0.f || cf.y != 0.f;                     // an unselected edge has both coefficients 0
            if (il >= 0 && (FUSE || sel)) g.gv = ldg4(a.g + (int64_t)il * a.ldg);
            if (sel) g.hv = ldg4(ht + (int64_t)il * a.ld);
            g.ir = __ldg(a.inv_r + item);
            if (fin_ok) {
                g.hj = __ldg(a.h + (int64_t)item * a.ld + fc);
                if (owns_row(a, item)) g.dn = __ldg(a.dnT + (int64_t)(item - a.row_offset) * a.ld + fc);
            }
        }
    };
    int begA, degA, begB, degB, begC, degC, begD, degD;
    load_rp(row0, begA, degA);
    load_rp(row0 + stride, begB, degB);
    load_rp(row0 + 2 * stride, begC, degC);
    int ilA, ilB; float2 cfA, cfB;
    load_edges(begA, degA, ilA, cfA);
    load_edges(begB, degB, ilB, cfB);
    Gs gA, gB;
    gather(row0, degA, ilA, cfA, gA);
    for (int row = row0; row < a.n_total; row += stride) {
        load_rp(row + 3 * stride, begD, degD);
        int ilC; float2 cfC;
        load_edges(begC, degC, ilC, cfC);
        gather(row + stride, degB, ilB, cfB, gB);
        if ((unsigned)degA <= 32u) {
            float v[8] = {cfA.x * gA.gv.x, cfA.x * gA.gv.y, cfA.x * gA.gv.z, cfA.x * gA.gv.w,
                          cfA.y * gA.hv.x, cfA.y * gA.hv.y, cfA.y * gA.hv.z, cfA.y * gA.hv.w};
            const float tot = lane_reduce_scatter<8>(v, lane);
            const float dval = __shfl_xor_sync(kFull, tot, 16);              // for the finishing lanes: dval of their channel
            // dh_j = dval + (dn - n_j (n_j . dn)) / r_j with dn = the target-side part (dnT) + the source-side part
            const float nj = gA.hj * gA.ir;
            const float dn = gA.dn + tot;
            float proj = fin_ok ? nj * dn : 0.f;
            proj += __shfl_xor_sync(kFull, proj, 4);
            proj += __shfl_xor_sync(kFull, proj, 8);
            if (fin_ok) a.dh[(int64_t)row * a.ld + fc] = dval + (dn - nj * proj) * gA.ir;
            if (FUSE) {
                float u[4] = {gA.gv.x, gA.gv.y, gA.gv.z, gA.gv.w};
                const float dw = lane_reduce_scatter<4>(u, lane);
                if (wwriter) a.dwt[(int64_t)row * a.lddw + wc] = dw * beta;
            }
        }
        begA = begB; degA = degB; ilA = ilB; cfA = cfB; gA = gB;
        begB = begC; degB = degC; ilB = ilC; cfB = cfC;
        begC = begD; degC = degD;
    }
}

// long source rows: sum of the chunk partials + the same finish (warp per row, lane = channel)
template <int G, bool FUSE>
__global__ void __launch_bounds__(kThreads) edge_bwd_source_merge_kernel(const EdgeBwdArgs a) {
    constexpr int C = 4 * G;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ch = lane % C;
    const bool ch_ok = ch < a.c;
    const float beta = FUSE ? __ldg(a.beta) : 0.f;
    for (int li = blockIdx.x * kWarpsPerBlock + warp; li < a.n_lrows; li += gridDim.x * kWarpsPerBlock) {
        const int row = __ldg(a.lrows + li);                                 // true source id
        const int c0 = __ldg(a.lrow_ptr + li), c1 = __ldg(a.lrow_ptr + li + 1);
        float dval = 0.f, dnj = 0.f, dw = 0.f;
#pragma unroll 4
        for (int ci = c0; ci < c1; ++ci) {
            const float* o = a.tmp_part + (int64_t)ci * 3 * C + ch;
            dval += __ldg(o); dnj += __ldg(o + C);
            if (FUSE) dw += __ldg(o + 2 * C);
        }
        const float ir = __ldg(a.inv_r + row);
        const float nj = ch_ok ? __ldg(a.h + (int64_t)row * a.ld + ch) * ir : 0.f;
        const float dn = (ch_ok && owns_row(a, row) ? __ldg(a.dnT + (int64_t)(row - a.row_offset) * a.ld + ch) : 0.f) + dnj;
        float proj = (lane < C && ch_ok) ? nj * dn : 0.f;
        proj = group_sum<32>(proj);
        if (lane < C && ch_ok) {
            a.dh[(int64_t)row * a.ld + ch] = dval + (dn - nj * proj) * ir;
            if (FUSE) a.dwt[(int64_t)row * a.lddw + ch] = dw * beta;
        }
    }
}

// fixed-order sum of per-block partials (deterministic replacement of a float atomicAdd)
__global__ void __launch_bounds__(256) sum_partials_kernel(const float* __restrict__ part, int n, float* __restrict__ out) {
    __shared__ float red[256];
    float t = 0.f;
    for (int i = threadIdx.x; i < n; i += 256) t += part[i];
    red[threadIdx.x] = t;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = red[0];
}

// ------------------------------------------------------------------------------------------ K3 / K4
// acc[s] = sum over the row's edges of val[e] x[col[e]], slot s of the lane (c4[s] = its first channel, ok[s] = it holds data)
template <int G>
__device__ __forceinline__ void gather_sum(const float* __restrict__ x, int64_t ldx, const int* __restrict__ col,
                                           const float* __restrict__ val, int beg, int end, const int (&c4)[RowShape<G>::V],
                                           const bool (&ok)[RowShape<G>::V], int grp, int lane, float4 (&acc)[RowShape<G>::V]) {
    using S = RowShape<G>;
    constexpr int EPW = S::EPW, V = S::V;
    constexpr int U = Unroll<G>::value;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int s = 0; s < V; ++s) acc[s] = z4;
    for (int base = beg; base < end; base += 32) {
        const int nchunk = min(32, end - base);
        const int jl = lane < nchunk ? __ldg(col + base + lane) : -1;
        const float wl = (val && lane < nchunk) ? __ldg(val + base + lane) : 1.f;
        for (int st = 0; st < nchunk; st += EPW * U) {
            float4 v[U][V]; float w[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = st + u * EPW + grp;
                int j = __shfl_sync(0xffffffffu, jl, e & 31);
                w[u] = __shfl_sync(0xffffffffu, wl, e & 31);
                if (e >= nchunk) j = -1;
#pragma unroll
                for (int s = 0; s < V; ++s) v[u][s] = (j >= 0 && ok[s]) ? ldg4(x + (int64_t)j * ldx + c4[s]) : z4;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
#pragma unroll
                for (int s = 0; s < V; ++s) fma4(acc[s], w[u], v[u][s]);
            }
        }
    }
#pragma unroll
    for (int s = 0; s < V; ++s) {
        acc[s].x = cross_group_sum<G>(acc[s].x); acc[s].y = cross_group_sum<G>(acc[s].y);
        acc[s].z = cross_group_sum<G>(acc[s].z); acc[s].w = cross_group_sum<G>(acc[s].w);
    }
}

template <int G>
__global__ void __launch_bounds__(kThreads) spmm_fwd_kernel(const float* __restrict__ x, int n_rows, int c, int64_t ldx,
                                                           const int* __restrict__ rowptr, const int* __restrict__ col,
                                                           const float* __restrict__ val, const float* __restrict__ rowscale,
                                                           const float* __restrict__ bias, float* __restrict__ out, int64_t ldo) {
    using S = RowShape<G>;
    constexpr int V = S::V;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    int c4[V];
    bool ok[V];
#pragma unroll
    for (int s = 0; s < V; ++s) { c4[s] = slot_c4(q, s); ok[s] = c4[s] < c; }
    for (int row = blockIdx.x * kWarpsPerBlock + warp; row < n_rows; row += gridDim.x * kWarpsPerBlock) {
        const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
        float4 acc[V];
        gather_sum<G>(x, ldx, col, val, beg, end, c4, ok, grp, lane, acc);
#pragma unroll
        for (int s = 0; s < V; ++s) {
            if (grp == 0 && ok[s]) {
                if (rowscale) acc[s] = scale4(acc[s], __ldg(rowscale + row));
                if (bias) { const float4 b = ldg4(bias + c4[s]); acc[s].x += b.x; acc[s].y += b.y; acc[s].z += b.z; acc[s].w += b.w; }
                *reinterpret_cast<float4*>(out + (int64_t)row * ldo + c4[s]) = acc[s];
            }
        }
    }
}

template <int G>
__global__ void __launch_bounds__(kThreads) pp_fuse_fwd_kernel(const float* __restrict__ wt, int n, int c, int64_t ld,
                                                              const int* __restrict__ rowptr, const int* __restrict__ col,
                                                              const float* __restrict__ b_w, const float* __restrict__ beta_p,
                                                              const float* __restrict__ out1, const float* __restrict__ bias,
                                                              float* __restrict__ out0, float* __restrict__ out) {
    using S = RowShape<G>;
    constexpr int V = S::V;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = lane % S::L, grp = lane / S::L;
    int c4[V];
    bool ok[V];
#pragma unroll
    for (int s = 0; s < V; ++s) { c4[s] = slot_c4(q, s); ok[s] = c4[s] < c; }
    const float beta = __ldg(beta_p);
    for (int row = blockIdx.x * kWarpsPerBlock + warp; row < n; row += gridDim.x * kWarpsPerBlock) {
        const int beg = __ldg(rowptr + row), end = __ldg(rowptr + row + 1);
        float4 acc[V];
        gather_sum<G>(wt, ld, col, nullptr, beg, end, c4, ok, grp, lane, acc);
#pragma unroll
        for (int s = 0; s < V; ++s) {
            if (grp == 0 && ok[s]) {
                float4 a = acc[s];
                const float4 b = ldg4(b_w + c4[s]);
                a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
                const int64_t o = (int64_t)row * ld + c4[s];
                *reinterpret_cast<float4*>(out0 + o) = a;
                const float4 o1 = ldg4(out1 + o);
                float4 r;
                r.x = beta * a.x + (1.f - beta) * o1.x; r.y = beta * a.y + (1.f - beta) * o1.y;
                r.z = beta * a.z + (1.f - beta) * o1.z; r.w = beta * a.w + (1.f - beta) * o1.w;
                if (bias) { const float4 bb = ldg4(bias + c4[s]); r.x += bb.x; r.y += bb.y; r.z += bb.z; r.w += bb.w; }
                *reinterpret_cast<float4*>(out + o) = r;
            }
        }
    }
}

__global__ void __launch_bounds__(256) pp_beta_grad_kernel(const float* __restrict__ out0, const float* __restrict__ out1,
                                                          const float* __restrict__ g, int64_t numel, float* __restrict__ part) {
    float acc = 0.f;
    const int64_t n4 = numel / 4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 a = ldg4(out0 + 4 * i), b = ldg4(out1 + 4 * i), gg = ldg4(g + 4 * i);
        acc = fmaf(a.x - b.x, gg.x, fmaf(a.y - b.y, gg.y, fmaf(a.z - b.z, gg.z, fmaf(a.w - b.w, gg.w, acc))));
    }
    acc = group_sum<32>(acc);
    __shared__ float red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {                                  // fixed order: one partial per block, summed by sum_partials_kernel
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        part[blockIdx.x] = t;
    }
}

// ------------------------------------------------------------------------------------------ loss
// Mean negative log-likelihood over the rows whose label is >= 0 (R: train.py:81 `F.nll_loss(out[mask], y[mask])` -- a masked
// row is a label of -1 here), forward and backward, with fixed-order reductions.  torch's nll_loss spends 1.5 + 0.9 ms on
// the 1.6 M rows of the pokec shape (one CTA walks them); this is one streaming pass each way.
__global__ void __launch_bounds__(256) nll_loss_fwd_kernel(const float* __restrict__ logp, int64_t n, int c, int64_t ld, const int64_t* __restrict__ y,
                                                          float* __restrict__ part_sum, float* __restrict__ part_cnt) {
    float acc = 0.f, cnt = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = __ldg(y + i);
        if (t >= 0 && t < c) { acc -= __ldg(logp + i * ld + t); cnt += 1.f; }
    }
    acc = group_sum<32>(acc); cnt = group_sum<32>(cnt);
    __shared__ float ra[8], rc[8];
    if ((threadIdx.x & 31) == 0) { ra[threadIdx.x >> 5] = acc; rc[threadIdx.x >> 5] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, b = 0.f;
        for (int w = 0; w < 8; ++w) { a += ra[w]; b += rc[w]; }
        part_sum[blockIdx.x] = a; part_cnt[blockIdx.x] = b;
    }
}

__global__ void __launch_bounds__(256) nll_loss_finish_kernel(const float* __restrict__ part_sum, const float* __restrict__ part_cnt, int n,
                                                             float* __restrict__ loss, float* __restrict__ count) {
    __shared__ float ra[256], rc[256];
    float a = 0.f, b = 0.f;
    for (int i = threadIdx.x; i < n; i += 256) { a += part_sum[i]; b += part_cnt[i]; }
    ra[threadIdx.x] = a; rc[threadIdx.x] = b;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { ra[threadIdx.x] += ra[threadIdx.x + o]; rc[threadIdx.x] += rc[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { *count = rc[0]; *loss = rc[0] > 0.f ? ra[0] / rc[0] : 0.f; }
}

// dlogp[i, t] = -gscale / count for t = y[i], 0 elsewhere (the whole [n, c] gradient is written: no memset needed)
__global__ void __launch_bounds__(256) nll_loss_bwd_kernel(int64_t n, int c, int64_t ld, const int64_t* __restrict__ y, const float* __restrict__ gscale,
                                                          const float* __restrict__ count, float* __restrict__ dlogp) {
    const float cntv = __ldg(count);
    const float g = cntv > 0.f ? -__ldg(gscale) / cntv : 0.f;
    const int64_t total = n * (int64_t)c;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = e / c;
        const int t = (int)(e - i * c);
        dlogp[i * ld + t] = (__ldg(y + i) == t) ? g : 0.f;
    }
}

// ------------------------------------------------------------------------------------------ SDDMM
__global__ void __launch_bounds__(kThreads) sddmm_dot_kernel(const float* __restrict__ xh, int d, int64_t ld,
                                                            const int* __restrict__ a, const int* __restrict__ b,
                                                            int64_t ne, float* __restrict__ s) {
    const int lane = threadIdx.x & 31;
    int64_t e = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const bool vec = (ld % 4 == 0) && (d % 4 == 0);
    for (; e < ne; e += (int64_t)gridDim.x * kWarpsPerBlock) {
        const float* pa = xh + (int64_t)__ldg(a + e) * ld;
        const float* pb = xh + (int64_t)__ldg(b + e) * ld;
        float acc = 0.f;
        if (vec) for (int k = lane * 4; k < d; k += 128) acc += dot4(ldg4(pa + k), ldg4(pb + k));
        else for (int k = lane; k < d; k += 32) acc = fmaf(__ldg(pa + k), __ldg(pb + k), acc);
        acc = group_sum<32>(acc);
        if (lane == 0) s[e] = acc;
    }
}

#define SNG_DISPATCH_G(cexpr, ...)                                              \
    switch (group_lanes(cexpr)) {                                               \
        case 1: { constexpr int G = 1; __VA_ARGS__; } break;                    \
        case 2: { constexpr int G = 2; __VA_ARGS__; } break;                    \
        case 4: { constexpr int G = 4; __VA_ARGS__; } break;                    \
        case 8: { constexpr int G = 8; __VA_ARGS__; } break;                    \
        case 16: { constexpr int G = 16; __VA_ARGS__; } break;                  \
        case 32: { constexpr int G = 32; __VA_ARGS__; } break;                  \
        case 64: { constexpr int G = 64; __VA_ARGS__; } break;                  \
        case 128: { constexpr int G = 128; __VA_ARGS__; } break;                \
        default: set_error("c=%lld: no edge kernel for this width", (long long)(cexpr)); return SNG_ERR_UNSUPPORTED; \
    }
static_assert(SNG_MAX_CHANNELS == 4 * 128, "SNG_DISPATCH_G instantiates the edge kernels up to G = 128 float4 slots per row");

static int check_rows(const char* fn, int64_t n, int64_t c, int64_t ld) {
    if (n < 0 || n >= (1ll << 31)) { set_error("%s: n=%lld out of range", fn, (long long)n); return SNG_ERR_ARG; }
    if (c <= 0 || c % 4 != 0 || ld % 4 != 0 || ld < c) { set_error("%s: c=%lld ld=%lld must be multiples of 4, ld>=c", fn, (long long)c, (long long)ld); return SNG_ERR_ARG; }
    if (c > SNG_MAX_CHANNELS) {
        set_error("%s: c=%lld > %d channels (SNG_MAX_CHANNELS) not supported by the edge kernels", fn, (long long)c, SNG_MAX_CHANNELS);
        return SNG_ERR_UNSUPPORTED;
    }
    return SNG_OK;
}

}  // namespace sng

using namespace sng;

extern "C" int sng_rownorm_f32(const float* x, int64_t n, int64_t d, int64_t ldx, float* xhat_f32, int64_t ld_f32,
                               uint16_t* xhat_f16, int64_t ld_f16, float* inv_norm, void* stream) {
    SNG_REQUIRE(x && n >= 0 && d > 0 && ldx >= d && d < (1ll << 30), "sng_rownorm_f32: bad x/n/d/ldx");
    SNG_REQUIRE(!xhat_f32 || (ld_f32 >= d && ld_f32 < (1ll << 30)), "sng_rownorm_f32: ld_f32 < d");
    SNG_REQUIRE(!xhat_f16 || (ld_f16 >= d && ld_f16 < (1ll << 30)), "sng_rownorm_f32: ld_f16 < d");
    if (n == 0) return SNG_OK;
    rownorm_kernel<<<grid_resident(rownorm_kernel, n, kWarpsPerBlock), kThreads, 0, (cudaStream_t)stream>>>(
        x, n, (int)d, ldx, xhat_f32, (int)ld_f32, reinterpret_cast<__half*>(xhat_f16), (int)ld_f16, inv_norm);
    return check_launch("sng_rownorm_f32");
}

namespace sng {
// dynamic shared memory of the long-row / hub kernels (see their carve-up)
static size_t long_smem(int top_k) { return (size_t)kWarpsPerBlock * 2 * (top_k > 0 ? top_k : 1) * sizeof(float); }
// (the partial sums take 128 V channels per warp: 8 KB for C <= 128, 32 KB at C = 512, inside the 48 KB default)
template <int G>
static size_t hub_smem(int top_k) {
    const size_t k1 = top_k > 0 ? top_k : 1;
    return ((size_t)kWarpsPerBlock * 2 * k1 + 2 * k1 + kWarpsPerBlock + (size_t)kWarpsPerBlock * 2 * 128 * RowShape<G>::V) * sizeof(float);
}

// row slots per warp of the staged forward kernel (see there); any single item (33 / fused 65 slots) must fit
static int forward_slots(bool fuse) {
    return fuse ? 66 : 40;                  // measured (pokec shape, C = 32): smaller pools win -- occupancy beats prefetch depth
}
template <int G, bool FUSE, bool SELECT_ALL, bool DSEL>
static void launch_edge_fwd(EdgeFwdArgs a, const int32_t* rows_hub, int64_t n_hub, cudaStream_t st) {
    const size_t ls = long_smem(a.top_k), hs = hub_smem<G>(a.top_k);
    if constexpr (G <= 8) {
        if (a.n_chunks >= 0) {
            // degree lists known, rows of <= 128 bytes: staged kernel over the short rows, then over the <= 32-edge chunks of the
            // long rows, then the per-row merge of the chunk candidates
            a.slots = forward_slots(FUSE);
            const size_t ss = (size_t)kStWarps * a.slots * staged_row_bytes<G>();
            if constexpr (G == 1) {
                // 16-byte rows: everything in registers (edge_fwd_narrow_kernel); the chunk pass of the long rows stays staged
                edge_fwd_narrow_kernel<FUSE, SELECT_ALL, DSEL><<<grid_resident(edge_fwd_narrow_kernel<FUSE, SELECT_ALL, DSEL>, a.n, kWarpsPerBlock), kThreads, 0, st>>>(a);
            } else {
                cudaFuncSetAttribute(edge_fwd_staged_kernel<G, FUSE, SELECT_ALL, false, DSEL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss);
                edge_fwd_staged_kernel<G, FUSE, SELECT_ALL, false, DSEL><<<grid_resident(edge_fwd_staged_kernel<G, FUSE, SELECT_ALL, false, DSEL>, a.n, kStWarps, ss, kStWarps * 32), kStWarps * 32, ss, st>>>(a);
            }
            if (a.n_chunks > 0) {
                cudaFuncSetAttribute(edge_fwd_staged_kernel<G, FUSE, SELECT_ALL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss);
                edge_fwd_staged_kernel<G, FUSE, SELECT_ALL, true><<<grid_resident(edge_fwd_staged_kernel<G, FUSE, SELECT_ALL, true>, a.n_chunks, kStWarps, ss, kStWarps * 32), kStWarps * 32, ss, st>>>(a);
                edge_fwd_merge_kernel<G, FUSE, SELECT_ALL, DSEL><<<grid_resident(edge_fwd_merge_kernel<G, FUSE, SELECT_ALL, DSEL>, a.n_lrows, kWarpsPerBlock, ls), kThreads, ls, st>>>(a);
            }
            return;
        }
    }
    // wide rows (C > 32) or no degree lists: the chunked kernel runs every row; listed hubs still get their block kernel
    a.rows = nullptr; a.n_rows = 0;
    a.skip_deg = n_hub > 0 ? 1024 : 0;
    edge_fwd_long_kernel<G, FUSE, SELECT_ALL, DSEL><<<grid_resident(edge_fwd_long_kernel<G, FUSE, SELECT_ALL, DSEL>, a.n, kWarpsPerBlock, ls), kThreads, ls, st>>>(a);
    if (a.skip_deg) {
        a.rows = rows_hub; a.n_rows = (int)n_hub; a.skip_deg = 0;
        edge_fwd_hub_kernel<G, FUSE, SELECT_ALL, DSEL><<<grid_capped(n_hub, 1, 4), kThreads, hs, st>>>(a);
    }
}
}  // namespace sng

extern "C" size_t sng_edge_fwd_workspace_bytes(int64_t n_chunks, int64_t c, int top_k) {
    if (n_chunks <= 0 || c <= 0 || c > 32) return 0;
    const int64_t kk = top_k > 0 ? (top_k < 32 ? top_k : 32) : 0, cg = 4 * group_lanes(c);
    return (size_t)n_chunks * (size_t)(2 * kk + 1 + 2 * cg) * 4 + 1024;
}

extern "C" int sng_edge_fwd_denom(const float* h, int64_t n_total, int64_t n, int64_t row_offset, int64_t c, int64_t ldh,
                                  const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                                  const int32_t* chunk_tab, int64_t n_chunks, const int32_t* lrows, const int32_t* lrow_ptr, int64_t n_lrows,
                                  const int32_t* rows_hub, int64_t n_hub, void* workspace, size_t workspace_bytes,
                                  int top_k, float thr, float* out, int64_t ldo,
                                  int32_t* sel_src, float* sel_w, int32_t* sel_q, int32_t* sel_cnt, float* inv_norm, int inv_norm_ready,
                                  const float* wt, int64_t ldw, const float* b_w, const float* beta, const float* bias, float* diff,
                                  int denominator, float* inv_denom, void* stream) {
    if (int rc = check_rows("sng_edge_fwd", n, c, ldh)) return rc;
    SNG_REQUIRE(denominator == 0 || (denominator == 1 && top_k > 0), "sng_edge_fwd: denominator=%d must be 0 (candidates) or 1 (selected, needs top_k > 0)", denominator);
    SNG_REQUIRE(!inv_denom || denominator == 1, "sng_edge_fwd: inv_denom is an output of denominator=1 (selected)");
    SNG_REQUIRE(h && rowptr && ((col && out) || n == 0) && ldo % 4 == 0 && ldo >= c, "sng_edge_fwd: null pointer or bad ldo");   // (an empty shard has no edges, no rows)
    SNG_REQUIRE(row_offset >= 0 && row_offset + n <= n_total && n_total < (1ll << 31) && ldh < (1ll << 31) && ldo < (1ll << 31),
                "sng_edge_fwd: bad row_offset / n_total");
    SNG_REQUIRE(inv_norm, "sng_edge_fwd: inv_norm [n_total] is required");
    SNG_REQUIRE(top_k <= SNG_MAX_TOPK, "sng_edge_fwd: top_k=%d > %d", top_k, SNG_MAX_TOPK);
    SNG_REQUIRE(top_k <= 0 || thr > -1.1f, "sng_edge_fwd: thr must be > -1.1 (knock-out sentinel of R models.py:153)");
    SNG_REQUIRE(!sel_cnt || (top_k > 0 && sel_src && sel_w), "sng_edge_fwd: sel_src / sel_w / sel_cnt go together and need top_k > 0");
    SNG_REQUIRE(!sel_q || (sel_cnt && tpos), "sng_edge_fwd: sel_q needs sel_cnt and tpos");
    SNG_REQUIRE(n_chunks <= 0 || (chunk_tab && lrows && lrow_ptr && n_lrows > 0 && n_chunks < (1ll << 31)), "sng_edge_fwd: chunk tables missing");
    SNG_REQUIRE(n_hub >= 0 && (n_hub == 0 || rows_hub), "sng_edge_fwd: hub list missing");
    SNG_REQUIRE(!wt || (b_w && beta && ldw % 4 == 0 && ldw >= c && ldw < (1ll << 31)), "sng_edge_fwd: fused epilogue needs b_w, beta and a 16-byte aligned wt");
    SNG_REQUIRE(wt || !diff, "sng_edge_fwd: diff is an output of the fused epilogue");
    if (n == 0 && (inv_norm_ready || n_total == 0)) return SNG_OK;     // (an empty row shard still fills inv_norm: the backward reads it)
    const bool staged = c <= 32 && n_chunks >= 0;
    if (staged && n_chunks > 0) {
        if (!workspace || workspace_bytes < sng_edge_fwd_workspace_bytes(n_chunks, c, top_k)) { set_error("sng_edge_fwd: workspace too small"); return SNG_ERR_WORKSPACE; }
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (!inv_norm_ready)                                     // (sng_lin_norm_fwd already produced it with h)
        SNG_DISPATCH_G(c, row_inv_norm_kernel<G><<<grid_resident(row_inv_norm_kernel<G>, n_total, kWarpsPerBlock * RowShape<G>::EPW * 4), kThreads, 0, st>>>(h, n_total, (int)c, ldh, inv_norm));
    if (n == 0) return check_launch("sng_edge_fwd");
    EdgeFwdArgs a;
    a.h = h; a.inv_r = inv_norm; a.n = (int)n; a.row_offset = (int)row_offset; a.c = (int)c; a.ldh = (int)ldh;
    a.rowptr = rowptr; a.col = col; a.tpos = tpos; a.rows = nullptr; a.n_rows = 0; a.skip_deg = 0;
    a.top_k = top_k > 0 ? top_k : 0; a.thr = thr; a.out = out; a.ldo = (int)ldo;
    a.inv_denom = inv_denom;
    a.sel_src = sel_src; a.sel_w = sel_w; a.sel_q = sel_q; a.sel_cnt = sel_cnt;
    a.wt = wt; a.ldw = (int)ldw; a.b_w = b_w; a.beta = beta; a.bias = bias; a.diff = diff;
    a.chunk_tab = reinterpret_cast<const int4*>(chunk_tab); a.n_chunks = staged ? (int)n_chunks : -1;
    a.lrows = lrows; a.lrow_ptr = lrow_ptr; a.n_lrows = (int)n_lrows;
    a.tmp_s = nullptr; a.tmp_p = nullptr; a.tmp_cnt = nullptr; a.tmp_acc = nullptr; a.tmp_a0 = nullptr;
    if (staged && n_chunks > 0) {
        const int64_t kk = a.top_k < 32 ? a.top_k : 32, cg = 4 * group_lanes(c);
        float* w = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
        a.tmp_s = w; w += n_chunks * kk;
        a.tmp_p = reinterpret_cast<int*>(w); w += n_chunks * kk;
        a.tmp_cnt = reinterpret_cast<int*>(w); w += n_chunks;
        a.tmp_acc = w; w += n_chunks * cg;
        a.tmp_a0 = w;
    }
    SNG_DISPATCH_G(c,
        if (wt) { if (top_k <= 0) launch_edge_fwd<G, true, true, false>(a, rows_hub, n_hub, st);
                  else if (denominator) launch_edge_fwd<G, true, false, true>(a, rows_hub, n_hub, st);
                  else launch_edge_fwd<G, true, false, false>(a, rows_hub, n_hub, st); }
        else { if (top_k <= 0) launch_edge_fwd<G, false, true, false>(a, rows_hub, n_hub, st);
               else if (denominator) launch_edge_fwd<G, false, false, true>(a, rows_hub, n_hub, st);
               else launch_edge_fwd<G, false, false, false>(a, rows_hub, n_hub, st); });
    return check_launch("sng_edge_fwd");
}

extern "C" int sng_edge_fwd(const float* h, int64_t n_total, int64_t n, int64_t row_offset, int64_t c, int64_t ldh,
                            const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                            const int32_t* chunk_tab, int64_t n_chunks, const int32_t* lrows, const int32_t* lrow_ptr, int64_t n_lrows,
                            const int32_t* rows_hub, int64_t n_hub, void* workspace, size_t workspace_bytes,
                            int top_k, float thr, float* out, int64_t ldo,
                            int32_t* sel_src, float* sel_w, int32_t* sel_q, int32_t* sel_cnt, float* inv_norm, int inv_norm_ready,
                            const float* wt, int64_t ldw, const float* b_w, const float* beta, const float* bias, float* diff,
                            void* stream) {
    return sng_edge_fwd_denom(h, n_total, n, row_offset, c, ldh, rowptr, col, tpos, chunk_tab, n_chunks, lrows, lrow_ptr, n_lrows,
                              rows_hub, n_hub, workspace, workspace_bytes, top_k, thr, out, ldo, sel_src, sel_w, sel_q, sel_cnt,
                              inv_norm, inv_norm_ready, wt, ldw, b_w, beta, bias, diff, 0, nullptr, stream);
}

namespace sng {
// row slots per warp of the staged source pass (see edge_bwd_source_staged_kernel); >= 64 so that any single item fits
constexpr int kSourceSlots = 64;            // measured (pokec shape, C = 32): 64 / 72 equal, 80+ slower in both modes (occupancy)
template <int G>
static int launch_bwd_target_staged(const EdgeBwdArgs& a, cudaStream_t st) {
    const size_t ss = (size_t)kStWarps * 2 * (size_t)((a.top_k < 32 ? a.top_k : 32) + 2) * staged_row_bytes<G>();
    cudaFuncSetAttribute(edge_bwd_target_staged_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss);
    const int grid = grid_resident(edge_bwd_target_staged_kernel<G>, a.n, kStWarps, ss, kStWarps * 32);
    edge_bwd_target_staged_kernel<G><<<grid, kStWarps * 32, ss, st>>>(a);
    return grid;
}
template <int G, bool FUSE>
static void launch_bwd_source_staged(EdgeBwdArgs a, cudaStream_t st) {
    a.slots = kSourceSlots;
    const size_t ss = (size_t)kStWarps * a.slots * 16 * G;
    if constexpr (G == 1) {
        edge_bwd_source_narrow_kernel<FUSE><<<grid_resident(edge_bwd_source_narrow_kernel<FUSE>, a.n_total, kWarpsPerBlock), kThreads, 0, st>>>(a);
    } else {
        cudaFuncSetAttribute(edge_bwd_source_staged_kernel<G, FUSE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss);
        edge_bwd_source_staged_kernel<G, FUSE, false><<<grid_resident(edge_bwd_source_staged_kernel<G, FUSE, false>, a.n_total, kStWarps, ss, kStWarps * 32), kStWarps * 32, ss, st>>>(a);
    }
    if (a.n_chunks > 0) {
        cudaFuncSetAttribute(edge_bwd_source_staged_kernel<G, FUSE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ss);
        edge_bwd_source_staged_kernel<G, FUSE, true><<<grid_resident(edge_bwd_source_staged_kernel<G, FUSE, true>, a.n_chunks, kStWarps, ss, kStWarps * 32), kStWarps * 32, ss, st>>>(a);
        edge_bwd_source_merge_kernel<G, FUSE><<<grid_resident(edge_bwd_source_merge_kernel<G, FUSE>, a.n_lrows, kWarpsPerBlock), kThreads, 0, st>>>(a);
    }
}

// launch body of sng_edge_bwd and sng_list_bwd: pass T (by target), pass S (by source), then the fixed-order dbeta sum
static int launch_edge_bwd(const EdgeBwdArgs& a, float* dbeta, cudaStream_t st, const char* fn) {
    const int c = a.c, top_k = a.top_k, n = a.n, n_total = a.n_total;
    const bool fuse = a.dwt != nullptr;
    // n == 0 (an empty shard) still runs both passes: pass T writes no row but its one block writes a zero dbeta partial,
    // pass S writes the zero contribution of every row
    const bool staged_t = c <= 32 && top_k > 0 && top_k <= 32;      // pass T from the saved lists, rows staged in shared memory
    const bool staged_s = c <= 32 && a.n_chunks >= 0;               // pass S with the by-source chunk tables
    int grid_t = 1;
    SNG_DISPATCH_G(c,
        if constexpr (G == 1) {
            if (staged_t) {
                grid_t = grid_resident(edge_bwd_target_narrow_kernel, n, kWarpsPerBlock);
                edge_bwd_target_narrow_kernel<<<grid_t, kThreads, 0, st>>>(a);
            }
        } else if constexpr (G <= 8) {
            if (staged_t) grid_t = launch_bwd_target_staged<G>(a, st);
        }
        if (!staged_t || G > 8) {
            if (a.inv_denom) { grid_t = grid_resident(edge_bwd_target_kernel<G, false, true>, n, kWarpsPerBlock); edge_bwd_target_kernel<G, false, true><<<grid_t, kThreads, 0, st>>>(a); }
            else if (top_k > 0) { grid_t = grid_resident(edge_bwd_target_kernel<G, false>, n, kWarpsPerBlock); edge_bwd_target_kernel<G, false><<<grid_t, kThreads, 0, st>>>(a); }
            else { grid_t = grid_resident(edge_bwd_target_kernel<G, true>, n, kWarpsPerBlock); edge_bwd_target_kernel<G, true><<<grid_t, kThreads, 0, st>>>(a); }
        }
        bool done_s = false;
        if constexpr (G <= 8) {
            if (staged_s) { if (fuse) launch_bwd_source_staged<G, true>(a, st); else launch_bwd_source_staged<G, false>(a, st); done_s = true; }
        }
        if (!done_s) {
            if (fuse) edge_bwd_source_kernel<G, true><<<grid_resident(edge_bwd_source_kernel<G, true>, n_total, kWarpsPerBlock), kThreads, 0, st>>>(a);
            else edge_bwd_source_kernel<G, false><<<grid_resident(edge_bwd_source_kernel<G, false>, n_total, kWarpsPerBlock), kThreads, 0, st>>>(a);
        });
    if (dbeta) sum_partials_kernel<<<1, 256, 0, st>>>(a.dbeta_part, grid_t, dbeta);
    return check_launch(fn);
}
}  // namespace sng

extern "C" int sng_edge_bwd_denom(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                                  int64_t c, int64_t ld, int64_t ldg,
                                  const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                                  const int32_t* rowptr_out, const int32_t* col_out, int64_t src_shift, int64_t num_edges,
                                  int top_k, const int32_t* sel_src, const float* sel_w, const int32_t* sel_q, const int32_t* sel_cnt,
                                  const float* beta, const float* diff, int64_t lddiff, float* dbeta,
                                  float* coef, float* dn_target, float* partials, float* dh, float* dwt, int64_t lddw,
                                  const int32_t* chunk_tab_out, int64_t n_chunks_out, const int32_t* lrows_out, const int32_t* lrow_ptr_out,
                                  int64_t n_lrows_out, float* chunk_partials, const float* inv_denom, void* stream) {
    if (int rc = check_rows("sng_edge_bwd", n_total, c, ld)) return rc;
    SNG_REQUIRE(!inv_denom || top_k > 0, "sng_edge_bwd: inv_denom (denominator='selected') needs the selection lists (top_k > 0)");
    SNG_REQUIRE(n >= 0 && row_offset >= 0 && row_offset + n <= n_total, "sng_edge_bwd: bad n / row_offset / n_total");
    // (an empty shard, n == 0, has no rows of g / dn_target / the lists, and possibly no edges: those may be NULL)
    SNG_REQUIRE(h && inv_norm && rowptr && rowptr_out && (col_out || num_edges == 0) && coef && dh && ldg % 4 == 0 && ldg >= c &&
                (n == 0 || (g && dn_target)), "sng_edge_bwd: null pointer or bad ldg");
    SNG_REQUIRE(n == 0 || (top_k > 0 ? (sel_src && sel_w && sel_q && sel_cnt) : (col && tpos)), "sng_edge_bwd: missing selection lists / CSR + tpos");
    SNG_REQUIRE(!dwt || (beta && lddw % 4 == 0 && lddw >= c), "sng_edge_bwd: dwt needs beta and a 16-byte aligned leading dimension");
    SNG_REQUIRE(!dwt || (row_offset == 0 && n == n_total),
                "sng_edge_bwd: dwt needs a call over all rows (row_offset = 0, n = n_total); a row shard's pass S sees only its own out-edges");
    SNG_REQUIRE(!dbeta || (beta && (diff || n == 0) && partials && lddiff % 4 == 0 && lddiff >= c), "sng_edge_bwd: dbeta needs beta, diff and the partials workspace");
    SNG_REQUIRE(src_shift >= 0 && num_edges >= 0, "sng_edge_bwd: bad src_shift / num_edges");
    SNG_REQUIRE(n_chunks_out <= 0 || (chunk_tab_out && lrows_out && lrow_ptr_out && n_lrows_out > 0 && chunk_partials),
                "sng_edge_bwd: by-source chunk tables / partials workspace missing");
    if (n_total == 0) return SNG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (top_k > 0 && num_edges > 0 &&                                // unselected edges keep both coefficients 0
        cudaMemsetAsync(coef, 0, (size_t)num_edges * sizeof(float2), st) != cudaSuccess) return check_launch("sng_edge_bwd memset");
    EdgeBwdArgs a;
    a.h = h; a.inv_r = inv_norm; a.g = g; a.n_total = (int)n_total; a.n = (int)n; a.row_offset = (int)row_offset;
    a.c = (int)c; a.ld = (int)ld; a.ldg = (int)ldg;
    a.rowptr = rowptr; a.col = col; a.tpos = tpos; a.top_k = top_k > 0 ? top_k : 0;
    a.sel_src = sel_src; a.sel_w = sel_w; a.sel_q = sel_q; a.sel_cnt = sel_cnt; a.inv_denom = inv_denom;
    a.beta = beta; a.diff = dbeta ? diff : nullptr; a.lddiff = (int)lddiff; a.dbeta_part = dbeta ? partials : nullptr;
    a.coef = reinterpret_cast<float2*>(coef); a.dnT = dn_target;
    a.rowptr_out = rowptr_out; a.col_out = col_out; a.shift = (int)src_shift;
    a.dh = dh; a.dwt = dwt; a.lddw = (int)lddw;
    a.chunk_tab = reinterpret_cast<const int4*>(chunk_tab_out); a.n_chunks = (int)n_chunks_out; a.lrows = lrows_out; a.lrow_ptr = lrow_ptr_out;
    a.n_lrows = (int)n_lrows_out; a.tmp_part = chunk_partials;
    return launch_edge_bwd(a, dbeta, st, "sng_edge_bwd");
}

extern "C" int sng_edge_bwd(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                            int64_t c, int64_t ld, int64_t ldg,
                            const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                            const int32_t* rowptr_out, const int32_t* col_out, int64_t src_shift, int64_t num_edges,
                            int top_k, const int32_t* sel_src, const float* sel_w, const int32_t* sel_q, const int32_t* sel_cnt,
                            const float* beta, const float* diff, int64_t lddiff, float* dbeta,
                            float* coef, float* dn_target, float* partials, float* dh, float* dwt, int64_t lddw,
                            const int32_t* chunk_tab_out, int64_t n_chunks_out, const int32_t* lrows_out, const int32_t* lrow_ptr_out,
                            int64_t n_lrows_out, float* chunk_partials, void* stream) {
    return sng_edge_bwd_denom(h, inv_norm, g, n_total, n, row_offset, c, ld, ldg, rowptr, col, tpos, rowptr_out, col_out, src_shift,
                              num_edges, top_k, sel_src, sel_w, sel_q, sel_cnt, beta, diff, lddiff, dbeta, coef, dn_target, partials,
                              dh, dwt, lddw, chunk_tab_out, n_chunks_out, lrows_out, lrow_ptr_out, n_lrows_out, chunk_partials,
                              nullptr, stream);
}

extern "C" int sng_list_bwd(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                            int64_t c, int64_t ld, int64_t ldg,
                            int top_k, const int32_t* idx, const float* sim, const int32_t* cnt, const float* inv_denom,
                            const int32_t* sel_q, const int32_t* rowptr_tr, const int32_t* col_tr,
                            float* coef, float* dn_target, float* dh,
                            const int32_t* chunk_tab, int64_t n_chunks, const int32_t* lrows, const int32_t* lrow_ptr, int64_t n_lrows,
                            float* chunk_partials, void* stream) {
    if (int rc = check_rows("sng_list_bwd", n_total, c, ld)) return rc;
    SNG_REQUIRE(n >= 0 && row_offset >= 0 && row_offset + n <= n_total, "sng_list_bwd: bad n / row_offset / n_total");
    SNG_REQUIRE(top_k > 0 && top_k <= SNG_MAX_TOPK, "sng_list_bwd: list width top_k=%d must be in [1, %d]", top_k, SNG_MAX_TOPK);
    // (an empty shard, n == 0, has no rows of g / dn_target / the lists, and no transposed entries: those may be NULL)
    SNG_REQUIRE(h && inv_norm && rowptr_tr && dh && ldg % 4 == 0 && ldg >= c, "sng_list_bwd: null pointer or bad ldg");
    SNG_REQUIRE(n == 0 || (g && idx && sim && cnt && inv_denom && sel_q && col_tr && coef && dn_target), "sng_list_bwd: missing lists / transpose / workspace");
    SNG_REQUIRE(n_chunks <= 0 || (chunk_tab && lrows && lrow_ptr && n_lrows > 0 && chunk_partials),
                "sng_list_bwd: by-source chunk tables / partials workspace missing");
    if (n_total == 0) return SNG_OK;
    EdgeBwdArgs a;
    a.h = h; a.inv_r = inv_norm; a.g = g; a.n_total = (int)n_total; a.n = (int)n; a.row_offset = (int)row_offset;
    a.c = (int)c; a.ld = (int)ld; a.ldg = (int)ldg;
    a.rowptr = nullptr; a.col = nullptr; a.tpos = nullptr; a.top_k = top_k;
    a.sel_src = idx; a.sel_w = sim; a.sel_q = sel_q; a.sel_cnt = cnt; a.inv_denom = inv_denom;
    a.beta = nullptr; a.diff = nullptr; a.lddiff = 0; a.dbeta_part = nullptr;
    a.coef = reinterpret_cast<float2*>(coef); a.dnT = dn_target;            // every list entry writes its coefficient: no memset
    a.rowptr_out = rowptr_tr; a.col_out = col_tr; a.shift = 0;
    a.dh = dh; a.dwt = nullptr; a.lddw = 0;
    a.chunk_tab = reinterpret_cast<const int4*>(chunk_tab); a.n_chunks = (int)n_chunks; a.lrows = lrows; a.lrow_ptr = lrow_ptr;
    a.n_lrows = (int)n_lrows; a.tmp_part = chunk_partials;
    return launch_edge_bwd(a, nullptr, (cudaStream_t)stream, "sng_list_bwd");
}

extern "C" int sng_list_agg_fwd(const float* h, int64_t n_rows, int64_t c, int64_t ldh, int list_k, const int32_t* sel_src,
                                const float* sel_w, const int32_t* sel_cnt, const float* inv_denom, float* out, int64_t ldo,
                                void* stream) {
    if (int rc = check_rows("sng_list_agg_fwd", n_rows, c, ldh)) return rc;
    SNG_REQUIRE(h && sel_src && sel_w && sel_cnt && out && list_k > 0 && ldo % 4 == 0 && ldo >= c, "sng_list_agg_fwd: bad arguments");
    if (n_rows == 0) return SNG_OK;
    SNG_DISPATCH_G(c, list_agg_fwd_kernel<G><<<grid_resident(list_agg_fwd_kernel<G>, n_rows, kWarpsPerBlock), kThreads, 0, (cudaStream_t)stream>>>(h, (int)n_rows, (int)c, ldh, list_k, sel_src, sel_w, sel_cnt, inv_denom, out, ldo));
    return check_launch("sng_list_agg_fwd");
}

extern "C" int sng_edge_agg_bwd(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset, int64_t c, int64_t ld,
                                const int32_t* rowptr, const int32_t* col, int top_k, const int32_t* sel_src, const float* sel_w, const int32_t* sel_cnt,
                                const float* inv_denom, float* dval, float* dnrm, float* dh, void* stream) {
    if (int rc = check_rows("sng_edge_agg_bwd", n_total, c, ld)) return rc;
    SNG_REQUIRE(h && inv_norm && g && dval && dnrm && dh, "sng_edge_agg_bwd: null pointer");
    SNG_REQUIRE(n >= 0 && row_offset >= 0 && row_offset + n <= n_total, "sng_edge_agg_bwd: bad n / row_offset / n_total");
    SNG_REQUIRE(top_k > 0 ? (sel_src && sel_w && sel_cnt && inv_denom) : (rowptr && col), "sng_edge_agg_bwd: missing selection list / CSR");
    if (n_total == 0) return SNG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    SNG_DISPATCH_G(c,
        if (n > 0 && top_k > 0) edge_agg_bwd_scatter_kernel<G, false><<<grid_resident(edge_agg_bwd_scatter_kernel<G, false>, n, kWarpsPerBlock), kThreads, 0, st>>>(h, inv_norm, g, (int)n, (int)row_offset, (int)c, ld, rowptr, col, top_k, sel_src, sel_w, sel_cnt, inv_denom, dval, dnrm);
        else if (n > 0) edge_agg_bwd_scatter_kernel<G, true><<<grid_resident(edge_agg_bwd_scatter_kernel<G, true>, n, kWarpsPerBlock), kThreads, 0, st>>>(h, inv_norm, g, (int)n, (int)row_offset, (int)c, ld, rowptr, col, 0, nullptr, nullptr, nullptr, nullptr, dval, dnrm);
        norm_bwd_finish_kernel<G><<<grid_resident(norm_bwd_finish_kernel<G>, n_total, kWarpsPerBlock * RowShape<G>::EPW), kThreads, 0, st>>>(h, inv_norm, (int)n_total, (int)c, ld, dval, dnrm, dh));
    return check_launch("sng_edge_agg_bwd");
}

extern "C" int sng_spmm_fwd(const float* x, int64_t n_rows, int64_t c, int64_t ldx, const int32_t* rowptr, const int32_t* col,
                            const float* val, const float* rowscale, const float* bias, float* out, int64_t ldo, void* stream) {
    if (int rc = check_rows("sng_spmm_fwd", n_rows, c, ldx)) return rc;
    SNG_REQUIRE(x && rowptr && col && out && ldo % 4 == 0 && ldo >= c, "sng_spmm_fwd: null pointer or bad ldo");
    if (n_rows == 0) return SNG_OK;
    SNG_DISPATCH_G(c, spmm_fwd_kernel<G><<<grid_resident(spmm_fwd_kernel<G>, n_rows, kWarpsPerBlock), kThreads, 0, (cudaStream_t)stream>>>(x, (int)n_rows, (int)c, ldx, rowptr, col, val, rowscale, bias, out, ldo));
    return check_launch("sng_spmm_fwd");
}

extern "C" int sng_pp_fuse_fwd(const float* wt, int64_t n, int64_t c, int64_t ld, const int32_t* rowptr_out, const int32_t* col_out,
                               const float* b_w, const float* beta, const float* out1, const float* bias, float* out0, float* out,
                               void* stream) {
    if (int rc = check_rows("sng_pp_fuse_fwd", n, c, ld)) return rc;
    SNG_REQUIRE(wt && rowptr_out && col_out && b_w && beta && out1 && out0 && out, "sng_pp_fuse_fwd: null pointer");
    if (n == 0) return SNG_OK;
    SNG_DISPATCH_G(c, pp_fuse_fwd_kernel<G><<<grid_resident(pp_fuse_fwd_kernel<G>, n, kWarpsPerBlock), kThreads, 0, (cudaStream_t)stream>>>(wt, (int)n, (int)c, ld, rowptr_out, col_out, b_w, beta, out1, bias, out0, out));
    return check_launch("sng_pp_fuse_fwd");
}

extern "C" int sng_pp_beta_grad(const float* out0, const float* out1, const float* g, int64_t numel, float* dbeta, float* partials,
                                void* stream) {
    SNG_REQUIRE(out0 && out1 && g && dbeta && partials && numel >= 0 && numel % 4 == 0, "sng_pp_beta_grad: bad arguments (numel must be a multiple of 4)");
    int grid = grid_capped(numel / 4, 256, 8);
    if (grid > SNG_PARTIALS) grid = SNG_PARTIALS;
    if (numel == 0) { return cudaMemsetAsync(dbeta, 0, sizeof(float), (cudaStream_t)stream) == cudaSuccess ? SNG_OK : check_launch("sng_pp_beta_grad"); }
    pp_beta_grad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out0, out1, g, numel, partials);
    sum_partials_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(partials, grid, dbeta);
    return check_launch("sng_pp_beta_grad");
}

extern "C" int sng_nll_loss_fwd(const float* logp, int64_t n, int64_t c, int64_t ld, const int64_t* y, float* loss, float* count,
                               float* partials, void* stream) {
    SNG_REQUIRE(logp && y && loss && count && partials && n >= 0 && c > 0 && ld >= c && c < (1ll << 30), "sng_nll_loss_fwd: bad arguments");
    int grid = grid_capped(n, 256, 8);
    if (grid > SNG_PARTIALS / 2) grid = SNG_PARTIALS / 2;
    nll_loss_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(logp, n, (int)c, ld, y, partials, partials + SNG_PARTIALS / 2);
    nll_loss_finish_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(partials, partials + SNG_PARTIALS / 2, grid, loss, count);
    return check_launch("sng_nll_loss_fwd");
}

extern "C" int sng_nll_loss_bwd(int64_t n, int64_t c, int64_t ld, const int64_t* y, const float* gscale, const float* count, float* dlogp,
                               void* stream) {
    SNG_REQUIRE(y && gscale && count && dlogp && n >= 0 && c > 0 && ld >= c, "sng_nll_loss_bwd: bad arguments");
    if (n == 0) return SNG_OK;
    nll_loss_bwd_kernel<<<grid_capped(n * c, 256, 8), 256, 0, (cudaStream_t)stream>>>(n, (int)c, ld, y, gscale, count, dlogp);
    return check_launch("sng_nll_loss_bwd");
}

extern "C" int sng_sddmm_dot(const float* xhat, int64_t n, int64_t d, int64_t ld, const int32_t* a, const int32_t* b,
                             int64_t num_edges, float* s, void* stream) {
    SNG_REQUIRE(xhat && a && b && s && n >= 0 && d > 0 && ld >= d && num_edges >= 0, "sng_sddmm_dot: bad arguments");
    if (num_edges == 0) return SNG_OK;
    sddmm_dot_kernel<<<grid_resident(sddmm_dot_kernel, num_edges, kWarpsPerBlock), kThreads, 0, (cudaStream_t)stream>>>(xhat, (int)d, ld, a, b, num_edges, s);
    return check_launch("sng_sddmm_dot");
}

// ------------------------------------------------------------------------------------------ toolbox helpers
namespace sng {
// Per-class sums of unit rows, S[c] = sum_{i: y_i = c} xhat_i  (FP64 accumulation): the closed form behind every
// "sum of all pairwise similarities" metric, sum_{i in a, j in b} <xhat_i, xhat_j> = <S_a, S_b>
// (R: SimGFAToolbox/dense.py:9-30, 104-130, 167-179 compute the same sums by materialising N x N blocks).
__global__ void __launch_bounds__(256) class_sum_kernel(const float* __restrict__ xh, const int* __restrict__ y, int64_t n, int d, int64_t ld,
                                                       int num_classes, double* __restrict__ sums, double* __restrict__ counts) {
    // grid.x tiles rows, grid.y tiles columns (256 per block): each thread owns one column for a slab of rows
    const int col = blockIdx.y * 256 + threadIdx.x;
    const int64_t rows_per = (n + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per, r1 = min(n, r0 + rows_per);
    const bool counter = counts && blockIdx.y == 0 && threadIdx.x == 0;
    int cur = -1;
    double acc = 0.0, run = 0.0;
    for (int64_t r = r0; r < r1; ++r) {
        int c = y ? __ldg(y + r) : 0;
        if (c < 0 || c >= num_classes) c = -1;                         // rows with an out-of-range label are ignored
        if (c != cur) {
            if (cur >= 0 && col < d) atomicAdd(sums + (int64_t)cur * d + col, acc);
            if (cur >= 0 && counter) atomicAdd(counts + cur, run);
            cur = c; acc = 0.0; run = 0.0;
        }
        if (c >= 0 && col < d) acc += (double)__ldg(xh + r * ld + col);
        run += 1.0;
    }
    if (cur >= 0 && col < d) atomicAdd(sums + (int64_t)cur * d + col, acc);
    if (cur >= 0 && counter) atomicAdd(counts + cur, run);
}
}  // namespace sng

extern "C" int sng_class_sums_f64(const float* xhat, const int32_t* y, int64_t n, int64_t d, int64_t ld, int num_classes, double* sums,
                                  double* counts, void* stream) {
    SNG_REQUIRE(xhat && sums && n >= 0 && d > 0 && ld >= d && num_classes >= 1 && (y || num_classes == 1), "sng_class_sums_f64: bad arguments");
    if (n == 0) return SNG_OK;
    const int gx = (int)(n < 4096 ? (n + 63) / 64 : 2048);
    dim3 grid((unsigned)(gx > 0 ? gx : 1), (unsigned)((d + 255) / 256));
    sng::class_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(xhat, y, n, (int)d, ld, num_classes, sums, counts);
    return check_launch("sng_class_sums_f64");
}
