// Counter-based row dropout (include/sng.h): the keep bit of element (row, channel) is a pure function of (seed, call, global row,
// channel), so row shards of any size draw exactly the masks of the unsharded layer, and the backward regenerates the mask from
// the same counters instead of reading a stored [N, C] mask.
//   e = (row_offset + i) * c + j; words = Philox4x32-10(counter = (e >> 2, call), key = seed); w = words[e & 3]
//   keep = (w >> 8) >= t, t = round(p 2^24);  forward y = keep ? a s : 0, a = relu ? max(z, 0) : z, s = 1 / (1 - p)
//                                             backward dz = keep && (!relu || z > 0) ? g s : 0
#include "sng_common.cuh"

#include <math.h>

namespace sng {
constexpr int kDoThreads = 256;

struct Philox4 {
    uint32_t w[4];
    // word k without a dynamically indexed (local memory) array
    __device__ __forceinline__ uint32_t word(uint32_t k) const { return k == 0 ? w[0] : k == 1 ? w[1] : k == 2 ? w[2] : w[3]; }
};

// Philox4x32-10 with the Random123 multipliers and Weyl key increments
__device__ __forceinline__ Philox4 philox4x32_10(uint64_t ctr_lo, uint64_t ctr_hi, uint64_t key) {
    uint32_t c0 = (uint32_t)ctr_lo, c1 = (uint32_t)(ctr_lo >> 32), c2 = (uint32_t)ctr_hi, c3 = (uint32_t)(ctr_hi >> 32);
    uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return Philox4{{c0, c1, c2, c3}};
}

struct DropArgs {
    const float* z; const float* g; float* out;
    int64_t n, ldz, ldg, ldo, row_offset;
    int c;
    uint64_t seed, call;
    uint32_t t;
    float s;
    int relu;
};

// forward: out = keep ? a s : 0; backward: out = keep && (!relu || z > 0) ? g s : 0
template <bool BWD>
__device__ __forceinline__ float drop_one(const DropArgs& A, uint32_t w, float z, float g) {
    const bool keep = (w >> 8) >= A.t;
    if (BWD) return keep && (!A.relu || z > 0.f) ? g * A.s : 0.f;
    return keep ? (A.relu ? fmaxf(z, 0.f) : z) * A.s : 0.f;
}

// c % 4 == 0 with 16-byte aligned rows: a thread owns 4 channels of a row, which are exactly the 4 words of one Philox call.
// tpr = smallest power of two >= c / 4 (at most 256) threads per row, rpb = 256 / tpr rows per block step.
template <bool BWD>
__global__ void __launch_bounds__(kDoThreads) row_dropout_vec_kernel(const DropArgs A) {
    const int cq = A.c >> 2;
    int tpr_log = 0;
    while ((1 << tpr_log) < cq && tpr_log < 8) ++tpr_log;
    const int rpb = kDoThreads >> tpr_log;
    const int lane = threadIdx.x & ((1 << tpr_log) - 1);
    const bool need_z = !BWD || A.relu;
    for (int64_t r = (int64_t)blockIdx.x * rpb + (threadIdx.x >> tpr_log); r < A.n; r += (int64_t)gridDim.x * rpb) {
        for (int q = lane; q < cq; q += 1 << tpr_log) {
            const int j = q << 2;
            const float4 zv = need_z ? ldg4(A.z + r * A.ldz + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 gv = BWD ? ldg4(A.g + r * A.ldg + j) : zv;
            const uint64_t e4 = ((uint64_t)(A.row_offset + r) * (uint64_t)A.c + (uint64_t)j) >> 2;
            const Philox4 P = philox4x32_10(e4, A.call, A.seed);
            float4 o;
            o.x = drop_one<BWD>(A, P.w[0], zv.x, gv.x);
            o.y = drop_one<BWD>(A, P.w[1], zv.y, gv.y);
            o.z = drop_one<BWD>(A, P.w[2], zv.z, gv.z);
            o.w = drop_one<BWD>(A, P.w[3], zv.w, gv.w);
            *reinterpret_cast<float4*>(A.out + r * A.ldo + j) = o;
        }
    }
}

// any c and stride: a thread owns one Philox call = the up to 4 elements of the flat global range [e0, e0 + 4) inside this shard
// (a ragged c splits a group across two rows); one division per group finds the first element's row.
template <bool BWD>
__global__ void __launch_bounds__(kDoThreads) row_dropout_scalar_kernel(const DropArgs A, uint64_t q_begin, uint64_t q_end) {
    const uint64_t base = (uint64_t)A.row_offset * (uint64_t)A.c, end = base + (uint64_t)A.n * (uint64_t)A.c;
    const bool need_z = !BWD || A.relu;
    for (uint64_t q = q_begin + (uint64_t)blockIdx.x * kDoThreads + threadIdx.x; q < q_end; q += (uint64_t)gridDim.x * kDoThreads) {
        const Philox4 P = philox4x32_10(q, A.call, A.seed);
        const uint64_t e0 = q << 2 > base ? q << 2 : base;
        int64_t r = (int64_t)(e0 / (uint64_t)A.c) - A.row_offset;
        int j = (int)(e0 % (uint64_t)A.c);
        for (uint64_t e = e0; e < (q << 2) + 4 && e < end; ++e) {
            const float z = need_z ? __ldg(A.z + r * A.ldz + j) : 0.f;
            const float g = BWD ? __ldg(A.g + r * A.ldg + j) : 0.f;
            A.out[r * A.ldo + j] = drop_one<BWD>(A, P.word((uint32_t)e & 3u), z, g);
            if (++j == A.c) { j = 0; ++r; }
        }
    }
}

inline bool aligned16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

template <bool BWD>
static int row_dropout(const char* what, DropArgs A, double p, cudaStream_t st) {
    SNG_REQUIRE(p >= 0.0 && p <= 1.0, "%s: p must be in [0, 1] (p=%g)", what, p);
    SNG_REQUIRE(A.n >= 0 && A.c >= 1 && A.row_offset >= 0, "%s: bad arguments (n=%lld c=%d row_offset=%lld)", what, (long long)A.n, A.c,
                (long long)A.row_offset);
    SNG_REQUIRE(A.ldz >= A.c && A.ldo >= A.c && (!BWD || A.ldg >= A.c), "%s: leading dimensions must be >= c (c=%d ldz=%lld ldg=%lld ld_out=%lld)",
                what, A.c, (long long)A.ldz, (long long)A.ldg, (long long)A.ldo);
    // e = (row_offset + n) c must fit in 64 bits, with room for the e >> 2 group counter's last group
    SNG_REQUIRE((uint64_t)A.row_offset + (uint64_t)A.n <= (uint64_t)(INT64_MAX - 4) / (uint64_t)A.c,
                "%s: (row_offset + n) * c overflows 64 bits (row_offset=%lld n=%lld c=%d)", what, (long long)A.row_offset, (long long)A.n, A.c);
    const bool need_z = !BWD || A.relu;
    SNG_REQUIRE((A.z || !need_z || A.n == 0) && (A.g || !BWD || A.n == 0) && (A.out || A.n == 0), "%s: NULL operand with n=%lld", what,
                (long long)A.n);
    if (A.n == 0) return SNG_OK;
    A.t = (uint32_t)floor(p * 16777216.0 + 0.5);
    A.s = 1.0f / (1.0f - (float)p);
    const bool vec = A.c % 4 == 0 && A.ldz % 4 == 0 && A.ldo % 4 == 0 && (!BWD || A.ldg % 4 == 0) && aligned16(need_z ? A.z : nullptr) &&
                     aligned16(A.out) && aligned16(BWD ? A.g : nullptr);
    if (vec) {
        int tpr = 1;
        while (tpr < A.c / 4 && tpr < kDoThreads) tpr <<= 1;
        const int grid = grid_resident(row_dropout_vec_kernel<BWD>, A.n, kDoThreads / tpr, 0, kDoThreads);
        row_dropout_vec_kernel<BWD><<<grid, kDoThreads, 0, st>>>(A);
    } else {
        const uint64_t base = (uint64_t)A.row_offset * (uint64_t)A.c;
        const uint64_t q_begin = base >> 2, q_end = ((base + (uint64_t)A.n * (uint64_t)A.c - 1) >> 2) + 1;
        const int grid = grid_resident(row_dropout_scalar_kernel<BWD>, (int64_t)(q_end - q_begin), kDoThreads, 0, kDoThreads);
        row_dropout_scalar_kernel<BWD><<<grid, kDoThreads, 0, st>>>(A, q_begin, q_end);
    }
    return check_launch(what);
}
}  // namespace sng

using namespace sng;

extern "C" int sng_row_dropout_fwd(const float* z, int64_t n, int64_t c, int64_t ldz, int64_t row_offset, uint64_t seed, uint64_t call,
                                   float p, int relu, float* y, int64_t ldy, void* stream) {
    SNG_REQUIRE(c >= 1 && c <= INT32_MAX, "sng_row_dropout_fwd: bad arguments (c=%lld)", (long long)c);
    DropArgs A{z, nullptr, y, n, ldz, 0, ldy, row_offset, (int)c, seed, call, 0u, 0.f, relu != 0};
    return row_dropout<false>("sng_row_dropout_fwd", A, (double)p, (cudaStream_t)stream);
}

extern "C" int sng_row_dropout_bwd(const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, int64_t row_offset,
                                   uint64_t seed, uint64_t call, float p, int relu, float* dz, int64_t lddz, void* stream) {
    SNG_REQUIRE(c >= 1 && c <= INT32_MAX, "sng_row_dropout_bwd: bad arguments (c=%lld)", (long long)c);
    // z is read only with relu: without it the caller may pass NULL and ldz is not checked
    DropArgs A{z, g, dz, n, relu ? ldz : c, ldg, lddz, row_offset, (int)c, seed, call, 0u, 0.f, relu != 0};
    return row_dropout<true>("sng_row_dropout_bwd", A, (double)p, (cudaStream_t)stream);
}
