// BatchNorm over row shards, fused with the ReLU that precedes it in every model (R: models/models.py:81-84: relu -> bn).
// Four streaming passes over z = the conv output (pre-activation), a = max(z, 0):
//   forward  stats: this shard's per-channel (sum a, sum a^2)          apply: y = gamma (a - mu) rstd + beta, mu, rstd
//   backward stats: (sum g, sum g ahat), ahat = (a - mu) rstd           apply: dz = 1[z > 0] gamma rstd (g - sum g / N - ahat sum g ahat / N)
// The sums are FP64: per-CTA partials in a fixed order, then one warp per output over the CTAs in a fixed order -- no atomics, so
// a shard's sums repeat bit for bit on a given device (the grid is grid_resident's), and the caller's all-reduce of the [2, c] sums
// sees the same operands on every run.
#include "sng_common.cuh"

namespace sng {
constexpr int kBnThreads = 256;
constexpr int kBnLoads = 8;                  // loads in flight per thread and operand: 8 / NC rows of NC channels

// Thread layout of every kernel here: tpr = smallest power of two >= c (at most 256) threads per row, channel col0 = t % tpr and,
// for NC = 2 (c > 256), col0 + tpr; rpb = 256 / tpr rows per block step.
struct BnLayout {
    int tpr_log, col0, rl, rpb;
    __device__ BnLayout(int c) {
        tpr_log = 0;
        while ((1 << tpr_log) < c && tpr_log < 8) ++tpr_log;
        col0 = threadIdx.x & ((1 << tpr_log) - 1);
        rl = threadIdx.x >> tpr_log;
        rpb = kBnThreads >> tpr_log;
    }
};

inline int bn_rows_per_block(int64_t c) {
    int tpr = 1;
    while (tpr < c && tpr < kBnThreads) tpr <<= 1;
    return kBnThreads / tpr;
}

// part [gridDim.x, 2, c]: BWD = false: (sum a, sum a^2); BWD = true: (sum g, sum g ahat).  Rows a thread does not own add exact zeros.
template <bool BWD, int NC>
__global__ void __launch_bounds__(kBnThreads) bn_stats_kernel(const float* __restrict__ z, const float* __restrict__ g, int64_t n, int c,
                                                             int64_t ldz, int64_t ldg, const float* __restrict__ mean,
                                                             const float* __restrict__ rstd, double* __restrict__ part) {
    const BnLayout L(c);
    const int tpr = 1 << L.tpr_log;
    bool ok[NC];
    float mu[NC], rs[NC];
    double s1[NC], s2[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int col = L.col0 + k * tpr;
        ok[k] = col < c;
        mu[k] = BWD && ok[k] ? __ldg(mean + col) : 0.f;
        rs[k] = BWD && ok[k] ? __ldg(rstd + col) : 0.f;
        s1[k] = 0.0; s2[k] = 0.0;
    }
    const int64_t step = (int64_t)gridDim.x * L.rpb;
    for (int64_t r0 = (int64_t)blockIdx.x * L.rpb + L.rl; r0 < n; r0 += kBnLoads / NC * step) {
        float v[kBnLoads / NC][NC], w[kBnLoads / NC][NC];
#pragma unroll
        for (int u = 0; u < kBnLoads / NC; ++u) {
            const int64_t r = r0 + u * step;
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const bool in = ok[k] && r < n;
                const int col = L.col0 + k * tpr;
                v[u][k] = in ? __ldg(z + r * ldz + col) : 0.f;
                w[u][k] = BWD && in ? __ldg(g + r * ldg + col) : 0.f;
            }
        }
#pragma unroll
        for (int u = 0; u < kBnLoads / NC; ++u) {
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const float a = fmaxf(v[u][k], 0.f);
                if (BWD) {
                    const float ahat = (a - mu[k]) * rs[k];
                    s1[k] += (double)w[u][k];
                    s2[k] = fma((double)w[u][k], (double)ahat, s2[k]);
                } else {
                    s1[k] += (double)a;
                    s2[k] = fma((double)a, (double)a, s2[k]);
                }
            }
        }
    }
    __shared__ double red[NC][2][kBnThreads];
#pragma unroll
    for (int k = 0; k < NC; ++k) { red[k][0][threadIdx.x] = s1[k]; red[k][1][threadIdx.x] = s2[k]; }
    __syncthreads();
    if (L.rl == 0) {                                            // row lanes of a channel, summed in a fixed order
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            if (!ok[k]) continue;
            double t1 = 0.0, t2 = 0.0;
            for (int q = 0; q < L.rpb; ++q) { t1 += red[k][0][q * tpr + L.col0]; t2 += red[k][1][q * tpr + L.col0]; }
            const int col = L.col0 + k * tpr;
            part[((int64_t)blockIdx.x * 2 + 0) * c + col] = t1;
            part[((int64_t)blockIdx.x * 2 + 1) * c + col] = t2;
        }
    }
}

// sums [2, c] = sum over the nblk partials, one warp per output: lanes stride over the blocks, then a fixed shuffle tree
__global__ void __launch_bounds__(256) bn_sums_kernel(const double* __restrict__ part, int nblk, int c, double* __restrict__ sums) {
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= 2 * c) return;
    const int j = i / c, col = i % c;
    double s = 0.0;
    for (int b = lane; b < nblk; b += 32) s += part[((int64_t)b * 2 + j) * c + col];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) sums[i] = s;
}

// mu = S1 / N, var = S2 / N - mu^2 (biased, as torch normalises), in FP64.  The cancellation loses about 2 log10(|mu| / sigma)
// of FP64's 16 digits: still FP32-exact for |mu| / sigma up to about 1e4, which post-ReLU activations stay far below.
__device__ __forceinline__ void bn_moments(const double* __restrict__ sums, int c, int col, int64_t n_total, double eps, float& mu, float& rs) {
    const double m = sums[col] / (double)n_total;
    const double var = fmax(sums[c + col] / (double)n_total - m * m, 0.0);
    mu = (float)m;
    rs = (float)(1.0 / sqrt(var + eps));
}

// y = gamma (a - mu) rstd + beta.  sums != NULL: mu / rstd from the global sums, written to mean / rstd by block 0;
// sums == NULL: mu / rstd read from mean / rstd (eval mode: the running statistics).
template <int NC>
__global__ void __launch_bounds__(kBnThreads) bn_fwd_apply_kernel(const float* __restrict__ z, int64_t n, int c, int64_t ldz,
                                                                 const double* __restrict__ sums, int64_t n_total, double eps,
                                                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                 float* __restrict__ mean, float* __restrict__ rstd, float* __restrict__ y, int64_t ldy) {
    const BnLayout L(c);
    const int tpr = 1 << L.tpr_log;
    bool ok[NC];
    float mu[NC], rs[NC], gm[NC], bt[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int col = L.col0 + k * tpr;
        ok[k] = col < c;
        mu[k] = rs[k] = gm[k] = bt[k] = 0.f;
        if (!ok[k]) continue;
        if (sums) {
            bn_moments(sums, c, col, n_total, eps, mu[k], rs[k]);
            if (blockIdx.x == 0 && L.rl == 0) { mean[col] = mu[k]; rstd[col] = rs[k]; }
        } else {
            mu[k] = __ldg(mean + col); rs[k] = __ldg(rstd + col);
        }
        gm[k] = __ldg(gamma + col); bt[k] = __ldg(beta + col);
    }
    const int64_t step = (int64_t)gridDim.x * L.rpb;
    for (int64_t r0 = (int64_t)blockIdx.x * L.rpb + L.rl; r0 < n; r0 += kBnLoads / NC * step) {
        float v[kBnLoads / NC][NC];
#pragma unroll
        for (int u = 0; u < kBnLoads / NC; ++u)
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const int64_t r = r0 + u * step;
                v[u][k] = ok[k] && r < n ? __ldg(z + r * ldz + L.col0 + k * tpr) : 0.f;
            }
#pragma unroll
        for (int u = 0; u < kBnLoads / NC; ++u)
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const int64_t r = r0 + u * step;
                if (ok[k] && r < n) y[r * ldy + L.col0 + k * tpr] = fmaf(gm[k], (fmaxf(v[u][k], 0.f) - mu[k]) * rs[k], bt[k]);
            }
    }
}

// dz = 1[z > 0] gamma rstd (g - S_g / N - ahat S_gahat / N); sums == NULL (eval mode: constant statistics): dz = 1[z > 0] gamma rstd g
template <int NC>
__global__ void __launch_bounds__(kBnThreads) bn_bwd_apply_kernel(const float* __restrict__ z, const float* __restrict__ g, int64_t n, int c,
                                                                 int64_t ldz, int64_t ldg, const double* __restrict__ sums, int64_t n_total,
                                                                 const float* __restrict__ gamma, const float* __restrict__ mean,
                                                                 const float* __restrict__ rstd, float* __restrict__ dz, int64_t lddz) {
    const BnLayout L(c);
    const int tpr = 1 << L.tpr_log;
    bool ok[NC];
    float mu[NC], rs[NC], gr[NC], k1[NC], k2[NC];
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const int col = L.col0 + k * tpr;
        ok[k] = col < c;
        mu[k] = rs[k] = gr[k] = k1[k] = k2[k] = 0.f;
        if (!ok[k]) continue;
        mu[k] = __ldg(mean + col); rs[k] = __ldg(rstd + col);
        gr[k] = __ldg(gamma + col) * rs[k];
        if (sums) { k1[k] = (float)(sums[col] / (double)n_total); k2[k] = (float)(sums[c + col] / (double)n_total); }
    }
    const int64_t step = (int64_t)gridDim.x * L.rpb;
    for (int64_t r0 = (int64_t)blockIdx.x * L.rpb + L.rl; r0 < n; r0 += kBnLoads / NC * step) {
        float v[kBnLoads / NC][NC], w[kBnLoads / NC][NC];
#pragma unroll
        for (int u = 0; u < kBnLoads / NC; ++u)
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const int64_t r = r0 + u * step;
                const bool in = ok[k] && r < n;
                const int col = L.col0 + k * tpr;
                v[u][k] = in ? __ldg(z + r * ldz + col) : 0.f;
                w[u][k] = in ? __ldg(g + r * ldg + col) : 0.f;
            }
#pragma unroll
        for (int u = 0; u < kBnLoads / NC; ++u)
#pragma unroll
            for (int k = 0; k < NC; ++k) {
                const int64_t r = r0 + u * step;
                if (!(ok[k] && r < n)) continue;
                const float zz = v[u][k];
                const float ahat = (fmaxf(zz, 0.f) - mu[k]) * rs[k];
                dz[r * lddz + L.col0 + k * tpr] = zz > 0.f ? gr[k] * (w[u][k] - k1[k] - ahat * k2[k]) : 0.f;
            }
    }
}

template <bool BWD, int NC>
static int bn_stats_nc(const char* what, const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, const float* mean,
                    const float* rstd, double* sums, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    const int grid = grid_resident(bn_stats_kernel<BWD, NC>, n, bn_rows_per_block(c) * (kBnLoads / NC), 0, kBnThreads);
    SNG_REQUIRE(workspace && workspace_bytes >= (size_t)grid * 2 * c * sizeof(double) + 256, "%s: workspace too small (%zu bytes)",
                what, workspace_bytes);
    double* part = reinterpret_cast<double*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    bn_stats_kernel<BWD, NC><<<grid, kBnThreads, 0, st>>>(z, g, n, (int)c, ldz, ldg, mean, rstd, part);
    bn_sums_kernel<<<(unsigned)((2 * c + 7) / 8), 256, 0, st>>>(part, grid, (int)c, sums);
    return check_launch(what);
}

// channels per thread: 2 only for rows wider than the block
template <bool BWD>
static int bn_stats(const char* what, const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, const float* mean,
                    const float* rstd, double* sums, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    return c > kBnThreads ? bn_stats_nc<BWD, 2>(what, z, g, n, c, ldz, ldg, mean, rstd, sums, workspace, workspace_bytes, st)
                          : bn_stats_nc<BWD, 1>(what, z, g, n, c, ldz, ldg, mean, rstd, sums, workspace, workspace_bytes, st);
}

template <int NC>
static void bn_fwd_apply_launch(const float* z, int64_t n, int64_t c, int64_t ldz, const double* sums, int64_t n_total, double eps,
                                const float* gamma, const float* beta, float* mean, float* rstd, float* y, int64_t ldy, cudaStream_t st) {
    const int grid = grid_resident(bn_fwd_apply_kernel<NC>, n, bn_rows_per_block(c) * (kBnLoads / NC), 0, kBnThreads);
    bn_fwd_apply_kernel<NC><<<grid, kBnThreads, 0, st>>>(z, n, (int)c, ldz, sums, n_total, eps, gamma, beta, mean, rstd, y, ldy);
}

template <int NC>
static void bn_bwd_apply_launch(const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, const double* sums,
                                int64_t n_total, const float* gamma, const float* mean, const float* rstd, float* dz, int64_t lddz, cudaStream_t st) {
    const int grid = grid_resident(bn_bwd_apply_kernel<NC>, n, bn_rows_per_block(c) * (kBnLoads / NC), 0, kBnThreads);
    bn_bwd_apply_kernel<NC><<<grid, kBnThreads, 0, st>>>(z, g, n, (int)c, ldz, ldg, sums, n_total, gamma, mean, rstd, dz, lddz);
}
}  // namespace sng

using namespace sng;

extern "C" size_t sng_bn_workspace_bytes(int64_t n, int64_t c) {
    (void)n;
    if (c <= 0 || c > SNG_MAX_CHANNELS) return 0;
    // at most one resident wave of 256-thread CTAs: 2048 / 256 per SM
    return (size_t)sm_count() * (2048 / kBnThreads) * 2 * (size_t)c * sizeof(double) + 256;
}

extern "C" int sng_bn_fwd_stats(const float* z, int64_t n, int64_t c, int64_t ldz, double* sums, void* workspace, size_t workspace_bytes,
                                void* stream) {
    SNG_REQUIRE(sums && n >= 0 && c > 0 && c <= SNG_MAX_CHANNELS && ldz >= c && (z || n == 0),
                "sng_bn_fwd_stats: bad arguments (n=%lld c=%lld ldz=%lld; c <= %d)", (long long)n, (long long)c, (long long)ldz, SNG_MAX_CHANNELS);
    return bn_stats<false>("sng_bn_fwd_stats", z, nullptr, n, c, ldz, 0, nullptr, nullptr, sums, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int sng_bn_fwd_apply(const float* z, int64_t n, int64_t c, int64_t ldz, const double* sums, int64_t n_total, double eps,
                                const float* gamma, const float* beta, float* mean, float* rstd, float* y, int64_t ldy, void* stream) {
    SNG_REQUIRE(n >= 0 && c > 0 && c <= SNG_MAX_CHANNELS && ldz >= c && ldy >= c && gamma && beta && mean && rstd && ((z && y) || n == 0),
                "sng_bn_fwd_apply: bad arguments (n=%lld c=%lld ldz=%lld ldy=%lld)", (long long)n, (long long)c, (long long)ldz, (long long)ldy);
    SNG_REQUIRE(!sums || (n_total > 0 && eps >= 0.0), "sng_bn_fwd_apply: n_total must be positive with sums (n_total=%lld)", (long long)n_total);
    cudaStream_t st = (cudaStream_t)stream;
    // block 0 writes mean / rstd, so the kernel runs (one block) for an empty shard too
    if (c > kBnThreads) bn_fwd_apply_launch<2>(z, n, c, ldz, sums, n_total, eps, gamma, beta, mean, rstd, y, ldy, st);
    else bn_fwd_apply_launch<1>(z, n, c, ldz, sums, n_total, eps, gamma, beta, mean, rstd, y, ldy, st);
    return check_launch("sng_bn_fwd_apply");
}

extern "C" int sng_bn_bwd_stats(const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, const float* mean,
                                const float* rstd, double* sums, void* workspace, size_t workspace_bytes, void* stream) {
    SNG_REQUIRE(sums && mean && rstd && n >= 0 && c > 0 && c <= SNG_MAX_CHANNELS && ldz >= c && ldg >= c && ((z && g) || n == 0),
                "sng_bn_bwd_stats: bad arguments (n=%lld c=%lld ldz=%lld ldg=%lld)", (long long)n, (long long)c, (long long)ldz, (long long)ldg);
    return bn_stats<true>("sng_bn_bwd_stats", z, g, n, c, ldz, ldg, mean, rstd, sums, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int sng_bn_bwd_apply(const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, const double* sums,
                                int64_t n_total, const float* gamma, const float* mean, const float* rstd, float* dz, int64_t lddz,
                                void* stream) {
    SNG_REQUIRE(gamma && mean && rstd && n >= 0 && c > 0 && c <= SNG_MAX_CHANNELS && ldz >= c && ldg >= c && lddz >= c && ((z && g && dz) || n == 0),
                "sng_bn_bwd_apply: bad arguments (n=%lld c=%lld ldz=%lld ldg=%lld lddz=%lld)", (long long)n, (long long)c, (long long)ldz,
                (long long)ldg, (long long)lddz);
    SNG_REQUIRE(!sums || n_total > 0, "sng_bn_bwd_apply: n_total must be positive with sums (n_total=%lld)", (long long)n_total);
    if (n == 0) return SNG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (c > kBnThreads) bn_bwd_apply_launch<2>(z, g, n, c, ldz, ldg, sums, n_total, gamma, mean, rstd, dz, lddz, st);
    else bn_bwd_apply_launch<1>(z, g, n, c, ldz, ldg, sums, n_total, gamma, mean, rstd, dz, lddz, st);
    return check_launch("sng_bn_bwd_apply");
}
