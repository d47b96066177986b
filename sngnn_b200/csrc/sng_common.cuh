// Shared helpers for libsng.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/sng.h"

namespace sng {

void set_error(const char* fmt, ...);
int check_launch(const char* what);   // cudaPeekAtLastError -> SNG_ERR_CUDA + message
int sm_count();                       // cached; 148 (a B200's) if there is no device, see sng_api.cu

#define SNG_REQUIRE(cond, ...)                                  \
    do {                                                        \
        if (!(cond)) {                                          \
            ::sng::set_error(__VA_ARGS__);                      \
            return SNG_ERR_ARG;                                 \
        }                                                       \
    } while (0)

constexpr float kNormEps = 1e-12f;   // F.normalize eps, R: models/models.py:122

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
    return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}
__device__ __forceinline__ float4 scale4(const float4& a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ void fma4(float4& acc, float s, const float4& v) {
    acc.x = fmaf(s, v.x, acc.x); acc.y = fmaf(s, v.y, acc.y); acc.z = fmaf(s, v.z, acc.z); acc.w = fmaf(s, v.w, acc.w);
}
// butterfly sum over the G lanes of a group (G power of two, groups are lane-aligned)
template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// sum over the 32/G groups of a warp (lanes with equal lane % G)
template <int G>
__device__ __forceinline__ float cross_group_sum(float v) {
#pragma unroll
    for (int o = 16; o >= G; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// 1 / max(||x||, 1e-12) from the squared norm (one MUFU.RSQ; 2 ulp, far inside the 1e-5 contract)
__device__ __forceinline__ float inv_norm_of(float ss) { return rsqrtf(fmaxf(ss, kNormEps * kNormEps)); }

// lanes-per-row group size for a padded channel count c (multiple of 4): smallest power of two >= c/4
inline int group_lanes(int64_t c) {
    int g = 1;
    while (g * 4 < c) g <<= 1;
    return g;
}

// Grid of a grid-stride kernel: the blocks `items` need, at most ctas_per_sm CTAs per SM, at least one.
inline int grid_capped(int64_t items, int64_t items_per_block, int64_t ctas_per_sm) {
    const int64_t need = (items + items_per_block - 1) / items_per_block, cap = sm_count() * ctas_per_sm;
    const int64_t g = need < cap ? need : cap;
    return (int)(g < 1 ? 1 : g);
}
// Grid of a grid-stride row kernel = exactly the number of CTAs that are resident at once (SMs x occupancy of THIS kernel):
// every CTA then gets the same share of rows and there is no partial second wave (a fixed 8 CTAs per SM left the gather
// kernels, which fit 5-6, with a 1.3-1.6 wave launch whose tail ran on a half-empty GPU).
template <typename Kernel>
int grid_resident(Kernel kernel, int64_t items, int items_per_block, size_t smem = 0, int threads = 256) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem) != cudaSuccess || occ < 1) { cudaGetLastError(); occ = 1; }
    return grid_capped(items, items_per_block, occ);
}

}  // namespace sng
