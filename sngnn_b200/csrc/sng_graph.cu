// Graph preparation on the GPU (SURVEY.md §8(f) rank 1): what the reference redoes in Python every forward
// (R: models/models.py:117-127, :234-236, :323) -- append N self loops, optionally drop every src == dst edge, build the
// COO of A[src - min(src), dst] -- done once per edge_index and turned into the int32 CSR arrays the edge kernels consume:
//   CSR by TARGET   (rowptr_in,  col_in  = sources in ORIGINAL EDGE-POSITION order: the tie-break order of the selection)
//   CSR by SOURCE   (rowptr_out, col_out = targets of node (src - min src)), col_in_shift = col_in - min src
//   tpos            position of by-target edge p in the by-source arrays (the transpose index of the deterministic backward)
//   long_rows       target rows with more than 32 / 1024 in-edges (the forward runs them on their own kernels)
// A stable LSD radix sort (cub::DeviceRadixSort -- a library sort, the only library call of the edge path) of
// (key = target | source, value = edge id) keeps equal keys in input order, which is exactly the position order the
// selection rule needs; dropped edges get a sentinel key and sort to the end.
#include "sng_common.cuh"
#include <cub/device/device_radix_sort.cuh>

namespace sng {

__global__ void __launch_bounds__(256) graph_keys_kernel(const int64_t* __restrict__ ei, int64_t ne, int n, int remove_self,
                                                        int* __restrict__ key_dst, int* __restrict__ key_src, int* __restrict__ eid,
                                                        int* __restrict__ min_src) {
    int local_min = 0x7fffffff;
    const int64_t total = ne + n;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        int s, d;
        if (e < ne) { s = (int)__ldg(ei + e); d = (int)__ldg(ei + ne + e); }
        else { s = d = (int)(e - ne); }                                   // the appended self loops (R: add_self_loops appends at the end)
        const bool keep = !(remove_self && s == d);
        key_dst[e] = keep ? d : n;                                        // sentinel bucket n sorts behind every node
        if (key_src) key_src[e] = keep ? s : n;
        eid[e] = (int)e;
        if (keep) local_min = min(local_min, s);
    }
    if (min_src) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) local_min = min(local_min, __shfl_xor_sync(0xffffffffu, local_min, o));
        if ((threadIdx.x & 31) == 0 && local_min != 0x7fffffff) atomicMin(min_src, local_min);
    }
}

// other end of every sorted edge: by == 0 -> source of edge perm[p] (col_in), by == 1 -> target (col_out, and inv[perm[q]] = q)
__global__ void __launch_bounds__(256) graph_ends_kernel(const int64_t* __restrict__ ei, int64_t ne, int64_t total, const int* __restrict__ perm,
                                                        int by, int* __restrict__ col, int* __restrict__ inv) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
        const int e = __ldg(perm + p);
        col[p] = e < ne ? (int)__ldg(ei + (by ? ne : 0) + e) : (int)(e - ne);
        if (inv) inv[e] = (int)p;
    }
}

// rowptr[r] = first position whose key is >= r + shift  (keys ascending; r = 0..n)
__global__ void __launch_bounds__(256) graph_rowptr_kernel(const int* __restrict__ keys, int64_t total, int n, const int* __restrict__ shift_p,
                                                          int* __restrict__ rowptr) {
    const int shift = (shift_p && *shift_p < n) ? *shift_p : 0;          // (no kept edge: the memset pattern stays, shift 0)
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r <= n; r += gridDim.x * blockDim.x) {
        const int want = (r == n) ? n : min(r + shift, n);               // row n = number of kept edges (sentinel keys are n)
        int64_t lo = 0, hi = total;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (__ldg(keys + mid) < want) lo = mid + 1; else hi = mid;
        }
        rowptr[r] = (int)lo;
    }
}

// info = {kept edges, min src, symmetric (in-lists == out-lists, shift 0), rows with 32 < deg <= 1024, rows with deg > 1024, max in-degree}
__global__ void __launch_bounds__(256) graph_finish_kernel(const int* __restrict__ rowptr_in, int n, float* __restrict__ inv_deg,
                                                          const int* __restrict__ col_in, int* __restrict__ col_in_shift,
                                                          const int* __restrict__ min_src, const int* __restrict__ rowptr_out,
                                                          const int* __restrict__ col_out, const int* __restrict__ perm_in,
                                                          const int* __restrict__ inv_out, int* __restrict__ tpos,
                                                          int* __restrict__ long_rows, int* __restrict__ info) {
    const int kept = rowptr_in[n];
    const int shift = (min_src && *min_src < n) ? *min_src : 0;
    bool sym = shift == 0;
    int max_deg = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int deg = rowptr_in[i + 1] - rowptr_in[i];
        inv_deg[i] = 1.0f / (float)max(deg, 1);                           // PyG aggr='mean' denominator
        max_deg = max(max_deg, deg);
        if (long_rows && deg > 32) {
            if (deg <= 1024) long_rows[atomicAdd(info + 3, 1)] = i;       // filled from the front
            else long_rows[n - 1 - atomicAdd(info + 4, 1)] = i;           // hubs from the back
        }
        if (rowptr_out && (rowptr_out[i] != rowptr_in[i] || rowptr_out[i + 1] != rowptr_in[i + 1])) sym = false;
    }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kept; i += gridDim.x * blockDim.x) {
        const int j = col_in[i];
        if (col_in_shift) col_in_shift[i] = j - shift;
        if (col_out && col_out[i] != j) sym = false;
        if (tpos) tpos[i] = inv_out[perm_in[i]];
    }
    if (rowptr_out && !sym) atomicAnd(info + 2, 0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) max_deg = max(max_deg, __shfl_xor_sync(0xffffffffu, max_deg, o));
    if ((threadIdx.x & 31) == 0) atomicMax(info + 5, max_deg);
    if (blockIdx.x == 0 && threadIdx.x == 0) { info[0] = kept; info[1] = shift; }
}

// ---- transpose of fixed-width neighbour lists (the by-source index of sng_list_bwd).  Entry p = i * k + s of the lists is
// keyed by its column idx[p] (padding, s >= cnt[i]: the sentinel n_total); the stable sort of (key, p) orders every source
// row's entries by p, i.e. by (target row, rank).
__global__ void __launch_bounds__(256) list_keys_kernel(const int* __restrict__ idx, const int* __restrict__ cnt, int64_t total, int k,
                                                       int n_total, int* __restrict__ key, int* __restrict__ pos) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(p / k), s = (int)(p - (int64_t)i * k);
        key[p] = s < __ldg(cnt + i) ? __ldg(idx + p) : n_total;
        pos[p] = (int)p;
    }
}

// col_tr[q] = local target row of sorted entry q, sel_q[p] = its position q (-1 for padding)
__global__ void __launch_bounds__(256) list_place_kernel(const int* __restrict__ key_sorted, const int* __restrict__ pos_sorted, int64_t total,
                                                        int k, int n_total, int* __restrict__ col_tr, int* __restrict__ sel_q) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
        const int p = __ldg(pos_sorted + q);
        const bool valid = __ldg(key_sorted + q) < n_total;
        if (valid) col_tr[q] = p / k;
        sel_q[p] = valid ? (int)q : -1;
    }
}

static int key_bits(int64_t n) { int b = 1; while ((1ll << b) <= n) ++b; return b; }      // keys are in [0, n]

static size_t sort_temp_bytes(int64_t total, int bits) {
    size_t t = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, total, 0, bits);
    return t;
}

}  // namespace sng

using namespace sng;

static size_t al256(size_t x) { return (x + 255) / 256 * 256; }

extern "C" size_t sng_graph_prepare_workspace_bytes(int64_t num_edges, int64_t n) {
    if (num_edges < 0 || n <= 0 || num_edges + n >= (1ll << 31)) return 0;
    const int64_t total = num_edges + n;
    return 7 * al256((size_t)total * 4) + al256(sort_temp_bytes(total, key_bits(n))) + 512;
}

extern "C" int sng_graph_prepare(const int64_t* edge_index, int64_t num_edges, int64_t n, int remove_self_loops,
                                 int32_t* rowptr_in, int32_t* col_in, float* inv_deg, int32_t* rowptr_out, int32_t* col_out,
                                 int32_t* col_in_shift, int32_t* tpos, int32_t* long_rows, int32_t* info, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    SNG_REQUIRE(n > 0 && num_edges >= 0 && num_edges + n < (1ll << 31), "sng_graph_prepare: graph too large for int32 CSR");
    SNG_REQUIRE((edge_index || num_edges == 0) && rowptr_in && col_in && inv_deg && info && workspace, "sng_graph_prepare: null pointer");
    SNG_REQUIRE(rowptr_out && col_out && col_in_shift, "sng_graph_prepare: by-source outputs missing");
    if (workspace_bytes < sng_graph_prepare_workspace_bytes(num_edges, n)) { set_error("sng_graph_prepare: workspace too small"); return SNG_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t total = num_edges + n;
    const int bits = key_bits(n);
    uint8_t* w = reinterpret_cast<uint8_t*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    int* key_dst = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* key_src = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* eid = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* key_sorted = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* perm_in = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* perm_out = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* inv_out = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* min_src = reinterpret_cast<int*>(w); w += 256;
    void* temp = w;
    size_t temp_bytes = sort_temp_bytes(total, bits);
    const int grid = grid_capped(total, 256, 16);
    if (cudaMemsetAsync(min_src, 0x7f, sizeof(int), st) != cudaSuccess) return check_launch("sng_graph_prepare memset");   // 0x7f7f7f7f
    if (cudaMemsetAsync(info, 0, 8 * sizeof(int), st) != cudaSuccess) return check_launch("sng_graph_prepare memset");
    if (cudaMemsetAsync(info + 2, 0xff, sizeof(int), st) != cudaSuccess) return check_launch("sng_graph_prepare memset");
    graph_keys_kernel<<<grid, 256, 0, st>>>(edge_index, num_edges, (int)n, remove_self_loops, key_dst, key_src, eid, min_src);
    if (int rc = check_launch("sng_graph_prepare keys")) return rc;
    if (cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_dst, key_sorted, eid, perm_in, total, 0, bits, st) != cudaSuccess)
        return check_launch("sng_graph_prepare sort by target");
    graph_ends_kernel<<<grid, 256, 0, st>>>(edge_index, num_edges, total, perm_in, 0, col_in, nullptr);
    const int rgrid = grid_capped(n + 1, 256, 16);
    graph_rowptr_kernel<<<rgrid, 256, 0, st>>>(key_sorted, total, (int)n, nullptr, rowptr_in);
    if (cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_src, key_sorted, eid, perm_out, total, 0, bits, st) != cudaSuccess)
        return check_launch("sng_graph_prepare sort by source");
    graph_ends_kernel<<<grid, 256, 0, st>>>(edge_index, num_edges, total, perm_out, 1, col_out, inv_out);
    graph_rowptr_kernel<<<rgrid, 256, 0, st>>>(key_sorted, total, (int)n, min_src, rowptr_out);
    graph_finish_kernel<<<grid, 256, 0, st>>>(rowptr_in, (int)n, inv_deg, col_in, col_in_shift, min_src, rowptr_out, col_out, perm_in,
                                             inv_out, tpos, long_rows, info);
    return check_launch("sng_graph_prepare");
}

extern "C" size_t sng_list_transpose_workspace_bytes(int64_t nq, int64_t k, int64_t n_total) {
    if (nq < 0 || k <= 0 || k > SNG_MAX_TOPK || n_total < 0 || n_total >= (1ll << 31) || nq * k >= (1ll << 31)) return 0;
    const int64_t total = nq * k;
    return 4 * al256((size_t)total * 4) + al256(sort_temp_bytes(total, key_bits(n_total))) + 256;
}

extern "C" int sng_list_transpose(const int32_t* idx, const int32_t* cnt, int64_t nq, int64_t k, int64_t n_total,
                                  int32_t* rowptr_tr, int32_t* col_tr, int32_t* sel_q, void* workspace, size_t workspace_bytes,
                                  void* stream) {
    const size_t need = sng_list_transpose_workspace_bytes(nq, k, n_total);
    SNG_REQUIRE(need > 0, "sng_list_transpose: bad nq=%lld / k=%lld / n_total=%lld", (long long)nq, (long long)k, (long long)n_total);
    SNG_REQUIRE(rowptr_tr && (nq == 0 || (idx && cnt && col_tr && sel_q)), "sng_list_transpose: null pointer");
    if (!workspace || workspace_bytes < need) { set_error("sng_list_transpose: workspace too small"); return SNG_ERR_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t total = nq * k;
    const int bits = key_bits(n_total);
    uint8_t* w = reinterpret_cast<uint8_t*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    int* key = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* pos = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* key_sorted = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    int* pos_sorted = reinterpret_cast<int*>(w); w += al256((size_t)total * 4);
    size_t temp_bytes = sort_temp_bytes(total, bits);
    if (total > 0) {
        const int grid = grid_capped(total, 256, 16);
        list_keys_kernel<<<grid, 256, 0, st>>>(idx, cnt, total, (int)k, (int)n_total, key, pos);
        if (int rc = check_launch("sng_list_transpose keys")) return rc;
        if (cub::DeviceRadixSort::SortPairs(w, temp_bytes, key, key_sorted, pos, pos_sorted, total, 0, bits, st) != cudaSuccess)
            return check_launch("sng_list_transpose sort");
        list_place_kernel<<<grid, 256, 0, st>>>(key_sorted, pos_sorted, total, (int)k, (int)n_total, col_tr, sel_q);
    }
    graph_rowptr_kernel<<<grid_capped(n_total + 1, 256, 16), 256, 0, st>>>(key_sorted, total, (int)n_total, nullptr, rowptr_tr);
    return check_launch("sng_list_transpose");
}
