/*
 * sng.h -- C ABI of libsng.so, the B200 (sm_100a) implementation of SNGNN's similarity-navigated
 *          aggregation hot path.
 *
 * The reference (MinhZou/SNGNN) is pure Python; it has no FFI.  What this library replaces are the
 * torch / torch_scatter / torch_sparse / PyG calls issued by the functions cited at each entry point
 * ("R:" = /root/reference).  The Python binding a maintainer adds is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (row-major, contiguous unless an `ld*`
 *     leading dimension in ELEMENTS is given); the library never allocates and keeps no reference
 *     after return, except work enqueued on `stream`
 *   - `stream` is a cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); all calls are
 *     asynchronous with respect to the host
 *   - sizes are int64_t; node / edge ids on the device are int32_t (N, E < 2^31)
 *   - return value: 0 ok, <0 error; sng_last_error() gives a thread-local message
 *   - feature rows handed to the edge kernels must be padded to a multiple of 4 floats (16-byte rows);
 *     padding columns must be zero (the host layer does this, sngnn_b200/functional.py)
 */
#ifndef SNG_H_
#define SNG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SNG_API __attribute__((visibility("default")))
#else
#define SNG_API
#endif

#define SNG_OK 0
#define SNG_ERR_ARG (-1)         /* bad argument */
#define SNG_ERR_UNSUPPORTED (-2) /* shape not supported by this build */
#define SNG_ERR_CUDA (-3)        /* CUDA runtime/driver error */
#define SNG_ERR_WORKSPACE (-4)   /* workspace too small */

#define SNG_MAX_TOPK 64          /* edge path lists: top_k <= 64 (larger: sng_edge_fwd_wide); top_k <= 0 means "select every edge" */
#define SNG_MAX_CHANNELS 512     /* padded row width c of sng_edge_fwd / _bwd, sng_edge_agg_bwd, sng_list_agg_fwd, sng_spmm_fwd,
                                    sng_pp_fuse_fwd / _bwd; wider rows return SNG_ERR_UNSUPPORTED */
#define SNG_KNN_MAX_TOPK 64      /* all-pairs builder sng_simknn_build (larger top_k: sng_simknn_wide_count / _select) */
#define SNG_SIMHIST_MAX_BINS 4096 /* sng_simhist_f16: two 32-bit sub-histograms of this many bins take half of its 64 KiB */

SNG_API int sng_version(void);
SNG_API const char* sng_last_error(void);
/* SM count / compute capability of the current device; fails (SNG_ERR_CUDA) when there is no GPU. */
SNG_API int sng_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Tests / experiments only: while enabled, the similarity-kNN build honours four environment overrides: SNG_KNN_CAND
 * (candidate slots per row), SNG_KNN_SEED_S / SNG_KNN_SEED_Q (seed stride / quantile) and SNG_KNN_NORETRY (no retry pass).
 * Off by default: the library then never reads the environment.  Returns the previous setting. */
SNG_API int sng_set_debug_env(int enabled);

/* ------------------------------------------------------------------------------------------------
 * K0  row normalisation: xhat = x / max(||x||_2, 1e-12)
 * replaces F.normalize(x, p=2, dim=-1) at R: models/models.py:122,238,325 and
 * R: SimGFAToolbox/dense.py:15,35,67,106,139,159.
 * Any of the three outputs may be NULL.  Output rows are zero-padded up to their leading dimension
 * (ld_f32 >= d, ld_f16 >= d); xhat_f16 is IEEE binary16 (the tensor-core operand of K1).
 */
SNG_API int sng_rownorm_f32(const float* x, int64_t n, int64_t d, int64_t ldx,
                    float* xhat_f32, int64_t ld_f32,
                    uint16_t* xhat_f16, int64_t ld_f16,
                    float* inv_norm, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2 (+K4)  fused edge-restricted similarity / selection / mean aggregation, forward
 * replaces SNConv_plus(_plus).message + PyG propagate(aggr='mean')
 *   R: models/models.py:132,139-158 (++), :239,244-263 (+), :326,331-334 (base, top_k <= 0)
 * and, when `wt` is given, the structural term and the beta blend of R: models/models.py:124-136 in the SAME pass.
 * For every target row i with in-edge list [rowptr[i], rowptr[i+1]) of CSR-by-target (sources in `col`,
 * kept in original edge-position order):
 *   s_e    = <h_i/r_i , h_j/r_j>,  r = max(||h||, 1e-12)
 *   S_i    = first min(top_k, deg) edges under (s desc, position asc), cut at the first s < thr
 *   out_1[i] = (1/max(deg_i,1)) * sum_{e in S_i} s_e * h[src_e]                 denominator 0 ('candidates', PyG aggr='mean')
 *   out_1[i] = (1/max(|S_i|,1)) * sum_{e in S_i} s_e * h[src_e]                 denominator 1 ('selected', sng_edge_fwd_denom)
 *              (a row that selects nothing outputs 0)
 *   wt == NULL:  out = out_1
 *   wt != NULL:  out_0[i] = sum_{e in-list of i} wt[src_e] + b_w ;  out = beta*out_0 + (1-beta)*out_1 (+ bias) ;
 *                diff (may be NULL) = out_0 - out_1 = d out / d beta.  Only valid when the in-list of every node equals its
 *                out-list (symmetric graph, src shift 0: info[2] of sng_graph_prepare); otherwise use sng_pp_fuse_fwd.
 * Saved for backward (all may be NULL in inference): sel_src [n,top_k] (source ids, rank order, -1 padded),
 * sel_w [n,top_k] (s_e), sel_cnt [n], sel_q [n,top_k] = tpos of the selected edges (needs tpos; input of sng_edge_bwd).
 * Degree dispatch (tables built once per graph by the caller, sngnn_b200/graph.py): rows with more than 32 in-edges are cut
 * into chunks of <= 32 consecutive edges.  chunk_tab [n_chunks, 4] int32 = (first edge position, edges, local row id, 0);
 * lrows [n_lrows] = those rows in ascending order, lrow_ptr [n_lrows + 1] = their chunk ranges (both used for c <= 32 only);
 * rows_hub [n_hub] = the rows with more than 1024 in-edges (used for 32 < c <= SNG_MAX_CHANNELS, where one general kernel
 * runs every other row).  workspace >= sng_edge_fwd_workspace_bytes(n_chunks, c, top_k) holds the per-chunk candidates.
 * n_chunks < 0 = tables unknown: the general kernel then runs every row.
 * Row sharding: the call covers target rows [row_offset, row_offset + n) of `h`, which holds ALL n_total nodes
 * (sources are arbitrary); rowptr / out / sel_* / the chunk tables are local to the shard, `col` holds global source ids.
 * inv_norm [n_total] is filled with 1/max(||h_i||, 1e-12) (a pre-pass of this call, skipped when inv_norm_ready != 0: the
 * caller -- sng_lin_norm_fwd -- already produced it) and is an input of the backward.
 */
SNG_API size_t sng_edge_fwd_workspace_bytes(int64_t n_chunks, int64_t c, int top_k);
SNG_API int sng_edge_fwd(const float* h, int64_t n_total, int64_t n, int64_t row_offset, int64_t c, int64_t ldh,
                 const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                 const int32_t* chunk_tab, int64_t n_chunks, const int32_t* lrows, const int32_t* lrow_ptr, int64_t n_lrows,
                 const int32_t* rows_hub, int64_t n_hub, void* workspace, size_t workspace_bytes,
                 int top_k, float thr, float* out, int64_t ldo,
                 int32_t* sel_src, float* sel_w, int32_t* sel_q, int32_t* sel_cnt, float* inv_norm, int inv_norm_ready,
                 const float* wt, int64_t ldw, const float* b_w, const float* beta, const float* bias, float* diff,
                 void* stream);
/* sng_edge_fwd with the mean's denominator as an argument (sng_edge_fwd = this with denominator 0, inv_denom NULL).
 * denominator: 0 = candidates (1/max(deg_i,1)), 1 = selected (1/max(|S_i|,1); needs top_k > 0), in inference and training,
 * with and without the fused epilogue (diff then holds out_0 - out_1 of this out_1).  inv_denom [n] (may be NULL; only with
 * denominator 1) receives the factor 1/max(|S_i|,1) each row was scaled by: pass it to sng_edge_bwd_denom, which then uses the
 * same floats.  Row sharding: inv_denom is indexed by LOCAL row, like out and sel_cnt. */
SNG_API int sng_edge_fwd_denom(const float* h, int64_t n_total, int64_t n, int64_t row_offset, int64_t c, int64_t ldh,
                 const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                 const int32_t* chunk_tab, int64_t n_chunks, const int32_t* lrows, const int32_t* lrow_ptr, int64_t n_lrows,
                 const int32_t* rows_hub, int64_t n_hub, void* workspace, size_t workspace_bytes,
                 int top_k, float thr, float* out, int64_t ldo,
                 int32_t* sel_src, float* sel_w, int32_t* sel_q, int32_t* sel_cnt, float* inv_norm, int inv_norm_ready,
                 const float* wt, int64_t ldw, const float* b_w, const float* beta, const float* bias, float* diff,
                 int denominator, float* inv_denom, void* stream);

/* K2b (+K4b) backward of the above w.r.t. h -- and, under the fused epilogue, w.r.t. wt and beta -- WITHOUT float atomics:
 * two gather passes (by target, then by source through the transpose index tpos), every sum in a fixed order, so the
 * result is bit-reproducible (closed form of SURVEY.md §3.4).  g = dL/dout [n, ldg] (dL/dout_1 when beta == NULL).
 *   top_k > 0: uses the saved lists (sel_src, sel_w, sel_q, sel_cnt);  top_k <= 0: every edge of the CSR (col, tpos).
 *   rowptr_out [n_total + 1] / col_out = CSR by (source - src_shift) of the same edges, num_edges of them.
 *   beta != NULL: g is scaled by (1 - beta) for the aggregation; dbeta (may be NULL) = sum(diff * g) (needs diff, partials);
 *                 dwt (may be NULL) [n, lddw] = beta * sum over out-edges (j -> i) of g_i = dL/dwt.
 * Workspaces (caller-allocated, contents irrelevant): coef [2 * num_edges] floats, dn_target [n, ld], partials [SNG_PARTIALS].
 * chunk_tab_out / lrows_out / lrow_ptr_out: the degree tables of sng_edge_fwd built over the BY-SOURCE CSR (rows with more
 * than 32 out-edges cut into <= 32-edge chunks; lrows_out holds true source ids), chunk_partials [n_chunks_out, 3, 4*ceil_pow2(c/4)]
 * floats; n_chunks_out < 0 = tables unknown (the unstaged source pass then runs every row).
 * Output dh [n_total, ld]: every row is written.
 * Row sharding (the convention of sng_edge_fwd): the call covers target rows [row_offset, row_offset + n) of `h`, which holds
 * ALL n_total nodes, as does inv_norm; g, diff, the selection lists, rowptr / col / tpos and the by-source CSR are local to the
 * shard -- the by-source CSR holds only the shard's in-edges, over all source rows, with targets as LOCAL ids.  dh is then
 * this shard's CONTRIBUTION to dL/dh of every node (the map to dh is linear: the contributions of the shards add, e.g. in a
 * reduce-scatter across ranks), dbeta its part of dL/dbeta.  n = 0 gives a zero contribution.  dwt needs a call over all rows
 * (row_offset = 0, n = n_total); a row shard assembles dL/dwt from g elsewhere.  row_offset = 0, n = n_total: the whole graph. */
#define SNG_PARTIALS 4096
SNG_API int sng_edge_bwd(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                 int64_t c, int64_t ld, int64_t ldg,
                 const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                 const int32_t* rowptr_out, const int32_t* col_out, int64_t src_shift, int64_t num_edges,
                 int top_k, const int32_t* sel_src, const float* sel_w, const int32_t* sel_q, const int32_t* sel_cnt,
                 const float* beta, const float* diff, int64_t lddiff, float* dbeta,
                 float* coef, float* dn_target, float* partials, float* dh, float* dwt, int64_t lddw,
                 const int32_t* chunk_tab_out, int64_t n_chunks_out, const int32_t* lrows_out, const int32_t* lrow_ptr_out,
                 int64_t n_lrows_out, float* chunk_partials, void* stream);
/* sng_edge_bwd with the forward's per-row factor (sng_edge_bwd = this with inv_denom NULL).  inv_denom NULL: 1/max(deg_i,1)
 * from rowptr (denominator 0); else inv_denom [n] as sng_edge_fwd_denom wrote it (denominator 1, needs top_k > 0), per LOCAL
 * row under row sharding.  Everything else, the fused epilogue included, as sng_edge_bwd. */
SNG_API int sng_edge_bwd_denom(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                 int64_t c, int64_t ld, int64_t ldg,
                 const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                 const int32_t* rowptr_out, const int32_t* col_out, int64_t src_shift, int64_t num_edges,
                 int top_k, const int32_t* sel_src, const float* sel_w, const int32_t* sel_q, const int32_t* sel_cnt,
                 const float* beta, const float* diff, int64_t lddiff, float* dbeta,
                 float* coef, float* dn_target, float* partials, float* dh, float* dwt, int64_t lddw,
                 const int32_t* chunk_tab_out, int64_t n_chunks_out, const int32_t* lrows_out, const int32_t* lrow_ptr_out,
                 int64_t n_lrows_out, float* chunk_partials, const float* inv_denom, void* stream);

/* Per-edge selection form of sng_edge_fwd_denom / sng_edge_bwd_denom for top_k > SNG_MAX_TOPK (any top_k: every value
 * >= max_deg selects the same set, so callers clamp to that).  The selection rule is the same, S_i = {e : s_e >= thr and
 * rank_i(e) < top_k} with ranks by (s desc, position asc); it is saved as one flag per in-edge instead of [n, top_k] lists.
 * A row with deg <= top_k selects {e : s_e >= thr} in the aggregation pass itself.  A row with deg > top_k (only rows with
 * more than 32 in-edges can be: lrows, when given, lists them) is cut first, once: one block per row scores its edges,
 * radix-selects the top_k-th key and flags the winners, ties at the cut going to the lowest positions.  The aggregation reads
 * those flags and weights edge e by s_e when selected, with the denominator 0 (1/max(deg_i,1)) or 1 (1/max(|S_i|,1), written
 * to inv_denom [n] when given).
 * num_edges = rowptr[n] (edges of the call's rows), max_deg >= every row's in-degree: no row is cut when top_k >= max_deg.
 * sel_flag [num_edges] uint8 (CSR-by-target positions): required when top_k < max_deg or train != 0; with train != 0 every
 * edge's flag is written (the input of sng_edge_bwd_wide).  workspace >= sng_edge_fwd_wide_workspace_bytes(n_chunks, c,
 * num_edges, max_deg) (may be 0).  Other arguments, the fused epilogue and row sharding as sng_edge_fwd_denom; no selection
 * lists are written. */
SNG_API size_t sng_edge_fwd_wide_workspace_bytes(int64_t n_chunks, int64_t c, int64_t num_edges, int64_t max_deg);
SNG_API int sng_edge_fwd_wide(const float* h, int64_t n_total, int64_t n, int64_t row_offset, int64_t c, int64_t ldh,
                 const int32_t* rowptr, const int32_t* col, int64_t num_edges,
                 const int32_t* chunk_tab, int64_t n_chunks, const int32_t* lrows, const int32_t* lrow_ptr, int64_t n_lrows,
                 const int32_t* rows_hub, int64_t n_hub, void* workspace, size_t workspace_bytes,
                 int top_k, int64_t max_deg, float thr, float* out, int64_t ldo, uint8_t* sel_flag, int train,
                 float* inv_norm, int inv_norm_ready,
                 const float* wt, int64_t ldw, const float* b_w, const float* beta, const float* bias, float* diff,
                 int denominator, float* inv_denom, void* stream);
/* Backward of sng_edge_fwd_wide: sng_edge_bwd_denom's two gather passes over every in-edge of the CSR (col, tpos), an edge
 * counting only when sel_flag (the forward's, written with train != 0) marks it selected -- also when its score is 0.
 * inv_denom: the forward's factors (denominator 1) or NULL (1/max(deg_i,1)).  No float atomics, bit-reproducible; workspaces,
 * fused epilogue and row sharding as sng_edge_bwd. */
SNG_API int sng_edge_bwd_wide(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                 int64_t c, int64_t ld, int64_t ldg,
                 const int32_t* rowptr, const int32_t* col, const int32_t* tpos,
                 const int32_t* rowptr_out, const int32_t* col_out, int64_t src_shift, int64_t num_edges,
                 const uint8_t* sel_flag, const float* inv_denom,
                 const float* beta, const float* diff, int64_t lddiff, float* dbeta,
                 float* coef, float* dn_target, float* partials, float* dh, float* dwt, int64_t lddw,
                 const int32_t* chunk_tab_out, int64_t n_chunks_out, const int32_t* lrows_out, const int32_t* lrow_ptr_out,
                 int64_t n_lrows_out, float* chunk_partials, void* stream);

/* Gather form of the backward of sng_list_agg_fwd (explicit neighbour lists: the all-pairs mode) -- the same two passes and
 * kernels as sng_edge_bwd, no float atomics, bit-reproducible.  Any list width top_k >= 1 (n * top_k < 2^31): lists longer
 * than 32 are walked from memory by pass T.  The lists are those of sng_simknn_build / _wide_select: idx / sim [n, top_k]
 * (global column ids in rank order, sim = cosine of h_i and h_j), cnt [n]; entries t < cnt[i] <= top_k are node ids, the
 * rest is padding.  inv_denom [n] = the forward's per-row factor (1 / denominator).  g = dL/dout [n, ldg].
 * sel_q / rowptr_tr / col_tr: the transpose of the lists (sng_list_transpose), the by-source CSR over all n_total nodes.
 * chunk_tab / lrows / lrow_ptr: the degree tables of sng_edge_bwd over rowptr_tr (source rows with more than 32 list entries
 * cut into <= 32-entry chunks), chunk_partials as there; n_chunks < 0 = tables unknown (used for c <= 32 only).
 * Workspaces (contents irrelevant): coef [2 * rowptr_tr[n_total]] floats, dn_target [n, ld].  Output dh [n_total, ld]: every
 * row is written.  Row sharding as sng_edge_bwd: the lists are rows [row_offset, row_offset + n) of `h` (all n_total nodes,
 * as is inv_norm), dh is their CONTRIBUTION to dL/dh of every node; n = 0 gives a zero contribution. */
SNG_API int sng_list_bwd(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                 int64_t c, int64_t ld, int64_t ldg,
                 int top_k, const int32_t* idx, const float* sim, const int32_t* cnt, const float* inv_denom,
                 const int32_t* sel_q, const int32_t* rowptr_tr, const int32_t* col_tr,
                 float* coef, float* dn_target, float* dh,
                 const int32_t* chunk_tab, int64_t n_chunks, const int32_t* lrows, const int32_t* lrow_ptr, int64_t n_lrows,
                 float* chunk_partials, void* stream);

/* Transpose of fixed-width neighbour lists idx [nq, k] / cnt [nq] (entries t < cnt[i] are column ids in [0, n_total), the
 * rest padding) into the by-source index of sng_list_bwd: rowptr_tr [n_total + 1], col_tr [nq * k capacity; rowptr_tr[n_total]
 * used] = the LOCAL row i of every entry whose column is the source, ordered by (i, rank) within a source -- a stable radix
 * sort (cub::DeviceRadixSort), so the result is a pure function of the lists; sel_q [nq, k] = position of entry (i, t) in
 * col_tr (-1 for padding).  workspace >= sng_list_transpose_workspace_bytes(nq, k, n_total) (0 = shape rejected). */
SNG_API size_t sng_list_transpose_workspace_bytes(int64_t nq, int64_t k, int64_t n_total);
SNG_API int sng_list_transpose(const int32_t* idx, const int32_t* cnt, int64_t nq, int64_t k, int64_t n_total,
                       int32_t* rowptr_tr, int32_t* col_tr, int32_t* sel_q, void* workspace, size_t workspace_bytes, void* stream);

/* Scatter form of the backward (float atomics, so not bit-reproducible).  No layer of the package calls it since sng_list_bwd
 * covers explicit neighbour lists; it is kept as the comparison baseline of the timing scripts (scripts/k2_time.py,
 * scripts/shard_bwd_time.py, scripts/allpairs_bwd_time.py).
 * Pass 1 scatters into the two zero-initialised accumulators dval, dnrm [n_total, c];
 * pass 2 writes dh [n_total, c] = dval + (dnrm - n (n . dnrm)) / r.   `g` = dL/dout_1 [n, c].
 * top_k > 0: uses the saved selection lists (inv_denom[i] = 1/max(deg_i,1));
 * top_k <= 0: iterates the CSR (every edge selected).  inv_norm [n_total] = the array the forward filled
 * (or sng_rownorm_f32's inv_norm output for selection lists that did not come from the edge forward).
 * Row sharding: the call covers target rows [row_offset, row_offset + n) of `h` (all n_total nodes); g, the lists, inv_denom
 * and rowptr are local to the shard.  dh is then this shard's CONTRIBUTION to dL/dh of every node -- the map
 * (dval, dnrm) -> dh is linear, so the per-shard results simply add (reduce-scatter across ranks). */
SNG_API int sng_edge_agg_bwd(const float* h, const float* inv_norm, const float* g, int64_t n_total, int64_t n, int64_t row_offset,
                     int64_t c, int64_t ld,
                     const int32_t* rowptr, const int32_t* col,
                     int top_k, const int32_t* sel_src, const float* sel_w, const int32_t* sel_cnt,
                     const float* inv_denom,
                     float* dval, float* dnrm, float* dh, void* stream);

/* Aggregation from a selection list only (all-pairs mode: list = emitted kNN):
 * out[i] = inv_denom[i] * sum_{t<cnt[i]} w[i,t] * h[src[i,t]]. */
SNG_API int sng_list_agg_fwd(const float* h, int64_t n_rows, int64_t c, int64_t ldh,
                     int list_k, const int32_t* sel_src, const float* sel_w, const int32_t* sel_cnt,
                     const float* inv_denom, float* out, int64_t ldo, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K3  CSR x dense gather-reduce ("mean-aggregation SpMM")
 *   out[i] = rowscale[i] * sum_{e in row i} val[e] * x[col[e]]  + bias
 * val / rowscale / bias may be NULL (1 / 1 / 0).  Replaces torch.sparse mm at R: models/models.py:130
 * (A @ W^T), its transpose in backward, and scatter(reduce='mean') on an emitted kNN CSR.
 */
SNG_API int sng_spmm_fwd(const float* x, int64_t n_rows, int64_t c, int64_t ldx,
                 const int32_t* rowptr, const int32_t* col, const float* val,
                 const float* rowscale, const float* bias,
                 float* out, int64_t ldo, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K4  SNGNN++ fusion: out0 = A @ Wt + b_w (gather of Wt rows over OUT-neighbours), then
 *     out = beta*out0 + (1-beta)*out1 (+ bias).   R: models/models.py:124-136.
 * `beta` is a device scalar (the learnable parameter).  out0 is written too (needed for dL/dbeta).
 */
SNG_API int sng_pp_fuse_fwd(const float* wt, int64_t n, int64_t c, int64_t ld,
                    const int32_t* rowptr_out, const int32_t* col_out,
                    const float* b_w, const float* beta, const float* out1, const float* bias,
                    float* out0, float* out, void* stream);

/* dbeta = sum((out0 - out1) * g), summed in a fixed order (bit-reproducible); partials = workspace of SNG_PARTIALS floats. */
SNG_API int sng_pp_beta_grad(const float* out0, const float* out1, const float* g, int64_t numel,
                     float* dbeta, float* partials, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Mean negative log-likelihood of the rows with a label in [0, c) (a masked row carries the label -1), forward and
 * backward, fixed-order reductions.  replaces F.nll_loss(out[mask], y[mask]) at R: train.py:81,99,113.
 *   fwd: loss (device float) = -(1/count) sum_i logp[i, y[i]], count (device float) = labelled rows; partials = SNG_PARTIALS floats.
 *   bwd: dlogp [n, ld] = -gscale/count at (i, y[i]), 0 elsewhere (gscale = dL/dloss, a device scalar).
 */
SNG_API int sng_nll_loss_fwd(const float* logp, int64_t n, int64_t c, int64_t ld, const int64_t* y, float* loss, float* count,
                     float* partials, void* stream);
SNG_API int sng_nll_loss_bwd(int64_t n, int64_t c, int64_t ld, const int64_t* y, const float* gscale, const float* count, float* dlogp,
                     void* stream);

/* ------------------------------------------------------------------------------------------------
 * ReLU + BatchNorm1d over the rows of a shard (R: models/models.py:81-84 `x = F.relu(conv(x)); x = self.bns[i](x)`), with the
 * batch statistics taken over all n_total rows of every shard: each rank computes its shard's sums, the caller all-reduces the
 * FP64 [2, c] sums, every rank applies.  z [n, ldz] = the conv output (pre-activation), a = max(z, 0); 1 <= c <= SNG_MAX_CHANNELS.
 * Sums are FP64 with per-CTA partials added in a fixed order (no atomics): bit-reproducible on a given device.  An empty shard
 * (n = 0) writes zero sums.  workspace >= sng_bn_workspace_bytes(n, c) (0 = c rejected).
 *   sng_bn_fwd_stats: sums [2, c] = (sum_i a_i, sum_i a_i^2) over this shard.
 *   sng_bn_fwd_apply: y [n, ldy] = gamma (a - mu) rstd + beta.  sums != NULL (training): the global sums over n_total rows give
 *     mu = S1 / N and rstd = 1 / sqrt(S2 / N - mu^2 + eps) (biased variance, as torch normalises), written to mean / rstd [c];
 *     sums == NULL (eval): mean / rstd are INPUTS (running_mean, 1 / sqrt(running_var + eps)); n_total and eps are unused.
 *   sng_bn_bwd_stats: sums [2, c] = (sum_i g_i, sum_i g_i ahat_i) over this shard, ahat = (a - mean) rstd recomputed from z.
 *   sng_bn_bwd_apply: dz [n, lddz] = 1[z > 0] gamma rstd (g - S1 / N - ahat S2 / N) with the global backward sums over n_total rows;
 *     sums == NULL (eval-mode statistics, constants): dz = 1[z > 0] gamma rstd g.
 *   The global backward sums are also dL/dbeta (S1) and dL/dgamma (S2).
 */
SNG_API size_t sng_bn_workspace_bytes(int64_t n, int64_t c);
SNG_API int sng_bn_fwd_stats(const float* z, int64_t n, int64_t c, int64_t ldz, double* sums, void* workspace, size_t workspace_bytes,
                     void* stream);
SNG_API int sng_bn_fwd_apply(const float* z, int64_t n, int64_t c, int64_t ldz, const double* sums, int64_t n_total, double eps,
                     const float* gamma, const float* beta, float* mean, float* rstd, float* y, int64_t ldy, void* stream);
SNG_API int sng_bn_bwd_stats(const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, const float* mean,
                     const float* rstd, double* sums, void* workspace, size_t workspace_bytes, void* stream);
SNG_API int sng_bn_bwd_apply(const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, const double* sums,
                     int64_t n_total, const float* gamma, const float* mean, const float* rstd, float* dz, int64_t lddz, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Counter-based dropout over the rows [row_offset, row_offset + n) of a layer of logical width c (R: models/models.py:85
 * `x = self.dropout(x)`, optionally fused with the ReLU before it).  The mask depends only on (seed, call, global row, channel):
 * element e = (row_offset + i) c + j keeps iff (w >> 8) >= round(p 2^24), w = word (e & 3) of Philox4x32-10 (Random123 constants)
 * with key (seed lo, seed hi) and counter (e >> 2 lo, e >> 2 hi, call lo, call hi).  Row shards of any split therefore draw the
 * masks of the whole layer, and the backward regenerates the mask: no [n, c] mask is stored.  s = 1.0f / (1.0f - p) in FP32.
 *   sng_row_dropout_fwd: y [n, ldy] = keep ? a s : 0, a = relu ? max(z, 0) : z (a select: p = 1 gives zeros).
 *   sng_row_dropout_bwd: dz [n, lddz] = keep && (!relu || z > 0) ? g s : 0; z is read only with relu (else it may be NULL).
 * 0 <= p <= 1, c >= 1, every ld >= c, n >= 0 (n = 0 launches nothing), row_offset >= 0, (row_offset + n) c < 2^63 - 4.
 * Rows whose pointers and strides are 16-byte aligned with c % 4 == 0 take float4 accesses; others a scalar path.
 */
SNG_API int sng_row_dropout_fwd(const float* z, int64_t n, int64_t c, int64_t ldz, int64_t row_offset, uint64_t seed, uint64_t call,
                     float p, int relu, float* y, int64_t ldy, void* stream);
SNG_API int sng_row_dropout_bwd(const float* z, const float* g, int64_t n, int64_t c, int64_t ldz, int64_t ldg, int64_t row_offset,
                     uint64_t seed, uint64_t call, float p, int relu, float* dz, int64_t lddz, void* stream);

/* ------------------------------------------------------------------------------------------------
 * lin + bias + 1/norm in one pass (SURVEY.md §8(f) 2):  h [n, cp] = x W^T + b with cp = 4 * ceil(c / 4) zero-padded channels,
 * inv_norm[i] = 1 / max(||h_i||, 1e-12).  replaces `x = self.lin(x); norm = F.normalize(x)` at R: models/models.py:121-122,
 * 237-238, 324-325 (FP32 FMA; supported when cp is a power of two in [4, 128] and f * cp <= 24576 -- sng_lin_norm_supported --
 * otherwise the caller keeps the library GEMM and lets sng_edge_fwd compute inv_norm).  x [n, ldx], w [c, ldw], bias [c] or NULL.
 */
SNG_API int sng_lin_norm_supported(int64_t f, int64_t c);
SNG_API int sng_lin_norm_fwd(const float* x, int64_t n, int64_t f, int64_t ldx, const float* w, int64_t c, int64_t ldw, const float* bias,
                     float* h, float* inv_norm, void* stream);

/* Weight / bias gradient of the same layer: dw [c, lddw] = g^T x, db [c] (or NULL) = column sums of g, for g [n, ldg] (the first c
 * columns are used), x [n, ldx].  One streaming pass over g and x, per-CTA partials summed in a fixed order (bit-reproducible).
 * replaces the autograd GEMMs of `self.lin` (R: models/models.py:121).  workspace >= sng_lin_bwd_workspace_bytes(n, f, c).
 * Supported for f <= 128 and ceil(f/4) * ceil(c/4) <= 256 (sng_lin_bwd_supported); wider layers keep the library GEMM. */
SNG_API int sng_lin_bwd_supported(int64_t f, int64_t c);
SNG_API size_t sng_lin_bwd_workspace_bytes(int64_t n, int64_t f, int64_t c);
SNG_API int sng_lin_bwd(const float* g, int64_t ldg, const float* x, int64_t ldx, int64_t n, int64_t f, int64_t c, float* dw, int64_t lddw,
                float* db, void* workspace, size_t workspace_bytes, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Data formats either side of the path.
 * sng_knn_to_csr: fixed-width neighbour lists (idx / sim [nq, top_k], cnt [nq], the outputs of sng_simknn_build or the saved
 *   lists of sng_edge_fwd) -> CSR: rowptr [nq+1] = exclusive scan of cnt (cub::DeviceScan), col [sum cnt] in rank order,
 *   val (may be NULL) = the similarities.  This is "then emits CSR neighbour lists" of the all-pairs builder.
 * sng_pp_fuse_bwd: backward of sng_pp_fuse_fwd: dbeta = sum((out0 - out1) g) (fixed order), g0 = beta g, dout1 = (1 - beta) g,
 *   dwt [n, c] = A^T g0 (row t gathers g0 over col_in_shift of t's in-edges).  Rows contiguous (ld == c).
 * sng_segment_mean: out[s] = mean of val[e] over seg[e] == s (0 for an empty segment), FP64 accumulation;
 *   replaces torch_scatter.scatter_mean at R: SimGFAToolbox/dense.py:163.  workspace >= 12 * n_seg + 256 bytes.
 */
SNG_API size_t sng_knn_to_csr_workspace_bytes(int64_t nq);
SNG_API int sng_knn_to_csr(const int32_t* idx, const float* sim, const int32_t* cnt, int64_t nq, int top_k, int32_t* rowptr, int32_t* col,
                   float* val, void* workspace, size_t workspace_bytes, void* stream);
SNG_API int sng_pp_fuse_bwd(const float* out0, const float* out1, const float* g, const float* beta, int64_t n, int64_t c, int64_t ld,
                    const int32_t* rowptr_in, const int32_t* col_in_shift, float* dbeta, float* partials, float* g0, float* dout1,
                    float* dwt, void* stream);
SNG_API int sng_segment_mean(const float* val, const int32_t* seg, int64_t num, int64_t n_seg, float* out, void* workspace,
                     size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SDDMM cosine at given edges: s[e] = <xhat[a[e]], xhat[b[e]]> (xhat already normalised, FP32).
 * replaces index_select x2 + mul + sum at R: SimGFAToolbox/dense.py:152-164 and the per-node mm of :53-58.
 */
SNG_API int sng_sddmm_dot(const float* xhat, int64_t n, int64_t d, int64_t ld,
                  const int32_t* a, const int32_t* b, int64_t num_edges, float* s, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Toolbox helpers (Sim-GFA metrics that are not neighbour selection).
 * sng_gemm_nt_f16: out[i, j] = row_scale[i] col_scale[j] sum_k A[i, k] B[j, k] on the tensor cores (tcgen05 / TMEM / TMA), FP16
 *   operands (row-major, lda / ldb % 8 == 0, 16-byte aligned), FP32 accumulation and output; scales may be NULL.  The N x N
 *   producer of the *_small metrics that RETURN the matrix (R: SimGFAToolbox/dense.py:138-149): with A = [hi | hi | lo],
 *   B = [hi | lo | hi] of the FP16 split x-hat = hi + lo the product equals the FP32 one to ~2^-22; and of the
 *   adjacency-as-features metrics (R: SimGFAToolbox/sparse.py:8-41): 0/1 columns are exact in FP16, the accumulators hold
 *   exact common-neighbour counts and the scales apply 1 / (|a_i| |a_j|).
 * sng_simhist_f16: counts[b] += number of ORDERED pairs i != j (i, j < n) whose score s = sum_k A[i, k] B[j, k] falls in bin b
 *   of [lo, hi) cut into `bins` equal bins, without the n x n matrix (tcgen05 contraction, binning epilogue).  s is
 *   clamped to [-1, 1]; bin = floor((s - lo) * bins / (hi - lo)), s == hi goes into the last bin (numpy.histogram), scores
 *   outside [lo, hi] are not counted.  With A = [hi | hi | lo], B = [hi | lo | hi] of the FP16 split of x-hat (as for
 *   sng_gemm_nt_f16) this is the distribution of the off-diagonal cosines of R: SimGFAToolbox/dense.py:144-149.  Each
 *   unordered pair of 128-row tiles is scored once: row tile I pairs with (I + s) mod T, s = 0 .. floor(T / 2), T = ceil(n
 *   / 128), the pair at s = T / 2 (T even) only for I < T / 2.  Only row tiles [tile_lo, tile_hi) are run (shards, split
 *   calls; an empty range adds nothing), so the counts of a split add up to those of [0, T).  Integer counting: the result
 *   is the same bits whatever the split.  counts [bins] uint64 is zeroed by the caller.  Requires 0 < n < 2^31,
 *   1 <= bins <= SNG_SIMHIST_MAX_BINS, lo < hi finite, lda / ldb % 8 == 0, 16-byte aligned operands.
 * sng_sparse_col_cos: the same cosine between two COLUMNS of a CSC matrix (sorted, duplicate-free indices) at given column
 *   pairs, by merging the two index lists -- the edge metrics of R: SimGFAToolbox/sparse.py:44-119 without densifying.
 * sng_class_sums_f64: sums[c, :] += sum_{i: y[i]==c} xhat[i, :] and counts[c] += |class c| (both zero-initialised,
 *   FP64); y may be NULL when num_classes == 1.  Every "sum over all pairs" metric is <S_a, S_b>
 *   (R: SimGFAToolbox/dense.py:9-30, 104-130, 167-179 materialise N x N blocks for the same sums).
 */
SNG_API int sng_gemm_nt_f16(const uint16_t* a, int64_t lda, const uint16_t* b, int64_t ldb, int64_t m, int64_t n, int64_t k,
                    const float* row_scale, const float* col_scale, float* out, int64_t ldo, void* stream);
SNG_API int sng_simhist_f16(const uint16_t* a, int64_t lda, const uint16_t* b, int64_t ldb, int64_t n, int64_t k, int64_t tile_lo,
                    int64_t tile_hi, float lo, float hi, int bins, uint64_t* counts, void* stream);
SNG_API int sng_sparse_col_cos(const int32_t* indptr, const int32_t* indices, const float* data, const float* inv_norm,
                       const int32_t* a, const int32_t* b, int64_t num_pairs, float* s, void* stream);
SNG_API int sng_class_sums_f64(const float* xhat, const int32_t* y, int64_t n, int64_t d, int64_t ld, int num_classes,
                       double* sums, double* counts, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Graph preparation (once per edge_index; the reference redoes it every forward in Python/PyG:
 * R: models/models.py:117-127 (++), :234-236 (+), :323 (base)).
 *   edge_index [2, num_edges] int64 (row 0 = sources, row 1 = targets), n nodes.
 *   N self loops are appended at the END; with remove_self_loops every src == dst edge is then dropped.
 *   rowptr_in [n+1], col_in [num_edges + n capacity]: CSR by target, sources in original edge-position order (the
 *   tie-break order of the selection); inv_deg [n] = 1/max(in-degree, 1).
 *   rowptr_out [n+1], col_out [capacity] = CSR by (src - min src) holding the targets (A of R: models.py:124-127),
 *   col_in_shift [capacity] = col_in - min src (its transpose).
 *   tpos [capacity] (may be NULL) = position of by-target edge p in the by-source arrays (the transpose
 *   index of sng_edge_bwd).  long_rows [n] (may be NULL): local ids of the rows with 32 < in-degree <= 1024 from the
 *   front, of the rows with in-degree > 1024 from the back, in no particular order (the caller sorts them and derives the
 *   chunk tables of sng_edge_fwd).
 *   info (device int32[8]) = {number of kept edges E', min src, 1 if every in-list equals the out-list and min src == 0,
 *   rows in (32, 1024], rows > 1024, max in-degree, 0, 0}.  Only the first E' entries of col_* / tpos
 *   are meaningful.  The two stable sorts are cub::DeviceRadixSort (a library sort); everything else is kernels of this library.
 */
SNG_API size_t sng_graph_prepare_workspace_bytes(int64_t num_edges, int64_t n);
SNG_API int sng_graph_prepare(const int64_t* edge_index, int64_t num_edges, int64_t n, int remove_self_loops,
                      int32_t* rowptr_in, int32_t* col_in, float* inv_deg,
                      int32_t* rowptr_out, int32_t* col_out, int32_t* col_in_shift,
                      int32_t* tpos, int32_t* long_rows,
                      int32_t* info, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K1  all-pairs similarity-kNN builder (tcgen05 / TMA / TMEM), never materialising the N x N matrix.
 *   xq_f16  [nq , ldh]  normalised query rows  (FP16, zero padded, ldh % 8 == 0, 16*ceil(d/16) <= ldh <= 16*ceil(d/16) + 64,
 *                       16-byte aligned; d <= 4096 -- beyond d ~ 640 the query block is streamed instead of resident)
 *   xall_f16[n  , ldh]  normalised database rows
 *   query row r is global node q_offset + r (used for remove_self and for sharding by query rows)
 * Stage 1 (tensor cores; a seed pass over a column sample first sets every row's starting threshold) keeps, per query
 * row, the `cand` best FP16-scored column TRIPLES {c, c+1, c+2} (two columns when c % 32 == 30), cand >= top_k + margin.
 * Stage 2 rescores their columns in FP32 (xq_f32 / xall_f32, leading dim ld32 % 4 == 0, zero padded), orders them by
 * (sim desc, index asc), applies thr / top_k and PROVES exactness: a row whose k-th exact score is not clear
 * of the best possible score of any dropped column is flagged.
 * Flagged rows first get a RETRY pass (a second tensor-core pass over just those rows, with long candidate lists and a
 * much lower starting threshold); only rows that fail that proof too are recomputed by an exact FP32 scan (stage 3).
 * The retry pass is sized from the number of flagged rows: the call reads that 4-byte count back and synchronises `stream`
 * once, after stage 2 (nothing else in the library synchronises); on a stream that is being captured it launches one retry
 * round of at most 16 K rows with the count on the device instead.  All-zero query rows are answered by rule in stage 2.
 * Outputs: idx [nq, top_k] int32 (-1 padded), sim [nq, top_k], cnt [nq]; n_fallback (device int32) counts
 * rows that needed stage 3, n_retry (device int32, may be NULL) rows that needed the retry pass.
 * Replaces (as "the reference rule on the complete graph", SURVEY.md §0) the selection of
 * R: models/models.py:145-156 and the blocked X X^T of R: SimGFAToolbox/dense.py:17-27.
 */
SNG_API size_t sng_simknn_workspace_bytes(int64_t nq, int64_t n, int64_t d, int top_k);
SNG_API int sng_simknn_build(const uint16_t* xq_f16, const uint16_t* xall_f16, int64_t ldh,
                     const float* xq_f32, const float* xall_f32, int64_t ld32,
                     int64_t nq, int64_t q_offset, int64_t n, int64_t d,
                     int top_k, float thr, int remove_self,
                     int32_t* idx, float* sim, int32_t* cnt, int32_t* n_fallback, int32_t* n_retry,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Stage 1 only (profiling / tests): cand_idx [nq, lists, cand] = first column of a kept column triple (-1 = empty slot),
 * cand_val = the triple's largest FP16 score, cand_min [nq, lists] = upper bound of every score that list dropped (-inf if
 * it dropped nothing above thr_lo); lists = column splits (one list per row and split).  force_ew in {0,1,2,4} picks the
 * epilogue warps per TMEM lane quarter (0 = auto; 4 = the four-accumulator split mode, K <= 128), force_nsplit > 0 the
 * number of column splits; *lists_out receives lists (size the outputs for lists * cand <= 192 slots per row).
 * seeds (may be NULL) = output of sng_simknn_seed with the same seed_stride: every row then starts pruning at the
 * seed_q-th largest of its 16 group maxima instead of thr_lo.
 * sweep_phase (may be NULL) = [column splits] int32, zero-initialised by the caller: the CTAs of a launch use it to start
 * their sweep over the database tiles where the other resident CTAs currently are, which keeps the tiles in L2. */
SNG_API int sng_simknn_stage1(const uint16_t* xq_f16, const uint16_t* xall_f16, int64_t ldh,
                      int64_t nq, int64_t q_offset, int64_t n, int64_t d,
                      int cand, float thr_lo, int remove_self,
                      int32_t* cand_idx, float* cand_val, float* cand_min,
                      int force_ew, int force_nsplit, int* lists_out,
                      const float* seeds, int seed_q, int seed_stride, int32_t* sweep_phase, void* stream);

/* Seed pass only (profiling / tests): the same tensor-core pipeline over every seed_stride-th database row with a
 * branch-free epilogue; seeds_out [nq, 16] = maxima of the row's FP16 scores over 16 disjoint groups of sampled columns
 * (group of sample column c: ((c >> 8) & 1) * 8 + ((c & 255) >> 5)).  sng_simknn_build runs it first (when the plan
 * says so) to start every row's pruning threshold near its final value. */
SNG_API int sng_simknn_seed(const uint16_t* xq_f16, const uint16_t* xall_f16, int64_t ldh,
                    int64_t nq, int64_t n, int64_t d, int seed_stride, int force_ew,
                    float* seeds_out, void* stream);

/* Launch plan of sng_simknn_build for a shape: out8 = {epilogue warps per lane quarter, candidate slots per list,
 * column splits, seed stride (0 = no seed pass), seed quantile, B ring stages, K blocks of 64, lists per row}. */
SNG_API int sng_simknn_plan(int64_t nq, int64_t n, int64_t d, int top_k, int32_t* out8);

/* Wide all-pairs build: any top_k >= 1 (int64; 2^40 = every column with cosine >= thr), the selection rule of
 * sng_simknn_build.  Lists have k_eff = min(top_k, n - remove_self) entries: idx / sim [nq, k_eff], cnt [nq]; nq * k_eff
 * must be < 2^31.  Query rows [q_offset, q_offset + nq) must be rows of the database.  Two calls on the same workspace
 * (>= sng_simknn_wide_workspace_bytes(nq, n, d, top_k); the second call reads what the first left there):
 *   sng_simknn_wide_count: seed pass (its stride chosen from k_eff) -> every row's emission threshold T_i -> a tensor-core
 *     sweep counting the columns whose FP16 score is >= T_i -> offsets [nq + 1] int64 = their exclusive scan (a row with more
 *     than 16384 candidates gets none); offsets[nq] = the candidate total.
 *   sng_simknn_wide_select: a second sweep writes the candidate column ids into cand [offsets[nq]] int32 (allocated by the
 *     caller from the total), then every row is rescored in FP32 (the exact score of sng_simknn_build), sorted by
 *     (sim desc, index asc) and proven; rows that cannot be proven, or have too many candidates, are recomputed by an exact
 *     FP32 scan of all n columns.  n_exact (device int32, may be NULL) = the number of such rows.
 * Neither call synchronises; the caller reads offsets[nq] back to size cand. */
SNG_API size_t sng_simknn_wide_workspace_bytes(int64_t nq, int64_t n, int64_t d, int64_t top_k);
SNG_API int sng_simknn_wide_count(const uint16_t* xq_f16, const uint16_t* xall_f16, int64_t ldh,
                      int64_t nq, int64_t q_offset, int64_t n, int64_t d, int64_t top_k, float thr, int remove_self,
                      int64_t* offsets, void* workspace, size_t workspace_bytes, void* stream);
SNG_API int sng_simknn_wide_select(const uint16_t* xq_f16, const uint16_t* xall_f16, int64_t ldh,
                      const float* xq_f32, const float* xall_f32, int64_t ld32,
                      int64_t nq, int64_t q_offset, int64_t n, int64_t d, int64_t top_k, float thr, int remove_self,
                      const int64_t* offsets, int32_t* cand, int32_t* idx, float* sim, int32_t* cnt, int32_t* n_exact,
                      void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SNG_H_ */
