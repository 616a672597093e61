/*
 * wdgh_b200.h -- C ABI of the B200-native graph-statistics hot path.
 *
 * Drop-in boundary for the path BASELINE.json `north_star` names in
 * SitaoLuan/When-Do-GNNs-Help:  A_hat X aggregation (SGC-1 / GCN propagation)
 * plus the homophily / node-distinguishability metrics of
 *     utils/homophily_metrics.py   and   utils/util_funcs.py.
 * Each entry point cites the reference lines it replaces.  The reference is
 * pure Python; its "FFI" for this path is a ctypes binding (see
 * INTEGRATION.md), so every signature is plain pointers + sizes, no torch
 * types.
 *
 * Conventions
 *   - Pointers are DEVICE pointers on the current CUDA device unless the name
 *     ends in `_host`.  `stream` is a cudaStream_t passed as void* (NULL = the
 *     legacy default stream).  Calls are asynchronous on `stream` unless stated.
 *   - A graph is CSR: rowptr int64[n+1], col int32[nnz] (row-major, the order
 *     `A.coalesce().indices()` yields), optional val float32[nnz] (NULL = all 1).
 *   - Labels are int32[n]; negative = unlabelled (LINKX convention, hm.py:48).
 *   - Return value: 0 on success, a positive cudaError_t, or a negative
 *     WDGH_E* code; wdgh_last_error() gives the message of the calling thread.
 *   - There is NO CPU fallback anywhere behind this ABI.
 */
#ifndef WDGH_B200_H
#define WDGH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WDGH_VERSION 100

#define WDGH_EINVAL (-1)  /* bad argument                                   */
#define WDGH_ENODEV (-2)  /* no sm_100 device / kernel image not loadable  */
#define WDGH_ESTATE (-3)  /* plan / workspace too small or stale            */

/* normalisation applied on the fly inside wdgh_spmm_csr */
#define WDGH_NORM_NONE 0 /* Y = A X                       (torch.spmm(adj, x), hm.py:192,199,234)          */
#define WDGH_NORM_RW   1 /* Y = D^-1 (A [+I]) X           (row_normalized_adjacency, util_funcs.py:383-390) */
#define WDGH_NORM_SYM  2 /* Y = D^-1/2 (A [+I]) D^-1/2 X  (sys_normalized_adjacency, util_funcs.py:418-426) */
/* scale modes of wdgh_degree_scale / wdgh_scale_values only (the other util_funcs.py normalisers; not valid for the SpMM) */
#define WDGH_NORM_RW_SUM  3 /* r_i = 1 / rowsum_i (signed sum), inf -> 0   (normalize :29-36, preprocess_features :39-46) */
#define WDGH_NORM_SYM_RAW 4 /* r_i = rowsum_i^-1/2, inf -> 0, no 0 -> 1 substitution       (normalize_adj :429-436)    */

/* ---- library ------------------------------------------------------------ */
int         wdgh_version(void);
const char *wdgh_last_error(void);
/* sm count and compute capability of the current device */
int         wdgh_device_info(int *sm_count, int *cc_major, int *cc_minor);
/* kernels this library has launched since load (bench.py's "gpu_launches") */
uint64_t    wdgh_launch_count(void);

/* ---- formats (A.coalesce().indices() -> CSR; hm.py:50,63,127) ------------ */
/* indices: torch COO layout int64[2][nnz], row-major sorted (coalesced).
 * Writes rowptr int64[n+1] and col int32[nnz]. */
int wdgh_coo_to_csr(const int64_t *indices, int64_t nnz, int64_t n,
                    int64_t *rowptr, int32_t *col, void *stream);
/* CSR -> explicit int64 row ids (the inverse; for handing indices back to torch) */
int wdgh_csr_to_coo_rows(const int64_t *rowptr, int64_t n, int64_t nnz, int64_t *row, void *stream);
/* int64 labels (torch.LongTensor) -> int32; *max_label (device int32) = max over n */
int wdgh_pack_labels(const int64_t *labels, int64_t n, int32_t *out, int32_t *max_label, void *stream);
/* argmax over the columns of a dense one-hot / score matrix -> int32 labels (hm.py:193) */
int wdgh_argmax_rows(const float *m, int64_t n, int64_t c, int64_t ld, int32_t *out, void *stream);

/* ---- load-balance plan (degree binning for skewed graphs) ---------------- */
/* Rows with more than `heavy_threshold` entries are split into chunks of that
 * many entries; everything else is handled one row per warp / sub-warp group.
 * The plan lives in caller-provided device memory and is reused by
 * wdgh_spmm_csr and wdgh_structure_counts for the same rowptr.
 *   plan_i64  : int64[WDGH_PLAN_WORDS(capacity)]  (device).  Words 8..11 of the header are the ticket counters of
 *               the persistent row-group kernels (zeroed here, re-armed by the last CTA of every launch): the plan
 *               is therefore written by wdgh_spmm_csr* / wdgh_structure_counts, and one plan must not be used by two
 *               launches that run concurrently on different streams (they would also share `partial`).
 *   capacity  : >= 2 * nnz / heavy_threshold + 2       (upper bound on the number of chunks)
 *   plan_host : int64[8] HOST array the later calls take alongside plan_i64
 * SYNCHRONOUS (reads the two counters back to size the later launches). */
#define WDGH_PLAN_HEADER 16
#define WDGH_PLAN_WORDS(capacity) (WDGH_PLAN_HEADER + 3 * (capacity))
int wdgh_plan_build(const int64_t *rowptr, int64_t n, int64_t nnz, int64_t heavy_threshold,
                    int64_t *plan_i64, int64_t capacity,
                    int64_t *plan_host /* int64[8] out: n_heavy, n_chunks, threshold, capacity, 0, 0, nnz, 0 */,
                    void *stream);

/* ---- normalisation (util_funcs.py:365-390, 418-426) ---------------------- */
/* dinv[i] = (rowsum_i + self_loop)^p, p=-1 (RW) / -1/2 (SYM), inf -> 0, row sums
 * of an all-zero row become 1 for SYM as in util_funcs.py:422.  val NULL = binary. */
int wdgh_degree_scale(const int64_t *rowptr, const float *val, int64_t n,
                      int norm, int add_self_loop, float *dinv /* nullable */,
                      double *dinv64 /* nullable: the same scale before the float32 cast */,
                      uint8_t *deg_code /* nullable, binary adjacency only: min(row length, 255) per node; lets
                                           wdgh_spmm_csr replace the per-entry float gather by an L2-resident
                                           1-byte lookup (255 = fall back to dinv) */,
                      void *stream);
/* Materialise the normalised values of a CSR that ALREADY contains its diagonal:
 * out[e] = f32( dinv64_i * val[e] * dinv64_j ) (SYM) or f32( dinv64_i * val[e] ) (RW), i.e. the float64
 * products scipy forms before sparse_mx_to_torch_sparse_tensor casts them (util_funcs.py:402). */
int wdgh_scale_values(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                      int norm, const double *dinv64, float *out, void *stream);
/* CSR of (A + I): merges / inserts the diagonal, keeping columns sorted.
 * out_rowptr int64[n+1]; out_col / out_val sized nnz + n (upper bound);
 * scratch int64[n + 2*ceil(n/1024) + 8].  The new nnz is out_rowptr[n]. */
int wdgh_add_self_loops(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                        int64_t *out_rowptr, int32_t *out_col, float *out_val,
                        int64_t *scratch, void *stream);
/* Dense row normalisation, normalize_tensor(mx, symmetric) (util_funcs.py:365-380).
 * symmetric != 0 needs a square matrix (n == d).  scratch_n: float32[n]. */
int wdgh_normalize_dense(const float *x, int64_t n, int64_t d, int64_t ld,
                         int symmetric, float *scratch_n, float *out, int64_t ldo, void *stream);

/* ---- A_hat X aggregation: CSR SpMM, float32 ------------------------------ */
/* y[n][d] = norm(A [+ I]) x.   norm != NONE with val == NULL computes
 * D^-1/2 / D^-1 from the row lengths on the fly -- A_hat is never materialised.
 *   dinv     : float32[n] from wdgh_degree_scale (required iff norm != NONE)
 *   plan_i64 / plan_host : from wdgh_plan_build (required)
 *   partial  : float32[n_chunks * roundup(d,4)] scratch for the partial sums of split rows, n_chunks =
 *              plan_host[1] (may be NULL if 0).
 *   row_offset : 0 for a whole graph.  For a 1-D row shard (multi-GPU) the CSR holds rows
 *              [row_offset, row_offset + n) of the global matrix: `col`, `x` and `dinv` use global
 *              node ids, `y` is local ([n][d]).
 * Replaces torch.spmm / torch.mm(adj, features) at hm.py:192,199,234,299,315. */
int wdgh_spmm_csr(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                  const float *x, int64_t d, int64_t ldx, float *y, int64_t ldy,
                  int norm, int add_self_loop, const float *dinv,
                  const uint8_t *deg_code /* nullable: from wdgh_degree_scale, global ids like dinv */,
                  int64_t *plan_i64, const int64_t *plan_host, float *partial,
                  int64_t row_offset, void *stream);

/* Element types of the output of wdgh_spmm_csr_bf16 / _f16 and wdgh_pipeline_host_bf16 / _f16: float32, or the half
 * type of the features (a bf16 entry rejects WDGH_DTYPE_F16, an f16 entry WDGH_DTYPE_BF16) */
#define WDGH_DTYPE_F32  0
#define WDGH_DTYPE_BF16 1
#define WDGH_DTYPE_F16  2
/* wdgh_spmm_csr with a bfloat16 feature matrix (raw bf16 bits), fp32 accumulation, y float32 or bf16 (y_dtype).
 * ldx / ldy in elements; plan, dinv, deg_code, partial (float32) exactly as for wdgh_spmm_csr.
 * Every row is summed in the order of wdgh_spmm_csr, and bf16 -> fp32 is exact: fp32 output is bit-identical to
 * wdgh_spmm_csr on the upcast matrix, bf16 output is that result rounded to nearest even.  Rows of x starting on an
 * 8-byte boundary with d and ldx multiples of 4 take the vectorised kernels; any other width or alignment works. */
int wdgh_spmm_csr_bf16(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                       const uint16_t *x, int64_t d, int64_t ldx, void *y, int64_t ldy, int y_dtype,
                       int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                       int64_t *plan_i64, const int64_t *plan_host, float *partial,
                       int64_t row_offset, void *stream);
/* wdgh_spmm_csr with a float16 feature matrix (raw IEEE binary16 bits), fp32 accumulation, y float32 or float16
 * (y_dtype WDGH_DTYPE_F32 / WDGH_DTYPE_F16).  Every row is summed in the order of wdgh_spmm_csr, and fp16 -> fp32 is
 * exact for every value (subnormals, +-0, +-inf, NaN): fp32 output is bit-identical to wdgh_spmm_csr on the upcast
 * matrix, fp16 output is that result rounded to nearest even (overflow to +-inf).  Alignment rules as for
 * wdgh_spmm_csr_bf16. */
int wdgh_spmm_csr_f16(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                      const uint16_t *x, int64_t d, int64_t ldx, void *y, int64_t ldy, int y_dtype,
                      int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                      int64_t *plan_i64, const int64_t *plan_host, float *partial,
                      int64_t row_offset, void *stream);

/* ---- phased aggregation (overlap of the feature all-gather with compute, N > 1) ---- */
/* seg[b][r] (int64[num_bounds][n]) = first stored entry of row r whose column id is >= bounds_dev[b]; with
 * bounds = the partition's node-id boundaries, [seg[b][r], seg[b+1][r]) are the entries of row r whose source
 * node lives on rank b (columns are sorted inside a row). */
int wdgh_column_segments(const int64_t *rowptr, const int32_t *col, int64_t n,
                         const int64_t *bounds_dev, int32_t num_bounds, int64_t *seg, void *stream);
/* flags[r] = 1 for the rows the plan splits into chunks (uint8[n]) */
int wdgh_plan_heavy_flags(const int64_t *plan_i64, const int64_t *plan_host, int64_t n, uint8_t *flags, void *stream);
/* wdgh_spmm_csr restricted to the entries [range_begin[r], range_end[r]) of every row r:
 *   accumulate != 0 : y += (instead of y =);   finalize != 0 : apply the self loop and the row scale now
 *   (earlier phases store raw partial sums);   run_split_rows != 0 : afterwards compute the split rows over their
 *   full column range (they need all of x; finalized or raw like the call).
 *   extra_parts : n_extra (<= 8) raw partial sums of the SAME rows in one device buffer, part q at
 *   extra_parts + q * extra_part_rows * ld_extra (float32[extra_part_rows][ld_extra] each, local row index like y).
 *   They are added to every row as virtual trailing stream entries of weight 1 (fetched in the same gather batches
 *   as the feature rows): the partial of an earlier column range kept in another buffer and, in the 2-D multi-GPU
 *   partition, the row slices the peers stored into this rank's memory over NVLink -- the last phase of a row slice
 *   is also its reduction + epilogue, and with range_begin == range_end the call is a pure streaming reduction.
 *   The split-row pass adds only the LAST n_extra_split parts (an earlier phase never stores split rows).  d >= 128.
 *   ctas_per_sm : 0 = default grid; a smaller value leaves SM capacity to a kernel running concurrently on another
 *   stream (the NVLink-bound foreign-slice launches of the 2-D partition run next to the HBM-bound own slice).
 *   `y` (and the extra parts) may be peer-mapped memory of another GPU.
 * Needs 16-byte aligned rows and d in {32, 64} or d >= 128. */
int wdgh_spmm_csr_ranged(const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end,
                         const int32_t *col, const float *val, int64_t n,
                         const float *x, int64_t d, int64_t ldx, float *y, int64_t ldy,
                         int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                         const uint8_t *skip_rows, int accumulate, int finalize, int run_split_rows,
                         const float *extra_parts, int32_t n_extra, int32_t n_extra_split,
                         int64_t extra_part_rows, int64_t ld_extra, int32_t ctas_per_sm,
                         int64_t *plan_i64, const int64_t *plan_host, float *partial,
                         int64_t row_offset, void *stream);
/* wdgh_spmm_csr_ranged with a bfloat16 feature matrix (raw bf16 bits, ldx in elements) and float32 y: every phase
 * accumulates in fp32 and stores fp32 (raw partial sums are never rounded), so each call is bit-identical to
 * wdgh_spmm_csr_ranged on the upcast matrix with the same arguments.  No extra partial sums and no ctas_per_sm (the
 * 2-D multi-GPU partition is fp32).  Needs rows on 8-byte boundaries (d and ldx multiples of 4) and d in {32, 64} or
 * d >= 128. */
int wdgh_spmm_csr_ranged_bf16(const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end,
                              const int32_t *col, const float *val, int64_t n,
                              const uint16_t *x, int64_t d, int64_t ldx, float *y, int64_t ldy,
                              int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                              const uint8_t *skip_rows, int accumulate, int finalize, int run_split_rows,
                              int64_t *plan_i64, const int64_t *plan_host, float *partial,
                              int64_t row_offset, void *stream);
/* wdgh_spmm_csr_ranged with a float16 feature matrix (raw binary16 bits, ldx in elements) and float32 y: fp32 partial
 * sums, so each call is bit-identical to wdgh_spmm_csr_ranged on the upcast matrix with the same arguments.  No extra
 * partial sums and no ctas_per_sm; alignment and widths as for wdgh_spmm_csr_ranged_bf16. */
int wdgh_spmm_csr_ranged_f16(const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end,
                             const int32_t *col, const float *val, int64_t n,
                             const uint16_t *x, int64_t d, int64_t ldx, float *y, int64_t ldy,
                             int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                             const uint8_t *skip_rows, int accumulate, int finalize, int run_split_rows,
                             int64_t *plan_i64, const int64_t *plan_host, float *partial,
                             int64_t row_offset, void *stream);

/* ---- label metrics: one pass over the edges ------------------------------ */
/* Integer statistics every label metric of homophily_metrics.py is a ratio of
 * (edge / node / class / adjusted homophily, label informativeness; hm.py:43-161).
 *   counters int64[WDGH_SC_WORDS(C)], zeroed by the call:
 *     [WDGH_SC_MATCH_ALL]  stored entries with equal endpoint labels (self-loops included)   hm.py:51
 *     [WDGH_SC_MATCH_LAB]  same, both endpoints labelled >= 0                               hm.py:52-54
 *     [WDGH_SC_N_LAB]      stored entries with both endpoints labelled >= 0
 *     [WDGH_SC_N_SELF]     stored diagonal entries
 *     [WDGH_SC_N_EMPTY]    rows without any stored entry            (class_distribution IndexError)
 *     [WDGH_SC_NBINS]      1 + max row id having an off-diagonal entry (node_homophily RuntimeError)
 *     [WDGH_SC_N_NODES_NSL] rows with >= 1 off-diagonal entry                               hm.py:78
 *     [WDGH_SC_HEADER + c]           nodes of class c                                        hm.py:114,137
 *     [WDGH_SC_HEADER + C + c]       sum over class-c nodes of stored entries per row        hm.py:141
 *     [WDGH_SC_HEADER + 2C + a*C+b]  off-diagonal entries a->b, both labelled                hm.py:97-100,144
 *     [WDGH_SC_HEADER + 2C + C*C + c] class-c nodes without any off-diagonal entry (homophily_plot.py our_measure :131-132)
 *   node_sum double[2]: [0] sum_i f32(match_i)/f32(deg_i) over rows with deg_i > 0, diagonal excluded (hm.py:77-78);
 *                       [1] the same with the stored diagonal counted as a matching entry
 *                           (utils/homophily_plot.py:92-100, which does not strip self-loops)
 *   deg_nsl / match_nsl int32[n]: per-row off-diagonal entry count / label matches (scratch AND output)
 * A label counts as labelled when 0 <= l < num_classes.  Any other value -- negative, or >= num_classes -- is
 * unlabelled: it indexes no class table and no pair bin, but the match counts (MATCH_ALL, match_nsl) still compare
 * raw labels, so two such values match only when equal (hm.py:51).
 */
#define WDGH_SC_MATCH_ALL   0
#define WDGH_SC_MATCH_LAB   1
#define WDGH_SC_N_LAB       2
#define WDGH_SC_N_SELF      3
#define WDGH_SC_N_EMPTY     4
#define WDGH_SC_NBINS       5
#define WDGH_SC_N_NODES_NSL 6
#define WDGH_SC_N_MULTI_NEG 7 /* labels the 1-byte copy cannot represent exactly (< -1 or >= num_classes) seen
                                 while packing: re-run without labels_u8_scratch */
#define WDGH_SC_HEADER      8
#define WDGH_SC_WORDS(C)    (WDGH_SC_HEADER + 3 * (C) + (C) * (C))
int wdgh_structure_counts(const int64_t *rowptr, const int32_t *col, int64_t n, int64_t nnz,
                          const int32_t *labels, int32_t num_classes,
                          int64_t *plan_i64, const int64_t *plan_host,
                          int64_t *counters, double *node_sum,
                          int32_t *deg_nsl, int32_t *match_nsl,
                          uint8_t *labels_u8_scratch /* nullable: uint8[n_labels]; when given and C <= 254 the
                                                        neighbour-label gathers use a 1-byte copy (L2-resident) */,
                          int64_t n_labels /* length of `labels` (= n for a whole graph, n_global for a shard) */,
                          int64_t row_offset /* as in wdgh_spmm_csr: labels are global, deg/match local */,
                          void *stream);
/* A_hat X aggregation AND the label statistics in one call (binary adjacency): wdgh_spmm_csr followed by
 * wdgh_structure_counts on the same stream, same arguments, same results. */
int wdgh_spmm_structure_fused(const int64_t *rowptr, const int32_t *col, int64_t n, int64_t nnz,
                              const float *x, int64_t d, int64_t ldx, float *y, int64_t ldy,
                              int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                              const int32_t *labels, int32_t num_classes,
                              int64_t *plan_i64, const int64_t *plan_host, float *partial,
                              int64_t *counters, double *node_sum, int32_t *deg_nsl, int32_t *match_nsl,
                              uint8_t *labels_u8_scratch, int64_t n_labels, int64_t row_offset, void *stream);
/* Same statistics from an arbitrary edge list (torch `edge_index` int64[2][E]: unsorted, repeats
 * counted with multiplicity), as node_homophily_edge_idx / compact_matrix_edge_idx / our_measure
 * receive it (hm.py:71,81,105).  Row lengths are unknown here, so the per-class degree mass
 * [WDGH_SC_HEADER + C + c] and [WDGH_SC_N_EMPTY] stay 0. */
int wdgh_structure_counts_coo(const int64_t *edge_index, int64_t num_edges, int64_t n,
                              const int32_t *labels, int32_t num_classes,
                              int64_t *counters, double *node_sum,
                              int32_t *deg_nsl, int32_t *match_nsl,
                              int hist_includes_self_loops /* homophily_plot.py compact_matrix_edge_idx keeps (i,i) */,
                              void *stream);
/* edge_homophily with a 2-D label matrix (hm.py:50-56 as called from
 * homophily_tests.py:115-116): counts elementwise-equal label entries over all
 * stored (i,j); *equal_count (device uint64) out of nnz*c comparisons. */
int wdgh_edge_label_rows_equal(const int64_t *rowptr, const int32_t *col, int64_t n,
                               const float *label_rows, int64_t c, int64_t ld,
                               unsigned long long *equal_count, void *stream);

/* ---- generalised edge homophily: feature cosine over edges (hm.py:164-187) */
/* mode bit 1 (value 2) set: plain dot products <x_i, x_j> instead of cosines (homophily_plot.py:48-52
 * edge_homophily with a label matrix).
 * mode 0: all off-diagonal stored entries whose value is > 0 (val NULL = all);
 *         out_sum[0] += sum of cosines, out_cnt[0] += entries counted.
 * mode 1: the `n_ids` stored-entry ids in `entry_ids` (position in the coalesced COO,
 *         diagonal included); same outputs.  NaN cosines count as 0 (hm.py:168,185). */
int wdgh_edge_cosine(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                     const float *x, int64_t d, int64_t ldx,
                     int mode, const int64_t *entry_ids, int64_t n_ids,
                     double *out_sum, unsigned long long *out_cnt, void *stream);

/* ---- dense contractions: aggregation similarity and the KR Gram ---------- */
/* g[m][m] = z z^T for z float32[m][d]  ((A X)(A X)^T, hm.py:192,199-200,234-235,246).
 *   mode WDGH_GRAM_TC / WDGH_GRAM_TC_FAITHFUL: TMA-fed tcgen05 kernel, 3xTF32 operand split (fp32-level products),
 *     128 x 256 tiles, upper triangle only; the k-blocks are accumulated in TMEM in chunks that the epilogue warps add in
 *     fp32 registers: 4 k-blocks per chunk (TC, ~5e-7 relative) or 1 (TC_FAITHFUL, fp32 level: the KR metric feeds the
 *     Gram to pinv(rcond=1e-15), which amplifies rounding noise).  Needs `workspace` =
 *     float32[wdgh_gram_workspace_floats(m, d)], 16-byte aligned.  d <= 32 is routed to the SIMT kernel (faster there).
 *   mode WDGH_GRAM_SIMT: SIMT fp32 tile kernel (cross-check), workspace may be NULL. */
#define WDGH_GRAM_SIMT        0
#define WDGH_GRAM_TC          1
#define WDGH_GRAM_TC_FAITHFUL 2
int64_t wdgh_gram_workspace_floats(int64_t m, int64_t d);
int wdgh_gram(const float *z, int64_t m, int64_t d, int64_t ldz,
              float *g, int64_t ldg, int mode, float *workspace, void *stream);
/* gather rows: out[k][:] = x[ids[k]][:]  (torch indexing `[sample, :]`, hm.py:199,234,246) */
int wdgh_gather_rows(const float *x, int64_t d, int64_t ldx, const int64_t *ids, int64_t m,
                     float *out, int64_t ldo, void *stream);
/* w[m][C]: w[i][c] = sum (is_mean=0) or mean (is_mean=1) over j with labels[j]==c of g[i][j] (hm.py:201-206) */
int wdgh_class_colsum(const float *g, int64_t m, int64_t ldg, const int32_t *labels, int32_t num_classes,
                      int is_mean, float *w, void *stream);
/* The same w without the m x m matrix g = z z^T: w[i][c] = sum (is_mean = 0) / mean (is_mean = 1) over j with
 * labels[j] == c of <z_i, z_j>, computed as <z_i, s_c> with the class sums s_c = sum_{j: labels[j] == c} z_j
 * (hm.py:192,199-206; homophily_plot.py similarity, non-NTK branch :196-206).  z float32[m][d] with row stride ldz >= d,
 * any d >= 1, any C >= 1; m = 0 does nothing.  w float32[m][C] row-major, as wdgh_las_score takes it.
 *   Summation order: s and the class counts are accumulated in fp64.  The rows are cut into contiguous segments
 *   (their number and bounds depend on m, d and C only); each segment is summed in row order into its own partial
 *   table, and the partials are added in segment order (8 contiguous runs, then the run sums).  w[i][c] =
 *   f32(sum_k z[i][k] * s[c][k]) with products and sum in fp64 in k order, or f32(that sum / count) -- one rounding
 *   to float32 for the sum, fp64 division then one rounding for the mean.  No atomics: the result is a function of
 *   the inputs alone, independent of the device's SM count and of scheduling.
 *   A label outside [0, C) joins no class (as in wdgh_class_colsum).  An empty class gives 0 (sum) and NaN (mean).
 *   workspace: double[wdgh_class_inner_workspace_doubles(m, d, C)], at most C (d + 1) + max(C (d + 1), 2^22)
 *   doubles (32 MiB plus two [C][d + 1] tables); the size function returns -1 for invalid sizes. */
int64_t wdgh_class_inner_workspace_doubles(int64_t m, int64_t d, int32_t num_classes);
int wdgh_class_inner_sums(const float *z, int64_t m, int64_t d, int64_t ldz, const int32_t *labels,
                          int32_t num_classes, int is_mean, double *workspace, float *w, void *stream);
/* aggregation-similarity score from w (hm.py:207-229).  label_rows: float32[m][C] (the `label` argument).
 * *count (device uint64) = number of nodes whose indicator is true; the score is count / m.
 * scratch_c: float32[C]. */
int wdgh_las_score(const float *w, const int32_t *labels, const float *label_rows, int64_t m, int32_t num_classes,
                   int hard, int lp, int is_sum, float *scratch_c, unsigned long long *count, void *stream);
/* in place: g <- k (pi - acos k) / (2 pi) with k = clamp(g, 0, 1)   (homophily_plot.py similarity NTK branch :191-193) */
int wdgh_ntk_clamp_transform(float *g, int64_t m, int64_t ldg, void *stream);
/* in place: g <- arccos-kernel(g)/2 for n_layers==1, g/2 for n_layers==0 (hm.py:236-244,257).
 * scratch_m: float32[m]. */
int wdgh_gntk_transform(float *g, int64_t m, int64_t ldg, int n_layers, float *scratch_m, void *stream);

/* ---- end-to-end entry with HOST buffers (bench.py "e2e") ------------------ */
/* One pass of the hot path from host memory: H2D copy of the CSR, labels and
 * features, plan + normaliser, Y = norm(A+I) X, the label statistics, D2H copy of
 * the counters (+ node_sum) and, if y_host != NULL, of Y.  SYNCHRONOUS.
 *   counters_host int64[WDGH_SC_WORDS(C)], node_sum_host double[2].
 * Device buffers are allocated once and cached inside the library between calls. */
int wdgh_pipeline_host(const int64_t *rowptr_host, const int32_t *col_host, int64_t n, int64_t nnz,
                       const float *x_host, int64_t d, const int32_t *labels_host, int32_t num_classes,
                       int norm, int add_self_loop,
                       float *y_host, int64_t *counters_host, double *node_sum_host);
/* wdgh_pipeline_host with a bfloat16 feature matrix (raw bf16 bits, [n][d] contiguous): half the bytes of X on the
 * link.  y_host (NULL = counters only) is [n][d] of y_dtype: WDGH_DTYPE_F32, or WDGH_DTYPE_BF16 (half the bytes back).
 * Aggregation is fp32; a bf16 Y is the fp32 Y of the same call rounded to nearest even.  The copy / compute schedule
 * depends on (n, nnz, d, feature type, y_host != NULL), not on y_dtype.  Shares the cached pipeline (and
 * wdgh_pipeline_host_release) with wdgh_pipeline_host.  SYNCHRONOUS. */
int wdgh_pipeline_host_bf16(const int64_t *rowptr_host, const int32_t *col_host, int64_t n, int64_t nnz,
                            const uint16_t *x_host, int64_t d, const int32_t *labels_host, int32_t num_classes,
                            int norm, int add_self_loop,
                            void *y_host, int y_dtype, int64_t *counters_host, double *node_sum_host);
/* wdgh_pipeline_host with a float16 feature matrix (raw binary16 bits, [n][d] contiguous): half the bytes of X on the
 * link.  y_host (NULL = counters only) is [n][d] of y_dtype: WDGH_DTYPE_F32, or WDGH_DTYPE_F16 (the fp32 Y of the same
 * call rounded to nearest even, overflow to +-inf).  Same schedule, cache and ordering as wdgh_pipeline_host_bf16: an
 * fp32 Y is bit-identical to wdgh_pipeline_host on the upcast matrix.  SYNCHRONOUS. */
int wdgh_pipeline_host_f16(const int64_t *rowptr_host, const int32_t *col_host, int64_t n, int64_t nnz,
                           const uint16_t *x_host, int64_t d, const int32_t *labels_host, int32_t num_classes,
                           int norm, int add_self_loop,
                           void *y_host, int y_dtype, int64_t *counters_host, double *node_sum_host);
/* free the buffers cached by wdgh_pipeline_host / _bf16 / _f16 */
int wdgh_pipeline_host_release(void);

#ifdef __cplusplus
}
#endif
#endif /* WDGH_B200_H */
