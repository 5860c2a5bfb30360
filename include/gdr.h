/*
 * gdr.h — C ABI of the B200-native graph-distillation core (libgdr_b200.so).
 *
 * The reference (Tyler-Linchenwei/Graph-Distillation-for-Recommendation) is pure
 * Python and has no FFI surface; its hot path is reached through Python call
 * sites that hand torch / numpy / scipy objects to torch-sparse, scipy
 * sparsetools and scikit-learn.  This header is the boundary a maintainer would
 * bind instead (ctypes stub: see INTEGRATION.md).  Every entry point names the
 * reference call site it replaces as  file:line  relative to
 * /root/reference/ClustGDD/ ("sklearn/" = scikit-learn's cluster package, the
 * third-party dependency that owns stage 3's arithmetic).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - every function returns int: 0 = ok, <0 = GDR_E* ; text via gdr_last_error().
 *   - all data pointers are DEVICE pointers owned by the caller unless the
 *     parameter name ends in _host.  The library never frees caller memory and
 *     never allocates outputs; scratch comes from the caller through the
 *     two-phase  *_ws_bytes() / run(ws, ws_bytes)  pattern.
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); nothing
 *     synchronises unless the doc of the function says so.
 *   - dense matrices are row-major float32 with an explicit leading dimension
 *     in ELEMENTS; CSR is (rowptr int32[n+1], colidx int32[nnz], vals f32[nnz]).
 *   - thread-safe for distinct streams; no global mutable state except the
 *     thread-local error string.
 */
#ifndef GDR_H_
#define GDR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
/* the library is built with -fvisibility=hidden; only this header is exported */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define GDR_ABI_VERSION 1

#define GDR_OK            0
#define GDR_EINVAL      (-1)  /* bad argument (null pointer, negative size, misalignment) */
#define GDR_EWORKSPACE  (-2)  /* ws_bytes smaller than *_ws_bytes() asked for            */
#define GDR_ECUDA       (-3)  /* a CUDA runtime/driver call failed                        */
#define GDR_ERANGE      (-4)  /* index out of range / size exceeds int32 CSR limits       */
#define GDR_EUNSUPPORTED (-5) /* shape not supported by this kernel (see doc)             */

typedef void* gdr_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------- */
int         gdr_abi_version(void);
const char* gdr_last_error(void);
/* Fills sm_count / compute capability of the CURRENT device. */
int         gdr_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Counter of kernels this library has launched in the calling process since
 * load (all threads); used by bench.py for "gpu_launches". */
int64_t     gdr_launch_count(void);

/* Optional kernel timing for bench.py's roofline leg: kind 1 = the k-means E-step main
 * kernel, 2 = the CSR SpMM; 0 = off.  Every launch of that kind is bracketed by a CUDA
 * event pair on its stream; collect() synchronises those events and returns the summed
 * device time and the number of launches. */
int gdr_profile_enable(int kind);
int gdr_profile_collect(double* total_ms_host, int64_t* launches_host);

/* Path selectors and test knobs; not a stable surface: keys may change between versions, and an unknown key
 * fails with GDR_EINVAL.  keys:
 * "tc_screen" (E-step of gdr_kmeans_assign_tc: 0 [default] automatic, 1 direct 3xTF32, any value >= 2 the
 * two-level screen whatever N); "tc_gate" (first-level epilogue gate of the two-level screen: 0 off, any other
 * value [default 1] on; the same labels either way); "tc_cand" (second level of the two-level screen: 1 [default]
 * seeded 1xTF32 candidate pass + exact re-score of the candidates, 0 3xTF32 over all centres; same labels);
 * "tc_cand_cap" (candidate list capacity per row and column half, 1..16; 0 = 16);
 * "lloyd_graph" (0: no CUDA-graph replay of the Lloyd iteration); "coarsen_dense" (0: stage 4 always on the sort
 * path); "sparsify_batch" (cap on the classes per batch of gdr_sparsify_classes); "kpp_dist_skip_score" (1: the
 * k-means++ rounds of gdr_kmeans_plusplus_dist without their score pass, for exchange timing only);
 * "rs_match" (radix-sort ranking: 0 [default] per-bit warp ballots, 1 MATCH.ANY); "rs_max_bits" (digit width cap
 * of large sorts; 0 [default] = 9); "topk_path" (gdr_topk_scores: 0 automatic, 1 exact SIMT path,
 * 2 tensor-core screen); "topk_condensed_path" (gdr_topk_condensed: 1 every row on the exact fallback). */
int gdr_debug_set(const char* key, int value);
/* Debug read-back (synchronises the device).  keys: "tc_level2_rows" = rows the last two-level
 * tensor-core screen (gdr_kmeans_assign_tc) left undecided after its first level; -1 if none ran.
 * "tc_cand_rows" / "tc_cand_overflow_rows" / "tc_cand_entries" = of those, the rows the last run decided on their
 * candidate centres / the rows whose candidate list overflowed (they took the 3xTF32 fallback) / the candidates
 * recorded for the rows read (-1 if the last two-level run did not use candidate lists).
 * "topk_overflow_rows" = rows the last tensor-core gdr_topk_scores finished on the exact path; -1 if none ran.
 * "topk_condensed_fallback_rows" = rows the last gdr_topk_condensed finished on the exact path; -1 if it wrote
 * nothing.  An unknown key fails with GDR_EINVAL. */
int gdr_debug_get(const char* key, int64_t* value_host);

/* ---- generic device primitives (used by stages 1, 3, 4) -------------- */
/* Stable LSD radix sort of (uint64 key, uint32 payload) pairs on the low
 * `key_bits` bits.  Result is left in keys_io / vals_io. */
int64_t gdr_sort_pairs_ws_bytes(int64_t n);
int     gdr_sort_pairs(int64_t n, int key_bits, uint64_t* keys_io, uint32_t* vals_io,
                       void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* ---- stage 1: adjacency build ---------------------------------------- */
/* COO -> CSR with duplicate (row,col) entries SUMMED and column indices
 * sorted inside each row.
 *   replaces  scipy  sp.csr_matrix((ones,(r,c)))          utils.py:66-67
 *             sp.coo_matrix((vals,(u,i))).tocsr()          distill_recsys.py:116-117
 *             adj + adj.T ; adj[adj>1] = 1                 utils_graphsaint.py:20-22
 *   val == NULL means all ones.  symmetrize: also insert (col,row) for every
 *   entry (n_rows must equal n_cols).  binarize: every stored value becomes 1.
 *   Capacity of colidx/vals must be nnz_in * (symmetrize ? 2 : 1).
 *   *nnz_out_dev (device int64) receives the number of stored entries
 *   (= rowptr[n_rows]).  Indices outside [0,n_rows)x[0,n_cols) set
 *   status_dev[0] != 0 (device int32, caller checks after sync) and are dropped. */
int64_t gdr_coo_to_csr_ws_bytes(int64_t n_rows, int64_t n_cols, int64_t nnz_in, int symmetrize);
int     gdr_coo_to_csr(int64_t n_rows, int64_t n_cols, int64_t nnz_in,
                       const int64_t* row, const int64_t* col, const float* val,
                       int symmetrize, int binarize,
                       int32_t* rowptr, int32_t* colidx, float* vals,
                       int64_t* nnz_out_dev, int32_t* status_dev,
                       void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* Symmetric normalisation  D^-1/2 (A [+ I]) D^-1/2  of a CSR matrix.
 *   replaces  normalize_adj_tensor(adj, sparse=True)       deep_robust_utils.py:245-256
 *             -> to_scipy :408-417 -> normalize_adj :180-207
 *   self_loop_mode: 0 never add I, 1 always add I, 2 = the reference's rule
 *   "add I iff A[0,0] == 0" (deep_robust_utils.py:199-200).
 *   Degrees are row sums in fp64 (deg_out, nullable); r = deg^-1/2 in fp64 with
 *   inf -> 0; value = fp32((r_i * a_ij) * r_j)  — bit-exact with scipy.
 *   Output capacity: nnz + n.  *nnz_out_dev = stored entries of the result. */
int64_t gdr_sym_normalize_ws_bytes(int64_t n, int64_t nnz);
int     gdr_sym_normalize(int64_t n, int64_t nnz,
                          const int32_t* rowptr, const int32_t* colidx, const float* vals,
                          int self_loop_mode,
                          int32_t* rowptr_out, int32_t* colidx_out, float* vals_out,
                          double* deg_out, int64_t* nnz_out_dev,
                          void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* Row-block form of gdr_sym_normalize for the row-partitioned build (one rank owns rows
 * [row_offset, row_offset + n_local) with GLOBAL column ids; replaces the same reference lines,
 * deep_robust_utils.py:180-207, on a block).  Phase 1: degrees of the block (fp64, +1 when
 * add_identity) and the output row pointer (a diagonal slot is inserted where the block has none).
 * The caller all-gathers the degrees into deg_global[n].  Phase 2 writes the block of
 * D^-1/2 (A [+ I]) D^-1/2 — bit-identical to the rows gdr_sym_normalize produces on the whole matrix.
 * add_identity is the caller's global decision (self_loop_mode 2: A[0,0] == 0 on the owner of row 0). */
int64_t gdr_sym_normalize_block_ws_bytes(int64_t n_local);
int     gdr_sym_normalize_block_degrees(int64_t n_local, int64_t row_offset, const int32_t* rowptr,
                                        const int32_t* colidx, const float* vals, int add_identity,
                                        double* deg_local_out, int32_t* rowptr_out /* n_local + 1 */,
                                        void* ws, int64_t ws_bytes, gdr_stream_t stream);
int     gdr_sym_normalize_block_fill(int64_t n_local, int64_t row_offset, const int32_t* rowptr,
                                     const int32_t* colidx, const float* vals, int add_identity,
                                     const double* deg_global, const int32_t* rowptr_out,
                                     int32_t* colidx_out, float* vals_out, int64_t* nnz_out_dev,
                                     void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* Dense n x n variant:  D^-1/2 (A + I) D^-1/2  in fp32, O(n^2).
 *   replaces  normalize_adj_tensor(adj) dense branch       deep_robust_utils.py:257-264 */
int gdr_sym_normalize_dense(int64_t n, const float* A, int64_t lda, float* out, int64_t ldo,
                            void* ws, int64_t ws_bytes, gdr_stream_t stream);
int64_t gdr_sym_normalize_dense_ws_bytes(int64_t n);

/* Bipartite edge normalisation  norm_e = w_e / (sqrt(du[cu_e]+eps) * sqrt(di[ci_e]+eps)),
 * du = scatter-sum of w over cu, di over ci (fp32, deterministic order = CSR order).
 *   replaces  LightGCNCondensed.propagate degree/norm part distill_recsys.py:329-335
 *   Input is the CSR of the cu x ci weight matrix (rowptr/colidx/w) plus the
 *   transposed CSR built by gdr_csr_transpose; outputs norm in BOTH orders. */
int gdr_bipartite_normalize(int64_t n_u, int64_t n_i, int64_t nnz,
                            const int32_t* rowptr, const int32_t* colidx, const float* w,
                            const int32_t* t_rowptr, const int32_t* t_perm,
                            float eps, float* norm_out, float* t_norm_out,
                            float* deg_u, float* deg_i, gdr_stream_t stream);

/* Backward of the bipartite LightGCN propagation w.r.t. the edge weights (the condensed model's trained edge
 * weights, distill_recsys.py:319-353 under the refinement loop :684-733).  Notation: CSR entry e = (a, b) of the
 * n_u x n_i weight matrix, A_ab = norm_e, M = [[0, A], [A^T, 0]], X_l = M^l [u0; i0], out = c sum_{l<=L} X_l,
 * Y_m = M^m dL/dout (the adjoint propagation: gdr_spmm_prop on A / A^T), c = 1/(L+1).
 *
 * gdr_csr_locate: edge_pos_out[k] = position of the pair (row[k], col[k]) in the CSR (columns sorted inside a row),
 *   -1 when missing.  status_dev (device int32, zeroed by the caller): bit 0 = a pair outside the matrix,
 *   bit 1 = a pair not stored.  With E == nnz and status 0, edge_pos is a permutation of [0, nnz).
 * gdr_lightgcn_edge_grad: from the stacked layers Xu [L][n_u][ld], Xi [L][n_i][ld] (X_0 .. X_{L-1}) and Yu, Yi
 *   (Y_0 .. Y_{L-1}), all 16-byte aligned with ld a multiple of 4:
 *     G_out[e]   = dL/dA_ab = c sum_{j<L} ( Xi_j[b] . PY_{L-1-j}[a] + Yi_j[b] . PX_{L-1-j}[a] ),
 *                  PY_k = sum_{m<=k} Yu_m, PX_k = sum_{m<=k} Xu_m   (fp32)
 *     S_u_out[a] = sum_{e in row a} G_e norm_e                                  (fp64)
 *   L == 0 or d == 0 gives zeros.  Deterministic: one fixed summation order, no float atomics.
 * gdr_bipartite_normalize_backward: with the forward's norm and fp32 degrees (gdr_bipartite_normalize),
 *     S_i[b] = sum over the transposed row b, ascending, of G_e norm_e                 (fp64)
 *     dw_out[k] = G_e / (sqrt(du[a]+eps) sqrt(di[b]+eps)) - S_u[a] / (2 (du[a]+eps)) - S_i[b] / (2 (di[b]+eps)),
 *   e = edge_pos[k], evaluated in fp64 and rounded once; dw_out is in input edge order. */
int     gdr_csr_locate(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                       int64_t E, const int64_t* row, const int64_t* col, int32_t* edge_pos_out,
                       int32_t* status_dev, gdr_stream_t stream);
int     gdr_lightgcn_edge_grad(int64_t n_u, int64_t n_i, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                               const float* norm, int num_layers, int64_t d, const float* Xu, const float* Xi,
                               const float* Yu, const float* Yi, int64_t ld, float c, float* G_out,
                               double* S_u_out, gdr_stream_t stream);
int64_t gdr_bipartite_normalize_backward_ws_bytes(int64_t n_i, int64_t nnz);
int     gdr_bipartite_normalize_backward(int64_t n_u, int64_t n_i, int64_t nnz, const int32_t* rowptr,
                                         const int32_t* colidx, const int32_t* t_rowptr, const int32_t* t_perm,
                                         const float* norm, const float* deg_u, const float* deg_i, float eps,
                                         const float* G, const double* S_u, int64_t E, const int32_t* edge_pos,
                                         float* dw_out, void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* Rankformer GCN edge weights (Rankformer/code/rec.py:118-124, the teacher's propagation the
 * reference's LightGCN mirrors): du / di = interaction counts clamped to >= 1,
 *   out_e = w_e / du^a / di^b   (users <- items),   t_out = w_e / du^b / di^a (items <- users,
 *   in transposed order).  scratch: nnz floats. */
int gdr_bipartite_pow_normalize(int64_t n_u, int64_t n_i, int64_t nnz,
                                const int32_t* rowptr, const int32_t* colidx, const float* w,
                                const int32_t* t_rowptr, const int32_t* t_perm, float a, float b,
                                float* out, float* t_out, float* deg_u, float* deg_i,
                                float* scratch, gdr_stream_t stream);

/* CSR transpose: t_rowptr[n_cols+1], t_colidx[nnz] (= source row ids, ascending
 * inside each transposed row), t_perm[nnz] = position of that entry in the input. */
int64_t gdr_csr_transpose_ws_bytes(int64_t n_rows, int64_t n_cols, int64_t nnz);
int     gdr_csr_transpose(int64_t n_rows, int64_t n_cols, int64_t nnz,
                          const int32_t* rowptr, const int32_t* colidx,
                          int32_t* t_rowptr, int32_t* t_colidx, int32_t* t_perm,
                          void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* CSR -> COO index expansion (row-major, int64) — the layout the reference's
 * sparse_mx_to_torch_sparse_tensor produces     deep_robust_utils.py:389-396.
 * col_out nullable. */
int gdr_csr_to_coo(int64_t n_rows, const int32_t* rowptr, const int32_t* colidx,
                   int64_t* row_out, int64_t* col_out, gdr_stream_t stream);

/* ---- stage 2: propagation -------------------------------------------- */
/* One hop of   Y = (alpha * A) @ X ;  T += beta * Y   (T nullable).
 *   replaces  prop_feat = alpha*adj_norm @ prop_feat ;
 *             target_feat = target_feat + (1-alpha)*prop_feat
 *                                       clustgdd_agent_transduct.py:64-65
 *                                       clustgdd_agent_induct.py:77-78,85-86,93-94
 *   and the index_add_ message passing of distill_recsys.py:340-345 (alpha=1).
 *   The stored value used is fp32(vals[e] * alpha) exactly as `alpha*adj_norm`
 *   produces it.  A is rows_local x n_cols CSR; X has n_cols rows.
 *   Requirements: ldx, ldy, ldt multiples of 4 and X/Y/T 16-byte aligned
 *   (the host pads F up to a multiple of 4).  Row sums are accumulated in
 *   CSR order, one fp32 chain per output element => deterministic. */
int gdr_spmm_prop(int64_t rows_local, int64_t F,
                  const int32_t* rowptr, const int32_t* colidx, const float* vals,
                  float alpha, const float* X, int64_t ldx,
                  float* Y, int64_t ldy,
                  float* T, int64_t ldt, float beta,
                  gdr_stream_t stream);

/* nnz-balanced row blocks for the SpMM (hub-heavy graphs): block c owns the rows r with
 * rowptr[r] + 16 r in [2048 c, 2048 (c+1)) — equal work per CTA, at most 128 rows each.  The plan
 * depends on the sparsity pattern only; build it once per matrix (bounds_out: int32
 * [gdr_spmm_plan_blocks() + 1]) and pass it to gdr_spmm_prop_planned.  Same arithmetic and the
 * same results as gdr_spmm_prop. */
int64_t gdr_spmm_plan_blocks(int64_t n_rows, int64_t nnz);
int     gdr_spmm_plan(int64_t n_rows, int64_t nnz, const int32_t* rowptr, int32_t* bounds_out,
                      gdr_stream_t stream);
int     gdr_spmm_prop_planned(int64_t rows_local, int64_t F,
                              const int32_t* rowptr, const int32_t* colidx, const float* vals,
                              float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy,
                              float* T, int64_t ldt, float beta,
                              const int32_t* bounds, int64_t n_blocks, gdr_stream_t stream);

/* out = a * X  (dense, row-major; used for the t = 0 term (1-alpha)*X). */
int gdr_scale_rows(int64_t rows, int64_t F, float a, const float* X, int64_t ldx,
                   float* out, int64_t ldo, gdr_stream_t stream);

/* ---- stage 3: k-means ------------------------------------------------- */
/* Column mean / variance of X in fp64 -> mean_out f32[D], var_mean_out f64[1]
 * (= mean over columns of the population variance; sklearn/_kmeans.py:285-293),
 * and optionally Xc = X - mean (sklearn/_kmeans.py:1487-1489). */
int64_t gdr_center_columns_ws_bytes(int64_t N, int64_t D);
int     gdr_center_columns(int64_t N, int64_t D, const float* X, int64_t ldx,
                           float* mean_out, double* var_mean_out,
                           float* Xc /*nullable*/, int64_t ldxc,
                           void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* StandardScaler(with_mean, with_std).fit_transform of distill_recsys.py:172 — per-column mean and
 * population variance in fp64 (two passes), constant columns get scale 1, then
 * out = fp32((x - fp32(mean)) / fp32(scale)).  mean_out / scale_out: device f64[D], nullable. */
int64_t gdr_standard_scale_ws_bytes(int64_t N, int64_t D);
int     gdr_standard_scale(int64_t N, int64_t D, const float* X, int64_t ldx, float* out, int64_t ldo,
                           double* mean_out, double* scale_out, void* ws, int64_t ws_bytes,
                           gdr_stream_t stream);

/* Row-partitioned form of the two steps above (multi-GPU): per-rank fp64 column sums
 * (sums_out[0..D) = sum, [D..2D) = sum of squares; all-reduced by the host, which derives
 * mean and tol') and the centring pass with a given mean.  ws: gdr_center_columns_ws_bytes. */
int gdr_column_sums(int64_t N, int64_t D, const float* X, int64_t ldx, double* sums_out,
                    void* ws, int64_t ws_bytes, gdr_stream_t stream);
int gdr_center_apply(int64_t N, int64_t D, const float* X, int64_t ldx, const float* mean,
                     float* Xc, int64_t ldxc, gdr_stream_t stream);

/* E-step.  labels[i] = argmin_j ( |c_j|^2 - 2 x_i . c_j ), first index wins ties.
 *   replaces  _update_chunk_dense                 sklearn/_k_means_lloyd.pyx:196-213
 *   precision_mode 0: exact fp32 SIMT everywhere.
 *   precision_mode 1: tcgen05 3xTF32 tensor-core screen, rows whose best/second
 *                     margin is inside the error band are re-scored in exact fp32.
 *   n_changed_dev (nullable, device int32) += #rows whose label differs from
 *   labels_prev (nullable).  best_out (nullable) = the winning partial distance. */
int64_t gdr_kmeans_assign_ws_bytes(int64_t N, int64_t K, int64_t D, int precision_mode);
int     gdr_kmeans_assign(int64_t N, int64_t K, int64_t D,
                          const float* X, int64_t ldx, const float* C, int64_t ldc,
                          int32_t* labels, const int32_t* labels_prev,
                          int32_t* n_changed_dev, float* best_out,
                          int precision_mode,
                          void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* Tensor-core E-step with a cached operand split (the Lloyd loop calls prepare once per
 * fit, X being constant across iterations, then assign_tc every iteration):
 *   prepare: X -> (X_hi, X_lo) TF32 pair, rows zero-padded to a multiple of 32 floats, + |x_i|.
 *   assign_tc: 3xTF32 tcgen05/TMA GEMM with fused |c|^2 add and (best, second, argmin)
 *   epilogue; rows whose margin second-best is within 2^-15 |x_i| max|c_j| are re-scored by
 *   the exact fp32 kernel.  *n_refined_dev (nullable) receives how many rows have their margin between the
 *   two nearest centres within that band: judged on the exact fp32 distances for the rows the two-level screen
 *   decides on candidate centres, on the 3xTF32 distances for every other row.
 *   Supports D <= 128 (GDR_EUNSUPPORTED otherwise). */
int64_t gdr_kmeans_tc_xsplit_bytes(int64_t N, int64_t D);
int     gdr_kmeans_tc_prepare(int64_t N, int64_t D, const float* X, int64_t ldx,
                              void* xsplit, int64_t xsplit_bytes, gdr_stream_t stream);
int64_t gdr_kmeans_assign_tc_ws_bytes(int64_t N, int64_t K, int64_t D);
int     gdr_kmeans_assign_tc(int64_t N, int64_t K, int64_t D,
                             const float* X, int64_t ldx, const void* xsplit,
                             const float* C, int64_t ldc,
                             int32_t* labels, const int32_t* labels_prev,
                             int32_t* n_changed_dev, float* best_out, int32_t* n_refined_dev,
                             void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* MiniBatchKMeans centre update for one batch (sklearn/cluster/_k_means_minibatch.pyx:56-110, behind
 * clustgdd_agent_transduct.py:103, clustgdd_agent_induct.py:132, distill_recsys.py:174-176):
 * C_new[c] = (C_old[c] * weight_sums[c] + sum of the batch rows labelled c, in batch order) / (weight_sums[c] + count),
 * weight_sums[c] += count; a cluster without members in the batch keeps its old centre.  Same fp32 chain as sklearn. */
int gdr_minibatch_update(int64_t B, int64_t K, int64_t D, const float* Xb, int64_t ldx, const int32_t* labels,
                         const float* C_old, int64_t ldc_old, float* C_new, int64_t ldc_new, float* weight_sums,
                         gdr_stream_t stream);

/* One complete Lloyd run from given (already mean-centred) initial centres — the loop of
 * _kmeans_single_lloyd (sklearn/_kmeans.py:630-758) behind KMeans(...).fit()
 * (clustgdd_agent_transduct.py:105, distill_recsys.py:178).  C_inout holds the initial
 * centres on entry and the final centres on return; labels_out int32[N] (device).
 * inertia / n_iter / info[2] = {strict_convergence, relocation_rounds} are HOST outputs.
 * SYNCHRONISES the stream once per iteration (24-byte convergence status). */
int64_t gdr_kmeans_lloyd_ws_bytes(int64_t N, int64_t K, int64_t D, int precision_mode);
int     gdr_kmeans_lloyd(int64_t N, int64_t K, int64_t D, const float* Xc, int64_t ldx,
                         float* C_inout, int64_t ldc, int32_t* labels_out,
                         int max_iter, double tol_abs, int precision_mode,
                         double* inertia_out_host, int32_t* n_iter_out_host, int32_t* info_out_host,
                         int verbose, void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* Greedy k-means++ seeding (sklearn/_kmeans.py:180-278; the default init of the reference's
 * KMeans(n_clusters=n) at clustgdd_agent_transduct.py:105 and distill_recsys.py:178).
 * The caller draws the random numbers on the host exactly as sklearn consumes them:
 * first_center = random_state.choice(N, p=uniform) and, for each of the K-1 further centres,
 * rand_vals_host[(c-1)*n_trials ...] = random_state.uniform(size=n_trials), n_trials = 2 + int(ln K).
 * All distance / potential / cumulative-sum arithmetic runs on the device (fp64 accumulation,
 * fixed order).  centers_out [K][ldc] (device); indices_out_dev int64[K] nullable.
 * n_trials <= 16.  Synchronises the stream once at the end. */
int64_t gdr_kmeans_plusplus_ws_bytes(int64_t N, int64_t K, int64_t D, int n_trials);
int     gdr_kmeans_plusplus(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx,
                            int64_t first_center, const double* rand_vals_host, int n_trials,
                            float* centers_out, int64_t ldc, int64_t* indices_out_dev,
                            void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* M-step, part 1: per-cluster sums and counts.
 *   replaces  centers_new[label] += X[i]; weight[label] += 1
 *                                                 sklearn/_k_means_lloyd.pyx:215-218
 *             and the Python cluster-mean loop    clustgdd_agent_transduct.py:121-125
 *             and index_add_/bincount pooling     distill_recsys.py:628-636
 *   Deterministic: members of a cluster are summed in ascending row order, one
 *   fp32 chain per output element (== np.add.at order).  gdr_segment_sum_dist (with the
 *   communicator calls below) gives the same bits on a row partition. */
int64_t gdr_segment_sum_ws_bytes(int64_t N, int64_t K, int64_t D);
int     gdr_segment_sum(int64_t N, int64_t K, int64_t D,
                        const float* X, int64_t ldx, const int32_t* labels,
                        float* sums, int64_t lds, int32_t* counts,
                        void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* counts[k] = #{i : labels[i] == k}  (cluster sizes: torch.bincount at
 * distill_recsys.py:630, column sums of the one-hot at transduct :238).
 * Labels outside [0,K) set status_dev[0] (nullable) and are skipped. */
int gdr_label_histogram(int64_t N, int64_t K, const int32_t* labels, int32_t* counts,
                        int32_t* status_dev, gdr_stream_t stream);

/* M-step, part 2: average + centre shift.
 *   replaces  _average_centers / _center_shift    sklearn/_k_means_common.pyx:274-311
 *   C_new[j] = sums[j] * (1.0f / counts[j]); an empty cluster takes the centre of
 *   the (first) largest cluster.  stats_dev f64[2 + K]: [0] = sum_j |C_new_j-C_old_j|^2,
 *   [1] = number of empty clusters, [2..] scratch (per-cluster shift).  mean_mode 1: empty -> NaN row, no shift
 *   (the reference's torch `.mean(dim=0)` of an empty selection, transduct :122). */
int gdr_kmeans_finalize(int64_t K, int64_t D, const float* sums, int64_t lds,
                        const int32_t* counts, const float* C_old, int64_t ldc_old,
                        float* C_new, int64_t ldc_new, double* stats_dev, int mean_mode,
                        gdr_stream_t stream);

/* Empty-cluster relocation  (sklearn/_k_means_common.pyx:167-211): for the idx-th
 * empty cluster move the idx-th farthest sample (distance to its centre in
 * C_old) out of its cluster.  Mutates sums/counts in place.  SYNCHRONISES. */
int64_t gdr_kmeans_relocate_ws_bytes(int64_t N, int64_t K, int64_t D);
int     gdr_kmeans_relocate(int64_t N, int64_t K, int64_t D,
                            const float* X, int64_t ldx, const float* C_old, int64_t ldc,
                            const int32_t* labels, float* sums, int64_t lds, int32_t* counts,
                            void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* inertia = sum_i |x_i - c_label(i)|^2  accumulated in fp64 (deterministic).
 *   replaces  _inertia_dense                      sklearn/_k_means_common.pyx:94-124 */
int64_t gdr_inertia_ws_bytes(int64_t N, int64_t D);
int     gdr_inertia(int64_t N, int64_t D, const float* X, int64_t ldx,
                    const float* C, int64_t ldc, const int32_t* labels, double* out_dev,
                    void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* out[i, :] = X[i, :] + sign * v[:]   (centres += X_mean, sklearn/_kmeans.py:1546) */
int gdr_add_row_vector(int64_t rows, int64_t D, float* X, int64_t ldx, const float* v,
                       float sign, gdr_stream_t stream);

/* ---- stage 4: cluster-coarsened graph -------------------------------- */
/* Segmented edge counting:  for every input edge e (src,dst[,w]) form the key
 * (labels_src[src], labels_dst[dst]); output the CSR (n_src x n_dst) of
 *   counts[a,b] = #edges with that key   (int32, exact)
 *   wsum[a,b]   = sum of w over them     (fp32; nullable).  CSR input whose coarse row fits in shared memory (n_dst
 *                 <= ~17 K with weights): one CTA per coarse row accumulates the cells there, the weights as 64-bit
 *                 fixed-point integers with a step q ~ 2^-48 of the cluster's largest |w| -> bit-reproducible, within
 *                 n_cell * q / 2 plus one fp32 rounding of the exact sum (one ulp only when the cell is at least about
 *                 n_cell * q * 2^24).  Otherwise (COO input,
 *                 wider rows, gdr_debug_set("coarsen_dense", 0)): radix sort by cell, fp32 sums in input order.
 *   replaces  build_condensed_bipartite           distill_recsys.py:184-201
 *             graph_compress (P^T A P)            clustgdd_agent_transduct.py:234-250
 *                                                 clustgdd_agent_induct.py:258-274
 *   Edges come either as COO (src/dst int64) or, when src == NULL, as CSR
 *   (csr_rowptr/csr_colidx int32 with n_rows rows).  drop_diag removes a == b.
 *   Output capacity: min(E, n_src*n_dst).  *nnz_out_dev = stored entries. */
int64_t gdr_coarsen_ws_bytes(int64_t E, int64_t n_src, int64_t n_dst);
int     gdr_coarsen(int64_t E, const int64_t* src, const int64_t* dst,
                    int64_t n_rows, const int32_t* csr_rowptr, const int32_t* csr_colidx,
                    const float* w,
                    const int32_t* labels_src, const int32_t* labels_dst,
                    int64_t n_src, int64_t n_dst, int drop_diag,
                    int32_t* rowptr, int32_t* colidx, int32_t* counts, float* wsum,
                    int64_t* nnz_out_dev,
                    void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* Multi-GPU merge of per-rank coarsened graphs (row-partitioned stage 4): every rank scatters
 * its local result into a dense n_src x n_dst pair (int32 counts, f32 weight sums; both are
 * zeroed first), the host all-reduces them (NCCL sum), and dense_to_coarse compacts the
 * merged matrices back to CSR (cells with count 0 are dropped, columns ascending). */
int gdr_coarse_scatter_dense(int64_t n_src, int64_t n_dst, const int32_t* rowptr, const int32_t* colidx,
                             const int32_t* counts, const float* wsum /*nullable*/,
                             int32_t* dense_counts, float* dense_wsum /*nullable*/, gdr_stream_t stream);
int64_t gdr_dense_to_coarse_ws_bytes(int64_t n_src);
int gdr_dense_to_coarse(int64_t n_src, int64_t n_dst, const int32_t* dense_counts,
                        const float* dense_wsum /*nullable*/, int32_t* rowptr, int32_t* colidx,
                        int32_t* counts, float* wsum /*nullable*/, int64_t* nnz_out_dev,
                        void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* graph_compress value pass: vals[e] = wsum[e] / (size[a] * size[b])  computed as
 * fp32 (wsum * (1/size[a])) * (1/size[b])  (transduct :237-244). */
int gdr_coarsen_scale(int64_t n_src, const int32_t* rowptr, const int32_t* colidx,
                      const float* wsum, const int32_t* size_src, const int32_t* size_dst,
                      float* vals_out, gdr_stream_t stream);

/* Multi-GPU propagation helper: remap the (global) column ids of a row block to the rows of the chunk-major
 * gathered operand used by the row-chunk pipelined hop: node (rank r, local row i = c*chunk_rows + o) ->
 * c*world*chunk_rows + r*chunk_rows + o. */
int gdr_remap_chunk_major(int64_t nnz, const int32_t* colidx_in, int64_t rows_per, int64_t chunk_rows,
                          int64_t world, int32_t* colidx_out, gdr_stream_t stream);

/* ---- edge scoring + top-k sparsification (SURVEY §8f item 1; between stages 3 and 4) ----
 * All on a device CSR whose stored order is the reference's coalesced COO order
 * (rows = src, colidx = dst).
 *   gdr_row_sums_f32        degree = adj @ ones, fp32, stored order   utils_clustgdd.py:153-154
 *   gdr_er_lower            ER_estimator  v/deg[src] + v/deg[dst]      utils_clustgdd.py:151-162
 *                           (deg_scratch: n floats, receives the degrees)
 *   gdr_edge_cosine_scale   vals_out = vals * cosine_similarity(ebd[src], ebd[dst], eps)
 *                           (attaw_ER_estimator, utils_clustgdd.py:168-172; inv_norm_scratch: n floats)
 *   gdr_softmax_rows        F.softmax(ebd, dim=-1)                     clustgdd_agent_transduct.py:158
 *   gdr_class_edge_weight   (prob[src,cls] * prob[dst,cls]) * er       clustgdd_agent_transduct.py:164-167
 *   gdr_topk_filter_csr     torch.topk(weight, k) + COO rebuild        clustgdd_agent_transduct.py:142-151,168-181
 *                           keeps every entry above the k-th largest weight plus the first entries (stored
 *                           order) equal to it, exactly k in total; output is a sorted CSR (capacity k);
 *                           radix select + two scans, no host synchronisation, no sort.
 * Row-block forms (one rank's rows [row_lo, row_lo + n_local) of a row-partitioned graph, column ids global): per-row
 * operands are read at row_lo + r, per-column operands at colidx[j]; every value has the bits of the whole-graph call.
 *   gdr_er_lower_rows           er with a caller-supplied GLOBAL degree vector deg [n_global]
 *   gdr_edge_cosine_scale_rows  global ebd [n_global][ld]; inv_norm_scratch: n_global floats (all norms are computed)
 * gdr_sparsify_classes_dist (below, with gdr_sparsify_classes) runs the top-k across the ranks. */
int gdr_row_sums_f32(int64_t n, const int32_t* rowptr, const float* vals, float* deg_out, gdr_stream_t stream);
int gdr_er_lower(int64_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx, const float* vals,
                 float* deg_scratch, float* er_out, gdr_stream_t stream);
int gdr_edge_cosine_scale(int64_t n, int64_t nnz, int64_t C, const int32_t* rowptr, const int32_t* colidx,
                          const float* vals, const float* ebd, int64_t ld, float eps,
                          float* inv_norm_scratch, float* vals_out, gdr_stream_t stream);
int gdr_er_lower_rows(int64_t n_local, int64_t nnz, int64_t row_lo, const int32_t* rowptr, const int32_t* colidx,
                      const float* vals, const float* deg, float* er_out, gdr_stream_t stream);
int gdr_edge_cosine_scale_rows(int64_t n_local, int64_t nnz, int64_t C, int64_t row_lo, int64_t n_global,
                               const int32_t* rowptr, const int32_t* colidx, const float* vals, const float* ebd,
                               int64_t ld, float eps, float* inv_norm_scratch, float* vals_out, gdr_stream_t stream);
int gdr_softmax_rows(int64_t n, int64_t C, const float* X, int64_t ld, float* out, int64_t ldo,
                     gdr_stream_t stream);
int gdr_class_edge_weight(int64_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                          const float* er, const float* prob, int64_t ldp, int64_t cls, float* w_out,
                          gdr_stream_t stream);
/* ---- multi-GPU exchange steps (SURVEY 8e; one process per GPU, NCCL over NVLink) -------------------
 * The reference is single-device (clustgdd_agent_transduct.py:38-129 runs every stage on one `device`), so
 * these entry points replace nothing in it: they are the exchanges a row partition of the same path needs.
 * NCCL is bound at run time (dlopen of the already mapped libnccl.so.2, else the system copy / $GDR_NCCL_LIB).
 * Protocol: rank 0 calls gdr_comm_unique_id, the host framework broadcasts the 128 bytes, every rank calls
 * gdr_comm_init (collective).  All exchange calls are collective and are enqueued on `stream`.
 * Collective entry check of the row-partitioned entry points (gdr_kmeans_plusplus_dist, gdr_dense_gram_dist,
 * gdr_sparsify_classes_dist, gdr_segment_sum_dist): a rank does not return on its own argument checks.  Every rank all-gathers its verdict,
 * its row block and the values every rank must pass alike (listed with each entry point) through a small buffer the
 * communicator owns (allocated by gdr_comm_init), reads them back and synchronises the stream once.  A rank whose own
 * arguments are rejected returns its own code (GDR_EINVAL, GDR_EWORKSPACE, GDR_EUNSUPPORTED, GDR_ERANGE), every other
 * rank GDR_EINVAL.  Values that differ between ranks, a row block that does not start where the previous rank's ends,
 * or blocks that do not cover the global row count return GDR_EINVAL on every rank.  A failure of the exchange itself
 * returns GDR_ECUDA.  After any rejection the communicator stays usable. */
typedef struct gdr_comm gdr_comm_t;
int gdr_comm_unique_id(void* id128_host);
int gdr_comm_init(gdr_comm_t** comm_out, const void* id128_host, int rank, int world);
int gdr_comm_destroy(gdr_comm_t* comm);
int gdr_comm_info(const gdr_comm_t* comm, int* rank_host, int* world_host, int* nccl_version_host);
/* stage 2 (clustgdd_agent_transduct.py:59-65 on a row partition): full[r*rows_per_rank + i][:] = rank r's local[i][:];
 * rows are ld floats wide (padding columns travel with the row), every rank passes the same rows_per_rank. */
int gdr_allgather_rows(gdr_comm_t* comm, const float* local, int64_t rows_per_rank, int64_t ld, float* full,
                       gdr_stream_t stream);
int gdr_allgather_bytes(gdr_comm_t* comm, const void* local, int64_t bytes_per_rank, void* full, gdr_stream_t stream);
/* stage 3 (sklearn/_k_means_lloyd.pyx:124-152: the per-thread partial sums are reduced there; here per GPU):
 * sums[n_floats] (f32) and ints[n_ints] (i32: counts, n_changed) summed over the ranks IN PLACE as ONE grouped
 * NCCL operation; every rank receives bit-identical results. */
int gdr_allreduce_centroids(gdr_comm_t* comm, float* sums, int64_t n_floats, int32_t* ints, int64_t n_ints,
                            gdr_stream_t stream);
int gdr_allreduce_f64(gdr_comm_t* comm, double* buf, int64_t n, int op_max, gdr_stream_t stream);
/* stage 1 / 4: variable all-to-all of fixed-size elements (edge buckets by owner row, (cell, count, sum) runs by key
 * range).  Offsets / counts are HOST arrays of `world` entries, in elements of elem_bytes. */
int gdr_alltoallv(gdr_comm_t* comm, const void* send, const int64_t* send_off_host, const int64_t* send_cnt_host,
                  void* recv, const int64_t* recv_off_host, const int64_t* recv_cnt_host, int64_t elem_bytes,
                  gdr_stream_t stream);
/* One MiniBatchKMeans batch on a row partition (sklearn/_kmeans.py:2154-2166 behind distill_recsys.py:174-176): every
 * rank ends with Xb[j][0..ldb) = the bytes of global row idx[j] (columns D..ldb zero) and, when C != NULL,
 * labels_b[j] = that row's label against C with the bits of gdr_kmeans_assign(precision_mode = 0).  C == NULL
 * assembles the rows only (labels_b is then ignored).  Device arrays: idx[m] (global row ids, the same on every rank,
 * duplicates allowed), order[m] (the batch positions grouped by owning rank: rank order, ascending within a rank).
 * counts_host[world] = positions each rank owns (sum m).  Every rank derives idx, order and counts from the same host
 * draws and row offsets, so nothing about them is exchanged; X_local holds global rows [row_lo, row_lo + n_local).
 * Steps: the owned rows are packed into a compact buffer in batch order, labelled there by k_row_sqnorm +
 * k_assign_simt (each row tile scans all K, so a row's label does not depend on which rows share the launch), sent to
 * every rank in ONE group of NCCL sends / receives (none at world 1) and placed at their positions.
 * COLLECTIVE, but a per-step exchange like gdr_alltoallv: no collective entry check and no stream synchronisation.
 * The caller agrees on every argument once (DistMiniBatchKMeans does so at fit entry); every check here is local and
 * precedes the exchange, and the workspace size depends only on agreed values (m, K, D), so a workspace rejection is
 * the same on every rank.  The world argument of the size query is unused. */
int64_t gdr_minibatch_batch_dist_ws_bytes(int64_t m, int64_t K, int64_t D, int world);
int     gdr_minibatch_batch_dist(gdr_comm_t* comm, int64_t m, const int64_t* idx, const int32_t* order,
                                 const int64_t* counts_host, int64_t row_lo, int64_t n_local, int64_t K, int64_t D,
                                 const float* X_local, int64_t ldx, const float* C, int64_t ldc, float* Xb, int64_t ldb,
                                 int32_t* labels_b, void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* gdr_segment_sum on a row partition (the cluster means of clustgdd_agent_transduct.py:116-127 and the pooling of
 * distill_recsys.py:623-636 on row-partitioned features and labels).  COLLECTIVE over comm.  Each rank passes its rows
 * X[n_local][ldx] and labels, global rows [row_lo, row_lo + n_local) (n_local = 0 allowed, X and labels may then be
 * NULL).  sums[K][lds] and counts[K] come out on every rank with the bits gdr_segment_sum gives on the rows concatenated
 * in rank order (columns [D, lds) zero).  gdr_segment_sum sums each element as one fp32 chain from +0.0 over the
 * cluster's members in ascending row order, so cluster c's chain is rank 0's members, then rank 1's, and so on.
 * Steps: this rank's counts (gdr_label_histogram; a label outside [0, K) is this rank's GDR_ERANGE, read back with a
 * stream synchronisation); the collective entry check (see gdr_comm_init) on K, D and lds, with n_local < 2^31 per rank
 * and fewer than 2^31 rows in all; this rank's stable sort by label (gdr_segment_sum's code and digit count), before it
 * receives anything; then rank 0 zeroes sums and rank q > 0 receives K x lds floats from rank q - 1 into sums (NCCL
 * point-to-point), continues every chain over its members from the received value, and sends sums to rank q + 1 (an
 * empty rank hands on what it received).  The last rank's sums are sent to all, and the counts are all-reduced (exact
 * int32 sums).  Synchronises the stream twice: the label read-back and the entry check. */
int64_t gdr_segment_sum_dist_ws_bytes(int64_t n_local, int64_t K, int64_t D);
int     gdr_segment_sum_dist(gdr_comm_t* comm, int64_t row_lo, int64_t n_local, int64_t K, int64_t D, const float* X,
                             int64_t ldx, const int32_t* labels, float* sums, int64_t lds, int32_t* counts, void* ws,
                             int64_t ws_bytes, gdr_stream_t stream);
/* Symmetric buffers: the same device allocation on every rank, mapped into every peer over NVLink (CUDA IPC), so that a
 * kernel can store straight into the other GPUs' copies.  gdr_symm_create / _destroy are collective (and, with
 * gdr_comm_init's entry-check buffer, the only entry points of this library that allocate device memory).
 * gdr_symm_barrier is stream-ordered: when it completes on a rank, everything every rank enqueued before ITS barrier
 * call — including its stores into this rank's copy — is done and visible.  gdr_symm_put_rows: rows of `src` ->
 * offset dst_offset_bytes of every copy (one read, world posted stores).
 * gdr_symm_scatterv: the variable all-to-all / all-gather of stages 1 and 4 without NCCL — block p of `send`
 * (send_cnt_host[p] elements of elem_bytes at element send_off_host[p]) is stored at BYTE offset dst_off_bytes_host[p]
 * of rank p's copy (its own included), one kernel, 16-byte posted NVLink stores; bracket it with gdr_symm_barrier.
 * gdr_spmm_prop_mc: one hop of clustgdd_agent_transduct.py:59-65 on a row partition FUSED with the all-gather of its
 * result: the SpMM epilogue stores every output row into row dst_row_offset + r of the matrix at dst_offset_bytes of
 * EVERY copy, i.e. straight into the gathered operand of the next hop (Y, this rank's plain copy, is optional). */
typedef struct gdr_symm gdr_symm_t;
int gdr_symm_create(gdr_comm_t* comm, int64_t bytes, gdr_symm_t** symm_out);
int gdr_symm_destroy(gdr_symm_t* symm);
int gdr_symm_info(const gdr_symm_t* symm, void** local_ptr_host, int64_t* bytes_host);
int gdr_symm_barrier(gdr_symm_t* symm, gdr_stream_t stream);
int gdr_symm_put_rows(gdr_symm_t* symm, int64_t dst_offset_bytes, const float* src, int64_t rows, int64_t ld,
                      int include_self, gdr_stream_t stream);
int gdr_symm_scatterv(gdr_symm_t* symm, const void* send, const int64_t* send_off_host, const int64_t* send_cnt_host,
                      const int64_t* dst_off_bytes_host, int64_t elem_bytes, gdr_stream_t stream);
int gdr_spmm_prop_mc(gdr_symm_t* symm, int64_t dst_offset_bytes, int64_t dst_ld, int64_t dst_row_offset,
                     int64_t rows_local, int64_t F, const int32_t* rowptr, const int32_t* colidx, const float* vals,
                     float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy, float* T, int64_t ldt, float beta,
                     const int32_t* bounds, int64_t n_blocks, gdr_stream_t stream);
/* stage 4 on a row partition (clustgdd_agent_transduct.py:234-250): every rank coarsens its local edges
 * (gdr_coarsen), turns the result into 16-byte records [cell key = (a << bits(n_dst)) | b ; (count << 32) | weight-sum
 * bits] (gdr_coarse_records; uint64[m][2]), exchanges them by key range (coarse row a -> owner rank, gdr_alltoallv) and merges what it
 * receives: stable sort by cell, integer count sums (exact, independent of the rank count), fp32 weight sums in
 * source-rank order (deterministic).  Output: the CSR of coarse rows [a_lo, a_lo + n_rows). */
int     gdr_coarse_records(int64_t n_src, int64_t n_dst, const int32_t* rowptr, const int32_t* colidx,
                           const int32_t* counts, const float* wsum, uint64_t* records_out, gdr_stream_t stream);
int64_t gdr_coarse_merge_ws_bytes(int64_t m);
int     gdr_coarse_merge(int64_t m, const uint64_t* records, int64_t a_lo, int64_t n_rows, int64_t n_src,
                         int64_t n_dst, int32_t* rowptr, int32_t* colidx, int32_t* counts, float* wsum,
                         int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* distill_recsys on a row partition (users and items each split over the ranks):
 *   gdr_bipartite_norm_block   distill_recsys.py:329-335 for a row block of R (or of R^T): own row degrees
 *                              (gdr_row_sums_f32) + the all-gathered degrees of the other side
 *   gdr_column_moments         second pass of StandardScaler (distill_recsys.py:172) on a row block: fp64
 *                              [sum (x - mean) | sum (x - mean)^2], to be all-reduced (first pass: gdr_column_sums)
 *   gdr_standardize_apply      fp32((x - mean) / scale) with the reduced column parameters */
int gdr_bipartite_norm_block(int64_t n_rows, int64_t nnz, const int32_t* rowptr, const int32_t* colidx, const float* w,
                             const float* deg_rows, const float* deg_cols, float eps, float* norm_out,
                             gdr_stream_t stream);
int gdr_column_moments(int64_t N, int64_t D, const float* X, int64_t ldx, const double* mean64, double* sums_out,
                       void* ws, int64_t ws_bytes, gdr_stream_t stream);
int gdr_standardize_apply(int64_t N, int64_t D, const float* X, int64_t ldx, const float* mean32, const float* scale32,
                          float* out, int64_t ldo, gdr_stream_t stream);
/* stage 1 on a row partition, routing form (utils.py:66-67, utils_graphsaint.py:20-22, distill_recsys.py:110-117 from a
 * SLICE of the pair list per rank): gdr_edges_route packs every pair (and its mirror when symmetrize) into a key
 * (row << bits(n_cols)) | col tagged with the owner rank of the row (row / rows_per) in the top byte and groups the keys by
 * owner with one stable partition pass; owner_starts_dev[0..128] = first key of every owner; status bit 0 = index out of
 * range, bit 1 = the pair (0, 0) occurs (deep_robust_utils.py:199).  After the all-to-all gdr_csr_from_keys sorts the keys
 * a rank received and emits the CSR of its row block (binarised, or with the multiplicity of every pair as value). */
int64_t gdr_edges_route_ws_bytes(int64_t E, int symmetrize);
int     gdr_edges_route(int64_t E, const int64_t* row, const int64_t* col, int64_t n_rows, int64_t n_cols, int symmetrize,
                        int64_t rows_per, int world, uint64_t* keys_out, int64_t* owner_starts_dev, int32_t* status_dev,
                        void* ws, int64_t ws_bytes, gdr_stream_t stream);
int64_t gdr_csr_from_keys_ws_bytes(int64_t m);
int     gdr_csr_from_keys(int64_t m, const uint64_t* keys_in, int64_t row_lo, int64_t n_rows_local, int64_t n_cols,
                          int binarize, int32_t* rowptr, int32_t* colidx, float* vals, int64_t* nnz_out_dev, void* ws,
                          int64_t ws_bytes, gdr_stream_t stream);
/* stage 4 on a row partition, routing form (default): gdr_coarsen_route turns every local edge into a (cell key, weight)
 * pair tagged with the owner rank of its coarse row (top byte of the key; dropped diagonal pairs: bucket 127) and groups
 * the pairs by owner with ONE stable partition pass — keys_out / w_out sorted by owner, owner_starts_dev[0..128] the
 * first pair of every owner.  After the all-to-all the owner runs gdr_coarse_merge_edges: sort + integer run lengths +
 * fp32 sums in the exchange order, which is the global CSR order — counts AND sums are bit-identical to the SORT form of
 * the single-device gdr_coarsen (COO input, or a coarse row too wide for shared memory; its default for a CSR is the
 * shared-memory form, whose owner-side counterpart is gdr_coarse_merge_edges_dense below).  Output: CSR of the coarse
 * rows [a_lo, a_lo + n_rows).  (clustgdd_agent_transduct.py:234-250, distill_recsys.py:184-201) */
int64_t gdr_coarsen_route_ws_bytes(int64_t E);
int     gdr_coarsen_route(int64_t E, const int64_t* src, const int64_t* dst, int64_t n_rows, const int32_t* csr_rowptr,
                          const int32_t* csr_colidx, const float* w, const int32_t* labels_src, const int32_t* labels_dst,
                          int64_t n_src, int64_t n_dst, int drop_diag, int world, uint64_t* keys_out, float* w_out,
                          int64_t* owner_starts_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream);
int64_t gdr_coarse_merge_edges_ws_bytes(int64_t m);
int     gdr_coarse_merge_edges(int64_t m, const uint64_t* keys_in, const float* w_in, int64_t a_lo, int64_t n_rows,
                               int64_t n_src, int64_t n_dst, int32_t* rowptr, int32_t* colidx, int32_t* counts,
                               float* wsum, int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* The same merge without sorting the cells: the routed pairs are grouped by coarse row (a stable sort on the row bits
 * only) and one CTA per coarse row accumulates its cells in shared memory — integer counts and 64-bit fixed-point weight
 * sums, as gdr_coarsen does on one GPU.  cluster_edges / cluster_wmax_bits: per coarse row of the WHOLE graph, the number
 * of edges leaving it and the bit pattern of their largest |weight| (gdr_cluster_stats on every rank's rows, summed /
 * maxed over the ranks): they fix the fixed-point step, so every term is rounded as on one GPU and the sums are
 * bit-identical to gdr_coarsen's for any number of ranks.  _ok: 1 when a coarse row of n_dst cells fits in shared memory. */
int     gdr_cluster_stats(int64_t n_rows, const int32_t* rowptr, const float* w, const int32_t* labels, int64_t n_src,
                          int32_t* nodes_out, int32_t* edges_out, uint32_t* wmax_bits_out, int32_t* status_dev,
                          gdr_stream_t stream);
int     gdr_coarse_merge_edges_dense_ok(int64_t n_rows, int64_t n_dst, int has_weights);
int64_t gdr_coarse_merge_edges_dense_ws_bytes(int64_t m, int64_t n_rows);
int     gdr_coarse_merge_edges_dense(int64_t m, const uint64_t* keys_in, const float* w_in, int64_t a_lo, int64_t n_rows,
                                     int64_t n_src, int64_t n_dst, const int32_t* cluster_edges,
                                     const uint32_t* cluster_wmax_bits, int32_t* rowptr, int32_t* colidx, int32_t* counts,
                                     float* wsum, int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* gdr_kmeans_lloyd on a row partition: Xc_local = this rank's N_local rows (may be 0) of the mean-centred matrix of
 * N_total rows, centres replicated.  Each iteration all-reduces [K x ld sums | K counts | n_changed] inside the replayed
 * CUDA graph; the replicated centres stay bit-identical across ranks; empty clusters are relocated from the globally
 * farthest rows (_k_means_common.pyx:167-211).  Workspace: gdr_kmeans_lloyd_ws_bytes(N_local, ...).  inertia is the
 * global WCSS.  SYNCHRONISES the stream once per iteration (24-byte status), like gdr_kmeans_lloyd. */
int gdr_kmeans_lloyd_dist(gdr_comm_t* comm, int64_t N_local, int64_t N_total, int64_t K, int64_t D,
                          const float* Xc_local, int64_t ldx, float* C_inout, int64_t ldc, int32_t* labels_out,
                          int max_iter, double tol_abs, int precision_mode, double* inertia_out_host,
                          int32_t* n_iter_out_host, int32_t* info_out_host, int verbose, void* ws, int64_t ws_bytes,
                          gdr_stream_t stream);
/* gdr_kmeans_plusplus on a row partition: the same greedy D^2 seeding without gathering X.  COLLECTIVE over comm.
 * X_local = this rank's N_local rows (N_local = 0 allowed); the ranks' blocks in rank order are the global row order
 * (the call all-gathers N_local once and derives every rank's row offset and N_total).  first_center and
 * indices_out_dev hold global row ids.  Collective entry check (see gdr_comm_init) on first_center, n_trials, K, D and
 * a checksum of the host draws (rand_vals_host as for gdr_kmeans_plusplus).  Same checks as gdr_kmeans_plusplus:
 * n_trials <= 16, K <= N_total, and the shared-memory plan for n_trials * D.  centers_out [K][ldc] (device) comes out
 * bit-identical on every rank.
 * Per round: the owner of each draw (first rank with rows whose prefix P_r + T_r reaches u * pot) finds the row with
 * gdr_kmeans_plusplus's search and publishes it (all-gather A; the rows are copied, never summed); one pass over
 * X_local scores all candidates; each rank's fp64 totals per candidate are all-gathered (B) and added in rank order.
 * Every per-row fp32 distance has the one-GPU bits; only the fp64 totals are grouped by rank, so picks can differ
 * from gdr_kmeans_plusplus only where a draw or a comparison of two candidate potentials falls within fp64 rounding.
 * With one rank the indices and centres are bit-identical to gdr_kmeans_plusplus.  A draw no row reaches becomes row
 * N_total - 1 (np.clip).  One round is captured into a CUDA graph and replayed.  Synchronises the stream twice: after
 * the entry check and at the end. */
int64_t gdr_kmeans_plusplus_dist_ws_bytes(int64_t N_local, int64_t K, int64_t D, int n_trials, int world);
int     gdr_kmeans_plusplus_dist(gdr_comm_t* comm, int64_t N_local, int64_t K, int64_t D,
                                 const float* X_local, int64_t ldx, int64_t first_center,
                                 const double* rand_vals_host, int n_trials,
                                 float* centers_out, int64_t ldc, int64_t* indices_out_dev,
                                 void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* ---- dense fp64 steps of the truncated SVD embeddings (distill_recsys.py:124-155 compute_svd_embeddings; the reference
 * calls scipy's ARPACK svds on the host).  The block Krylov Rayleigh-Ritz of svd.py runs its sparse products on
 * gdr_spmm_prop and everything else here — hand-written, no cuSOLVER / cuBLAS, fixed-order reductions:
 *   gdr_dense_gram        C[p x r] = A^T B, A [N x p], B [N x r] tall-skinny (Gram matrices, projections Q^T Z)
 *   gdr_dense_chol        lower Cholesky factor of an n x n SPD matrix, n <= 128; info_dev[0] = 0 or 1 + failing pivot
 *   gdr_dense_trsm_rows   Y <- Y L^-T (CholeskyQR: Y becomes orthonormal)
 *   gdr_dense_gemm_small  Z <- (beta Z + alpha A P) * colscale, A [N x m] tall, P [m x r] small; fp64 and/or fp32 output
 *   gdr_sym_eig_jacobi    eigen-decomposition of an n x n symmetric matrix by parallel cyclic Jacobi (A is destroyed;
 *                         evals descending, order[k] = column of W holding the k-th eigenvector); SYNCHRONISES per sweep
 *   gdr_dense_gather_cols Wk[:, k] = W[:, order[k]], k < kcols */
int64_t gdr_dense_gram_ws_bytes(int64_t N, int64_t p, int64_t r);
int     gdr_dense_gram(int64_t N, int64_t p, int64_t r, const double* A, int64_t lda, const double* B, int64_t ldb,
                       double* C, int64_t ldc, void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* gdr_dense_gram on a row partition.  COLLECTIVE over comm.  Each rank passes its n_local rows of A and B, global rows
 * [row_lo, row_lo + n_local) of the N_global (n_local = 0 allowed, A and B may then be NULL); C[p x r] comes out on
 * every rank with the bits gdr_dense_gram gives on the concatenated rows, for any number of ranks.  The slabs are
 * gdr_dense_gram's, from N_global; a rank runs each slab's fp64 fma chain over its rows of that slab, continuing the
 * exact accumulators (the carry) handed on by the previous rank when the slab began there, and adds the slabs that end
 * on it to the slab-order running sum it receives (0.0 on rank 0).  Rank q sends rank q + 1 the carry and the running
 * sum (2 p r doubles, NCCL point-to-point); the last rank's sum is C and is sent to all.  Slabs that start on a rank
 * are summed before it receives anything.  Collective entry check (see gdr_comm_init) on N_global, p and r; the row
 * blocks must cover N_global.  Synchronises the stream once, after the entry check.  The `world` argument of
 * gdr_dense_gram_dist_ws_bytes is unused (the workspace does not depend on the rank count); it stays for the ABI. */
int64_t gdr_dense_gram_dist_ws_bytes(int64_t N_global, int64_t p, int64_t r, int world);
int     gdr_dense_gram_dist(gdr_comm_t* comm, int64_t N_global, int64_t row_lo, int64_t n_local, int64_t p, int64_t r,
                            const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc,
                            void* ws, int64_t ws_bytes, gdr_stream_t stream);
int     gdr_dense_chol(int64_t n, const double* S, int64_t lds, double* L, int64_t ldl, int32_t* info_dev, double rel_tol,
                       gdr_stream_t stream);
int     gdr_dense_trsm_rows(int64_t N, int64_t n, double* Y, int64_t ldy, const double* L, int64_t ldl,
                            gdr_stream_t stream);
int     gdr_dense_gemm_small(int64_t N, int64_t m, int64_t r, double alpha, const double* A, int64_t lda, const double* P,
                             int64_t ldp, double beta, double* Z, int64_t ldz, float* Zf, int64_t ldzf,
                             const double* colscale, gdr_stream_t stream);
int64_t gdr_sym_eig_jacobi_ws_bytes(int64_t n);
int     gdr_sym_eig_jacobi(int64_t n, double* A, double* W, double* evals, int32_t* order, int max_sweeps, double tol,
                           int32_t* sweeps_out_host, void* ws, int64_t ws_bytes, gdr_stream_t stream);
int     gdr_dense_gather_cols(int64_t n, int64_t kcols, const double* W, const int32_t* order, double* Wk,
                              gdr_stream_t stream);

/* Induced subgraph  adj[np.ix_(idx, idx)]  (utils_graphsaint.py:34-36, utils.py:127-129) as relabelled COO
 * triplets: row i of the result is node idx[i].  Outputs have the capacity of the source nnz; the caller turns
 * them into a CSR with gdr_coo_to_csr.  idx entries must lie in [0, n). */
int64_t gdr_induced_subgraph_ws_bytes(int64_t n, int64_t m);
int     gdr_induced_subgraph_coo(int64_t n, const int32_t* rowptr, const int32_t* colidx, const float* vals,
                                 int64_t m, const int64_t* idx, int64_t* out_row, int64_t* out_col,
                                 float* out_val, int64_t* nnz_out_dev, void* ws, int64_t ws_bytes,
                                 gdr_stream_t stream);
/* every class of the 'attaw' sparsifier in one call: slice c of rowptr_out [C][n+1], colidx_out / vals_out [C][k],
 * nnz_out_dev [C] receives the graph of class c (weights = (prob[src,c] * prob[dst,c]) * er, top-k, rebuild).
 * Classes are processed in batches (blockIdx.y = class) sized to ~1.5 GB of scratch: ~20 launches per batch. */
int64_t gdr_sparsify_classes_ws_bytes(int64_t n, int64_t nnz, int64_t C);
int     gdr_sparsify_classes(int64_t n, int64_t nnz, int64_t C, const int32_t* rowptr, const int32_t* colidx,
                             const float* vals, const float* er, const float* prob, int64_t ldp, int64_t k,
                             int32_t* rowptr_out, int32_t* colidx_out, float* vals_out, int64_t* nnz_out_dev,
                             void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* gdr_sparsify_classes on a row partition.  COLLECTIVE over comm.  Each rank passes its local CSR block (n_local rows
 * from global row row_lo, nnz local entries, global column ids; n_local = 0 and nnz = 0 allowed), the global er of its
 * local edges, the GLOBAL prob [n_global][ldp] (or NULL: the weight is er itself and C must be 1, for 'vanilla' /
 * 'single') and the GLOBAL k (0 <= k <= total nnz).  Output per class c: this rank's kept edges as a local CSR, slice
 * c of rowptr_out [C][n_local+1] and of colidx_out / vals_out [C][min(k, nnz)], count in nnz_out_dev[c].  The blocks
 * concatenated in rank order are byte-identical to gdr_sparsify_classes / gdr_topk_filter_csr on the whole graph for
 * any number of ranks: the row blocks in rank order are the global stored order, each radix pass sums the ranks'
 * histograms (64-bit counts, one all-reduce per pass and class batch), and the ties at the threshold are shared out
 * in rank order (one all-gather of the per-rank tie counts per batch): rank p keeps its first
 * clamp(k_rem - sum_{q<p} ties_q, 0, ties_p).  Collective entry check (see gdr_comm_init) on C, k, n_global, whether
 * prob is given and the "sparsify_batch" cap; the row blocks must cover n_global, and it also gathers every rank's
 * local nnz.  The class batch is sized from the largest local nnz.  The local nnz keeps the int32 CSR limit
 * (GDR_ERANGE).  Synchronises the stream once, after the entry check. */
int64_t gdr_sparsify_classes_dist_ws_bytes(int64_t n_local, int64_t nnz_local, int64_t C, int world);
int     gdr_sparsify_classes_dist(gdr_comm_t* comm, int64_t n_local, int64_t nnz_local, int64_t row_lo,
                                  int64_t n_global, int64_t C, const int32_t* rowptr, const int32_t* colidx,
                                  const float* vals, const float* er, const float* prob, int64_t ldp, int64_t k,
                                  int32_t* rowptr_out, int32_t* colidx_out, float* vals_out, int64_t* nnz_out_dev,
                                  void* ws, int64_t ws_bytes, gdr_stream_t stream);
int64_t gdr_topk_filter_ws_bytes(int64_t n, int64_t nnz);
int     gdr_topk_filter_csr(int64_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                            const float* vals, const float* weight, int64_t k, int32_t* rowptr_out,
                            int32_t* colidx_out, float* vals_out, int64_t* nnz_out_dev,
                            void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* ---- evaluation: full-ranking top-K recommendation and Recall / Precision / NDCG@K -------------------------
 * The protocol of the reference's recall_at_k (distill_recsys.py:446-497, called at :680 and :733) and of
 * Rankformer's metrics (Rankformer/code/model.py:27-53): score every item for a user, drop the user's training
 * items, keep the K best, count hits against the held-out items.  The definitions below are this library's.
 *
 * gdr_topk_scores: row r of the output is user u = rows[r] (rows == NULL: u = r, n_rows <= n_users).
 *   s(u, j) = fp32 chain  acc = 0; for t < d: acc = fmaf(U[u, t], I[j, t], acc)   (-0 reported as +0)
 *   items_out[r][0..k) = the k items j not in exclusion row u, by (score desc, j asc); a row with fewer eligible
 *   items is padded with item -1 / score -inf.  scores_out holds the exact scores.  Every stored entry of the
 *   exclusion CSR (n_users x n_items, both pointers NULL = none) excludes its item, whatever its value.
 *   The score matrix is never held: either an exact SIMT product one row slab at a time (scratch of a few hundred MB)
 *   or, for d <= 128 and k <= 256 on large products, a 3xTF32 tensor-core screen that keeps per user only the
 *   candidates within twice a proven error band of a running top-k threshold and re-scores them exactly (rows whose
 *   candidate list overflows finish on the exact path).  The choice is automatic (debug key "topk_path": 1 exact,
 *   2 tensor core); the tensor-core path SYNCHRONISES the stream once (to size the exact finish of overflowed rows).
 *   status_dev (device int32, zeroed by the caller): bit 0 = a non-finite value in a used row of U or in I,
 *   bit 1 = a user id outside [0, n_users).  Outputs are deterministic, identical on both paths, and bit-identical to
 *   the fmaf chain of a correctly rounding CPU fmaf (the test reference tests/topk_ref.c).
 * gdr_ranking_metrics: items [n_rows][ldit] (from gdr_topk_scores), test CSR n_users x n_items with sorted
 *   columns.  For every row with |test_u| > 0 and every K = ks_host[q] <= k:
 *     hits = |{i < K : items[r][i] in test_u}|, recall = hits / |test_u|, precision = hits / K,
 *     ndcg = sum_{i < K, hit} 1/log2(i+2) / sum_{i < min(K, |test_u|)} 1/log2(i+2).
 *   sums_out_dev[q*3 + {0,1,2}] = fp64 sums of (recall, precision, ndcg) over the evaluated rows in ascending
 *   row order; *n_eval_dev = rows with |test_u| > 0.  per_row_out (nullable) [n_ks][3][n_rows] f32, NaN for rows
 *   without test items.  n_ks <= 32. */
int64_t gdr_topk_scores_ws_bytes(int64_t n_rows, int64_t n_items, int64_t d, int64_t k);
int     gdr_topk_scores(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t d, int64_t k,
                        const float* U, int64_t ldu, const int64_t* rows /*nullable*/,
                        const float* I, int64_t ldi,
                        const int32_t* ex_rowptr, const int32_t* ex_colidx /*both nullable*/,
                        float* scores_out, int64_t lds, int32_t* items_out, int64_t ldit,
                        int32_t* status_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream);
int64_t gdr_ranking_metrics_ws_bytes(int64_t n_rows, int n_ks);
int     gdr_ranking_metrics(int64_t n_rows, int64_t n_users, int64_t k, const int32_t* items, int64_t ldit,
                            const int64_t* rows /*nullable*/, const int32_t* test_rowptr,
                            const int32_t* test_colidx, int n_ks, const int32_t* ks_host,
                            double* sums_out_dev, int64_t* n_eval_dev, float* per_row_out /*nullable*/,
                            void* ws, int64_t ws_bytes, gdr_stream_t stream);
/* gdr_topk_condensed: gdr_topk_scores for a condensed model, from its cluster tables.  U [n_cu][ldu] and I [n_ci][ldi]
 *   are the super-user and super-item rows; user_map [n_users] and item_map [n_items] (int64) give each original user
 *   and item its row, values in [0, n_cu) and [0, n_ci).  rows, the exclusion CSR (n_users x n_items, columns sorted
 *   inside each row) and the outputs are those of gdr_topk_scores, and the output bytes are those of gdr_topk_scores
 *   on the expanded tables U[user_map], I[item_map] (either of its paths): (score desc, item asc) across clusters,
 *   -0 reported as +0, (-1, -inf) padding.  Only the n_cu x n_ci distinct scores of the used super-users are
 *   computed: each super-user orders the clusters its rows can need, and each row walks that order, expanding
 *   clusters to their members in id order.  A row that meets a tie run of more than 32 clusters before it has k
 *   items is finished on gdr_topk_scores' exact path with its expanded row (debug key "topk_condensed_path": 1 sends
 *   every row there; gdr_debug_get("topk_condensed_fallback_rows") reads back how many rows the last call sent).
 *   status_dev (device int32, zeroed by the caller): bit 0 = a non-finite value in a super-user row of an evaluated
 *   row or in a super-item row with at least one member (a super-item without members is never read), bit 1 = a user
 *   id in rows outside [0, n_users), bit 2 = a map value outside its range; when any bit is set nothing is written.
 *   The workspace depends on the shapes only (slabs of super-users); the call SYNCHRONISES the stream twice (to size
 *   the slabs from the number of used super-users, and the fallback from its row count). */
int64_t gdr_topk_condensed_ws_bytes(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t n_cu, int64_t n_ci,
                                    int64_t d, int64_t k);
int     gdr_topk_condensed(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t n_cu, int64_t n_ci, int64_t d,
                           int64_t k, const float* U, int64_t ldu, const float* I, int64_t ldi,
                           const int64_t* user_map, const int64_t* item_map, const int64_t* rows /*nullable*/,
                           const int32_t* ex_rowptr, const int32_t* ex_colidx /*both nullable*/,
                           float* scores_out, int64_t lds, int32_t* items_out, int64_t ldit,
                           int32_t* status_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream);

/* ---- BPR training step: triplet sampling and the fused BPR loss + gradient -------------------------------------
 * The sampler, loss and gradient of the refinement loop (distill_recsys.py:684-733); with LightGCNPropagate a step
 * needs no host round trip.  Neither entry point synchronises.
 *
 * gdr_bpr_sample: R = the n_users x n_items interaction CSR, columns sorted and unique inside each row (values are
 *   not read).  eligible[0..n_eligible) = the users with 0 < deg(u) < n_items (the caller builds it once).  Triplet b
 *   of `step`, b < batch:
 *     Philox4x32-10, key = (seed & 0xffffffff, seed >> 32), counter = (b, step, j, 0); a 64-bit word x gives an
 *     integer in [0, n) as umulhi64(x, n).  Call j = 0 -> (w0..w3): user = eligible[draw((w1<<32)|w0, n_eligible)],
 *     pos = the draw((w3<<32)|w2, deg)-th entry of the user's row.  Call j = 1 -> (v0..v3): r = draw((v1<<32)|v0,
 *     n_items - deg), neg = r + #{t : c_t - t <= r} over the row's columns c_0 < ... < c_{deg-1} (the r-th item
 *     outside the row: the distribution of a rejection sampler, found by binary search).
 *   users_out, pos_out, neg_out: int64 [batch].  Output depends on (R, eligible, seed, step, b) only: the same on
 *   every run and every GPU.  batch in [1, 2^31/3], step in [0, 2^32), n_items >= 2.
 * gdr_bpr_loss: U [n_u][ldu], I [n_i][ldi] f32 (16-byte aligned, ld a multiple of 4 and >= d), triplets
 *   users / pos / neg int64 [batch], batch in [1, 2^31/3].  Per triplet
 *     x_b = dot(U[u], I[p]) - dot(U[u], I[n]), each dot the fp32 chain acc = fmaf(U[u,t], I[., t], acc), t ascending;
 *     l_b = softplus(-x_b) (fp32, max(z,0) + log1p(exp(-|z|))),  c_b = -sigmoid(-x_b) / B (fp32, one rounding).
 *   *loss_out (device f32) = (fp64 sum of l_b: per-CTA partials in a fixed tree, then a fixed-order combine) / B.
 *   gU / gI (each nullable; ld a multiple of 4, >= d, 16-byte aligned): overwritten with
 *     gU[u] = sum_b c_b (I[p_b] - I[n_b]) over u_b = u,  gI[j] = sum_{p_b = j} c_b U[u_b] - sum_{n_b = j} c_b U[u_b],
 *   zero in untouched rows.  Each row's terms are added in fp64 in (b, role) order and rounded once (rows with > 2048
 *   terms: fixed chunks in that order, fp64 partials added in chunk order), from a stable sort of the 3B
 *   (row, 3b + role) slots; no float atomics, so the gradients are bit-identical from run to run.
 *   status_dev (device int32, zeroed by the caller): bit 0 = an id out of range, bit 1 = a non-finite x_b (a
 *   non-finite value in a used row).  Such triplets add nothing; the outputs are then not meaningful. */
int     gdr_bpr_sample(int64_t n_users, int64_t n_items, const int32_t* rowptr, const int32_t* colidx,
                       int64_t n_eligible, const int32_t* eligible, uint64_t seed, int64_t step, int64_t batch,
                       int64_t* users_out, int64_t* pos_out, int64_t* neg_out, gdr_stream_t stream);
int64_t gdr_bpr_loss_ws_bytes(int64_t batch, int64_t n_u, int64_t n_i);
int     gdr_bpr_loss(int64_t batch, int64_t n_u, int64_t n_i, int64_t d, const float* U, int64_t ldu,
                     const float* I, int64_t ldi, const int64_t* users, const int64_t* pos, const int64_t* neg,
                     float* loss_out, float* gU /*nullable*/, int64_t ldgu, float* gI /*nullable*/, int64_t ldgi,
                     int32_t* status_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* GDR_H_ */
