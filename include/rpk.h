/*
 * rpk.h -- C ABI of the B200 item-similarity library (librpk.so).
 *
 * The reference (LienM/recpack, pure Python) has no native boundary on this path; these
 * entry points are what a binding for its hot path replaces, one per reference call site:
 *
 *   rpk_fit_topk        ItemKNN._fit: compute_cosine_similarity /
 *                       compute_conditional_probability + get_top_K_values
 *                       (recpack/algorithms/nearest_neighbour.py:22-84,204-224,
 *                        recpack/util.py:50-96)
 *   rpk_model_load_*    the fitted `similarity_matrix_` attribute
 *                       (recpack/algorithms/base.py:220-255)
 *   rpk_predict_topn    ItemSimilarityMatrixAlgorithm._predict (base.py:237-255) fused
 *                       with history removal (recpack/pipelines/pipeline.py:174-175) and
 *                       the top-K ranking of MetricTopK.calculate (metrics/base.py:189)
 *   rpk_predict_csr_*   _predict with the reference's full CSR output
 *   rpk_topk_csr        get_top_K_ranks on an arbitrary prediction matrix (util.py:50-77)
 *   rpk_metrics_topn    NDCGK / DCGK / RecallK / CalibratedRecallK._calculate
 *                       (metrics/dcg.py:21-128, metrics/recall.py:21-85)
 *   rpk_gram_dense_f64 / rpk_ease_from_inverse / rpk_predict_dense_*
 *                       EASE._fit and its dense X @ B predict (recpack/algorithms/ease.py:63-95)
 *   rpk_embed_topk      the similarity_matrix_ of Prod2Vec (cosine_similarity of the item embeddings +
 *                       get_top_K_values) and of any item-factor matrix
 *
 * Conventions
 *   - plain C types only; every call returns 0 on success, non-zero on failure, with a
 *     message available from rpk_last_error().  No C++ exception crosses the boundary.
 *   - every data pointer may be a HOST pointer or a DEVICE pointer of the context's device;
 *     the library detects which (cudaPointerGetAttributes).  Host inputs are copied to the
 *     device inside the call, host outputs are copied back and the call returns after the
 *     copy completed.  With device pointers only, calls are asynchronous on the context's
 *     stream (rpk_set_stream) and stream-ordered with each other.
 *   - the caller owns all inputs and outputs; the context owns only workspace and the
 *     loaded model.  A context is bound to one device and is not re-entrant; use one
 *     context per (process, device) -- multi-GPU is one process per GPU.
 *   - interaction matrices are CSR (users x items): indptr int64[U+1], indices int32[nnz],
 *     rows with strictly increasing column indices (scipy "canonical format").  Values are
 *     not passed: the path is defined on the binarised matrix (base.py:129-151).
 */
#ifndef RPK_H
#define RPK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RPK_ABI_VERSION 3

#if defined(__GNUC__)
#define RPK_EXPORT __attribute__((visibility("default")))
#else
#define RPK_EXPORT
#endif

typedef struct rpk_ctx rpk_ctx;

enum { RPK_SIM_COSINE = 0, RPK_SIM_CONDPROB = 1, RPK_SIM_DOT = 2 /* rpk_embed_topk only */ };
enum { RPK_METRIC_NDCG = 0, RPK_METRIC_RECALL = 1, RPK_METRIC_DCG = 2, RPK_METRIC_CALIBRATED_RECALL = 3,
       RPK_METRIC_PRECISION = 4,        /* hits / K (recpack/metrics/precision.py:41-50) */
       RPK_METRIC_RECIPROCAL_RANK = 5,  /* 1 / rank of the first hit, 0 without one (metrics/reciprocal_rank.py:37-40) */
       RPK_METRIC_HITS = 6              /* number of hits among the first K places = row sum of HitK's scores (metrics/hit.py:20-45) */ };

RPK_EXPORT int rpk_abi_version(void);

/* Create / destroy a context on CUDA device `device`. */
RPK_EXPORT int rpk_create(int device, rpk_ctx** out);
RPK_EXPORT void rpk_destroy(rpk_ctx* ctx);
/* Message of the last failed call on this context (or of a failed rpk_create when ctx is NULL). */
RPK_EXPORT const char* rpk_last_error(const rpk_ctx* ctx);
/* Use `cuda_stream` (a cudaStream_t, may be NULL for the default stream) for all later calls. */
RPK_EXPORT int rpk_set_stream(rpk_ctx* ctx, void* cuda_stream);
/* Block until everything queued on the context's stream has finished. */
RPK_EXPORT int rpk_sync(rpk_ctx* ctx);
/* Number of kernels this context has launched since creation (for the bench's gpu_launches). */
RPK_EXPORT int64_t rpk_launch_count(const rpk_ctx* ctx);
/* Test hook: force a code path.  bit 0: wide (64-bit CAS) score accumulators in predict;
 * bit 1: tiny candidate-list capacity in the selection routine (exercises its refinement and
 * tie paths on small inputs); bit 2: more than one item-range pass in fit/predict;
 * bit 3: the fit cuts its heaviest rows into pieces even on small inputs; bit 4: rpk_predict_topn computes exact
 * scores for every list even when out_val is NULL (it otherwise proves most lists from approximate sums). */
RPK_EXPORT int rpk_debug_flags(rpk_ctx* ctx, int flags);

/*
 * Fit: for every item row i in [item_begin, item_end) compute the co-occurrence counts
 * c_ij = |users(i) & users(j)| against ALL items j, and keep the K best j != i with c_ij > 0.
 *
 *   similarity = RPK_SIM_COSINE:   order by c_ij^2 / n_j   (exact rational; n_i is constant per row)
 *                                  value  = sum of c_ij copies of fl(a_i * a_j), a = 1/sqrt(n), added
 *                                  one at a time in float64 -- the reference's own operation order
 *   similarity = RPK_SIM_CONDPROB: order by c_ij, value = fl(fl(1/n_i) * c_ij)            (item_pow NULL)
 *                                  order by fl(c_ij * item_pow[j]), value = fl(fl(fl(1/n_i) * c_ij) * item_pow[j])
 *                                  item_pow[j] = (1/n_j)^pop_discount, float64[I], computed by the caller
 *   ties: ascending item index.
 *
 * Outputs (row-major, [item_end - item_begin] x K, rank order, best first):
 *   out_idx int32 (-1 padded), out_cnt int32 (c_ij, 0 padded), out_val float64 (0 padded),
 *   out_len int32[item_end - item_begin].  out_cnt / out_val may be NULL.
 */
RPK_EXPORT int rpk_fit_topk(rpk_ctx* ctx, int64_t U, int64_t I, int64_t nnz,
                 const int64_t* indptr, const int32_t* indices,
                 int similarity, const double* item_pow, int K,
                 int64_t item_begin, int64_t item_end,
                 int32_t* out_idx, int32_t* out_cnt, double* out_val, int32_t* out_len);

/*
 * Fit on a REAL-VALUED interaction matrix (values float64[nnz], one per stored entry, no explicit zeros):
 * ItemKNN(normalize_X=True) (nearest_neighbour.py:207-210: values = 1/d_u), compute_pearson_similarity
 * (nearest_neighbour.py:87-111: values = centred ratings) and the decayed matrices of the TARSItemKNN family
 * (time_aware_item_knn/base.py:166-201) reach the similarity functions with such a matrix.
 *
 *   similarity = RPK_SIM_COSINE:   s_ij = sum over users u (ascending) of fl(xh_ui * xh_uj), xh = x / ||x_.i||_2 with
 *                                  the norm as sklearn computes it (sequential sum of squares, sqrt, divide)
 *   similarity = RPK_SIM_CONDPROB: g_ij = sum over users of item i (ascending) of x_uj; s_ij = fl(fl(1/n_i) * g_ij)
 *                                  [* item_pow[j]], n_i = stored entries of column i (to_binary(X), :48-51)
 * Sums are float64 in the reference's operation order (scipy csr_matmat), so the values are bit-identical to the
 * reference's; sums that are exactly zero are not stored.  Per row the K best stored entries are kept by
 * (value descending, item ascending); the diagonal's explicit zero (setdiag, :64,81) competes and is then dropped,
 * as in get_top_K_values (util.py:80-96).  Outputs as rpk_fit_topk (no counts).  Deterministic.
 */
RPK_EXPORT int rpk_fit_topk_real(rpk_ctx* ctx, int64_t U, int64_t I, int64_t nnz,
                      const int64_t* indptr, const int32_t* indices, const double* values,
                      int similarity, const double* item_pow, int K,
                      int64_t item_begin, int64_t item_end,
                      int32_t* out_idx, double* out_val, int32_t* out_len);

/* Item popularities n_j of the matrix passed to the last rpk_fit_topk (int32[I]). */
RPK_EXPORT int rpk_fit_item_counts(rpk_ctx* ctx, int32_t* out_counts, int64_t I);

/*
 * Load the similarity model used by the predict calls.
 *   _topk: from [I x K] lists as rpk_fit_topk writes them (any order inside a row).
 *   _csr:  from a CSR item x item matrix (indptr int64[I+1], column indices unique per row).
 * Values must be finite and non-negative.  Scoring is defined in fixed point relative to the model's largest value
 * vmax: q = max(rint(v * 2^e), 1) with e = 39 - floor(log2(vmax)) (so vmax * 2^e lies in [2^39, 2^40)); a score is
 * the exact integer sum of q over the history, reported as sum * 2^-e.  |score - float64 sum| <= d_u * 2^-(e+1).
 */
RPK_EXPORT int rpk_model_load_topk(rpk_ctx* ctx, int64_t I, int K,
                        const int32_t* idx, const double* val, const int32_t* len);
/* As rpk_model_load_topk, for lists that live in a larger array (e.g. the all-gathered, padded per-rank
 * shards of a multi-GPU fit): model row i is read from input row row_src[i] (int64[I]); the input arrays
 * have rows_in rows. */
RPK_EXPORT int rpk_model_load_topk_rows(rpk_ctx* ctx, int64_t I, int K, int64_t rows_in,
                             const int32_t* idx, const double* val, const int32_t* len,
                             const int64_t* row_src);
/* Multi-GPU exchange in the model's own format (8 bytes per entry instead of 12, and no per-rank re-sort of
 * every row after the all-gather).  rpk_model_scale_exp returns the exponent e these lists would get as a model
 * of their own; the ranks agree on the smallest e (largest value anywhere) before packing.
 * rpk_model_pack_rows turns `rows` rank-ordered lists (as written by rpk_fit_topk; columns are item ids in
 * [0, I)) into packed rows out_ent[r*K + t] = column << 40 | q, q = max(rint(val * 2^scale_exp), 1), ascending
 * column, unused places all-ones.  rpk_model_load_packed_rows builds the model from such rows: model row i =
 * input row row_src[i] (int64[I], null = identity), len = entries per row, scale_exp as used for packing.
 * Replaces nothing in the reference (single process); it is the row exchange of SURVEY.md 8(e). */
RPK_EXPORT int rpk_model_scale_exp(rpk_ctx* ctx, int K, int64_t rows, const double* val, const int32_t* len,
                        int32_t* out_exp);
RPK_EXPORT int rpk_model_pack_rows(rpk_ctx* ctx, int64_t I, int K, int64_t rows,
                        const int32_t* idx, const double* val, const int32_t* len, int scale_exp, uint64_t* out_ent);
RPK_EXPORT int rpk_model_load_packed_rows(rpk_ctx* ctx, int64_t I, int K, int64_t rows_in,
                               const uint64_t* ent, const int32_t* len, const int64_t* row_src, int scale_exp);
/* The same exchange without a host round trip: rpk_model_vmax leaves the largest value of the lists as a double in
 * device memory, the ranks all-reduce it (MAX) on the stream, and the _v forms take that device scalar instead of an
 * exponent.  With device pointers only, nothing here synchronises; what the packing finds wrong with this rank's
 * values is reported by the next rpk_model_load_* call. */
RPK_EXPORT int rpk_model_vmax(rpk_ctx* ctx, int K, int64_t rows, const double* val, const int32_t* len, double* out_vmax);
RPK_EXPORT int rpk_model_pack_rows_v(rpk_ctx* ctx, int64_t I, int K, int64_t rows,
                          const int32_t* idx, const double* val, const int32_t* len, const double* vmax, uint64_t* out_ent);
RPK_EXPORT int rpk_model_load_packed_rows_v(rpk_ctx* ctx, int64_t I, int K, int64_t rows_in,
                                 const uint64_t* ent, const int32_t* len, const int64_t* row_src, const double* vmax);
/* Every rpk_fit_topk increments the context's fit token.  When the last fit covered all item rows and
 * produced values, its lists stay resident on the device and rpk_model_load_last_fit(token) builds the
 * model from them without any host round trip; it fails when `token` is not the current one. */
RPK_EXPORT int64_t rpk_fit_token(const rpk_ctx* ctx);
RPK_EXPORT int rpk_model_load_last_fit(rpk_ctx* ctx, int64_t token);
RPK_EXPORT int rpk_model_load_csr(rpk_ctx* ctx, int64_t I, int64_t nnz,
                       const int64_t* indptr, const int32_t* indices, const double* values);
/* A model of any sign (finite values, ascending unique columns per row), scored in float64 instead of fixed point:
 * rpk_predict_topn / _csr_count / _csr_fill then return scipy's X @ S bit for bit -- every score is the left fold of
 * s_ij over the user's history rows in their stored order, sums of exactly 0.0 are not stored, and the lists hold the
 * N largest stored scores (score desc, item index asc), negative ones included when fewer than N positive ones exist.
 * The history mask and the item filter apply as for the other models.  The rpk_model_load_* calls above keep
 * rejecting negative values. */
RPK_EXPORT int rpk_model_load_signed_csr(rpk_ctx* ctx, int64_t I, int64_t nnz,
                              const int64_t* indptr, const int32_t* indices, const double* values);

/*
 * Score U users: score_uj = sum over history items i of S_ij; optionally drop the user's own
 * history items; keep the N best (score desc, item index asc).
 *   out_idx int32 [U x N] (-1 padded), out_val float64 [U x N] (score, 0 padded; may be NULL),
 *   out_len int32 [U].
 * The lists are the same with and without out_val.  Without it the kernel stops at 32-bit approximate sums
 * wherever those already prove the order (gaps larger than the error bound) and computes exact sums only for the
 * remaining lists.
 * A model loaded with rpk_model_load_signed_csr is scored in float64 (scipy's X @ S, see there): out_val then holds the
 * exact float64 sums, and a sum of exactly 0.0 is not listed.
 */
RPK_EXPORT int rpk_predict_topn(rpk_ctx* ctx, int64_t U, int64_t nnz,
                     const int64_t* indptr, const int32_t* indices,
                     int N, int mask_history,
                     int32_t* out_idx, double* out_val, int32_t* out_len);

/*
 * Item filter of the predict calls (recpack/postprocessing/filters.py:58-101, ExcludeItems / SelectItems, applied
 * INSIDE predict so that a truncated list is refilled from the items that remain): allowed uint8[I], 1 = the item
 * may be recommended.  NULL removes the filter.  The mask is copied; it stays in force until changed.
 */
RPK_EXPORT int rpk_predict_item_filter(rpk_ctx* ctx, const uint8_t* allowed, int64_t I);

/* Full score matrix in CSR, as the reference's predict() returns it.  Two steps: _count fills
 * out_row_nnz int64[U]; the caller prefix-sums it into out_indptr and allocates; _fill writes
 * the column indices (ascending per row) and float64 scores. */
RPK_EXPORT int rpk_predict_csr_count(rpk_ctx* ctx, int64_t U, int64_t nnz,
                          const int64_t* indptr, const int32_t* indices,
                          int mask_history, int64_t* out_row_nnz);
RPK_EXPORT int rpk_predict_csr_fill(rpk_ctx* ctx, int64_t U, int64_t nnz,
                         const int64_t* indptr, const int32_t* indices,
                         int mask_history, const int64_t* out_indptr,
                         int32_t* out_indices, double* out_values);

/* Per row of an arbitrary CSR (values float64), the K best stored entries
 * (value desc, column asc): out_idx int32 [rows x K] (-1 padded), out_len int32[rows]. */
RPK_EXPORT int rpk_topk_csr(rpk_ctx* ctx, int64_t rows, int64_t nnz,
                 const int64_t* indptr, const int32_t* indices, const double* values,
                 int K, int32_t* out_idx, int32_t* out_len);

/*
 * Metrics on rank-ordered lists.  For every user u with a non-empty y_true row and every
 * metric m: per_user[m * U + u] = metric value (users with an empty y_true row get NaN and are
 * not counted).  sums[m] = sum over counted users, *n_users = number of counted users.
 *   discount float64[maxK] = 1/log2(r+2), idcg float64[maxK+1] -- tables computed by the caller
 *   (metrics/dcg.py:98-104) so that they are the reference's own numbers.
 */
RPK_EXPORT int rpk_metrics_topn(rpk_ctx* ctx, int64_t U, int N,
                     const int32_t* top_idx, const int32_t* top_len,
                     const int64_t* true_indptr, const int32_t* true_indices, int64_t true_nnz,
                     int n_metrics, const int32_t* kinds, const int32_t* Ks,
                     const double* discount, const double* idcg, int maxK,
                     double* per_user, double* sums, int64_t* n_users);

/*
 * CoverageK (recpack/metrics/coverage.py:13-40): *out_count = number of distinct items among the first K places of
 * the lists of users with a non-empty y_true row (users without true items are dropped first,
 * metrics/base.py:106-123); out_flags uint8[I] (may be NULL) marks those items.
 */
RPK_EXPORT int rpk_coverage_topn(rpk_ctx* ctx, int64_t U, int N, int K, int64_t I,
                      const int32_t* top_idx, const int32_t* top_len, const int64_t* true_indptr,
                      int64_t* out_count, uint8_t* out_flags);

/*
 * Scoring with a REAL-VALUED input matrix: C = A @ S for a CSR A [rows x I] (e.g. time-decayed histories) and the CSR
 * similarity matrix S [I x I] (ascending columns per row; values may be negative), float64 sums in scipy's csr_matmat
 * order -- bit-identical to the reference's `X_decayed @ similarity_matrix_` of TARSItemKNN._predict
 * (recpack/algorithms/time_aware_item_knn/base.py:137-149 -> algorithms/base.py:237-255).  Sums that are exactly zero
 * are not stored.  mask_history removes the columns of A's own row first (pipelines/pipeline.py:174-175).
 *   rpk_spgemm_topn   the N best stored entries per row by (value descending, column ascending); outputs as rpk_fit_topk_real
 *   rpk_spgemm_count  stored entries per row (int64[rows])
 *   rpk_spgemm_fill   the CSR rows (ascending columns) at out_indptr (int64[rows + 1], exclusive prefix of the counts)
 */
RPK_EXPORT int rpk_spgemm_topn(rpk_ctx* ctx, int64_t rows, int64_t a_nnz, const int64_t* a_indptr, const int32_t* a_indices,
                    const double* a_values, int64_t I, int64_t s_nnz, const int64_t* s_indptr, const int32_t* s_indices,
                    const double* s_values, int N, int mask_history, int32_t* out_idx, double* out_val, int32_t* out_len);
RPK_EXPORT int rpk_spgemm_count(rpk_ctx* ctx, int64_t rows, int64_t a_nnz, const int64_t* a_indptr, const int32_t* a_indices,
                     const double* a_values, int64_t I, int64_t s_nnz, const int64_t* s_indptr, const int32_t* s_indices,
                     const double* s_values, int mask_history, int64_t* out_row_nnz);
RPK_EXPORT int rpk_spgemm_fill(rpk_ctx* ctx, int64_t rows, int64_t a_nnz, const int64_t* a_indptr, const int32_t* a_indices,
                    const double* a_values, int64_t I, int64_t s_nnz, const int64_t* s_indptr, const int32_t* s_indices,
                    const double* s_values, int mask_history, const int64_t* out_indptr, int64_t out_nnz,
                    int32_t* out_indices, double* out_values);

/*
 * Data side: FractionInteractionSplitter.split (recpack/scenarios/splitters.py:233-263).  The interactions are given
 * grouped by user: user g has id uids[g] and the grouped positions seg[g] .. seg[g+1]-1, rows[] maps a grouped
 * position to the interaction's row in the caller's table (the reference's per-user order = table order).  For every
 * user the positions are shuffled exactly as np.random.RandomState(seed + uid).shuffle does (MT19937, Fisher-Yates
 * with masked rejection sampling) and the first ceil(n * in_frac) go to data_in: out_in_mask[row] = 1, else 0
 * (uint8[n_rows]).  seed + uid must fit 32 bits (numpy raises otherwise; the caller checks).
 */
RPK_EXPORT int rpk_split_fraction(rpk_ctx* ctx, int64_t n_users, const int64_t* uids, const int64_t* seg,
                       const int64_t* rows, int64_t n_rows, double in_frac, uint64_t seed, uint8_t* out_in_mask);

/*
 * Dense leg of the fit on the tensor cores (tcgen05 int8 MMA, int32 accumulation in TMEM):
 * G[i][j] = sum_k A[i][k] * A[j][k] for a 0/1 matrix A (uint8 [I x Kd] row-major, Kd <= 32768),
 * written as uint16 [I x I].  rpk_fit_topk uses this kernel for the densest user columns when
 * rpk_fit_config enables it; this entry point exposes it for verification.
 */
RPK_EXPORT int rpk_gram_dense_u16(rpk_ctx* ctx, int64_t I, int64_t Kd, const uint8_t* A, uint16_t* out_G);

/*
 * EASE (recpack/algorithms/ease.py:63-95).
 *   rpk_gram_dense_f64      XTX = (X.T @ X).toarray(): exact co-occurrence counts of ALL users as float64 [I x I]
 *                           (tensor-core Gram over 32,768-user chunks, summed).  out_G may be host or device memory.
 *   rpk_ease_from_inverse   B_ij = -P_ij / P_jj * w_j (i != j), B_ii = 0 from P = inv(XTX + l2 I): the closed form of
 *                           I - P @ diag(1 / diag(P)) followed by B @ diag(w), w_j = 1 / n_j^alpha (NULL: no scaling).
 *                           P and out_B are DEVICE matrices [I x I] float64 and may be the same buffer.  The inverse
 *                           itself is a library call on the caller's side (cuSOLVER potrf + potri).
 *   rpk_ease_prune          EASE._prune (ease.py:97-109): the min(keep, nnz(B)) entries of the DEVICE matrix B [I x I]
 *                           with the largest |B_ij| as a canonical CSR (ascending columns, values bit for bit).  The
 *                           entries are the values != 0.0; every NaN ranks above +inf; +x and -x tie; ties at the cut
 *                           go to the entries first in row-major order.  out_indptr int64[I + 1], out_indices int32
 *                           and out_values float64 sized keep, out_nnz int64[1] receives the count; outputs may be host
 *                           or device memory.  keep = 0 keeps nothing (the reference's "K = 0 keeps all" is the
 *                           caller's: pass keep = I * I).  Workspace: 16 bytes per entry of the top-digit bin that
 *                           holds the cut.
 *   rpk_predict_dense_topn  scores = X @ B for a dense float64 model B (device, [I x I] row-major): every score is
 *   rpk_predict_dense_full  the sum over the user's history in ascending item order, one float64 addition per term
 *                           (scipy's csr @ dense order).  _topn keeps the N best non-zero scores per user (score
 *                           desc, item index asc; history optionally removed first), _full writes all scores
 *                           float64 [U x I].
 */
RPK_EXPORT int rpk_gram_dense_f64(rpk_ctx* ctx, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr,
                       const int32_t* indices, double* out_G);
RPK_EXPORT int rpk_ease_from_inverse(rpk_ctx* ctx, int64_t I, const double* P, const double* w, double* out_B);
RPK_EXPORT int rpk_ease_prune(rpk_ctx* ctx, int64_t I, const double* B, int64_t keep, int64_t* out_indptr,
                   int32_t* out_indices, double* out_values, int64_t* out_nnz);
RPK_EXPORT int rpk_predict_dense_topn(rpk_ctx* ctx, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                           int64_t I, const double* B, int N, int mask_history,
                           int32_t* out_idx, double* out_val, int32_t* out_len);
RPK_EXPORT int rpk_predict_dense_full(rpk_ctx* ctx, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                           int64_t I, const double* B, int mask_history, double* out_scores);

/*
 * Item neighbours of a dense embedding matrix E (float64 [I x D] row-major, finite; 1 <= D <= 1024, I < 2^24,
 * 1 <= K <= 1024).  DESIGN.md 2, "Embedding neighbours":
 *   RPK_SIM_DOT:    s_ij = left fold over d = 0 .. D-1 of fl(e_id * e_jd), starting from the first product, separate
 *                   multiply and add (no FMA); every squared row norm must be below 2^1020
 *   RPK_SIM_COSINE: the same fold over xhat_i = fl(e_i / n_i), n_i = fl(sqrt(fold of fl(e_id * e_id))); a zero row stays zero
 * For every row i in [item_begin, item_end): over the columns j != i, the K largest stored values (an exact +-0.0 is not
 * stored), ordered by (value desc, column asc); negative values are kept when fewer than K larger ones exist.  Outputs
 * as rpk_fit_topk_real: out_idx int32 [rows x K] (-1 padded), out_val float64 (0 padded, may be NULL), out_len int32[rows].
 * NaN / inf in E and arguments outside the limits fail the call.  Synchronises once (the check of E).
 * The tensor cores (tf32) only screen candidates under the error bound of DESIGN.md 4.9; every value and every order
 * decision is made in float64 on the definition, so the result does not depend on the screen.
 *
 * rpk_embed_screen_f32: the screen's approximate matrix, out_S float32 [I x I] (I <= 65536), in the units of s.  For
 * verification of the bound only.
 */
RPK_EXPORT int rpk_embed_topk(rpk_ctx* ctx, int64_t I, int D, const double* E, int similarity, int K,
                   int64_t item_begin, int64_t item_end, int32_t* out_idx, double* out_val, int32_t* out_len);
RPK_EXPORT int rpk_embed_screen_f32(rpk_ctx* ctx, int64_t I, int D, const double* E, int similarity, float* out_S);

/* Device time (CUDA events on the context's stream) of the dominant kernels of the last calls:
 * out_ms[0] = tensor-core Gram of the last fit, out_ms[1] = sparse fit kernels of the last fit,
 * out_ms[2] = scoring kernel of the last predict; -1 where the kernel did not run;
 * out_ms[3] = users the last fit routed to the tensor cores, out_ms[4] = that number padded to the MMA
 * k-block.  out_ms must hold 5 doubles.  Synchronises. */
RPK_EXPORT int rpk_last_timings(rpk_ctx* ctx, double* out_ms);

/* Tracing: with `on` != 0 every later call records named marks (CUDA events) on the context's stream at its phase
 * boundaries.  rpk_trace_report synchronises, formats "name: ms since the previous mark" lines for all marks recorded
 * since the last report into an internal buffer (valid until the next call on the context), clears them and returns it. */
RPK_EXPORT int rpk_trace(rpk_ctx* ctx, int on);
RPK_EXPORT const char* rpk_trace_report(rpk_ctx* ctx);

/* Fit configuration.  dense_users: how many of the users with the longest histories go through the
 * tensor-core Gram (0 = none, -1 = automatic, at most 4096); the remaining users go through the
 * sparse kernel.  The result of rpk_fit_topk does not depend on this setting. */
RPK_EXPORT int rpk_fit_config(rpk_ctx* ctx, int dense_users);
/* rpk_fit_topk runs its item rows in strips so that only one strip of the dense leg's count matrix (uint16,
 * rows x I) exists at a time -- the item x item matrix is never materialised as a whole.  rows: rows per strip
 * (rounded down to a multiple of 128, at least 128); 0 = automatic (a strip of at most 8 GB).  The result does not
 * depend on this setting. */
RPK_EXPORT int rpk_fit_strip_rows(rpk_ctx* ctx, int64_t rows);

#ifdef __cplusplus
}
#endif
#endif /* RPK_H */
