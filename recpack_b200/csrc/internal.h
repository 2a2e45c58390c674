// Host-side drivers implemented in the .cu files; called by the C ABI in api.cu.
#pragma once
#include <stdint.h>

struct rpk_ctx;

namespace rpk {

void run_fit(rpk_ctx* c, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices, int similarity,
             const double* item_pow, int K, int64_t item_begin, int64_t item_end, int32_t* out_idx, int32_t* out_cnt,
             double* out_val, int32_t* out_len);
void run_fit_real(rpk_ctx* c, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                  const double* values, int similarity, const double* item_pow, int K, int64_t item_begin, int64_t item_end,
                  int32_t* out_idx, double* out_val, int32_t* out_len);
void run_fit_item_counts(rpk_ctx* c, int32_t* out_counts, int64_t I);

void run_model_load_topk(rpk_ctx* c, int64_t I, int K, const int32_t* idx, const double* val, const int32_t* len);
void run_model_load_last_fit(rpk_ctx* c, int64_t token);
void run_model_scale_exp(rpk_ctx* c, int K, int64_t rows, const double* val, const int32_t* len, int32_t* out_exp);
void run_model_vmax(rpk_ctx* c, int K, int64_t rows, const double* val, const int32_t* len, double* out_vmax);
void run_model_pack_rows(rpk_ctx* c, int64_t I, int K, int64_t rows, const int32_t* idx, const double* val,
                         const int32_t* len, int scale_exp, const double* vmax, uint64_t* out_ent);
void run_model_load_packed_rows(rpk_ctx* c, int64_t I, int K, int64_t rows_in, const uint64_t* ent, const int32_t* len,
                                const int64_t* row_src, int scale_exp, const double* vmax);
void run_model_load_topk_rows(rpk_ctx* c, int64_t I, int K, int64_t rows_in, const int32_t* idx, const double* val,
                              const int32_t* len, const int64_t* row_src);
void run_model_load_csr(rpk_ctx* c, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                        const double* values);
void run_predict_topn(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices, int N,
                      int mask_history, int32_t* out_idx, double* out_val, int32_t* out_len);
void run_predict_item_filter(rpk_ctx* c, const uint8_t* allowed, int64_t I);
void run_predict_csr_count(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                           int mask_history, int64_t* out_row_nnz);
void run_predict_csr_fill(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                          int mask_history, const int64_t* out_indptr, int32_t* out_indices, double* out_values);

void run_topk_csr(rpk_ctx* c, int64_t rows, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                  const double* values, int K, int32_t* out_idx, int32_t* out_len);
void run_metrics_topn(rpk_ctx* c, int64_t U, int N, const int32_t* top_idx, const int32_t* top_len,
                      const int64_t* true_indptr, const int32_t* true_indices, int64_t true_nnz, int n_metrics,
                      const int32_t* kinds, const int32_t* Ks, const double* discount, const double* idcg, int maxK,
                      double* per_user, double* sums, int64_t* n_users);

void run_coverage_topn(rpk_ctx* c, int64_t U, int N, int K, int64_t I, const int32_t* top_idx, const int32_t* top_len,
                       const int64_t* true_indptr, int64_t* out_count, uint8_t* out_flags);

void run_spgemm(rpk_ctx* c, int64_t rows, int64_t a_nnz, const int64_t* a_indptr, const int32_t* a_indices, const double* a_values,
                int64_t I, int64_t b_nnz, const int64_t* b_indptr, const int32_t* b_indices, const double* b_values, int N,
                int mask_history, int mode, int32_t* out_idx, double* out_val, int32_t* out_len, int64_t* out_row_nnz,
                const int64_t* out_indptr, int64_t out_nnz, int32_t* csr_indices, double* csr_values);
void spgemm_rows_device(rpk_ctx* c, int64_t rows, const int64_t* a_ptr, const int32_t* a_idx, const double* a_val, int64_t I,
                        const int64_t* b_ptr, const int32_t* b_idx, const double* b_val, const int* order, const int* n_order, int N,
                        int mask_history, const unsigned char* item_ok, int mode, int32_t* out_idx, double* out_val,
                        int32_t* out_len, int64_t* out_row_nnz, const int64_t* out_indptr, int32_t* csr_indices,
                        double* csr_values);
void run_model_load_signed_csr(rpk_ctx* c, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                               const double* values);
void run_split_fraction(rpk_ctx* c, int64_t n_users, const int64_t* uids, const int64_t* seg, const int64_t* rows,
                        int64_t n_rows, double in_frac, uint64_t seed, uint8_t* out_in_mask);
void run_gram_dense_f64(rpk_ctx* c, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices, double* out_G);
void run_ease_from_inverse(rpk_ctx* c, int64_t I, const double* P, const double* w, double* B);
void run_ease_prune(rpk_ctx* c, int64_t I, const double* B, int64_t keep, int64_t* out_indptr, int32_t* out_indices,
                    double* out_values, int64_t* out_nnz);
void run_predict_dense(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices, int64_t I, const double* B,
                       int N, int mask_history, int32_t* out_idx, double* out_val, int32_t* out_len, double* out_full);
void run_gram_dense_u16(rpk_ctx* c, int64_t I, int64_t Kd, const unsigned char* A, unsigned short* G);
void run_gram_dense_tc(rpk_ctx* c, const unsigned char* A, int64_t rows_pad, int64_t kd_pad, int64_t row_begin,
                       int64_t row_end, unsigned short* G, int64_t ldg);
// the same with uint8 counts: every row of A holds at most 255 ones
void run_gram_dense_tc(rpk_ctx* c, const unsigned char* A, int64_t rows_pad, int64_t kd_pad, int64_t row_begin,
                       int64_t row_end, unsigned char* G, int64_t ldg);
void run_embed_topk(rpk_ctx* c, int64_t I, int D, const double* E, int similarity, int K, int64_t item_begin,
                    int64_t item_end, int32_t* out_idx, double* out_val, int32_t* out_len);
void run_embed_screen_f32(rpk_ctx* c, int64_t I, int D, const double* E, int similarity, float* out_S);

}  // namespace rpk
