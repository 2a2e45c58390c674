// extern "C" surface of librpk.so (include/rpk.h).  Every entry point catches all C++ exceptions
// and turns them into a status code + message.
#include <stdio.h>
#include <string.h>

#include "common.cuh"
#include "internal.h"

static thread_local std::string g_create_error;

#define RPK_API_BEGIN(ctx)                       \
  if (!(ctx)) return 1;                          \
  try {                                          \
    if (cudaSetDevice((ctx)->device) != cudaSuccess) throw rpk::Error("cudaSetDevice failed");

#define RPK_API_END(ctx)                         \
  }                                              \
  catch (const std::exception& e) {              \
    (ctx)->err = e.what();                       \
    (ctx)->host_out_pending = false;             \
    cudaGetLastError();                          \
    return 1;                                    \
  }                                              \
  catch (...) {                                  \
    (ctx)->err = "unknown error";                \
    return 1;                                    \
  }                                              \
  return 0;

extern "C" {

int rpk_abi_version(void) { return RPK_ABI_VERSION; }

int rpk_create(int device, rpk_ctx** out) {
  if (!out) return 1;
  *out = nullptr;
  try {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess) throw rpk::Error(std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device < 0 || device >= ndev) throw rpk::Error("device index out of range");
    RPK_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RPK_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
      throw rpk::Error(std::string("librpk is built for sm_100a (Blackwell); device is ") + prop.name);
    rpk_ctx* c = new rpk_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_max = (int)prop.sharedMemPerBlockOptin;
    c->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
    c->dense_users = -1;  // automatic
    *out = c;
  } catch (const std::exception& e) {
    g_create_error = e.what();
    cudaGetLastError();
    return 1;
  }
  return 0;
}

void rpk_destroy(rpk_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto& kv : ctx->bufs)
    if (kv.second.p) cudaFree(kv.second.p);
  for (auto& e : ctx->ev)
    if (e) cudaEventDestroy(e);
  for (auto& e : ctx->side_ev)
    if (e) cudaEventDestroy(e);
  for (auto& m : ctx->marks) cudaEventDestroy(m.second);
  for (auto& e : ctx->mark_pool) cudaEventDestroy(e);
  ctx->span_reset();
  for (auto& e : ctx->span_pool) cudaEventDestroy(e);
  if (ctx->hist_ev) cudaEventDestroy(ctx->hist_ev);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->side) cudaStreamDestroy(ctx->side);
  delete ctx;
}

const char* rpk_last_error(const rpk_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int rpk_set_stream(rpk_ctx* ctx, void* cuda_stream) {
  RPK_API_BEGIN(ctx)
  ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  RPK_API_END(ctx)
}

int rpk_sync(rpk_ctx* ctx) {
  RPK_API_BEGIN(ctx)
  RPK_CUDA(cudaStreamSynchronize(ctx->stream));
  RPK_API_END(ctx)
}

int64_t rpk_launch_count(const rpk_ctx* ctx) { return ctx ? ctx->launches : 0; }

int rpk_debug_flags(rpk_ctx* ctx, int flags) {
  RPK_API_BEGIN(ctx)
  ctx->flags = flags;
  ctx->m_P = 0;  // predict geometry may change
  ctx->m_P2 = 0;
  RPK_API_END(ctx)
}

int rpk_fit_topk(rpk_ctx* ctx, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                 int similarity, const double* item_pow, int K, int64_t item_begin, int64_t item_end, int32_t* out_idx,
                 int32_t* out_cnt, double* out_val, int32_t* out_len) {
  RPK_API_BEGIN(ctx)
  rpk::run_fit(ctx, U, I, nnz, indptr, indices, similarity, item_pow, K, item_begin, item_end, out_idx, out_cnt, out_val,
               out_len);
  RPK_API_END(ctx)
}

int rpk_fit_topk_real(rpk_ctx* ctx, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                      const double* values, int similarity, const double* item_pow, int K, int64_t item_begin,
                      int64_t item_end, int32_t* out_idx, double* out_val, int32_t* out_len) {
  RPK_API_BEGIN(ctx)
  rpk::run_fit_real(ctx, U, I, nnz, indptr, indices, values, similarity, item_pow, K, item_begin, item_end, out_idx, out_val,
                    out_len);
  RPK_API_END(ctx)
}

int rpk_fit_item_counts(rpk_ctx* ctx, int32_t* out_counts, int64_t I) {
  RPK_API_BEGIN(ctx)
  rpk::run_fit_item_counts(ctx, out_counts, I);
  RPK_API_END(ctx)
}

int rpk_model_load_topk(rpk_ctx* ctx, int64_t I, int K, const int32_t* idx, const double* val, const int32_t* len) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_load_topk(ctx, I, K, idx, val, len);
  RPK_API_END(ctx)
}

int rpk_model_load_topk_rows(rpk_ctx* ctx, int64_t I, int K, int64_t rows_in, const int32_t* idx, const double* val,
                             const int32_t* len, const int64_t* row_src) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_load_topk_rows(ctx, I, K, rows_in, idx, val, len, row_src);
  RPK_API_END(ctx)
}

int rpk_model_scale_exp(rpk_ctx* ctx, int K, int64_t rows, const double* val, const int32_t* len, int32_t* out_exp) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_scale_exp(ctx, K, rows, val, len, out_exp);
  RPK_API_END(ctx)
}

int rpk_model_pack_rows(rpk_ctx* ctx, int64_t I, int K, int64_t rows, const int32_t* idx, const double* val,
                        const int32_t* len, int scale_exp, uint64_t* out_ent) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_pack_rows(ctx, I, K, rows, idx, val, len, scale_exp, nullptr, out_ent);
  RPK_API_END(ctx)
}

int rpk_model_load_packed_rows(rpk_ctx* ctx, int64_t I, int K, int64_t rows_in, const uint64_t* ent, const int32_t* len,
                               const int64_t* row_src, int scale_exp) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_load_packed_rows(ctx, I, K, rows_in, ent, len, row_src, scale_exp, nullptr);
  RPK_API_END(ctx)
}

int rpk_model_vmax(rpk_ctx* ctx, int K, int64_t rows, const double* val, const int32_t* len, double* out_vmax) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_vmax(ctx, K, rows, val, len, out_vmax);
  RPK_API_END(ctx)
}

int rpk_model_pack_rows_v(rpk_ctx* ctx, int64_t I, int K, int64_t rows, const int32_t* idx, const double* val,
                          const int32_t* len, const double* vmax, uint64_t* out_ent) {
  RPK_API_BEGIN(ctx)
  if (!vmax) throw rpk::Error("vmax must not be null");
  rpk::run_model_pack_rows(ctx, I, K, rows, idx, val, len, 0, vmax, out_ent);
  RPK_API_END(ctx)
}

int rpk_model_load_packed_rows_v(rpk_ctx* ctx, int64_t I, int K, int64_t rows_in, const uint64_t* ent, const int32_t* len,
                                 const int64_t* row_src, const double* vmax) {
  RPK_API_BEGIN(ctx)
  if (!vmax) throw rpk::Error("vmax must not be null");
  rpk::run_model_load_packed_rows(ctx, I, K, rows_in, ent, len, row_src, 0, vmax);
  RPK_API_END(ctx)
}

int64_t rpk_fit_token(const rpk_ctx* ctx) { return ctx ? ctx->lf_token : 0; }

int rpk_model_load_last_fit(rpk_ctx* ctx, int64_t token) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_load_last_fit(ctx, token);
  RPK_API_END(ctx)
}

int rpk_model_load_csr(rpk_ctx* ctx, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                       const double* values) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_load_csr(ctx, I, nnz, indptr, indices, values);
  RPK_API_END(ctx)
}

int rpk_model_load_signed_csr(rpk_ctx* ctx, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                              const double* values) {
  RPK_API_BEGIN(ctx)
  rpk::run_model_load_signed_csr(ctx, I, nnz, indptr, indices, values);
  RPK_API_END(ctx)
}

int rpk_predict_topn(rpk_ctx* ctx, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices, int N,
                     int mask_history, int32_t* out_idx, double* out_val, int32_t* out_len) {
  RPK_API_BEGIN(ctx)
  rpk::run_predict_topn(ctx, U, nnz, indptr, indices, N, mask_history, out_idx, out_val, out_len);
  RPK_API_END(ctx)
}

int rpk_predict_item_filter(rpk_ctx* ctx, const uint8_t* allowed, int64_t I) {
  RPK_API_BEGIN(ctx)
  rpk::run_predict_item_filter(ctx, allowed, I);
  RPK_API_END(ctx)
}

int rpk_predict_csr_count(rpk_ctx* ctx, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                          int mask_history, int64_t* out_row_nnz) {
  RPK_API_BEGIN(ctx)
  rpk::run_predict_csr_count(ctx, U, nnz, indptr, indices, mask_history, out_row_nnz);
  RPK_API_END(ctx)
}

int rpk_predict_csr_fill(rpk_ctx* ctx, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                         int mask_history, const int64_t* out_indptr, int32_t* out_indices, double* out_values) {
  RPK_API_BEGIN(ctx)
  rpk::run_predict_csr_fill(ctx, U, nnz, indptr, indices, mask_history, out_indptr, out_indices, out_values);
  RPK_API_END(ctx)
}

int rpk_topk_csr(rpk_ctx* ctx, int64_t rows, int64_t nnz, const int64_t* indptr, const int32_t* indices,
                 const double* values, int K, int32_t* out_idx, int32_t* out_len) {
  RPK_API_BEGIN(ctx)
  rpk::run_topk_csr(ctx, rows, nnz, indptr, indices, values, K, out_idx, out_len);
  RPK_API_END(ctx)
}

int rpk_metrics_topn(rpk_ctx* ctx, int64_t U, int N, const int32_t* top_idx, const int32_t* top_len,
                     const int64_t* true_indptr, const int32_t* true_indices, int64_t true_nnz, int n_metrics,
                     const int32_t* kinds, const int32_t* Ks, const double* discount, const double* idcg, int maxK,
                     double* per_user, double* sums, int64_t* n_users) {
  RPK_API_BEGIN(ctx)
  rpk::run_metrics_topn(ctx, U, N, top_idx, top_len, true_indptr, true_indices, true_nnz, n_metrics, kinds, Ks, discount,
                        idcg, maxK, per_user, sums, n_users);
  RPK_API_END(ctx)
}

int rpk_coverage_topn(rpk_ctx* ctx, int64_t U, int N, int K, int64_t I, const int32_t* top_idx, const int32_t* top_len,
                      const int64_t* true_indptr, int64_t* out_count, uint8_t* out_flags) {
  RPK_API_BEGIN(ctx)
  rpk::run_coverage_topn(ctx, U, N, K, I, top_idx, top_len, true_indptr, out_count, out_flags);
  RPK_API_END(ctx)
}

int rpk_gram_dense_f64(rpk_ctx* ctx, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr, const int32_t* indices, double* out_G) {
  RPK_API_BEGIN(ctx)
  rpk::run_gram_dense_f64(ctx, U, I, nnz, indptr, indices, out_G);
  RPK_API_END(ctx)
}

int rpk_ease_from_inverse(rpk_ctx* ctx, int64_t I, const double* P, const double* w, double* out_B) {
  RPK_API_BEGIN(ctx)
  rpk::run_ease_from_inverse(ctx, I, P, w, out_B);
  RPK_API_END(ctx)
}

int rpk_predict_dense_topn(rpk_ctx* ctx, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices, int64_t I,
                           const double* B, int N, int mask_history, int32_t* out_idx, double* out_val, int32_t* out_len) {
  RPK_API_BEGIN(ctx)
  rpk::run_predict_dense(ctx, U, nnz, indptr, indices, I, B, N, mask_history, out_idx, out_val, out_len, nullptr);
  RPK_API_END(ctx)
}

int rpk_predict_dense_full(rpk_ctx* ctx, int64_t U, int64_t nnz, const int64_t* indptr, const int32_t* indices, int64_t I,
                           const double* B, int mask_history, double* out_scores) {
  RPK_API_BEGIN(ctx)
  if (!out_scores) throw rpk::Error("out_scores must not be null");
  rpk::run_predict_dense(ctx, U, nnz, indptr, indices, I, B, 1, mask_history, nullptr, nullptr, nullptr, out_scores);
  RPK_API_END(ctx)
}

int rpk_gram_dense_u16(rpk_ctx* ctx, int64_t I, int64_t Kd, const uint8_t* A, uint16_t* out_G) {
  RPK_API_BEGIN(ctx)
  rpk::run_gram_dense_u16(ctx, I, Kd, A, out_G);
  RPK_API_END(ctx)
}

int rpk_last_timings(rpk_ctx* ctx, double* out_ms) {
  RPK_API_BEGIN(ctx)
  if (!out_ms) throw rpk::Error("out_ms must not be null");
  RPK_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 2; ++k) {  // fit: sums over the strips
    out_ms[k] = -1.0;
    double sum = 0.0;
    bool any = false;
    for (auto& pr : ctx->spans[k]) {
      if (!pr.second) continue;
      float ms = 0.f;
      RPK_CUDA(cudaEventElapsedTime(&ms, pr.first, pr.second));
      sum += ms;
      any = true;
    }
    if (any) out_ms[k] = sum;
  }
  out_ms[2] = -1.0;
  if (ctx->ev_valid[2]) {
    float ms = 0.f;
    RPK_CUDA(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
    out_ms[2] = ms;
  }
  out_ms[3] = ctx->last_dense_users;
  out_ms[4] = ctx->last_dense_kd;
  RPK_API_END(ctx)
}

int rpk_trace(rpk_ctx* ctx, int on) {
  RPK_API_BEGIN(ctx)
  ctx->tracing = on != 0;
  RPK_API_END(ctx)
}

const char* rpk_trace_report(rpk_ctx* ctx) {
  if (!ctx) return "";
  ctx->trace_text.clear();
  try {
    cudaSetDevice(ctx->device);
    RPK_CUDA(cudaStreamSynchronize(ctx->stream));
    char line[256];
    for (size_t k = 0; k < ctx->marks.size(); ++k) {
      float ms = 0.f;
      if (k > 0) RPK_CUDA(cudaEventElapsedTime(&ms, ctx->marks[k - 1].second, ctx->marks[k].second));
      snprintf(line, sizeof(line), "%-28s %9.3f ms\n", ctx->marks[k].first.c_str(), ms);
      ctx->trace_text += line;
    }
    for (auto& m : ctx->marks) ctx->mark_pool.push_back(m.second);
    ctx->marks.clear();
  } catch (const std::exception& e) {
    ctx->err = e.what();
  }
  return ctx->trace_text.c_str();
}

int rpk_fit_config(rpk_ctx* ctx, int dense_users) {
  RPK_API_BEGIN(ctx)
  if (dense_users < -1 || dense_users > 4096) throw rpk::Error("dense_users must be in [-1, 4096]");
  ctx->dense_users = dense_users;
  RPK_API_END(ctx)
}

int rpk_spgemm_topn(rpk_ctx* ctx, int64_t rows, int64_t a_nnz, const int64_t* a_indptr, const int32_t* a_indices,
                    const double* a_values, int64_t I, int64_t s_nnz, const int64_t* s_indptr, const int32_t* s_indices,
                    const double* s_values, int N, int mask_history, int32_t* out_idx, double* out_val, int32_t* out_len) {
  RPK_API_BEGIN(ctx)
  rpk::run_spgemm(ctx, rows, a_nnz, a_indptr, a_indices, a_values, I, s_nnz, s_indptr, s_indices, s_values, N, mask_history, 0,
                  out_idx, out_val, out_len, nullptr, nullptr, 0, nullptr, nullptr);
  RPK_API_END(ctx)
}

int rpk_spgemm_count(rpk_ctx* ctx, int64_t rows, int64_t a_nnz, const int64_t* a_indptr, const int32_t* a_indices,
                     const double* a_values, int64_t I, int64_t s_nnz, const int64_t* s_indptr, const int32_t* s_indices,
                     const double* s_values, int mask_history, int64_t* out_row_nnz) {
  RPK_API_BEGIN(ctx)
  rpk::run_spgemm(ctx, rows, a_nnz, a_indptr, a_indices, a_values, I, s_nnz, s_indptr, s_indices, s_values, 1, mask_history, 1,
                  nullptr, nullptr, nullptr, out_row_nnz, nullptr, 0, nullptr, nullptr);
  RPK_API_END(ctx)
}

int rpk_spgemm_fill(rpk_ctx* ctx, int64_t rows, int64_t a_nnz, const int64_t* a_indptr, const int32_t* a_indices,
                    const double* a_values, int64_t I, int64_t s_nnz, const int64_t* s_indptr, const int32_t* s_indices,
                    const double* s_values, int mask_history, const int64_t* out_indptr, int64_t out_nnz, int32_t* out_indices,
                    double* out_values) {
  RPK_API_BEGIN(ctx)
  rpk::run_spgemm(ctx, rows, a_nnz, a_indptr, a_indices, a_values, I, s_nnz, s_indptr, s_indices, s_values, 1, mask_history, 2,
                  nullptr, nullptr, nullptr, nullptr, out_indptr, out_nnz, out_indices, out_values);
  RPK_API_END(ctx)
}

int rpk_split_fraction(rpk_ctx* ctx, int64_t n_users, const int64_t* uids, const int64_t* seg, const int64_t* rows,
                       int64_t n_rows, double in_frac, uint64_t seed, uint8_t* out_in_mask) {
  RPK_API_BEGIN(ctx)
  rpk::run_split_fraction(ctx, n_users, uids, seg, rows, n_rows, in_frac, seed, out_in_mask);
  RPK_API_END(ctx)
}

int rpk_fit_strip_rows(rpk_ctx* ctx, int64_t rows) {
  RPK_API_BEGIN(ctx)
  if (rows < 0) throw rpk::Error("rows must be >= 0");
  ctx->strip_rows = rows;
  RPK_API_END(ctx)
}

}  // extern "C"
