// EASE on the GPU (recpack/algorithms/ease.py:63-95): the dense co-occurrence Gram on the tensor cores, the closed-form
// item-item model from the inverse, and scoring with a dense, signed model.
//
//   XTX = (X.T @ X).toarray()                         ease.py:79    -> rpk_gram_dense_f64: exact integer counts on tcgen05
//   P = inv(XTX + l2 * I)                              ease.py:80    -> the caller (cuSOLVER potrf / potri through torch)
//   B = I - P @ diag(1 / diag(P)); diag(B) = 0         ease.py:83-84 -> rpk_ease_from_inverse: B_ij = -P_ij / P_jj, B_ii = 0
//   B = B @ diag(1 / n_j^alpha)                        ease.py:86-88 -> the same kernel, column scale w_j
//   prune to the K largest |B_ij|                      ease.py:97-109 -> rpk_ease_prune: exact top-K by magnitude, canonical CSR
//   scores = X @ B                                     base.py:248   -> rpk_predict_dense_*: sum over the history in
//                                                                       ascending item order, float64, one add per term --
//                                                                       scipy's csr_matvecs order, so equal inputs give
//                                                                       bit-identical scores
#include <stdio.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "internal.h"
#include "prims.cuh"
#include "select.cuh"

namespace rpk {

// A[item][u - u0] = 1 for the interactions of users [u0, u1) (one warp per user).
__global__ void k_fill_dense_chunk(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t u0, int64_t u1,
                                   int64_t kd_pad, unsigned char* __restrict__ A) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = u0 + warp; u < u1; u += nwarps)
    for (int64_t k = indptr[u] + lane; k < indptr[u + 1]; k += 32) A[(int64_t)indices[k] * kd_pad + (u - u0)] = 1;
}

// G[i][j] (+)= G16[i][j]
__global__ void k_acc_g16(const unsigned short* __restrict__ g16, int64_t ldg, int64_t I, int first, double* __restrict__ G) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= I * I) return;
  const int64_t i = t / I, j = t - i * I;
  const double v = (double)g16[i * ldg + j];
  G[t] = first ? v : G[t] + v;
}

void run_gram_dense_f64(rpk_ctx* c, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
                        double* out_G_u) {
  RPK_REQUIRE(U >= 0 && I >= 1 && nnz >= 0 && out_G_u, "bad arguments");
  RPK_REQUIRE(I < ((int64_t)1 << 24), "item count must be below 2^24");
  cudaStream_t st = c->stream;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "fit_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "fit_indices");
  Out<double> o;
  o.init(c, out_G_u, (size_t)I * I, "ease_G");
  const int64_t rows_pad = (I + 255) / 256 * 256;
  const int64_t chunk = 32768;  // users per pass: their counts fit the kernel's 16-bit output
  const int64_t kd_max = std::min<int64_t>(chunk, (U + 127) / 128 * 128);
  unsigned char* A = c->buf<unsigned char>("ease_A", (size_t)rows_pad * std::max<int64_t>(kd_max, 128));
  unsigned short* G16 = c->buf<unsigned short>("ease_G16", (size_t)I * rows_pad);
  const int gblocks = (int)std::min<int64_t>(ceil_div(I * I, 256), 1 << 30);
  if (U == 0) RPK_CUDA(cudaMemsetAsync(o.dev, 0, sizeof(double) * (size_t)I * I, st));
  for (int64_t u0 = 0; u0 < U; u0 += chunk) {
    const int64_t u1 = std::min(U, u0 + chunk);
    const int64_t kd_pad = (u1 - u0 + 127) / 128 * 128;
    RPK_CUDA(cudaMemsetAsync(A, 0, (size_t)rows_pad * kd_pad, st));
    const int wblocks = (int)std::min<int64_t>(((u1 - u0) * 32 + 255) / 256, (int64_t)c->sm_count * 16);
    k_fill_dense_chunk<<<wblocks, 256, 0, st>>>(indptr, indices, u0, u1, kd_pad, A);
    RPK_LAUNCH_CHECK(c);
    run_gram_dense_tc(c, A, rows_pad, kd_pad, 0, I, G16, rows_pad);
    k_acc_g16<<<gblocks, 256, 0, st>>>(G16, rows_pad, I, u0 == 0 ? 1 : 0, o.dev);
    RPK_LAUNCH_CHECK(c);
  }
  o.finish(c);
  finish_call(c);
}

// B_ij = -P_ij / P_jj * w_j, B_ii = 0  (in place when B == P).  The division by the column's diagonal entry is the
// closed form of P @ diag(1 / diag(P)) (ease.py:83); the products are formed in the reference's order:
// fl(fl(P_ij * fl(1 / P_jj)) ...) -> negated -> * w_j.
__global__ void k_ease_finish(const double* P, const double* __restrict__ diag, const double* __restrict__ w, int64_t I, double* B) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= I * I) return;
  const int64_t i = t / I, j = t - i * I;
  double v = 0.0;
  if (i != j) {
    const double inv = __ddiv_rn(1.0, diag[j]);       // np.diag(1.0 / np.diag(P))
    v = -__dmul_rn(P[t], inv);                         // I - P @ diag(.), off the diagonal
    if (w) v = __dmul_rn(v, w[j]);                     // B @ diag(w)
  }
  B[t] = v;
}

void run_ease_from_inverse(rpk_ctx* c, int64_t I, const double* P_u, const double* w_u, double* B_u) {
  RPK_REQUIRE(I >= 1 && P_u && B_u, "bad arguments");
  RPK_REQUIRE(is_device_ptr(P_u) && is_device_ptr(B_u), "rpk_ease_from_inverse works on device matrices");
  const double* w = w_u ? stage_in(c, w_u, (size_t)I, "ease_w") : nullptr;
  // in place is fine except for the diagonal entries, which every column reads and the kernel zeroes: a copy first
  double* dg = c->buf<double>("ease_diag", (size_t)I);
  RPK_CUDA(cudaMemcpy2DAsync(dg, sizeof(double), P_u, sizeof(double) * ((size_t)I + 1), sizeof(double), (size_t)I,
                             cudaMemcpyDeviceToDevice, c->stream));
  k_ease_finish<<<ceil_div(I * I, 256), 256, 0, c->stream>>>(P_u, dg, w, I, B_u);
  RPK_LAUNCH_CHECK(c);
  finish_call(c);
}

// ------------------------------------------------------------------------------------------
// Pruning (EASE._prune, ease.py:97-109): the K largest-magnitude entries of a dense device B as a canonical CSR.
// Key of an entry: the bit pattern of |v| (sign cleared), every NaN mapped to one key above +inf; key 0 (+-0.0) is not
// an entry.  The K-th largest key T is found by a radix select: a histogram of the top 15 key bits over B, the
// entries of the boundary bin collected as candidates, four more digits over the candidates.  Kept: key > T, and the
// first K - #(key > T) entries with key == T in row-major order.  B is read three times: histogram, collect, fill.
// ------------------------------------------------------------------------------------------
static constexpr u64 PRUNE_NAN_KEY = 0x7ff0000000000001ull;  // +inf is 0x7ff0000000000000
static constexpr int PRUNE_BINS = 1 << 15;                  // top digit: key bits 62..48 (bit 63 is always 0)
static constexpr int PRUNE_TOP_SHIFT = 48;

__device__ __forceinline__ u64 prune_key(double v) {
  const u64 k = (u64)__double_as_longlong(v) & 0x7fffffffffffffffull;
  return k < PRUNE_NAN_KEY ? k : PRUNE_NAN_KEY;
}

__device__ __forceinline__ void prune_hist_flush(const unsigned* sh, int nbins, u64* __restrict__ hist) {
  __syncthreads();
  for (int b = threadIdx.x; b < nbins; b += blockDim.x)
    if (sh[b]) atomicAdd(hist + b, (u64)sh[b]);
}

// hist[key >> 48] over the non-zero entries of B [n = I*I] (one shared-memory histogram per CTA).
__global__ void __launch_bounds__(1024) k_prune_hist(const double* __restrict__ B, int64_t n, u64* __restrict__ hist) {
  extern __shared__ unsigned sh_hist[];
  for (int b = threadIdx.x; b < PRUNE_BINS; b += blockDim.x) sh_hist[b] = 0;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
#pragma unroll 4
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    const u64 k = prune_key(__ldg(B + t));
    if (k) atomicAdd(sh_hist + (k >> PRUNE_TOP_SHIFT), 1u);
  }
  prune_hist_flush(sh_hist, PRUNE_BINS, hist);
}

// One CTA per row: row_gt[i] = #(key >> 48 > bin); the entries of the bin are appended to the candidates
// (key, flat position), in no particular order.
__global__ void __launch_bounds__(256) k_prune_collect(const double* __restrict__ B, int64_t I, u64 bin, u64* __restrict__ cand_key,
                                                       int64_t* __restrict__ cand_pos, unsigned long long* __restrict__ n_cand,
                                                       int* __restrict__ row_gt) {
  __shared__ int wsum[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t i = blockIdx.x; i < I; i += gridDim.x) {
    const double* row = B + i * I;
    int gt = 0;
    for (int64_t j0 = 0; j0 < I; j0 += blockDim.x) {
      const int64_t j = j0 + threadIdx.x;
      const u64 k = j < I ? prune_key(__ldg(row + j)) : 0ull;
      gt += (k >> PRUNE_TOP_SHIFT) > bin;
      const bool in_bin = k != 0ull && (k >> PRUNE_TOP_SHIFT) == bin;
      const unsigned m = __ballot_sync(0xffffffffu, in_bin);
      if (m) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(n_cand, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (in_bin) {
          const unsigned long long at = base + __popc(m & ((1u << lane) - 1u));
          cand_key[at] = k;
          cand_pos[at] = i * I + j;
        }
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) gt += __shfl_xor_sync(0xffffffffu, gt, o);
    if (lane == 0) wsum[warp] = gt;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += wsum[w];
      row_gt[i] = s;
    }
    __syncthreads();
  }
}

// hist[(key >> shift) & (2^width - 1)] over the candidates whose key agrees with `prefix` above bit shift + width.
__global__ void __launch_bounds__(1024) k_prune_cand_hist(const u64* __restrict__ cand_key, int64_t n, u64 prefix, int shift,
                                                          int width, u64* __restrict__ hist) {
  extern __shared__ unsigned sh_hist[];
  const int nbins = 1 << width;
  for (int b = threadIdx.x; b < nbins; b += blockDim.x) sh_hist[b] = 0;
  __syncthreads();
  const int hi = shift + width;
  const u64 want = prefix >> hi;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    const u64 k = cand_key[t];
    if ((k >> hi) == want) atomicAdd(sh_hist + (int)((k >> shift) & (u64)(nbins - 1)), 1u);
  }
  prune_hist_flush(sh_hist, nbins, hist);
}

// Candidates above the threshold T add to their row's count, those equal to T to the row's tie count.
__global__ void k_prune_row_counts(const u64* __restrict__ cand_key, const int64_t* __restrict__ cand_pos, int64_t n, int64_t I,
                                   u64 T, int* __restrict__ row_gt, int* __restrict__ row_eq) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    const u64 k = cand_key[t];
    if (k > T) atomicAdd(row_gt + cand_pos[t] / I, 1);
    else if (k == T) atomicAdd(row_eq + cand_pos[t] / I, 1);
  }
}

// Row i takes the leftmost of the ties that the rows before it left over: min(row_eq, max(0, ties - eq_before)).
__global__ void k_prune_take(const int* __restrict__ row_gt, const int* __restrict__ row_eq, const int64_t* __restrict__ eq_before,
                             int64_t I, int64_t ties, int* __restrict__ row_take, int* __restrict__ row_keep) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= I) return;
  const int64_t left = ties - eq_before[i];
  const int take = left <= 0 ? 0 : (int)min(left, (int64_t)row_eq[i]);
  row_take[i] = take;
  row_keep[i] = row_gt[i] + take;
}

// One CTA per row: the kept entries in ascending column order at out_indptr[i] (ordered block-wide compaction).
__global__ void __launch_bounds__(256) k_prune_fill(const double* __restrict__ B, int64_t I, u64 T, const int* __restrict__ row_take,
                                                    const int64_t* __restrict__ indptr, int32_t* __restrict__ out_idx,
                                                    double* __restrict__ out_val) {
  __shared__ int wt[8], wk[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const unsigned below = (1u << lane) - 1u;
  for (int64_t i = blockIdx.x; i < I; i += gridDim.x) {
    const double* row = B + i * I;
    const int take = row_take[i];
    int64_t at = indptr[i];
    int ties_seen = 0;
    for (int64_t j0 = 0; j0 < I; j0 += blockDim.x) {
      const int64_t j = j0 + threadIdx.x;
      const double v = j < I ? __ldg(row + j) : 0.0;
      const u64 k = prune_key(v);
      const bool tie = k == T;
      const unsigned mt = __ballot_sync(0xffffffffu, tie);
      if (lane == 0) wt[warp] = __popc(mt);
      __syncthreads();
      int tie_rank = ties_seen + __popc(mt & below), tie_tile = 0;
      for (int w = 0; w < nw; ++w) {
        tie_rank += w < warp ? wt[w] : 0;
        tie_tile += wt[w];
      }
      const bool keep = k > T || (tie && tie_rank < take);
      const unsigned mk = __ballot_sync(0xffffffffu, keep);
      if (lane == 0) wk[warp] = __popc(mk);
      __syncthreads();
      int pos = __popc(mk & below), kept_tile = 0;
      for (int w = 0; w < nw; ++w) {
        pos += w < warp ? wk[w] : 0;
        kept_tile += wk[w];
      }
      if (keep) {
        out_idx[at + pos] = (int32_t)j;
        out_val[at + pos] = v;
      }
      at += kept_tile;
      ties_seen += tie_tile;
      __syncthreads();
    }
  }
}

// Stream-ordered workspace sized per call (it can be as large as B), returned to the pool on every exit path.
template <class T>
struct StreamBuf {
  T* p = nullptr;
  cudaStream_t st;
  StreamBuf(cudaStream_t s, size_t count) : st(s) { RPK_CUDA(cudaMallocAsync((void**)&p, sizeof(T) * count, st)); }
  void release() {
    if (p) RPK_CUDA(cudaFreeAsync(p, st));
    p = nullptr;
  }
  ~StreamBuf() {
    if (p) cudaFreeAsync(p, st);  // an exception is already on its way: nothing to report here
  }
  StreamBuf(const StreamBuf&) = delete;
  StreamBuf& operator=(const StreamBuf&) = delete;
};

// Index of the bin that holds the need-th largest entry (counting from the top); need becomes its rank inside the bin.
static int prune_pick(const std::vector<u64>& h, u64& need) {
  for (int b = (int)h.size() - 1; b >= 0; --b) {
    if (h[b] >= need) return b;
    need -= h[b];
  }
  throw Error("internal: prune selection ran out of entries");
}

void run_ease_prune(rpk_ctx* c, int64_t I, const double* B, int64_t keep, int64_t* out_indptr_u, int32_t* out_indices_u,
                    double* out_values_u, int64_t* out_nnz_u) {
  RPK_REQUIRE(I >= 1 && keep >= 0 && B && out_indptr_u && out_nnz_u, "bad arguments");
  RPK_REQUIRE(I < ((int64_t)1 << 31), "item count must be below 2^31");
  RPK_REQUIRE(is_device_ptr(B), "rpk_ease_prune works on a device matrix B");
  cudaStream_t st = c->stream;
  const int64_t n = I * I;
  u64* hist = c->buf<u64>("prune_hist", PRUNE_BINS);
  std::vector<u64> h(PRUNE_BINS);
  const size_t hist_smem = sizeof(unsigned) * PRUNE_BINS;
  RPK_CUDA(cudaFuncSetAttribute(k_prune_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_smem));
  RPK_CUDA(cudaFuncSetAttribute(k_prune_cand_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_smem));
  auto read_hist = [&](int nbins) {
    h.assign(nbins, 0);
    RPK_CUDA(cudaMemcpyAsync(h.data(), hist, sizeof(u64) * nbins, cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));
  };
  c->mark("prune_hist");
  RPK_CUDA(cudaMemsetAsync(hist, 0, sizeof(u64) * PRUNE_BINS, st));
  k_prune_hist<<<c->sm_count, 1024, hist_smem, st>>>(B, n, hist);
  RPK_LAUNCH_CHECK(c);
  read_hist(PRUNE_BINS);
  u64 nnz = 0;
  for (u64 x : h) nnz += x;
  const int64_t K = std::min<int64_t>(keep, (int64_t)nnz);

  Out<int64_t> o_ptr, o_nnz;
  Out<int32_t> o_idx;
  Out<double> o_val;
  o_ptr.init(c, out_indptr_u, (size_t)I + 1, "prune_out_ptr");
  o_nnz.init(c, out_nnz_u, 1, "prune_out_nnz");
  if (K > 0) {
    RPK_REQUIRE(out_indices_u && out_values_u, "out_indices / out_values must not be null");
    o_idx.init(c, out_indices_u, (size_t)K, "prune_out_idx");
    o_val.init(c, out_values_u, (size_t)K, "prune_out_val");
  }
  RPK_CUDA(cudaMemcpyAsync(o_nnz.dev, &K, sizeof(int64_t), cudaMemcpyHostToDevice, st));
  if (K == 0) {
    RPK_CUDA(cudaMemsetAsync(o_ptr.dev, 0, sizeof(int64_t) * ((size_t)I + 1), st));
  } else {
    // the boundary bin of the top digit: its entries become the candidates
    u64 need = (u64)K;
    const int b1 = prune_pick(h, need);
    const int64_t n_cand = (int64_t)h[b1];
    StreamBuf<u64> cand_key_buf(st, (size_t)n_cand);
    StreamBuf<int64_t> cand_pos_buf(st, (size_t)n_cand);
    u64* cand_key = cand_key_buf.p;
    int64_t* cand_pos = cand_pos_buf.p;
    unsigned long long* n_cand_dev = c->buf<unsigned long long>("prune_ncand", 1);
    int* row_gt = c->buf<int>("prune_row_gt", (size_t)I);
    int* row_eq = c->buf<int>("prune_row_eq", (size_t)I);
    int* row_take = c->buf<int>("prune_row_take", (size_t)I);
    int* row_keep = c->buf<int>("prune_row_keep", (size_t)I);
    int64_t* eq_before = c->buf<int64_t>("prune_eq_before", (size_t)I + 1);
    RPK_CUDA(cudaMemsetAsync(n_cand_dev, 0, sizeof(unsigned long long), st));
    RPK_CUDA(cudaMemsetAsync(row_eq, 0, sizeof(int) * (size_t)I, st));
    const int row_grid = (int)std::min<int64_t>(I, (int64_t)c->sm_count * 8);
    c->mark("prune_collect");
    k_prune_collect<<<row_grid, 256, 0, st>>>(B, I, (u64)b1, cand_key, cand_pos, n_cand_dev, row_gt);
    RPK_LAUNCH_CHECK(c);
    // the remaining 48 key bits, digit by digit over the candidates
    c->mark("prune_select");
    u64 T = (u64)b1 << PRUNE_TOP_SHIFT;
    const int digits[4][2] = {{33, 15}, {18, 15}, {3, 15}, {0, 3}};
    const int cgrid = (int)std::min<int64_t>(ceil_div(n_cand, 1024), c->sm_count);
    for (auto& dg : digits) {
      const int nbins = 1 << dg[1];
      RPK_CUDA(cudaMemsetAsync(hist, 0, sizeof(u64) * nbins, st));
      k_prune_cand_hist<<<cgrid, 1024, sizeof(unsigned) * nbins, st>>>(cand_key, n_cand, T, dg[0], dg[1], hist);
      RPK_LAUNCH_CHECK(c);
      read_hist(nbins);
      T |= (u64)prune_pick(h, need) << dg[0];
    }
    // T is the K-th largest key; `need` of its ties are kept
    c->mark("prune_counts");
    k_prune_row_counts<<<(int)std::min<int64_t>(ceil_div(n_cand, 256), (int64_t)c->sm_count * 16), 256, 0, st>>>(
        cand_key, cand_pos, n_cand, I, T, row_gt, row_eq);
    RPK_LAUNCH_CHECK(c);
    cand_key_buf.release();
    cand_pos_buf.release();
    scan_i32_i64(c, row_eq, eq_before, I);
    k_prune_take<<<ceil_div(I, 256), 256, 0, st>>>(row_gt, row_eq, eq_before, I, (int64_t)need, row_take, row_keep);
    RPK_LAUNCH_CHECK(c);
    scan_i32_i64(c, row_keep, o_ptr.dev, I);
    int64_t total = -1;
    RPK_CUDA(cudaMemcpyAsync(&total, o_ptr.dev + I, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));
    RPK_REQUIRE(total == K, "internal: pruned row counts do not add up to K");
    c->mark("prune_fill");
    k_prune_fill<<<row_grid, 256, 0, st>>>(B, I, T, row_take, o_ptr.dev, o_idx.dev, o_val.dev);
    RPK_LAUNCH_CHECK(c);
    c->mark("prune_end");
  }
  o_ptr.finish(c);
  o_nnz.finish(c);
  o_idx.finish(c);
  o_val.finish(c);
  RPK_CUDA(cudaStreamSynchronize(st));  // the host value behind the out_nnz copy lives on this frame
  c->host_out_pending = false;
}

// ------------------------------------------------------------------------------------------
// Dense scoring
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ u64 ordered_bits_f64(double v) {
  u64 b = (u64)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double from_ordered_bits(u64 k) {
  const u64 b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

// Candidates of one (user, column range): the columns with a non-zero score (what csr_matrix(scores) stores).
struct DenseScoreSrc {
  const double* acc;
  int r0, ns;
  __device__ __forceinline__ bool has_queue() const { return false; }
  template <class F>
  __device__ __forceinline__ bool for_each_queued(F, int*, int, int*) const { return false; }
  __device__ __forceinline__ int nslots() const { return ns; }
  __device__ __forceinline__ u64 margin() const { return 0ull; }
  __device__ __forceinline__ void set_floor(u64) {}
  __device__ __forceinline__ void stats(SelShared* sh) const { generic_stats(*this, sh); }
  template <class F>
  __device__ __forceinline__ void visit(F f, int stride) const {
    for (int slot = threadIdx.x * stride; slot < ns; slot += blockDim.x * stride) {
      const double v = acc[slot];
      if (v != 0.0) f(slot, ordered_bits_f64(v));
    }
  }
  template <class F>
  __device__ __forceinline__ void for_each(F f) const { visit(f, 1); }
  template <class F>
  __device__ __forceinline__ void for_each_sampled(F f) const { visit(f, SEL_SAMPLE); }
  __device__ __forceinline__ void entry(int slot, Entry& e) const {
    e.key = ordered_bits_f64(acc[slot]);
    e.idx = r0 + slot;
    e.aux = 0;
  }
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const {
    if (a.key != b.key) return a.key > b.key ? 1 : -1;
    return 0;
  }
};

struct DenseParams {
  const int64_t* indptr;
  const int* indices;
  const double* B;  // [I x I] row-major
  int64_t I;
  int U, P, R, N, mask, cap, direct_cap;
  int* part_idx;    // [U*P x N]
  u64* part_key;    // ordered bit patterns of the scores
  int* part_len;
  double* full;     // non-null: write every score [U x I] instead of lists
  int* nan_flag;    // lists: set when a score to rank is NaN (it has no place in the order)
};

// One CTA per (user, column range): the scores of the range are accumulated in shared memory, a thread owns its
// columns and walks the history rows in ascending item order (no atomics: the order of the additions is scipy's).
__global__ void __launch_bounds__(1024, 1) k_predict_dense(DenseParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + SEL_BINS);
  double* acc = reinterpret_cast<double*>(smem + sel_smem_bytes(p.cap));
  const int tid = threadIdx.x, nt = blockDim.x;
  const int64_t total = (int64_t)p.U * p.P;
  for (int64_t w = blockIdx.x; w < total; w += gridDim.x) {
    const int u = (int)(w / p.P), pass = (int)(w % p.P);
    const int r0 = pass * p.R;
    const int ns = (int)min((int64_t)p.R, p.I - r0);
    const int64_t xb = p.indptr[u];
    const int d = (int)(p.indptr[u + 1] - xb);
    for (int s = tid; s < ns; s += nt) acc[s] = 0.0;
    // rows in ascending item order (the CSR is canonical); every thread adds the same rows in the same order
    for (int r = 0; r < d; ++r) {
      const double* row = p.B + (int64_t)p.indices[xb + r] * p.I + r0;
      for (int s = tid; s < ns; s += nt) acc[s] = __dadd_rn(acc[s], __ldg(row + s));
    }
    __syncthreads();
    if (p.mask) {
      for (int r = tid; r < d; r += nt) {
        const int j = p.indices[xb + r] - r0;
        if (j >= 0 && j < ns) acc[j] = 0.0;
      }
      __syncthreads();
    }
    if (p.full) {
      for (int s = tid; s < ns; s += nt) p.full[(int64_t)u * p.I + r0 + s] = acc[s];
      __syncthreads();
      continue;
    }
    bool nan = false;
    for (int s = tid; s < ns; s += nt) nan |= isnan(acc[s]);
    if (nan) atomicOr(p.nan_flag, 1);
    DenseScoreSrc src{acc, r0, ns};
    const int m = block_select_topk(src, p.N, list, p.cap, p.direct_cap, hist, sh);
    const int64_t slot_out = (int64_t)u * p.P + pass;
    for (int t = tid; t < p.N; t += nt) {
      p.part_idx[slot_out * p.N + t] = t < m ? list[t].idx : -1;
      p.part_key[slot_out * p.N + t] = t < m ? list[t].key : 0ull;
    }
    if (tid == 0) p.part_len[slot_out] = m;
    __syncthreads();
  }
}

// One warp per user: merge the P per-range lists (keys = ordered bit patterns of float64 scores).
__global__ void k_dense_finalize(const int* __restrict__ part_idx, const u64* __restrict__ part_key, const int* __restrict__ part_len,
                                 int64_t U, int P, int N, int* __restrict__ out_idx, double* __restrict__ out_val,
                                 int* __restrict__ out_len) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = warp; u < U; u += nwarps) {
    const int PN = P * N;
    const int* pi = part_idx + u * PN;
    const u64* ps = part_key + u * PN;
    int tot = 0;
    for (int q = 0; q < P; ++q) tot += part_len[u * P + q];
    const int m = min(N, tot);
    for (int e = lane; e < PN; e += 32) {
      const int je = pi[e];
      if (je < 0) continue;
      const u64 se = ps[e];
      int rank = 0;
      for (int f = 0; f < PN; ++f) {
        const int jf = pi[f];
        if (jf < 0) continue;
        const u64 sf = ps[f];
        rank += (sf > se) || (sf == se && jf < je);
      }
      if (rank < N) {
        out_idx[u * N + rank] = je;
        if (out_val) out_val[u * N + rank] = from_ordered_bits(se);
      }
    }
    for (int t = m + lane; t < N; t += 32) {
      out_idx[u * N + t] = -1;
      if (out_val) out_val[u * N + t] = 0.0;
    }
    if (lane == 0) out_len[u] = m;
  }
}

static int next_pow2_(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

void run_predict_dense(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u, int64_t I,
                       const double* B, int N, int mask_history, int32_t* out_idx_u, double* out_val_u, int32_t* out_len_u,
                       double* out_full_u) {
  RPK_REQUIRE(U >= 0 && nnz >= 0 && I >= 1 && B, "bad arguments");
  RPK_REQUIRE(is_device_ptr(B), "the dense model must live on the device");
  RPK_REQUIRE(U < ((int64_t)1 << 31), "too many users in one call");
  const bool full = out_full_u != nullptr;
  if (!full) {
    RPK_REQUIRE(N >= 1 && N <= 2048, "N must be in [1, 2048]");
    RPK_REQUIRE(out_idx_u && out_len_u, "out_idx / out_len must not be null");
  }
  cudaStream_t st = c->stream;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "p_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "p_indices");
  Out<int32_t> o_idx, o_len;
  Out<double> o_val, o_full;
  if (full) {
    o_full.init(c, out_full_u, (size_t)U * I, "d_full");
  } else {
    o_idx.init(c, out_idx_u, (size_t)U * N, "p_out_idx");
    o_val.init(c, out_val_u, (size_t)U * N, "p_out_val");
    o_len.init(c, out_len_u, (size_t)U, "p_out_len");
  }
  if (U > 0) {
    DenseParams p;
    const int Nn = full ? 1 : N;
    p.cap = std::max(256, next_pow2_(2 * Nn));
    p.direct_cap = std::min(p.cap, std::max(64, 2 * Nn));
    const size_t fixed = sel_smem_bytes(p.cap);
    RPK_REQUIRE((size_t)c->smem_max > fixed + 1024 + 8192, "N too large for shared memory");
    const size_t avail = (size_t)c->smem_max - fixed - 1024;
    int P = 1;
    int64_t R = 0;
    for (;; ++P) {
      R = ((I + P - 1) / P + 1) & ~(int64_t)1;
      if ((size_t)R * 8 <= avail) break;
    }
    const int p_min = (c->flags & DBG_MANY_PASS) ? 4 : ((c->flags & DBG_MULTI_PASS) ? 2 : 1);
    if (P < p_min && I >= 4 * p_min) {
      P = p_min;
      R = ((I + P - 1) / P + 1) & ~(int64_t)1;
      P = (int)((I + R - 1) / R);  // the even R can leave the last range empty at small I (I = 17: R = 6, three ranges)
    }
    p.indptr = indptr;
    p.indices = indices;
    p.B = B;
    p.I = I;
    p.U = (int)U;
    p.P = P;
    p.R = (int)R;
    p.N = Nn;
    p.mask = mask_history;
    p.full = full ? o_full.dev : nullptr;
    p.part_idx = full ? nullptr : c->buf<int>("d_part_idx", (size_t)U * P * N);
    p.part_key = full ? nullptr : c->buf<u64>("d_part_key", (size_t)U * P * N);
    p.part_len = full ? nullptr : c->buf<int>("d_part_len", (size_t)U * P);
    p.nan_flag = full ? nullptr : c->buf<int>("d_nan", 1);
    if (!full) RPK_CUDA(cudaMemsetAsync(p.nan_flag, 0, sizeof(int), st));
    const size_t smem = fixed + (size_t)R * 8;
    RPK_CUDA(cudaFuncSetAttribute(k_predict_dense, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int nt = R >= 8192 ? 1024 : (R >= 2048 ? 512 : 256);
    const int grid = (int)std::min<int64_t>(U * P, (int64_t)c->sm_count * 4);
    c->ev_record(4);
    k_predict_dense<<<grid, nt, smem, st>>>(p);
    RPK_LAUNCH_CHECK(c);
    c->ev_record(5);
    c->ev_valid[2] = true;
    if (!full) {
      const int fgrid = (int)std::min<int64_t>((U * 32 + 255) / 256, (int64_t)c->sm_count * 16);
      k_dense_finalize<<<fgrid, 256, 0, st>>>(p.part_idx, p.part_key, p.part_len, U, P, N, o_idx.dev, o_val.dev, o_len.dev);
      RPK_LAUNCH_CHECK(c);
      int nan = 0;
      RPK_CUDA(cudaMemcpyAsync(&nan, p.nan_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
      RPK_CUDA(cudaStreamSynchronize(st));
      RPK_REQUIRE(!nan, "dense model: a score to rank is NaN (a NaN in the model, e.g. EASE(alpha != 0) with an item "
                        "nobody interacted with); top-N is not defined, the full scores are");
    }
#ifdef RPK_PHASE_PROF
    fprintf(stderr, "[dense paths] P=%d R=%lld nt=%d smem=%zu users=%lld N=%d full=%d\n", P, (long long)R, nt, smem,
            (long long)U, Nn, full ? 1 : 0);
#endif
  }
  o_idx.finish(c);
  o_val.finish(c);
  o_len.finish(c);
  o_full.finish(c);
  finish_call(c);
}

}  // namespace rpk
