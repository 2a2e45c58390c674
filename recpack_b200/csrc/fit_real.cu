// Item-item Gram of a REAL-VALUED interaction matrix with the fused similarity epilogue and per-row top-K.
//
// Replaces (reference, /root/reference) for inputs whose values are not all one:
//   recpack/algorithms/nearest_neighbour.py:207-210   ItemKNN(normalize_X=True): X <- l1-normalised rows of X
//   recpack/algorithms/nearest_neighbour.py:69-84     compute_cosine_similarity (sklearn normalize + csr_matmat)
//   recpack/algorithms/nearest_neighbour.py:22-66     compute_conditional_probability: to_binary(X).T @ X, A @ . @ A^alpha
//   recpack/algorithms/nearest_neighbour.py:87-111    compute_pearson_similarity = cosine of the centred matrix
//   recpack/util.py:50-96                             get_top_K_values (the explicit diagonal zero competes, then drops out)
//
// Values follow the reference's floating-point operation order, so kept similarities are bit-identical float64:
// scipy's csr_matmat adds fl(a_ui * b_uj) to the running sum of (i, j) in ascending user order; sums that end at
// exactly 0 are not stored.  One CTA owns an item row; its warps own disjoint column slices of the row's float64
// accumulators in shared memory and walk the row's users in ascending order, so every accumulator sees its terms
// in the reference's order without atomics (deterministic).  Columns are processed in ranges of R accumulators;
// the non-zero sums of every range are scaled, appended to the CTA's scratch row in global memory together with the
// diagonal's explicit zero, and the exact block-wide selection of select.cuh picks the K best (value desc, item asc).
#include <math.h>

#include "common.cuh"
#include "internal.h"
#include "prims.cuh"
#include "select.cuh"

namespace rpk {

namespace {

__device__ __forceinline__ u64 ordered_bits_f64(double v) {
  u64 b = (u64)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double from_ordered_bits(u64 k) {
  const u64 b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

struct RealRowSrc {
  __device__ __forceinline__ bool has_queue() const { return false; }
  template <class F>
  __device__ __forceinline__ bool for_each_queued(F, int*, int, int*) const { return false; }
  const int* idx;
  const double* val;
  int ns;
  __device__ __forceinline__ u64 margin() const { return 0ull; }
  __device__ __forceinline__ void set_floor(u64) {}
  __device__ __forceinline__ void stats(SelShared* sh) const { generic_stats(*this, sh); }
  __device__ __forceinline__ u64 key_at(int slot) const {
    double v = val[slot];
    if (v == 0.0) v = 0.0;  // the diagonal's +0.0; a -0.0 sum is never stored
    return ordered_bits_f64(v);
  }
  template <class F>
  __device__ __forceinline__ void visit(F f, int stride) const {
    for (int slot = threadIdx.x * stride; slot < ns; slot += blockDim.x * stride) f(slot, key_at(slot));
  }
  template <class F>
  __device__ __forceinline__ void for_each(F f) const { visit(f, 1); }
  template <class F>
  __device__ __forceinline__ void for_each_sampled(F f) const { visit(f, SEL_SAMPLE); }
  __device__ __forceinline__ void entry(int slot, Entry& e) const {
    e.key = key_at(slot);
    e.idx = idx[slot];
    e.aux = 0;
  }
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const {
    if (a.key != b.key) return a.key > b.key ? 1 : -1;
    return 0;
  }
};

__global__ void k_real_item_counts(const int* __restrict__ indices, int64_t nnz, int* __restrict__ n) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(&n[indices[k]], 1);
}

// CSC user lists in arbitrary order (atomic cursors) + the row's work = sum of its users' history lengths.
__global__ void k_real_fill_csc(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t U,
                                const int64_t* __restrict__ cscptr, int* __restrict__ cursor, int* __restrict__ csc_users,
                                u64* __restrict__ work) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = warp; u < U; u += nwarps) {
    const int64_t b = indptr[u], e = indptr[u + 1];
    const u64 d = (u64)(e - b);
    for (int64_t t = b + lane; t < e; t += 32) {
      const int i = indices[t];
      const int pos = atomicAdd(&cursor[i], 1);
      csc_users[cscptr[i] + pos] = (int)u;
      atomicAdd(&work[i], d);
    }
  }
}

// Sorts every item's user list ascending (the reference's summation order).  Short lists: rank by counting in
// shared memory; long lists: a bitmap over all users (nwords 32-bit words, sized by the host), read back in order.
__global__ void __launch_bounds__(256) k_real_sort_csc(const int64_t* __restrict__ cscptr, int* __restrict__ csc_users, int64_t I,
                                                       int nwords) {
  extern __shared__ unsigned sm_words[];
  __shared__ int s_scan[256];
  const int tid = threadIdx.x;
  for (int64_t i = blockIdx.x; i < I; i += gridDim.x) {
    const int64_t b = cscptr[i];
    const int n = (int)(cscptr[i + 1] - b);
    if (n <= 1) continue;  // block-uniform
    int* seg = csc_users + b;
    if (n <= 512) {
      int* keys = reinterpret_cast<int*>(sm_words);
      for (int t = tid; t < n; t += 256) keys[t] = seg[t];
      __syncthreads();
      for (int t = tid; t < n; t += 256) {
        const int k = keys[t];
        int r = 0;
        for (int s = 0; s < n; ++s) r += keys[s] < k;
        seg[r] = k;  // the users of an item are distinct
      }
      __syncthreads();
      continue;
    }
    for (int w = tid; w < nwords; w += 256) sm_words[w] = 0u;
    __syncthreads();
    for (int t = tid; t < n; t += 256) {
      const int u = seg[t];
      atomicOr(&sm_words[u >> 5], 1u << (u & 31));
    }
    __syncthreads();
    // exclusive prefix of the popcounts: each thread owns a contiguous run of words
    const int per = (nwords + 255) / 256;
    const int w0 = min(nwords, tid * per), w1 = min(nwords, w0 + per);
    int cnt = 0;
    for (int w = w0; w < w1; ++w) cnt += __popc(sm_words[w]);
    s_scan[tid] = cnt;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
      const int v = tid >= o ? s_scan[tid - o] : 0;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    int pos = s_scan[tid] - cnt;
    for (int w = w0; w < w1; ++w) {
      unsigned m = sm_words[w];
      while (m) {
        const int bit = __ffs(m) - 1;
        m &= m - 1;
        seg[pos++] = (w << 5) + bit;
      }
    }
    __syncthreads();
  }
}

// Offset of item i inside the (sorted) history of each of its users: the value of entry (u, i) is values[indptr[u] + off].
__global__ void k_real_csc_pos(const int64_t* __restrict__ cscptr, const int* __restrict__ csc_users,
                               const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t I,
                               int* __restrict__ csc_off) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < I; i += nwarps) {
    const int64_t b = cscptr[i], e = cscptr[i + 1];
    for (int64_t k = b + lane; k < e; k += 32) {
      const int u = csc_users[k];
      const int64_t hb = indptr[u];
      int lo = 0, hi = (int)(indptr[u + 1] - hb);
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (indices[hb + mid] < (int)i) lo = mid + 1;
        else hi = mid;
      }
      csc_off[k] = lo;
    }
  }
}

// sklearn's inplace_csr_row_normalize_l2 on X^T (sparsefuncs_fast.pyx:578-604): per item the squares are summed
// sequentially in ascending user order, the root taken, every value divided by it; all-zero rows are left alone.
__global__ void k_real_item_norms(const int64_t* __restrict__ cscptr, const int* __restrict__ csc_users,
                                  const int* __restrict__ csc_off, const int64_t* __restrict__ indptr,
                                  const double* __restrict__ values, int64_t I, double* __restrict__ norm) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= I) return;
  double s = 0.0;
  for (int64_t k = cscptr[i]; k < cscptr[i + 1]; ++k) {
    const double x = values[indptr[csc_users[k]] + csc_off[k]];
    s = __dadd_rn(s, __dmul_rn(x, x));
  }
  norm[i] = s == 0.0 ? 0.0 : sqrt(s);
}
__global__ void k_real_normalise(const int* __restrict__ indices, const double* __restrict__ values,
                                 const double* __restrict__ norm, int64_t nnz, double* __restrict__ out) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
    const double nm = norm[indices[k]];
    out[k] = nm == 0.0 ? values[k] : __ddiv_rn(values[k], nm);
  }
}
__global__ void k_real_recip(const int* __restrict__ n, int64_t I, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < I) out[i] = n[i] > 0 ? __ddiv_rn(1.0, (double)n[i]) : 0.0;
}

// First position in a[0, n) whose value is >= key (per lane: every lane searches its own array).
__device__ __forceinline__ int lane_lower_bound(const int* __restrict__ a, int n, int key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// One kernel serves two products of the form  row(i) = sum over the entries k of a LIST of  a_k * B[k, :] :
//   fit      list = users of item i (CSC of X, ascending), a_k = left value of (user, i), B = X (right values);
//   scoring  list = row u of a real-valued matrix A (decayed histories), a_k = A's value, B = the similarity model.
struct RealParams {
  const int64_t* indptr;  // B: CSR with ascending columns
  const int* indices;
  const double* left;   // fit: per CSR entry of X, null = 1.0 (binary left operand)
  const double* right;  // B's values
  const int64_t* cscptr;  // the lists
  const int* csc_users;   // ... their entries (row ids of B), ascending per list
  const int* csc_off;     // fit: offset of item i inside each user's history (where `left` is read)
  const double* left_entry;  // non-null: a_k stored per list entry (scoring)
  const int* split;  // non-null: [rows of B x split_w] positions of the slice boundaries inside every row of B (k_real_split)
  int split_w;       // = P * (warps + 1)
  const double* row_scale;  // null = none
  const double* col_scale;  // null = none
  const int* order;         // rows of this call, heaviest first (absolute row ids)
  int nrows;
  int P, R, I, K;
  int64_t item_begin;
  int cap, direct_cap;
  int diag;       // 1: column i of row i is an explicit zero that competes in the selection (fit: setdiag)
  int mask_list;  // 1: the columns named by the list itself are removed (history removal in scoring)
  const unsigned char* item_ok;  // non-null: item filter of the scoring (1 = may be recommended)
  int mode;       // 0: top-K lists; 1: count the stored entries per row; 2: write CSR rows (ascending columns)
  const int* nrows_dev;  // non-null: device-side number of rows of `order` (replaces nrows)
  int* queue;
  int* scr_idx;  // [grid x (I + 1)]
  double* scr_val;
  int* out_idx;
  double* out_val;
  int* out_len;
  long long* out_row_nnz;     // mode 1
  const int64_t* out_indptr;  // mode 2
  int* csr_indices;
  double* csr_values;
};

__global__ void __launch_bounds__(1024, 1) k_real_rows(RealParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + SEL_BINS);
  double* acc = reinterpret_cast<double*>(smem + sel_smem_bytes(p.cap));
  __shared__ int s_row, s_cnt, s_diag;
  __shared__ int s_wc[32];
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  int* scr_idx = p.scr_idx + (int64_t)blockIdx.x * (p.I + 1);
  double* scr_val = p.scr_val + (int64_t)blockIdx.x * (p.I + 1);
  const int nrows = p.nrows_dev ? *p.nrows_dev : p.nrows;
  for (;;) {
    __syncthreads();
    if (tid == 0) {
      s_row = atomicAdd(p.queue, 1);
      s_cnt = 0;
      s_diag = -1;
    }
    __syncthreads();
    if (s_row >= nrows) break;
    const int i = p.order[s_row];
    const int64_t ub = p.cscptr[i];
    const int nu = (int)(p.cscptr[i + 1] - ub);
    for (int pass = 0; pass < p.P; ++pass) {
      const int r0 = pass * p.R, r1 = min(p.I, r0 + p.R);
      for (int t = tid; t < r1 - r0; t += nt) acc[t] = 0.0;
      __syncthreads();
      // this warp's column slice of the range
      const int per = (r1 - r0 + nw - 1) / nw;
      const int c0 = r0 + warp * per, c1 = min(r1, c0 + per);
      if (c0 < c1) {
        // 32 list entries at a time, one per lane: every lane finds the part of ITS row of B that falls into the warp's
        // slice (two binary searches, all lanes busy), then the warp applies the 32 parts one after the other in list
        // order -- the order the reference adds them in -- with its lanes spread over the part's entries.
        for (int k0 = 0; k0 < nu; k0 += 32) {
          const int k = k0 + lane;
          int64_t hb = 0;
          int lo = 0, cnt = 0;
          double a = 0.0;
          if (k < nu) {
            const int u = p.csc_users[ub + k];
            hb = p.indptr[u];
            const int d = (int)(p.indptr[u + 1] - hb);
            if (p.split) {
              const int* sp = p.split + (int64_t)u * p.split_w + pass * (nw + 1) + warp;
              lo = sp[0];
              cnt = sp[1] - lo;
            } else {
              const int* h = p.indices + hb;
              lo = lane_lower_bound(h, d, c0);
              if (lo < d && h[lo] < c1) cnt = lane_lower_bound(h + lo, d - lo, c1);
            }
            if (cnt > 0) a = p.left_entry ? p.left_entry[ub + k] : (p.left ? p.left[hb + p.csc_off[ub + k]] : 1.0);
          }
          unsigned todo = __ballot_sync(0xffffffffu, cnt > 0);
          while (todo) {
            const int l = __ffs(todo) - 1;
            todo &= todo - 1u;
            const int64_t hb_l = __shfl_sync(0xffffffffu, hb, l) + __shfl_sync(0xffffffffu, lo, l);
            const int cnt_l = __shfl_sync(0xffffffffu, cnt, l);
            const double a_l = __shfl_sync(0xffffffffu, a, l);
            for (int t = lane; t < cnt_l; t += 32) {
              const int j = p.indices[hb_l + t];
              const double b = p.right[hb_l + t];
              acc[j - r0] = __dadd_rn(acc[j - r0], __dmul_rn(a_l, b));
            }
            __syncwarp();
          }
        }
      }
      __syncthreads();
      if (p.mask_list) {  // pipelines/pipeline.py:174-175: scores of history items are removed
        for (int k = tid; k < nu; k += nt) {
          const int j = p.csc_users[ub + k];
          if (j >= r0 && j < r1) acc[j - r0] = 0.0;
        }
        __syncthreads();
      }
      if (p.item_ok) {  // postprocessing/filters.py:58-101, before the truncation
        for (int t = tid; t < r1 - r0; t += nt)
          if (!p.item_ok[r0 + t]) acc[t] = 0.0;
        __syncthreads();
      }
      if (p.mode == 0) {
        // non-zero sums -> scratch row (scaled); the diagonal is an explicit zero of the reference's matrix
        const double rs = p.row_scale ? p.row_scale[i] : 1.0;
        for (int t0 = 0; t0 < r1 - r0; t0 += nt) {
          const int t = t0 + tid;
          bool keep = false;
          double v = 0.0;
          const int j = r0 + t;
          if (t < r1 - r0) {
            if (p.diag && j == i) {
              keep = true;
            } else {
              v = acc[t];
              if (v != 0.0) {
                keep = true;
                if (p.row_scale) v = __dmul_rn(rs, v);
                if (p.col_scale) v = __dmul_rn(v, p.col_scale[j]);
                if (v == 0.0) keep = false;  // underflow to zero: a zero product is not stored either
              }
            }
          }
          const unsigned m = __ballot_sync(0xffffffffu, keep);
          int base = 0;
          if (lane == 0 && m) base = atomicAdd(&s_cnt, __popc(m));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (keep) {
            const int pos = base + __popc(m & ((1u << lane) - 1u));
            scr_idx[pos] = j;
            scr_val[pos] = v;
          }
        }
        __syncthreads();
      } else {
        // stored entries of the row in ascending column order: count them (mode 1) or write them (mode 2)
        const int64_t row_base = p.mode == 2 ? p.out_indptr[i] : 0;
        for (int t0 = 0; t0 < r1 - r0; t0 += nt) {
          const int t = t0 + tid;
          const double v = t < r1 - r0 ? acc[t] : 0.0;
          const bool keep = v != 0.0;
          const unsigned m = __ballot_sync(0xffffffffu, keep);
          if (lane == 0) s_wc[warp] = __popc(m);
          __syncthreads();
          int before = 0, all = 0;
          for (int w = 0; w < nw; ++w) {
            const int cw = s_wc[w];
            before += w < warp ? cw : 0;
            all += cw;
          }
          if (keep && p.mode == 2) {
            const int64_t pos = row_base + s_cnt + before + __popc(m & ((1u << lane) - 1u));
            p.csr_indices[pos] = r0 + t;
            p.csr_values[pos] = v;
          }
          __syncthreads();
          if (tid == 0) s_cnt += all;
        }
        __syncthreads();
      }
    }
    if (p.mode != 0) {
      if (p.mode == 1 && tid == 0) p.out_row_nnz[i] = s_cnt;
      continue;
    }
    const int ns = s_cnt;
    int m = 0;
    if (ns > 0) {
      RealRowSrc src{scr_idx, scr_val, ns};
      m = block_select_topk(src, p.K, list, p.cap, p.direct_cap, hist, sh);
    }
    __syncthreads();
    for (int t = tid; t < m; t += nt)
      if (p.diag && list[t].idx == i) s_diag = t;
    __syncthreads();
    const int dpos = s_diag;
    const int64_t ob = ((int64_t)i - p.item_begin) * p.K;
    const int len = dpos >= 0 ? m - 1 : m;
    for (int t = tid; t < p.K; t += nt) {
      const int s = (dpos >= 0 && t >= dpos) ? t + 1 : t;
      if (t < len) {
        p.out_idx[ob + t] = list[s].idx;
        p.out_val[ob + t] = from_ordered_bits(list[s].key);
      } else {
        p.out_idx[ob + t] = -1;
        p.out_val[ob + t] = 0.0;
      }
    }
    if (tid == 0) p.out_len[i - p.item_begin] = len;
  }
}

// split[r * W + p * (nw + 1) + w] = first position in row r of B whose column is >= the lower bound of the slice of warp w
// in column range p (w = nw: the end of the range): the row kernel then reads two table entries per (list entry, slice)
// instead of searching the row of B again for every row of the product that touches it.
__global__ void k_real_split(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t nrows_b, int I, int P, int R,
                             int nw, int* __restrict__ split) {
  const int W = P * (nw + 1);
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nrows_b * W) return;
  const int64_t r = t / W;
  const int s = (int)(t - r * W);
  const int pass = s / (nw + 1), w = s - pass * (nw + 1);
  const int r0 = pass * R, r1 = min(I, r0 + R);
  const int per = (r1 - r0 + nw - 1) / nw;
  const int bound = min(r1, r0 + w * per);
  const int64_t hb = indptr[r];
  split[t] = lane_lower_bound(indices + hb, (int)(indptr[r + 1] - hb), bound);
}

// Work of a scoring row: the entries of B it touches.
__global__ void k_spgemm_work(const int64_t* __restrict__ a_ptr, const int* __restrict__ a_idx, const int64_t* __restrict__ b_ptr,
                              int64_t rows, u64* __restrict__ work) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < rows; r += nwarps) {
    u64 w = 0;
    for (int64_t k = a_ptr[r] + lane; k < a_ptr[r + 1]; k += 32) w += (u64)(b_ptr[a_idx[k] + 1] - b_ptr[a_idx[k]]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
    if (lane == 0) work[r] = w + 1;
  }
}

// Slice-boundary table of B for the row kernel (null when it would not fit comfortably: the kernel then searches).
static const int* build_split(rpk_ctx* c, const int64_t* b_ptr, const int* b_idx, int64_t nrows_b, int64_t I, int P, int R, int nt,
                              int* split_w) {
  const int nw = nt / 32;
  const int64_t W = (int64_t)P * (nw + 1);
  *split_w = (int)W;
  if (nrows_b == 0 || nrows_b * W > ((int64_t)1 << 29)) return nullptr;  // > 2 GB of positions
  int* split = c->buf<int>("fr_split", (size_t)(nrows_b * W));
  k_real_split<<<ceil_div(nrows_b * W, 256), 256, 0, c->stream>>>(b_ptr, b_idx, nrows_b, (int)I, P, R, nw, split);
  RPK_LAUNCH_CHECK(c);
  return split;
}

int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

}  // namespace

void run_fit_real(rpk_ctx* c, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
                  const double* values_u, int similarity, const double* item_pow_u, int K, int64_t item_begin, int64_t item_end,
                  int32_t* out_idx_u, double* out_val_u, int32_t* out_len_u) {
  RPK_REQUIRE(U >= 0 && I >= 0 && nnz >= 0, "negative dimension");
  RPK_REQUIRE(I < (int64_t)1 << 24, "more than 2^24 items are not supported");
  RPK_REQUIRE(U < (int64_t)1 << 31, "more than 2^31 users are not supported");
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(0 <= item_begin && item_begin <= item_end && item_end <= I, "bad item range");
  RPK_REQUIRE(similarity == RPK_SIM_COSINE || similarity == RPK_SIM_CONDPROB, "unknown similarity");
  RPK_REQUIRE(out_idx_u && out_val_u && out_len_u, "out_idx / out_val / out_len must not be null");
  cudaStream_t st = c->stream;
  const int64_t nrows = item_end - item_begin;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "fr_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "fr_indices");
  const double* values = stage_in(c, values_u, (size_t)nnz, "fr_values");
  const double* pw = item_pow_u ? stage_in(c, item_pow_u, (size_t)I, "fr_pw") : nullptr;
  c->mark("fit_real: begin");

  int* n = c->buf<int>("fr_n", (size_t)I);
  int* cursor = c->buf<int>("fr_cursor", (size_t)I);
  u64* work = c->buf<u64>("fr_work", (size_t)I);
  int64_t* cscptr = c->buf<int64_t>("fr_cscptr", (size_t)I + 1);
  int* csc_users = c->buf<int>("fr_csc_users", (size_t)nnz);
  int* csc_off = c->buf<int>("fr_csc_off", (size_t)nnz);
  RPK_CUDA(cudaMemsetAsync(n, 0, sizeof(int) * (size_t)I, st));
  RPK_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * (size_t)I, st));
  RPK_CUDA(cudaMemsetAsync(work, 0, sizeof(u64) * (size_t)I, st));
  const int wide = c->sm_count * 16;
  if (nnz > 0) {
    k_real_item_counts<<<(int)std::min<int64_t>((nnz + 255) / 256, wide), 256, 0, st>>>(indices, nnz, n);
    RPK_LAUNCH_CHECK(c);
  }
  scan_i32_i64(c, n, cscptr, I);
  if (nnz > 0 && U > 0 && I > 0) {
    k_real_fill_csc<<<(int)std::min<int64_t>((U * 32 + 255) / 256, wide), 256, 0, st>>>(indptr, indices, U, cscptr, cursor,
                                                                                         csc_users, work);
    RPK_LAUNCH_CHECK(c);
    // the bitmap covers every user (U / 8 bytes); the 512-entry rank sort needs 2 KB
    const int nwords = (int)((U + 31) / 32);
    const size_t sort_smem = std::max<size_t>(2048, (size_t)nwords * 4);
    RPK_REQUIRE(sort_smem + 2048 <= (size_t)c->smem_max, "more than ~1.8M users are not supported on the real-valued fit path");
    RPK_CUDA(cudaFuncSetAttribute(k_real_sort_csc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
    k_real_sort_csc<<<(int)std::min<int64_t>(I, (int64_t)c->sm_count * 8), 256, sort_smem, st>>>(cscptr, csc_users, I, nwords);
    RPK_LAUNCH_CHECK(c);
    k_real_csc_pos<<<(int)std::min<int64_t>((I * 32 + 255) / 256, wide), 256, 0, st>>>(cscptr, csc_users, indptr, indices, I,
                                                                                        csc_off);
    RPK_LAUNCH_CHECK(c);
  }
  const double* left = nullptr;
  const double* right = values;
  const double* row_scale = nullptr;
  const double* col_scale = nullptr;
  if (similarity == RPK_SIM_COSINE) {
    double* norm = c->buf<double>("fr_norm", (size_t)I);
    double* xhat = c->buf<double>("fr_xhat", (size_t)nnz);
    if (I > 0) {
      k_real_item_norms<<<ceil_div(I, 128), 128, 0, st>>>(cscptr, csc_users, csc_off, indptr, values, I, norm);
      RPK_LAUNCH_CHECK(c);
    }
    if (nnz > 0) {
      k_real_normalise<<<(int)std::min<int64_t>((nnz + 255) / 256, wide), 256, 0, st>>>(indices, values, norm, nnz, xhat);
      RPK_LAUNCH_CHECK(c);
    }
    left = xhat;
    right = xhat;
  } else {
    double* rn = c->buf<double>("fr_recip", (size_t)I);
    if (I > 0) {
      k_real_recip<<<ceil_div(I, 256), 256, 0, st>>>(n, I, rn);
      RPK_LAUNCH_CHECK(c);
    }
    row_scale = rn;
    col_scale = pw;
  }
  c->mark("fit_real: CSC + operands");

  Out<int32_t> o_idx, o_len;
  Out<double> o_val;
  o_idx.init(c, out_idx_u, (size_t)nrows * K, "fr_out_idx");
  o_val.init(c, out_val_u, (size_t)nrows * K, "fr_out_val");
  o_len.init(c, out_len_u, (size_t)nrows, "fr_out_len");
  if (nrows > 0) {
    int* order = c->buf<int>("fr_order", (size_t)nrows);
    int* bcnt = c->buf<int>("fr_bcnt", 65 * 2 + 2);
    int* boff = bcnt + 65;
    int* queue = c->buf<int>("fr_queue", 4);
    RPK_CUDA(cudaMemsetAsync(bcnt, 0, sizeof(int) * (65 * 2 + 2), st));
    RPK_CUDA(cudaMemsetAsync(queue, 0, sizeof(int) * 4, st));
    k_bucket_count<<<ceil_div(nrows, 256), 256, 0, st>>>(work, item_begin, item_end, bcnt);
    RPK_LAUNCH_CHECK(c);
    k_bucket_offsets<<<1, 32, 0, st>>>(bcnt, boff);
    RPK_LAUNCH_CHECK(c);
    k_bucket_scatter<<<ceil_div(nrows, 256), 256, 0, st>>>(work, item_begin, item_end, boff, order);
    RPK_LAUNCH_CHECK(c);

    const bool tiny = c->flags & DBG_TINY_LIST;
    const int cap = std::max(tiny ? 64 : 1024, next_pow2(2 * K));
    const int direct_cap = tiny ? K : cap;
    const size_t fixed = sel_smem_bytes(cap);
    RPK_REQUIRE((size_t)c->smem_max > fixed + 4096 + 2048, "K too large for shared memory");
    const size_t avail = (size_t)c->smem_max - fixed - 2048;
    int64_t Rmax = (int64_t)(avail / sizeof(double)) & ~(int64_t)7;
    int P = (int)((I + Rmax - 1) / Rmax);
    if (P < 1) P = 1;
    if ((c->flags & DBG_MULTI_PASS) && P < 2 && I >= 16) P = 2;
    const int R = (int)(((I + P - 1) / P + 7) & ~(int64_t)7);
    const size_t smem = fixed + (size_t)R * sizeof(double);
    const int nt = R >= 8192 ? 1024 : (R >= 1024 ? 256 : 64);
    RPK_CUDA(cudaFuncSetAttribute(k_real_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(nrows, (int64_t)c->sm_count));
    RealParams rp;
    rp.indptr = indptr;
    rp.indices = indices;
    rp.left = left;
    rp.right = right;
    rp.cscptr = cscptr;
    rp.csc_users = csc_users;
    rp.csc_off = csc_off;
    rp.left_entry = nullptr;
    rp.split = build_split(c, indptr, indices, U, I, P, R, nt, &rp.split_w);
    rp.row_scale = row_scale;
    rp.col_scale = col_scale;
    rp.diag = 1;
    rp.mask_list = 0;
    rp.item_ok = nullptr;
    rp.mode = 0;
    rp.nrows_dev = nullptr;
    rp.out_row_nnz = nullptr;
    rp.out_indptr = nullptr;
    rp.csr_indices = nullptr;
    rp.csr_values = nullptr;
    rp.order = order;
    rp.nrows = (int)nrows;
    rp.P = P;
    rp.R = R;
    rp.I = (int)I;
    rp.K = K;
    rp.item_begin = item_begin;
    rp.cap = cap;
    rp.direct_cap = direct_cap;
    rp.queue = queue;
    rp.scr_idx = c->buf<int>("fr_scr_idx", (size_t)grid * (size_t)(I + 1));
    rp.scr_val = c->buf<double>("fr_scr_val", (size_t)grid * (size_t)(I + 1));
    rp.out_idx = o_idx.dev;
    rp.out_val = o_val.dev;
    rp.out_len = o_len.dev;
    k_real_rows<<<grid, nt, smem, st>>>(rp);
    RPK_LAUNCH_CHECK(c);
  }
  c->mark("fit_real: rows");
  o_idx.finish(c);
  o_val.finish(c);
  o_len.finish(c);
  finish_call(c);
}

// Rows of C = A @ B through k_real_rows, every operand in device memory (a_val null: every left value is 1.0, a binary
// history).  order null: all rows of A, heaviest first; else the rows order[0 .. *n_order) (n_order: device-side count,
// at most `rows`).  item_ok (non-null) removes the filtered columns before the truncation to N.
void spgemm_rows_device(rpk_ctx* c, int64_t rows, const int64_t* a_ptr, const int32_t* a_idx, const double* a_val, int64_t I,
                        const int64_t* b_ptr, const int32_t* b_idx, const double* b_val, const int* order, const int* n_order, int N,
                        int mask_history, const unsigned char* item_ok, int mode, int32_t* out_idx, double* out_val,
                        int32_t* out_len, int64_t* out_row_nnz, const int64_t* out_indptr, int32_t* csr_indices,
                        double* csr_values) {
  if (rows <= 0) return;
  cudaStream_t st = c->stream;
  int* queue = c->buf<int>("sg_queue", 4);
  RPK_CUDA(cudaMemsetAsync(queue, 0, sizeof(int) * 4, st));
  if (!order) {
    u64* work = c->buf<u64>("sg_work", (size_t)rows);
    int* ord = c->buf<int>("sg_order", (size_t)rows);
    int* bcnt = c->buf<int>("sg_bcnt", 65 * 2 + 2);
    int* boff = bcnt + 65;
    RPK_CUDA(cudaMemsetAsync(bcnt, 0, sizeof(int) * (65 * 2 + 2), st));
    k_spgemm_work<<<(int)std::min<int64_t>((rows * 32 + 255) / 256, (int64_t)c->sm_count * 16), 256, 0, st>>>(a_ptr, a_idx, b_ptr, rows,
                                                                                                        work);
    RPK_LAUNCH_CHECK(c);
    k_bucket_count<<<ceil_div(rows, 256), 256, 0, st>>>(work, 0, rows, bcnt);
    RPK_LAUNCH_CHECK(c);
    k_bucket_offsets<<<1, 32, 0, st>>>(bcnt, boff);
    RPK_LAUNCH_CHECK(c);
    k_bucket_scatter<<<ceil_div(rows, 256), 256, 0, st>>>(work, 0, rows, boff, ord);
    RPK_LAUNCH_CHECK(c);
    order = ord;
  }
  const bool tiny = c->flags & DBG_TINY_LIST;
  const int cap = std::max(tiny ? 64 : 1024, next_pow2(2 * N));
  const int direct_cap = tiny ? N : cap;
  const size_t fixed = sel_smem_bytes(cap);
  RPK_REQUIRE((size_t)c->smem_max > fixed + 4096 + 2048, "N too large for shared memory");
  const size_t avail = (size_t)c->smem_max - fixed - 2048;
  int64_t Rmax = (int64_t)(avail / sizeof(double)) & ~(int64_t)7;
  int P = (int)((std::max<int64_t>(I, 1) + Rmax - 1) / Rmax);
  if (P < 1) P = 1;
  if ((c->flags & DBG_MULTI_PASS) && P < 2 && I >= 16) P = 2;
  const int R = (int)(((std::max<int64_t>(I, 1) + P - 1) / P + 7) & ~(int64_t)7);
  const size_t smem = fixed + (size_t)R * sizeof(double);
  const int nt = R >= 8192 ? 1024 : (R >= 1024 ? 256 : 64);
  RPK_CUDA(cudaFuncSetAttribute(k_real_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(rows, (int64_t)c->sm_count));
  RealParams rp;
  rp.indptr = b_ptr;
  rp.indices = b_idx;
  rp.left = nullptr;
  rp.right = b_val;
  rp.cscptr = a_ptr;
  rp.csc_users = a_idx;
  rp.csc_off = nullptr;
  rp.left_entry = a_val;
  // a few handed-over rows search their slices instead of paying for the table of all rows of B
  rp.split = n_order ? nullptr : build_split(c, b_ptr, b_idx, I, I, P, R, nt, &rp.split_w);
  if (n_order) rp.split_w = 0;
  rp.row_scale = nullptr;
  rp.col_scale = nullptr;
  rp.order = order;
  rp.nrows = (int)rows;
  rp.nrows_dev = n_order;
  rp.P = P;
  rp.R = R;
  rp.I = (int)I;
  rp.K = N;
  rp.item_begin = 0;
  rp.cap = cap;
  rp.direct_cap = direct_cap;
  rp.diag = 0;
  rp.mask_list = mask_history ? 1 : 0;
  rp.item_ok = item_ok;
  rp.mode = mode;
  rp.queue = queue;
  rp.scr_idx = c->buf<int>("fr_scr_idx", mode == 0 ? (size_t)grid * (size_t)(I + 1) : 16);
  rp.scr_val = c->buf<double>("fr_scr_val", mode == 0 ? (size_t)grid * (size_t)(I + 1) : 16);
  rp.out_idx = out_idx;
  rp.out_val = out_val;
  rp.out_len = out_len;
  rp.out_row_nnz = reinterpret_cast<long long*>(out_row_nnz);
  rp.out_indptr = out_indptr;
  rp.csr_indices = csr_indices;
  rp.csr_values = csr_values;
  k_real_rows<<<grid, nt, smem, st>>>(rp);
  RPK_LAUNCH_CHECK(c);
}

// C = A @ B for a real-valued CSR A [rows x I] and a CSR B [I x I] with ascending columns (the similarity model), float64
// in scipy's csr_matmat order (bit-identical sums): per-row top-N lists (mode 0), stored entries per row (mode 1) or the
// CSR rows themselves (mode 2, out_indptr from the counts).  Replaces `X_decayed @ similarity_matrix_` of
// TARSItemKNN._predict (time_aware_item_knn/base.py:137-149 -> algorithms/base.py:237-255) and, with mask_history,
// pipelines/pipeline.py:174-175.
void run_spgemm(rpk_ctx* c, int64_t rows, int64_t a_nnz, const int64_t* a_indptr_u, const int32_t* a_indices_u,
                const double* a_values_u, int64_t I, int64_t b_nnz, const int64_t* b_indptr_u, const int32_t* b_indices_u,
                const double* b_values_u, int N, int mask_history, int mode, int32_t* out_idx_u, double* out_val_u,
                int32_t* out_len_u, int64_t* out_row_nnz_u, const int64_t* out_indptr_u, int64_t out_nnz, int32_t* csr_indices_u,
                double* csr_values_u) {
  RPK_REQUIRE(rows >= 0 && I >= 0 && a_nnz >= 0 && b_nnz >= 0, "negative dimension");
  RPK_REQUIRE(I < (int64_t)1 << 24, "more than 2^24 items are not supported");
  RPK_REQUIRE(rows < (int64_t)1 << 31, "more than 2^31 rows are not supported");
  RPK_REQUIRE(mode >= 0 && mode <= 2, "bad mode");
  if (mode == 0) {
    RPK_REQUIRE(N >= 1 && N <= 4096, "N must be in [1, 4096]");
    RPK_REQUIRE(out_idx_u && out_val_u && out_len_u, "out_idx / out_val / out_len must not be null");
  } else if (mode == 1) {
    RPK_REQUIRE(out_row_nnz_u, "out_row_nnz must not be null");
    N = 1;
  } else {
    RPK_REQUIRE(out_indptr_u && (out_nnz == 0 || (csr_indices_u && csr_values_u)), "CSR outputs must not be null");
    N = 1;
  }
  const int64_t* a_ptr = stage_in(c, a_indptr_u, (size_t)rows + 1, "sg_a_ptr");
  const int32_t* a_idx = stage_in(c, a_indices_u, (size_t)a_nnz, "sg_a_idx");
  const double* a_val = stage_in(c, a_values_u, (size_t)a_nnz, "sg_a_val");
  const int64_t* b_ptr = stage_in(c, b_indptr_u, (size_t)I + 1, "sg_b_ptr");
  const int32_t* b_idx = stage_in(c, b_indices_u, (size_t)b_nnz, "sg_b_idx");
  const double* b_val = stage_in(c, b_values_u, (size_t)b_nnz, "sg_b_val");
  const int64_t* o_ptr = mode == 2 ? stage_in(c, out_indptr_u, (size_t)rows + 1, "sg_o_ptr") : nullptr;
  Out<int32_t> o_idx, o_len, o_ci;
  Out<double> o_val, o_cv;
  Out<int64_t> o_cnt;
  if (mode == 0) {
    o_idx.init(c, out_idx_u, (size_t)rows * N, "sg_out_idx");
    o_val.init(c, out_val_u, (size_t)rows * N, "sg_out_val");
    o_len.init(c, out_len_u, (size_t)rows, "sg_out_len");
  } else if (mode == 1) {
    o_cnt.init(c, out_row_nnz_u, (size_t)rows, "sg_out_cnt");
  } else {
    o_ci.init(c, csr_indices_u, (size_t)out_nnz, "sg_out_ci");
    o_cv.init(c, csr_values_u, (size_t)out_nnz, "sg_out_cv");
  }
  c->mark("spgemm: begin");
  spgemm_rows_device(c, rows, a_ptr, a_idx, a_val, I, b_ptr, b_idx, b_val, nullptr, nullptr, N, mask_history, nullptr, mode, o_idx.dev,
                     o_val.dev, o_len.dev, o_cnt.dev, o_ptr, o_ci.dev, o_cv.dev);
  c->mark("spgemm: rows");
  o_idx.finish(c);
  o_val.finish(c);
  o_len.finish(c);
  o_cnt.finish(c);
  o_ci.finish(c);
  o_cv.finish(c);
  finish_call(c);
}

}  // namespace rpk
