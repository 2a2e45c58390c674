// ItemKNN fit on the GPU: exact co-occurrence counts per item row accumulated in shared memory,
// with the similarity ordering, diagonal removal and top-K selection fused on the row while it
// is still in shared memory -- the item x item matrix is never written to HBM.
//
// Replaces (reference, /root/reference):
//   recpack/algorithms/nearest_neighbour.py:22-84   compute_conditional_probability / compute_cosine_similarity
//   recpack/util.py:50-96                           get_top_K_ranks / get_top_K_values
// Row i of the Gram is  c_ij = sum_{u in users(i)} [j in hist(u)]: one CTA owns (row i, item range p),
// walks users(i) through the CSC copy of X and bumps 32-bit shared-memory counters (native ATOMS.ADD).
#include <stdio.h>

#include <vector>

#include "common.cuh"
#include "internal.h"
#include "prims.cuh"
#ifdef RPK_PHASE_PROF
__device__ unsigned long long g_sel_prof[16];
#define SEL_MARK_BEGIN() __shared__ long long sel_tprev; if (threadIdx.x == 0) sel_tprev = clock64()
#define SEL_MARK(k)                                                               \
  do {                                                                            \
    if (threadIdx.x == 0) {                                                       \
      const long long t_now = clock64();                                          \
      atomicAdd(&g_sel_prof[k], (unsigned long long)(t_now - sel_tprev));         \
      sel_tprev = t_now;                                                          \
    }                                                                             \
  } while (0)
// path counters of one fit call: the SelEvent branches taken by the row kernel's selections, then rows deferred to
// k_fit_sort_rows and rows merged by k_fit_merge
#define FIT_EV_DEFERRED 5
#define FIT_EV_MERGED 6
__device__ unsigned long long g_fit_ev[8];
#define SEL_EVENT(src, ev) sel_event(src, ev)
#endif
#include "select.cuh"

namespace rpk {

// ------------------------------------------------------------------------------------------
// CSR preparation: item popularities, CSC transpose, per-row work estimate
// ------------------------------------------------------------------------------------------
// Per-item number of users that stay on the sparse path: n_light starts as a copy of the item popularities
// and the (few) dense users' interactions are taken off it (one warp per user).
__global__ void k_item_counts_light(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t U,
                                    const int* __restrict__ dense_slot, int* __restrict__ n_light) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = warp; u < U; u += nwarps) {
    if (dense_slot[u] < 0) continue;
    for (int64_t k = indptr[u] + lane; k < indptr[u + 1]; k += 32) atomicSub(&n_light[indices[k]], 1);
  }
}

__global__ void k_item_counts(const int* __restrict__ indices, int64_t nnz, int* __restrict__ n) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) atomicAdd(&n[indices[e]], 1);
}

// One warp per user: scatter the user id into the lists of its items; work[j] += d_u.
__global__ void k_fill_csc(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t U,
                           const int* __restrict__ dense_slot, const int64_t* __restrict__ cscptr, int* __restrict__ cursor,
                           int* __restrict__ csc_users, u64* __restrict__ work, int item_begin, int item_end) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = warp; u < U; u += nwarps) {
    if (dense_slot && dense_slot[u] >= 0) continue;  // handled by the tensor-core Gram
    int64_t b = indptr[u], e = indptr[u + 1];
    u64 d = (u64)(e - b);
    for (int64_t k = b + lane; k < e; k += 32) {
      int j = indices[k];
      if (j < item_begin || j >= item_end) continue;  // only this shard's item rows are fitted
      int pos = atomicAdd(&cursor[j], 1);
      csc_users[cscptr[j] + pos] = (int)u;
      atomicAdd(&work[j], d);
    }
  }
}

// ---- hybrid split: the users with the longest histories go through the tensor-core Gram ----
__global__ void k_len_hist(const int64_t* __restrict__ indptr, int64_t U, int64_t I, int* __restrict__ hist) {
  int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u < U) {
    int64_t d = indptr[u + 1] - indptr[u];
    if (d > I) d = I;
    atomicAdd(&hist[d], 1);
  }
}
__global__ void k_assign_dense_slots(const int64_t* __restrict__ indptr, int64_t U, int* __restrict__ thr_cnt, int hmax,
                                     int* __restrict__ slot, int* __restrict__ dense_user) {
  int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= U) return;
  const int64_t d = indptr[u + 1] - indptr[u];
  int s = -1;
  if (d >= thr_cnt[0]) {
    s = atomicAdd(&thr_cnt[1], 1);
    if (s >= hmax) s = -1;  // cannot happen: the threshold admits at most hmax users
    else dense_user[s] = (int)u;
  }
  slot[u] = s;
}
// One block per dense user (their histories are the longest of all): A[item][slot] = 1 for its interactions, and the
// user is taken off the sparse path's item counts.
__global__ void k_fill_dense_users(const int64_t* __restrict__ indptr, const int* __restrict__ indices,
                                   const int* __restrict__ dense_user, const int* __restrict__ thr_cnt, int64_t kd_pad,
                                   unsigned char* __restrict__ A, int* __restrict__ n_light) {
  const int s = blockIdx.x;
  if (s >= thr_cnt[1]) return;
  const int u = dense_user[s];
  for (int64_t k = indptr[u] + threadIdx.x; k < indptr[u + 1]; k += blockDim.x) {
    const int j = indices[k];
    A[(int64_t)j * kd_pad + s] = 1;
    atomicSub(&n_light[j], 1);
  }
}
// A[item][slot] = 1 for every interaction of a dense user (one warp per user).
__global__ void k_fill_dense(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t U,
                             const int* __restrict__ slot, int64_t kd_pad, unsigned char* __restrict__ A) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = warp; u < U; u += nwarps) {
    const int s = slot[u];
    if (s < 0) continue;
    for (int64_t k = indptr[u] + lane; k < indptr[u + 1]; k += 32) A[(int64_t)indices[k] * kd_pad + s] = 1;
  }
}

// ---- items seen by >= 65536 users: a co-occurrence count between two of them may not fit 16 bits ----
constexpr int HEAVY_CAP = 32;
__global__ void k_find_heavy(const int* __restrict__ n, int64_t I, int* __restrict__ heavy_ids, int* __restrict__ heavy_n) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < I && n[j] >= 65536) {
    const int s = atomicAdd(heavy_n, 1);
    if (s < HEAVY_CAP) heavy_ids[s] = (int)j;
  }
}
// pair[a * HEAVY_CAP + b] = exact number of users with both heavy items a and b.  A group of G lanes
// (G = H rounded up to a power of two) takes one user, lane h looks heavy item h up in the user's sorted
// history; counts are kept per thread and flushed once.
__global__ void k_heavy_pairs(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t U,
                              const int* __restrict__ heavy_ids, const int* __restrict__ heavy_n, int* __restrict__ pair) {
  const int H = heavy_n[0];
  if (H < 2 || H > HEAVY_CAP) return;
  int G = 2;
  while (G < H) G <<= 1;
  const int lane = threadIdx.x & 31;
  const int h = lane & (G - 1), grp = lane / G, per_warp = 32 / G;
  const unsigned gmask = G == 32 ? 0xffffffffu : ((1u << G) - 1u);
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int target = h < H ? heavy_ids[h] : -1;
  // pair counts of this block in shared memory, added to the global table once at the end
  __shared__ int s_pair[HEAVY_CAP * HEAVY_CAP];
  for (int t = threadIdx.x; t < HEAVY_CAP * HEAVY_CAP; t += blockDim.x) s_pair[t] = 0;
  __syncthreads();
  for (int64_t u0 = warp * per_warp; u0 < U; u0 += nwarps * per_warp) {
    const int64_t u = u0 + grp;
    bool has = false;
    if (u < U && target >= 0) {
      int64_t lo = indptr[u], hi = indptr[u + 1];
      const int64_t end = hi;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int v = indices[mid];
        if (v < target) lo = mid + 1;
        else hi = mid;
      }
      has = lo < end && indices[lo] == target;
    }
    const unsigned m = (__ballot_sync(0xffffffffu, has) >> (grp * G)) & gmask;
    if (has) {
      unsigned others = m & ~(1u << h);
      while (others) {
        const int b = __ffs(others) - 1;
        others &= others - 1;
        atomicAdd(&s_pair[h * HEAVY_CAP + b], 1);
      }
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < HEAVY_CAP * HEAVY_CAP; t += blockDim.x)
    if (s_pair[t]) atomicAdd(&pair[t], s_pair[t]);
}

// pref[k] = sum of the history lengths of the users listed before position k of the same item
// (exclusive, in CSC order): lets the fit kernel cut a row's work into equal pieces per warp.
constexpr int CSC_PREFIX_LONG = 4096;  // items with more users than this are scanned by a whole block
__global__ void __launch_bounds__(1024) k_csc_prefix_long(const int64_t* __restrict__ cscptr, const int* __restrict__ csc_users,
                                                          const int64_t* __restrict__ indptr, int64_t item_begin,
                                                          int64_t item_end, unsigned* __restrict__ pref) {
  __shared__ unsigned s_warp[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int64_t i = item_begin + blockIdx.x; i < item_end; i += gridDim.x) {
    const int64_t b = cscptr[i], e = cscptr[i + 1];
    if (e - b <= CSC_PREFIX_LONG) continue;
    unsigned carry = 0;
    for (int64_t base = b; base < e; base += 4096) {  // 4 users per thread
      unsigned v[4], tot = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int64_t k = base + 4 * tid + q;
        v[q] = 0;
        if (k < e) {
          const int u = csc_users[k];
          v[q] = (unsigned)(indptr[u + 1] - indptr[u]);
        }
        tot += v[q];
      }
      unsigned incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (lane == 31) s_warp[warp] = incl;
      __syncthreads();
      unsigned wv = s_warp[lane];  // blockDim.x == 1024: 32 warp totals
      unsigned wincl = wv;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, wincl, o);
        if (lane >= o) wincl += t;
      }
      const unsigned before = __shfl_sync(0xffffffffu, wincl - wv, warp);
      const unsigned block_tot = __shfl_sync(0xffffffffu, wincl, 31);
      unsigned run = carry + before + incl - tot;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int64_t k = base + 4 * tid + q;
        if (k < e) pref[k] = run;
        run += v[q];
      }
      carry += block_tot;
      __syncthreads();
    }
  }
}

__global__ void k_csc_prefix(const int64_t* __restrict__ cscptr, const int* __restrict__ csc_users,
                             const int64_t* __restrict__ indptr, int64_t item_begin, int64_t item_end,
                             unsigned* __restrict__ pref) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = item_begin + warp; i < item_end; i += nwarps) {
    const int64_t b = cscptr[i], e = cscptr[i + 1];
    if (e - b > CSC_PREFIX_LONG) continue;  // long lists: k_csc_prefix_long (a whole block per item)
    unsigned carry = 0;
    for (int64_t base = b; base < e; base += 128) {  // 4 users per lane: four independent loads in flight
      unsigned v[4], tot = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int64_t k = base + 4 * lane + q;
        v[q] = 0;
        if (k < e) {
          const int u = csc_users[k];
          v[q] = (unsigned)(indptr[u + 1] - indptr[u]);
        }
        tot += v[q];
      }
      unsigned incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      unsigned run = carry + incl - tot;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int64_t k = base + 4 * lane + q;
        if (k < e) pref[k] = run;
        run += v[q];
      }
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
  }
}

// Largest popularity and (with pop_discount) the smallest item_pow among seen items: key bounds.
__global__ void k_item_extremes(const int* __restrict__ n, const double* __restrict__ pw, int64_t I, int* __restrict__ nmax,
                                u64* __restrict__ pwmin_bits) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int v = j < I ? n[j] : 0;
  v = __reduce_max_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && v > 0) atomicMax(nmax, v);
  if (pw) {
    u64 b = (j < I && n[j] > 0) ? (u64)__double_as_longlong(pw[j]) : ~0ull;  // positive doubles order like integers
    b = warp_min_u64(b);
    if ((threadIdx.x & 31) == 0) atomicMin(pwmin_bits, b);
  }
}

// code[j] = round(12 * log2(n_j)) clamped to [0, 255]: 1/n_j to within half a code step.
__global__ void k_pop_code(const int* __restrict__ n, unsigned char* __restrict__ code, int64_t I) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < I) {
    const int v = n[j] > 0 ? __float2int_rn(12.0f * log2f((float)n[j])) : 0;
    code[j] = (unsigned char)(v < 0 ? 0 : (v > 255 ? 255 : v));
  }
}

__global__ void k_recip_f32(const int* __restrict__ n, float* __restrict__ rnf, int64_t I) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < I) rnf[j] = n[j] > 0 ? __frcp_rn((float)n[j]) : 0.f;
}

// usplit[u*(P+1)+p] = first position in row u whose item id >= p*R  (p = 0..P)
__global__ void k_user_split(const int64_t* __restrict__ indptr, const int* __restrict__ indices, int64_t U, int P, int R,
                             int64_t* __restrict__ usplit) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= U * (P + 1)) return;
  int64_t u = t / (P + 1);
  int p = (int)(t % (P + 1));
  int64_t lo = indptr[u], hi = indptr[u + 1];
  if (p == P) {
    usplit[t] = hi;
    return;
  }
  int64_t target = (int64_t)p * R;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (indices[mid] < target) lo = mid + 1;
    else hi = mid;
  }
  usplit[t] = lo;
}

// ------------------------------------------------------------------------------------------
// Candidate sources for the selection routine
// ------------------------------------------------------------------------------------------
struct SimKey {
  const int* n;
  const float* rnf;
  const double* pw;
  const int* nmax;      // largest item popularity (device scalar)
  const double* pwmin;  // smallest item_pow among seen items (device scalar, mode 2)
  // cosine, inside k_fit_rows: 1/n_j rounded to a 12-steps-per-octave code (1 byte per item, kept in shared
  // memory) so that the selection scans need no global load per candidate; null: use rnf
  const unsigned char* code;
  const float* code_tab;  // [256] code -> 2^(-code/12)
  int mode;  // 0 cosine, 1 conditional probability, 2 conditional probability with pop_discount

  // Two keys can be mis-ordered only if their bit patterns differ by at most margin(): a few ulp with the
  // exact reciprocal; with the coded one each key is off by up to half a code step (2^(1/24)), so two keys
  // up to 2^(1/12) - 1 = 5.95 % apart can swap: 0.0595 * 2^24 patterns at most -> 2^20
  __device__ __forceinline__ u64 margin() const { return mode != 0 ? 0ull : (code ? (1ull << 20) : 32ull); }

  // cosine: approximate fp32 key c^2/n_j (a few ulp of error, covered by margin()); the exact order is
  // restored by cmp3 on (c, n_j).  conditional probability: the exact float64 key itself.
  __device__ __forceinline__ u64 akey(int c, int j) const {
    if (mode == 0) {
      const float a = (float)c;
      const float r = code ? code_tab[code[j]] : rnf[j];
      return (u64)__float_as_uint(__fmul_rn(__fmul_rn(a, a), r));
    }
    if (mode == 1) return (u64)__double_as_longlong((double)c);
    return (u64)__double_as_longlong(__dmul_rn((double)c, pw[j]));
  }
  // Every key of a row whose largest count is cmax lies in [lo, hi]  (rnf <= 1, item_pow <= 1).
  __device__ __forceinline__ void bounds(int cmax, u64& lo, u64& hi) const {
    if (mode == 0) {
      const float a = (float)cmax;
      hi = (u64)__float_as_uint(__fmul_rn(a, a));
      lo = (u64)__float_as_uint(__frcp_rn((float)nmax[0]) * 0.94f);  // 6 % slack for the coded reciprocal
    } else if (mode == 1) {
      hi = (u64)__double_as_longlong((double)cmax);
      lo = (u64)__double_as_longlong(1.0);
    } else {
      hi = (u64)__double_as_longlong((double)cmax);
      lo = (u64)__double_as_longlong(pwmin[0]);
    }
  }
  // Smallest count that can reach key thr (conservative): key <= c^2 (cosine) or key <= c.
  __device__ __forceinline__ int min_count(u64 thr) const {
    if (thr == 0) return 1;
    if (mode == 0) {
      const float t = __uint_as_float((unsigned)thr);
      const int c = (int)sqrtf(t) - 1;
      return c < 1 ? 1 : c;
    }
    const double t = __longlong_as_double((long long)thr);
    const int c = t > 2.0e9 ? 2000000000 : (int)t - 1;
    return c < 1 ? 1 : c;
  }
  __device__ __forceinline__ void entry(int c, int j, Entry& e) const {
    e.idx = j;
    e.aux = c;
    e.key = mode == 0 ? (u64)(unsigned)n[j] : akey(c, j);
  }
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const {
    if (mode == 0) {
      // c_a^2 / n_a  vs  c_b^2 / n_b   <=>   c_a^2 * n_b  vs  c_b^2 * n_a   (128-bit exact)
      u64 ca2 = (u64)(unsigned)a.aux * (u64)(unsigned)a.aux;
      u64 cb2 = (u64)(unsigned)b.aux * (u64)(unsigned)b.aux;
      u64 l_lo = ca2 * b.key, l_hi = __umul64hi(ca2, b.key);
      u64 r_lo = cb2 * a.key, r_hi = __umul64hi(cb2, a.key);
      if (l_hi != r_hi) return l_hi > r_hi ? 1 : -1;
      if (l_lo != r_lo) return l_lo > r_lo ? 1 : -1;
      return 0;
    }
    if (a.key != b.key) return a.key > b.key ? 1 : -1;
    return 0;
  }
};

// Dense shared-memory counters of one (row, item range).  PACK16: two 16-bit counters per word
// (rows with fewer than 65536 users cannot overflow them), else one 32-bit counter per item.
template <bool PACK16>
struct RowCountSrc {
  SimKey sk;
  const unsigned* cnt;
  int r0, ns, self;
  // "extra" candidates: columns whose count may not fit 16 bits (both items seen by >= 65536 users) carry an
  // exact 32-bit count from k_heavy_pairs; their packed counters are zeroed.  Slots ns .. ns+nex-1.
  const int* ex_idx;
  const int* ex_cnt;
  int nex;
  __device__ __forceinline__ int count(int slot) const {
    if (slot >= ns) return ex_cnt[slot - ns];
    if (PACK16) return (int)((cnt[slot >> 1] >> ((slot & 1) * 16)) & 0xffffu);
    return (int)cnt[slot];
  }
  __device__ __forceinline__ int item(int slot) const { return slot >= ns ? ex_idx[slot - ns] : r0 + slot; }
  __device__ __forceinline__ int nslots() const { return ns; }
  __device__ __forceinline__ u64 margin() const { return sk.margin(); }
  int cmin;  // set_floor(): counts below this cannot reach the requested key
  // cosine with coded popularities, packed counters: the smallest count that can reach the requested key, per
  // popularity code (key = c^2 * 2^(-code/12) >= thr  <=>  c >= sqrt(thr * 2^(code/12))).  One shared table of 256
  // entries, rebuilt by set_floor; the passes then test a counter against its item's entry with one load and one
  // compare instead of computing its key.  Null: only the global bound `cmin` is used.
  unsigned short* cm_tab;
  // the same bound without the slack of a whole count (rounding slack only): the queueing pass of for_each_queued tests
  // a counter against it instead of computing the counter's float key (no int -> float conversion, no multiplies)
  unsigned short* cq_tab;
  int count_bound;  // >= number of candidates of the row (0: unknown, stats() scans)
  const unsigned char* code_s;  // the coded popularities and their table again, as shared-memory pointers the compiler
  const float* tab_s;           // can see through (sk.code / sk.code_tab travel through the parameter struct: generic loads)
  u64 floor_key;                // set_floor(): candidates below this key may be skipped
  __device__ __forceinline__ void set_floor(u64 thr) {
    floor_key = thr;
    cmin = sk.min_count(thr);
    if (PACK16 && cm_tab) {
      __syncthreads();  // readers of the previous table are done
      if (threadIdx.x < 256) {
        int v = 1;
        if (thr) {
          const float need = __uint_as_float((unsigned)thr) / sk.code_tab[threadIdx.x];  // c^2 must reach this
          const float c = sqrtf(need) - 1.0f;                                            // one count of slack for rounding
          v = c < 1.0f ? 1 : (c > 65535.0f ? 65535 : (int)c);
        }
        cm_tab[threadIdx.x] = (unsigned short)v;
        int vq = 1;
        if (thr) {
          // key = fl(fl(c * c) * r) >= thr implies c >= sqrt(thr / r) * (1 - 2^-21); 1e-4 covers that with room to spare
          const float sq = sqrtf(__uint_as_float((unsigned)thr) / sk.code_tab[threadIdx.x]) * 0.9999f;
          vq = sq < 1.0f ? 1 : (sq > 65535.0f ? 65535 : (int)ceilf(sq));
        }
        cq_tab[threadIdx.x] = (unsigned short)vq;
      }
      __syncthreads();
    }
  }
  // Visit every candidate whose count reaches the floor.  The row's own slot (the diagonal) has been zeroed by the
  // caller, so no slot needs a self test.  Packed counters are read 16 bytes (eight counters) at a time and a
  // vector is skipped as a whole when none of its counters reaches the floor -- in the copy pass after a threshold
  // guess that is almost every vector, which is what makes the epilogue cheap next to the accumulation.
  // `nvec16`: number of 16-byte vectors of the counter array (the array is zero beyond the row's last counter).
  int nvec16;
  template <class F>
  __device__ __forceinline__ void visit(F f) const {
    const int tid = threadIdx.x, nt = blockDim.x;
    if (PACK16 && cm_tab) {
      // eight counters and the eight popularity codes of their items per iteration
      const uint4* c4 = reinterpret_cast<const uint4*>(cnt);
      const uint2* g8 = reinterpret_cast<const uint2*>(sk.code + r0);
      for (int v = tid; v < nvec16; v += nt) {
        const uint4 x = c4[v];
        if ((x.x | x.y | x.z | x.w) == 0u) continue;
        const uint2 g = g8[v];
        const unsigned xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int c = (int)((xs[q >> 1] >> ((q & 1) * 16)) & 0xffffu);
          const unsigned code = ((q < 4 ? g.x : g.y) >> ((q & 3) * 8)) & 0xffu;
          if (c >= (int)cm_tab[code]) f(8 * v + q, sk.akey(c, r0 + 8 * v + q));
        }
      }
    } else if (PACK16) {
      const uint4* c4 = reinterpret_cast<const uint4*>(cnt);
      const unsigned cm = (unsigned)(cmin > 65535 ? 65535 : (cmin < 1 ? 1 : cmin));
      const unsigned cm_hi = cm << 16;
      const bool none = cmin > 65535;  // no 16-bit counter can reach the floor
      for (int v = tid; v < nvec16; v += nt) {
        const uint4 x = c4[v];
        if ((x.x | x.y | x.z | x.w) == 0u || none) continue;
        const unsigned xs[4] = {x.x, x.y, x.z, x.w};
        bool any = false;
#pragma unroll
        for (int q = 0; q < 4; ++q) any |= (xs[q] >= cm_hi) | ((xs[q] & 0xffffu) >= cm);
        if (!any) continue;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c0 = (int)(xs[q] & 0xffffu), c1 = (int)(xs[q] >> 16);
          const int slot = 8 * v + 2 * q;
          if (c0 >= (int)cm) f(slot, sk.akey(c0, r0 + slot));
          if (c1 >= (int)cm) f(slot + 1, sk.akey(c1, r0 + slot + 1));
        }
      }
    } else {
      for (int w = tid; w < ns; w += nt) {
        const int c0 = (int)cnt[w];
        if (c0 >= cmin && c0 > 0) f(w, sk.akey(c0, r0 + w));
      }
    }
  }
  // Two-step visit (see compact_above).  Pass 1 computes the key of every counter without a branch -- eight counters
  // and their eight popularity codes per iteration, the same float operations as SimKey::akey -- and queues the
  // slots whose key reaches the floor, one shared-memory counter update per warp and iteration.  (Counts are small
  // numbers in most rows, so no cheap integer test separates the few survivors from the bulk: a test that lets a
  // fifth of the counters through makes every warp run the slow path at every step.)  Pass 2 hands the queued
  // slots to f, a candidate per thread.  Returns false (nothing visited) when the queue overflowed.
  __device__ __forceinline__ bool has_queue() const { return PACK16 && cm_tab != nullptr && floor_key > 0ull; }
  template <class F>
  __device__ bool for_each_queued(F f, int* queue, int qcap, int* qcount) const {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    if (tid == 0) *qcount = 0;
    __syncthreads();
    const uint4* c4 = reinterpret_cast<const uint4*>(cnt);
    const uint2* g8 = reinterpret_cast<const uint2*>(code_s + r0);
    for (int v0 = 0; v0 < nvec16; v0 += nt) {  // warp-uniform trip count: the warp queues together
      const int v = v0 + tid;
      unsigned hit = 0u;  // which of my eight counters reach the floor
      if (v < nvec16) {
        const uint4 x = c4[v];
        if ((x.x | x.y | x.z | x.w) != 0u) {
          const uint2 g = g8[v];
          const unsigned xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const unsigned cq = (xs[q >> 1] >> ((q & 1) * 16)) & 0xffffu;
            const unsigned need = cq_tab[((q < 4 ? g.x : g.y) >> ((q & 3) * 8)) & 0xffu];
            hit |= (cq >= need ? 1u : 0u) << q;
          }
        }
      }
      const int mine = __popc(hit);
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int wtot = __shfl_sync(0xffffffffu, incl, 31);
      if (wtot == 0) continue;
      int base = 0;
      if (lane == 31) base = atomicAdd(qcount, wtot);
      base = __shfl_sync(0xffffffffu, base, 31);
      int pos = base + incl - mine;
      while (hit) {
        const int q = __ffs(hit) - 1;
        hit &= hit - 1u;
        if (pos < qcap) queue[pos] = 8 * v + q;
        ++pos;
      }
    }
    __syncthreads();
    const int total = *qcount;
    if (total > qcap) return false;
    for (int t = tid; t < total; t += nt) {
      const int slot = queue[t];
      const int c = count(slot);
      f(slot, sk.akey(c, r0 + slot));
    }
    visit_extras(f);
    return true;
  }
  template <class F>
  __device__ __forceinline__ void visit_extras(F f) const {
    const int t = threadIdx.x;
    if (t < nex && ex_cnt[t] >= cmin && ex_cnt[t] > 0 && ex_idx[t] != self) f(ns + t, sk.akey(ex_cnt[t], ex_idx[t]));
  }
  template <class F>
  __device__ __forceinline__ void for_each(F f) const {
    visit(f);
    visit_extras(f);
  }
  // one slot in SEL_SAMPLE: the low counter of every 8th word (packed) / every 16th counter
  template <class F>
  __device__ __forceinline__ void for_each_sampled(F f) const {
    const int tid = threadIdx.x, nt = blockDim.x;
    if (PACK16) {
      const int nwords = (ns + 1) >> 1;
      for (int w = tid * (SEL_SAMPLE / 2); w < nwords; w += nt * (SEL_SAMPLE / 2)) {
        const int c0 = (int)(cnt[w] & 0xffffu);
        if (c0 >= cmin && c0 > 0) f(2 * w, sk.akey(c0, r0 + 2 * w));
      }
    } else {
      for (int w = tid * SEL_SAMPLE; w < ns; w += nt * SEL_SAMPLE) {
        const int c0 = (int)cnt[w];
        if (c0 >= cmin && c0 > 0) f(w, sk.akey(c0, r0 + w));
      }
    }
    visit_extras(f);
  }
  // Integer-only pass over the counters: candidate count and the largest count; the key bounds
  // follow from that (no popularity loads, no float math).
  __device__ void stats(SelShared* sh) const {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    if (PACK16 && cm_tab && count_bound > 0) {
      // no pass over the counters: a count is at most the row's own popularity, which bounds the keys; the number
      // of candidates is only needed as an upper bound (few real candidates under a large bound cost one
      // refinement pass more, nothing else)
      if (tid == 0) {
        u64 lo = 0, hi = 0;
        sk.bounds(sk.n[self], lo, hi);
        sh->count = count_bound;
        sh->kmin = lo;
        sh->kmax = hi;
      }
      __syncthreads();
      return;
    }
    if (tid == 0) {
      sh->count = 0;
      sh->bstar = 0;
    }
    __syncthreads();
    int cntc = 0;
    unsigned cmax = 0;
    if (PACK16) {
      const uint4* c4 = reinterpret_cast<const uint4*>(cnt);
      for (int v = tid; v < nvec16; v += nt) {
        const uint4 x = c4[v];
        if ((x.x | x.y | x.z | x.w) == 0u) continue;
        const unsigned xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const unsigned lo = xs[q] & 0xffffu, hi = xs[q] >> 16;
          cntc += (lo != 0u) + (hi != 0u);
          cmax = max(cmax, max(lo, hi));
        }
      }
    } else {
      for (int w = tid; w < ns; w += nt) {
        const unsigned c0 = cnt[w];
        cntc += c0 != 0u;
        cmax = max(cmax, c0);
      }
    }
    if (tid < nex && ex_cnt[tid] > 0 && ex_idx[tid] != self) {
      cntc++;
      cmax = max(cmax, (unsigned)ex_cnt[tid]);
    }
    cntc = __reduce_add_sync(0xffffffffu, cntc);
    cmax = __reduce_max_sync(0xffffffffu, cmax);
    if (lane == 0 && cntc) {
      atomicAdd(&sh->count, cntc);
      atomicMax(&sh->bstar, (int)cmax);
    }
    __syncthreads();
    if (tid == 0) {
      u64 lo = 0, hi = 0;
      if (sh->count) sk.bounds(sh->bstar, lo, hi);
      sh->kmin = lo;
      sh->kmax = hi;
    }
    __syncthreads();
  }
  __device__ __forceinline__ void entry(int slot, Entry& e) const { sk.entry(count(slot), item(slot), e); }
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const { return sk.cmp3(a, b); }
};

#ifdef RPK_PHASE_PROF
// only the selections of the row kernel (its counters are the source) are counted, not those of the merge and the sort
template <class Src>
__device__ __forceinline__ void sel_event(const Src&, int) {}
template <bool PACK16>
__device__ __forceinline__ void sel_event(const RowCountSrc<PACK16>&, int ev) { atomicAdd(&g_fit_ev[ev], 1ull); }
#endif

struct PairListSrc {  // (idx, cnt) pairs in global memory, idx < 0 = empty slot
  __device__ __forceinline__ bool has_queue() const { return false; }
  template <class F>
  __device__ __forceinline__ bool for_each_queued(F, int*, int, int*) const { return false; }
  SimKey sk;
  const int* idx;
  const int* cnt;
  int ns;
  __device__ __forceinline__ int nslots() const { return ns; }
  __device__ __forceinline__ u64 margin() const { return sk.margin(); }
  __device__ __forceinline__ void set_floor(u64) {}
  __device__ __forceinline__ void stats(SelShared* sh) const { generic_stats(*this, sh); }
  template <class F>
  __device__ __forceinline__ void visit(F f, int stride) const {
    for (int slot = threadIdx.x * stride; slot < ns; slot += blockDim.x * stride) {
      const int j = idx[slot];
      if (j >= 0) f(slot, sk.akey(cnt[slot], j));
    }
  }
  template <class F>
  __device__ __forceinline__ void for_each(F f) const { visit(f, 1); }
  template <class F>
  __device__ __forceinline__ void for_each_sampled(F f) const { visit(f, SEL_SAMPLE); }
  __device__ __forceinline__ void entry(int slot, Entry& e) const { sk.entry(cnt[slot], idx[slot], e); }
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const { return sk.cmp3(a, b); }
};

// ------------------------------------------------------------------------------------------
// The fit kernel
// ------------------------------------------------------------------------------------------
struct FitParams {
  const int64_t* indptr;
  const int* indices;
  const int64_t* usplit;  // null when P == 1
  const int64_t* cscptr;
  const int* csc_users;
  const unsigned* pref;   // per-item exclusive prefix of history lengths (CSC order)
  const u64* work;        // per-item total of history lengths
  const unsigned short* g16;  // dense-leg counts [I x ldg] (null: none); uint8 counts in the G8 kernel
  int64_t ldg;
  const int* pre;         // per item: slot of its pre-accumulated counters in `hbuf`, -1 = none (null: none at all)
  unsigned* hbuf;         // [slots x hstride] packed 16-bit counters summed over the pieces of a split row
  int64_t hstride;
  const int4* piece_tab;  // {item, piece, pieces, slot} of every piece, heaviest rows first
  const int* hcount;      // [0] number of pieces, [1] number of split rows
  const int* split_rows;  // the split rows (they are finished after everything else)
  int* hdone;             // per slot: pieces completed
  const int* hneed;       // per slot: pieces in all
  SimKey sk;
  const int* order;       // rows of this launch, heaviest first
  const int* nrows_dev;   // number of rows in `order` (device side: no host round trip)
  int P, R, I, K;
  int64_t item_begin;
  int cap, direct_cap;
  int direct_out;         // 1: P == 1, write final rows; 0: write per-(list position, pass) partial lists
  int* queue;
  int* out_idx;
  int* out_cnt;
  int* out_len;
  const unsigned char* pop_code;  // global [I], null: no coded reciprocals
  const int* heavy_ids;   // items seen by >= 65536 users (PACK16 launch only), null: none handled here
  const int* heavy_n;
  const int* heavy_pair;  // exact counts between them, [HEAVY_CAP x HEAVY_CAP]
  int defer_max;   // > 0: rows with at most this many survivors are sorted by k_fit_sort_rows instead
  int* scr_idx;    // [rows x defer_max] unsorted survivors (item, count)
  int* scr_cnt;
  int* scr_len;    // [rows] survivors in scratch, -1 = row already final in out_*
  unsigned long long* prof;  // RPK_PHASE_PROF builds: cycles of thread 0 per phase
};

#ifdef RPK_PHASE_PROF
#define FIT_MARK(k)                                                \
  do {                                                             \
    if (threadIdx.x == 0 && p.prof) {                              \
      const long long t_now = clock64();                           \
      atomicAdd(p.prof + (k), (unsigned long long)(t_now - t_prev)); \
      t_prev = t_now;                                              \
    }                                                              \
  } while (0)
#else
#define FIT_MARK(k) do {} while (0)
#endif

// Adds the histories of the users of item i whose work prefix lies in [lo, hi) to the counters (one warp;
// the window is a piece of the row's total work = sum of its users' history lengths).
template <bool PACK16>
__device__ __forceinline__ void accumulate_window(const FitParams& p, unsigned* cnt, int64_t ub, int nu, int r0,
                                                  unsigned lo, unsigned hi) {
  const int lane = threadIdx.x & 31;
  const unsigned* pf_row = p.pref + ub;
  int a = 0, b = nu;  // 32-ary search: last user whose prefix is <= lo
  while (b - a > 1) {
    const int step = (b - a + 31) / 32;
    const int k = a + lane * step;
    const bool ok = k < b && pf_row[k] <= lo;
    const unsigned mk = __ballot_sync(0xffffffffu, ok) | 1u;
    const int last = 31 - __clz(mk);
    const int na = a + last * step;
    b = min(b, na + step);
    a = na;
  }
  for (int kbase = a; kbase < nu; kbase += 32) {
    const int kk = kbase + lane;
    unsigned pf = 0xffffffffu;
    int64_t beg = 0;
    int len = 0;
    if (kk < nu) {
      const int u = p.csc_users[ub + kk];
      pf = pf_row[kk];
      beg = p.indptr[u];
      len = (int)(p.indptr[u + 1] - beg);
    }
    if (__shfl_sync(0xffffffffu, pf, 0) >= hi) break;
    // software pipeline over the users of the batch, three deep: while the counters of user l are updated the first
    // 128 indices of users l+1 and l+2 are already on their way (an index load is an L2 round trip: one user in
    // flight left every warp waiting most of the time)
    struct Stage {
      int j[4];
      int64_t b;
      int s, e;
    };
    auto fetch = [&](Stage& st, int l) {  // clip user l to [lo, hi) and issue its first loads
      st.s = 0;
      st.e = 0;
      st.b = 0;
      if (l < 32) {
        const unsigned pfl = __shfl_sync(0xffffffffu, pf, l);
        const int n = __shfl_sync(0xffffffffu, len, l);
        st.b = __shfl_sync(0xffffffffu, beg, l);
        if (pfl < hi) {
          st.s = lo > pfl ? (int)(lo - pfl) : 0;
          st.e = (int)min((unsigned)n, hi - pfl);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int e = st.s + lane + 32 * q;
        st.j[q] = e < st.e ? p.indices[st.b + e] - r0 : -1;
      }
    };
    auto apply = [&](const Stage& st) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (st.j[q] >= 0) {
          if (PACK16) atomicAdd(&cnt[st.j[q] >> 1], 1u << ((st.j[q] & 1) * 16));
          else atomicAdd(&cnt[st.j[q]], 1u);
        }
      // long histories: the rest, four loads in flight per lane
      for (int e = st.s + 128 + lane; e < st.e; e += 128) {
        int jj[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) jj[q] = e + 32 * q < st.e ? p.indices[st.b + e + 32 * q] - r0 : -1;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (jj[q] >= 0) {
            if (PACK16) atomicAdd(&cnt[jj[q] >> 1], 1u << ((jj[q] & 1) * 16));
            else atomicAdd(&cnt[jj[q]], 1u);
          }
      }
    };
    Stage A, B, C;
    fetch(A, 0);
    fetch(B, 1);
    for (int l = 0; l < 32; l += 3) {
      if (__shfl_sync(0xffffffffu, pf, l) >= hi) break;
      fetch(C, l + 2);
      apply(A);
      if (l + 1 >= 32 || __shfl_sync(0xffffffffu, pf, l + 1) >= hi) break;
      fetch(A, l + 3);
      apply(B);
      if (l + 2 >= 32 || __shfl_sync(0xffffffffu, pf, l + 2) >= hi) break;
      fetch(B, l + 4);
      apply(C);
    }
  }
}

// ---- very heavy rows: one CTA per row bounds the fit by the heaviest row once the rows of a shard are few
// (multi-GPU).  The work of such a row is cut into pieces.  Pieces are ordinary work items at the head of
// k_fit_rows' queue: a CTA counts its piece in shared memory and adds the counters into a global row; the
// split rows themselves come last in the queue, start from those counters and only run the epilogue.
constexpr int HEAVY_ROWS = 64;    // candidate rows (the first of the heaviest-first order)
constexpr int HEAVY_SPLITS = 16;  // pieces per row at most

__global__ void __launch_bounds__(1024) k_heavy_plan(const int* __restrict__ order, const int* __restrict__ nrows_dev,
                                                     const u64* __restrict__ work, int sm_count, u64 min_target,
                                                     int4* __restrict__ piece_tab, int* __restrict__ hcount,
                                                     int* __restrict__ split_rows, int* __restrict__ hneed,
                                                     int* __restrict__ pre) {
  __shared__ u64 s_tot;
  __shared__ int s_S[HEAVY_ROWS];
  const int tid = threadIdx.x, nrows = nrows_dev[0];
  if (tid == 0) s_tot = 0;
  __syncthreads();
  u64 t = 0;
  for (int k = tid; k < nrows; k += blockDim.x) t += work[order[k]];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  if ((tid & 31) == 0 && t) atomicAdd(&s_tot, t);
  __syncthreads();
  // a piece is about half of an SM's fair share of this launch; rows within 3/4 of the fair share stay whole
  u64 target = s_tot / (u64)(2 * sm_count);
  if (target < min_target) target = min_target;
  if (tid < HEAVY_ROWS) {
    int S = 1;
    if (tid < nrows) {
      const u64 w = work[order[tid]];
      if (2 * w > 3 * target && w < (1ull << 32)) {
        const u64 q = (w + target - 1) / target;
        S = q > (u64)HEAVY_SPLITS ? HEAVY_SPLITS : (int)q;
      }
    }
    s_S[tid] = S;
  }
  __syncthreads();
  if (tid == 0) {
    int np = 0, ns = 0;
    for (int r = 0; r < HEAVY_ROWS && r < nrows; ++r) {
      const int S = s_S[r];
      if (S < 2) continue;
      const int i = order[r];
      for (int q = 0; q < S; ++q) piece_tab[np++] = make_int4(i, q, S, ns);
      split_rows[ns] = i;
      hneed[ns] = S;
      pre[i] = ns;
      ++ns;
    }
    hcount[0] = np;
    hcount[1] = ns;
  }
}

// G8: the dense-leg counts are uint8 (at most 255 dense users); a separate instantiation, so that the uint16 kernel
// keeps its code
template <bool PACK16, bool G8>
__global__ void __launch_bounds__(1024, 1) k_fit_rows(FitParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + SEL_BINS);
  unsigned* cnt = reinterpret_cast<unsigned*>(smem + sel_smem_bytes(p.cap));
  __shared__ int s_work;
  __shared__ float s_code_tab[256];
  __shared__ unsigned short s_cm_tab[256];
  __shared__ unsigned short s_cq_tab[256];
  __shared__ int s_ex_idx[HEAVY_CAP], s_ex_cnt[HEAVY_CAP];

  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  const int nrow_items = p.nrows_dev[0] * p.P;
  const int n_pieces = (PACK16 && p.pre) ? p.hcount[0] : 0;
  const int total = n_pieces + nrow_items + ((PACK16 && p.pre) ? p.hcount[1] : 0);
  // coded item popularities for the selection keys: one byte per item behind the counters, loaded once
  if (p.pop_code) {
    unsigned char* code_s = reinterpret_cast<unsigned char*>(cnt) + (size_t)p.R * (PACK16 ? 2 : 4);
    for (int j = tid; j < p.R * p.P; j += nt) code_s[j] = j < p.I ? p.pop_code[j] : (unsigned char)0;
    for (int t = tid; t < 256; t += nt) s_code_tab[t] = exp2f(-(float)t / 12.0f);
    p.sk.code = code_s;
    p.sk.code_tab = s_code_tab;
    __syncthreads();
  }
#ifdef RPK_PHASE_PROF
  long long t_prev = clock64();
#endif
  for (;;) {
    if (tid == 0) s_work = atomicAdd(p.queue, 1);
    __syncthreads();
    const int w = s_work;
    __syncthreads();
    if (w >= total) break;
    FIT_MARK(0);
    if (PACK16 && w < n_pieces) {
      // ---- a piece of a split row: count it, add the counters into the row's global copy
      const int4 pc = p.piece_tab[w];
      const int nw_all = (p.I + 1) >> 1;
      for (int s = tid; s < nw_all; s += nt) cnt[s] = 0u;
      __syncthreads();
      const int64_t pub = p.cscptr[pc.x];
      const int pnu = (int)(p.cscptr[pc.x + 1] - pub);
      const unsigned T = (unsigned)p.work[pc.x];
      const unsigned pieces = (unsigned)pc.z * (unsigned)nwarps;
      unsigned share = (T + pieces - 1) / pieces;
      share = (share + 31u) & ~31u;
      const u64 lo64 = (u64)((unsigned)pc.y * (unsigned)nwarps + (unsigned)warp) * share;
      if (lo64 < T) accumulate_window<PACK16>(p, cnt, pub, pnu, 0, (unsigned)lo64, (unsigned)min((u64)T, lo64 + share));
      __syncthreads();
      unsigned* dst = p.hbuf + (int64_t)pc.w * p.hstride;
      for (int s = tid; s < nw_all; s += nt) {
        const unsigned v = cnt[s];
        if (v) atomicAdd(dst + s, v);
      }
      __threadfence();
      __syncthreads();
      if (tid == 0) atomicAdd(&p.hdone[pc.w], 1);
      continue;
    }
    int pos = 0, i, pass = 0;
    int pre_slot = -1;
    if (w < n_pieces + nrow_items) {
      pos = (w - n_pieces) / p.P;
      pass = (w - n_pieces) % p.P;
      i = p.order[pos];
      if (PACK16 && p.pre && p.pre[i] >= 0) continue;  // a split row: finished at the end of the queue
    } else {
      i = p.split_rows[w - n_pieces - nrow_items];
      pre_slot = p.pre[i];
      if (tid == 0) {  // its pieces were handed out long ago; wait for the last of them
        while (atomicAdd(&p.hdone[pre_slot], 0) < p.hneed[pre_slot]) __nanosleep(256);
      }
      __syncthreads();
    }
    const int r0 = pass * p.R;
    const int ns = min(p.R, p.I - r0);
    const int64_t ub = p.cscptr[i], ue = p.cscptr[i + 1];
    const int64_t orow = p.direct_out ? ((int64_t)i - p.item_begin) : ((int64_t)pos * p.P + pass);
    int* o_idx = p.out_idx + orow * p.K;
    int* o_cnt = p.out_cnt + orow * p.K;
    if (p.sk.n[i] == 0) {  // item never seen: empty row (base.py:257-279 warns about these)
      for (int t = tid; t < p.K; t += nt) {
        o_idx[t] = -1;
        o_cnt[t] = 0;
      }
      if (tid == 0) {
        p.out_len[orow] = 0;
        if (p.defer_max > 0) p.scr_len[orow] = -1;
      }
      continue;
    }
    const int nwords = PACK16 ? (ns + 1) >> 1 : ns;
    if (G8 && p.g16) {
      // start from the 8-bit counts of the dense leg: 8 counts (8 B, r0 is a multiple of 8) become 4 packed 16-bit
      // counter words; counts of columns >= ns (the next row, or padding) are masked off
      const unsigned char* g8 = reinterpret_cast<const unsigned char*>(p.g16);
      const uint2* gv = reinterpret_cast<const uint2*>(g8 + (int64_t)i * p.ldg + r0);
      const int nvec = (ns + 7) >> 3;
      if (PACK16) {
        // the row comes from HBM (59 KB at ML-25M shape): one bulk L2 prefetch puts all of it in flight at once, the
        // loads below then mostly hit L2 (the strip has a spare row at its end, so the rounded-up range stays inside)
        if (tid == 0) {
          const uintptr_t b = reinterpret_cast<uintptr_t>(gv) & ~(uintptr_t)15;
          const uintptr_t e = (reinterpret_cast<uintptr_t>(gv + nvec) + 15) & ~(uintptr_t)15;
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(b), "r"((unsigned)(e - b)) : "memory");
        }
        uint4* c4 = reinterpret_cast<uint4*>(cnt);
        for (int s0 = tid; s0 < nvec; s0 += 2 * nt) {  // two loads in flight per thread
          uint2 v[2];
#pragma unroll
          for (int q = 0; q < 2; ++q) v[q] = s0 + q * nt < nvec ? __ldcs(gv + s0 + q * nt) : make_uint2(0u, 0u);
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const int s = s0 + q * nt;
            if (s >= nvec) break;
            const int left = ns - 8 * s;  // valid counts in this vector
            if (left < 8) {
              v[q].x = left >= 4 ? v[q].x : v[q].x & ((1u << (8 * left)) - 1u);
              v[q].y = left <= 4 ? 0u : v[q].y & ((1u << (8 * (left - 4))) - 1u);
            }
            c4[s] = make_uint4(__byte_perm(v[q].x, 0u, 0x4140), __byte_perm(v[q].x, 0u, 0x4342),
                               __byte_perm(v[q].y, 0u, 0x4140), __byte_perm(v[q].y, 0u, 0x4342));
          }
        }
      } else {
        const unsigned char* grow = g8 + (int64_t)i * p.ldg + r0;
        for (int s = tid; s < nwords; s += nt) cnt[s] = grow[s];
      }
      for (int s = (PACK16 ? 4 * nvec : nwords) + tid; s < (PACK16 ? p.R >> 1 : p.R); s += nt) cnt[s] = 0u;
    } else if (p.g16) {
      // start from the counts of the dense leg (tensor-core Gram over the densest users)
      const unsigned short* grow = p.g16 + (int64_t)i * p.ldg + r0;
      if (PACK16) {
        // two uint16 counts = one packed word: the row is copied as it is, 16 B per cp.async, all copies of a
        // thread in flight at once (the row comes from HBM: 118 KB at ML-25M shape)
        const int nvec = nwords >> 2;
        const uint4* gv = reinterpret_cast<const uint4*>(grow);
        for (int s = tid; s < nvec; s += nt)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(cnt + 4 * s)), "l"(gv + s) : "memory");
        const unsigned* gw = reinterpret_cast<const unsigned*>(grow);
        for (int s = 4 * nvec + tid; s < nwords; s += nt) cnt[s] = gw[s];
        asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        if ((ns & 1) && tid == 0) cnt[nwords - 1] &= 0xffffu;
      } else {
        for (int s = tid; s < nwords; s += nt) cnt[s] = grow[s];
      }
      // the selection passes read whole 16-byte vectors: the tail of the array must be zero
      for (int s = nwords + tid; s < (PACK16 ? p.R >> 1 : p.R); s += nt) cnt[s] = 0u;
    } else {
      uint4* c4 = reinterpret_cast<uint4*>(cnt);
      const int nv = PACK16 ? p.R >> 3 : p.R >> 2;  // R is a multiple of 8
      for (int s = tid; s < nv; s += nt) c4[s] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    FIT_MARK(1);
    if (pre_slot >= 0) {  // the row's users were counted in pieces (P == 1 there): start from their sum
      const unsigned* hb = p.hbuf + (int64_t)pre_slot * p.hstride;
      for (int s = tid; s < nwords; s += nt) cnt[s] += __ldcg(hb + s);
    }
    const int64_t nu64 = ue - ub;
    if (pre_slot >= 0) {
    } else if (!p.usplit) {
      // ---- accumulate, single pass: the row's work (sum of its users' history lengths) is cut into equal
      //      pieces, one per warp, so that a single long history cannot stall the row on one warp
      const int nu = (int)nu64;
      const unsigned T = (unsigned)p.work[i];
      unsigned share = (T + nwarps - 1) / nwarps;
      share = (share + 31u) & ~31u;
      const unsigned lo = (unsigned)warp * share;
      const unsigned hi = min(T, lo + share);
      if (lo < hi) {
        accumulate_window<PACK16>(p, cnt, ub, nu, r0, lo, hi);
      }
    } else {
      // ---- accumulate, several item ranges: users are dealt to the warps in chunks (<= 32 users, one per
      //      lane, so that their row pointers are fetched in parallel)
      int chunk = (int)((nu64 + nwarps - 1) / nwarps);
      chunk = chunk < 1 ? 1 : (chunk > 32 ? 32 : chunk);
      for (int64_t base = ub + (int64_t)warp * chunk; base < ue; base += (int64_t)nwarps * chunk) {
        const int nvalid = (int)min((int64_t)chunk, ue - base);
        int64_t beg = 0;
        int len = 0;
        if (lane < nvalid) {
          const int u = p.csc_users[base + lane];
          const int64_t* us = p.usplit + (int64_t)u * (p.P + 1) + pass;
          beg = us[0];
          len = (int)(us[1] - beg);
        }
        for (int l = 0; l < nvalid; ++l) {
          const int64_t b = __shfl_sync(0xffffffffu, beg, l);
          const int n = __shfl_sync(0xffffffffu, len, l);
          for (int e = lane; e < n; e += 32) {
            const int j = p.indices[b + e] - r0;
            if (PACK16) atomicAdd(&cnt[j >> 1], 1u << ((j & 1) * 16));
            else atomicAdd(&cnt[j], 1u);
          }
        }
      }
    }
    __syncthreads();
    FIT_MARK(2);
    // ---- fused epilogue: similarity ordering, diagonal removal, top-K -- all on the shared-memory row
    // columns of a heavy row that are heavy themselves: their 16-bit counters may have wrapped -- zero them and
    // use the exact pair counts instead
    int nex = 0;
    if (PACK16 && p.heavy_ids && p.sk.n[i] >= 65536) {
      const int H = min(p.heavy_n[0], HEAVY_CAP);  // (more than HEAVY_CAP heavy items: those rows take the 32-bit launch)
      if (tid < H) {
        const int j = p.heavy_ids[tid];
        s_ex_idx[tid] = j;
        int me = 0;
        for (int h = 0; h < H; ++h) me = p.heavy_ids[h] == i ? h : me;
        const int sl = j - r0;
        const bool mine = sl >= 0 && sl < ns;  // a column belongs to exactly one item range
        const int exact = j != i ? p.heavy_pair[me * HEAVY_CAP + tid] : p.sk.n[i];  // what the counter summed to
        s_ex_cnt[tid] = (mine && j != i) ? exact : 0;
        // a low half that passed 65535 carried into its neighbour's half (exact >> 16 times): take that back,
        // unless the neighbour is a heavy column itself (its half is discarded below)
        if (mine && !(sl & 1) && sl + 1 < ns && (exact >> 16)) {
          bool nb_heavy = false;
          for (int h = 0; h < H; ++h) nb_heavy |= p.heavy_ids[h] == j + 1;
          if (!nb_heavy) atomicSub(&cnt[sl >> 1], (unsigned)(exact >> 16) << 16);
        }
      }
      __syncthreads();
      if (tid < H) {
        const int sl = p.heavy_ids[tid] - r0;
        if (sl >= 0 && sl < ns) atomicAnd(&cnt[sl >> 1], (sl & 1) ? 0x0000ffffu : 0xffff0000u);
      }
      nex = H;
      __syncthreads();
    }
    // the diagonal never survives (nearest_neighbour.py:64,81 + util.py:96): drop it here, once, instead of testing
    // every slot for it in the selection passes
    if (tid == 0) {
      const int sl = i - r0;
      if (sl >= 0 && sl < ns) {
        if (PACK16) cnt[sl >> 1] &= (sl & 1) ? 0x0000ffffu : 0xffff0000u;
        else cnt[sl] = 0u;
      }
    }
    __syncthreads();
    // upper bound of the row's candidates: every slot when dense counts were loaded, else one per counter update
    int cbound = ns + nex;
    if (!p.g16 && pre_slot < 0) cbound = (int)min((u64)cbound, p.work[i]);
    RowCountSrc<PACK16> src{p.sk, cnt, r0, ns, i, s_ex_idx, s_ex_cnt, nex, 1, (PACK16 && p.sk.code) ? s_cm_tab : nullptr, (PACK16 && p.sk.code) ? s_cq_tab : nullptr, cbound,
                            reinterpret_cast<const unsigned char*>(cnt) + (size_t)p.R * (PACK16 ? 2 : 4), s_code_tab, 0ull, p.R >> 3};
    bool sorted = true;
    FIT_MARK(3);
    const int m = block_select_topk(src, p.K, list, p.cap, p.direct_cap, hist, sh, p.defer_max, &sorted);
    FIT_MARK(4);
#ifdef RPK_PHASE_PROF
    if (tid == 0 && p.prof) {
      atomicAdd(p.prof + 8, 1ull);
      atomicAdd(p.prof + 9, (unsigned long long)m);
    }
#endif
    if (!sorted) {
      // hand the unsorted survivors to k_fit_sort_rows: many small CTAs sort rows concurrently there,
      // instead of this 1024-thread CTA idling through the sort's barriers
      int* s_idx = p.scr_idx + orow * p.defer_max;
      int* s_cnt = p.scr_cnt + orow * p.defer_max;
      for (int t = tid; t < m; t += nt) {
        s_idx[t] = list[t].idx;
        s_cnt[t] = list[t].aux;
      }
      if (tid == 0) p.scr_len[orow] = m;
#ifdef RPK_PHASE_PROF
      if (tid == 0) atomicAdd(&g_fit_ev[FIT_EV_DEFERRED], 1ull);
#endif
      __syncthreads();
      FIT_MARK(5);
      continue;
    }
    if (p.defer_max > 0 && tid == 0) p.scr_len[orow] = -1;
    for (int t = tid; t < p.K; t += nt) {
      o_idx[t] = t < m ? list[t].idx : -1;
      o_cnt[t] = t < m ? list[t].aux : 0;
    }
    if (tid == 0) p.out_len[orow] = m;
    __syncthreads();
  }
}

// Merge the P per-range lists of the rows that needed several passes.
struct MergeParams {
  SimKey sk;
  const int* part_idx;
  const int* part_cnt;
  const int* order;
  const int* nrows_dev;
  int64_t item_begin;
  int P, K, cap, direct_cap;
  int* out_idx;
  int* out_cnt;
  int* out_len;
};
__global__ void __launch_bounds__(256) k_fit_merge(MergeParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + SEL_BINS);
  const int tid = threadIdx.x, nt = blockDim.x;
  const int nrows = p.nrows_dev[0];
  for (int pos = blockIdx.x; pos < nrows; pos += gridDim.x) {
    const int64_t row = (int64_t)p.order[pos] - p.item_begin;
    PairListSrc src{p.sk, p.part_idx + (int64_t)pos * p.P * p.K, p.part_cnt + (int64_t)pos * p.P * p.K, p.P * p.K};
    const int m = block_select_topk(src, p.K, list, p.cap, p.direct_cap, hist, sh);
    for (int t = tid; t < p.K; t += nt) {
      p.out_idx[row * p.K + t] = t < m ? list[t].idx : -1;
      p.out_cnt[row * p.K + t] = t < m ? list[t].aux : 0;
    }
    if (tid == 0) p.out_len[row] = m;
#ifdef RPK_PHASE_PROF
    if (tid == 0) atomicAdd(&g_fit_ev[FIT_EV_MERGED], 1ull);
#endif
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// Finishing kernel: exact top K of the deferred survivors, and the similarity values of every row
// ------------------------------------------------------------------------------------------
// c-fold left sum ((x + x) + x) + ... in float64, round to nearest even: scipy's csr_matmat adds the c identical
// products of a cosine entry one at a time.  Inside one binade of the running sum s (fixed exponent, ulp u) every
// step from a multiple of u adds the same multiple d of u -- x rounded to u -- while the result stays in the binade.
// When x / u is a half-integer the tie goes to the even neighbour, so a step that starts inside the binade always
// lands on an even multiple of u; from there every step adds the same even d.  A step that enters the binade may land
// on an odd multiple, so the increment is read off two real steps after it, and the steps that stay below the binade's
// top are taken at once.  Inside a binade the bit patterns are consecutive multiples of u, so this is integer
// arithmetic on them.  About three real additions per binade: at most ~50 for c < 2^17.
__device__ __forceinline__ double repeat_sum(double x, int c) {
  double s = 0.0;
  int r = 0;
  while (r < c) {
    const double s0 = s;
    s = __dadd_rn(s, x);
    ++r;
    const long long b = __double_as_longlong(s);
    if (r == c || s0 == 0.0 || (__double_as_longlong(s0) >> 52) != (b >> 52)) continue;
    // s was reached by a step inside its binade
    const double s1 = __dadd_rn(s, x);
    ++r;
    const long long b1 = __double_as_longlong(s1);
    s = s1;
    if (r == c || (b1 >> 52) != (b >> 52)) continue;
    const long long d = b1 - b;                             // ulps per step until the binade ends
    const long long room = (((b >> 52) + 1) << 52) - 1 - b1;  // ulps from s1 to the binade's largest value
    long long t = c - r;
    if (d > 0) {
      // room, d < 2^53: the rounded quotient never reaches the next integer above the exact one
      const long long q = (long long)((double)room / (double)d);
      if (q < t) t = q;
    }
    s = __longlong_as_double(b1 + t * d);
    r += (int)t;
  }
  return s;
}

// Similarity values in the reference's floating-point operation order (include/rpk.h).  Row factor of item i: cosine
// a_i = 1/sqrt(n_i) -- sklearn row-normalises X^T (sparsefuncs_fast.pyx:578-604); conditional probability 1/n_i
// (algorithms/util.py:132).
__device__ __forceinline__ double row_factor(int mode, int n_i) {
  return mode == 0 ? __ddiv_rn(1.0, __dsqrt_rn((double)n_i)) : __ddiv_rn(1.0, (double)n_i);
}
// Value of entry (i, j) with count c, f_i = row_factor(i).
__device__ __forceinline__ double sim_value(int mode, double f_i, int n_j, int c, const double* pw, int j) {
  if (mode == 0) {
    // scipy's csr_matmat adds the c identical products fl(a_i a_j) one at a time
    const double aj = __ddiv_rn(1.0, __dsqrt_rn((double)n_j));
    return repeat_sum(__dmul_rn(f_i, aj), c);
  }
  double v = __dmul_rn(f_i, (double)c);    // A @ co_mat
  if (mode == 2) v = __dmul_rn(v, pw[j]);  // ... @ A.power(pop_discount)
  return v;
}

#ifdef RPK_PHASE_PROF
// rows sorted, rows given values only, comparisons settled exactly, then cycles of the first thread of a group in the
// phases of a sorted row: load + keys, select, compaction, sort, output + values
__device__ unsigned long long g_fit_sort[8];
#define SORT_MARK(k)                           \
  do {                                         \
    if (g == 0) {                              \
      const long long t_now = clock64();       \
      cyc[k] += (unsigned long long)(t_now - t_prev); \
      t_prev = t_now;                          \
    }                                          \
  } while (0)
#else
#define SORT_MARK(k) do {} while (0)
#endif

struct SortParams {
  const int* n;
  const double* pw;
  const int* scr_idx;
  const int* scr_cnt;
  const int* scr_len;
  int* queue;  // next row to take (zeroed before the launch)
  int defer_max, K, mode;
  int64_t nrows, item_begin;
  u64 key_mask;  // ~0, or the low 40 bits cleared (DBG_COARSE_SORT_KEY)
  u64 margin;    // two sort keys further apart than this many bit patterns are in exact order
  int* out_idx;
  int* out_cnt;
  int* out_len;
  double* out_val;  // null: no values asked for
};

constexpr int SORT_BINS = 256;  // radix of the threshold select
struct SortGroupShared {
  u64 w64[16];  // per-warp minima / maxima (256-thread groups)
  int wsum[8];  // per-warp sums
  u64 lo;       // the select's next bin
  int above, n_in;
  int row;
};
// per group: keys and (index, count) pairs of up to defer_max entries, the histogram, the scratch above
__host__ __device__ __forceinline__ size_t sort_group_bytes(int defer_max) {
  return (size_t)defer_max * 16 + SORT_BINS * 4 + (sizeof(SortGroupShared) + 15) / 16 * 16;
}

// The order of the deferred survivors.  Sort key: cosine fl((double)fl(c^2) / n_j) -- correctly rounded from exact
// operands while c^2 < 2^53, so it never inverts two exact values there; for c up to 2^31 each of the two roundings
// moves the key by at most 2^-53 relative, so two keys in the wrong order are at most 4 bit patterns apart (M = 4).
// Conditional probability: the float64 key is the definition (M = 0).  Keys further apart than M decide; otherwise
// the exact comparison (SimKey::cmp3), then the ascending index -- the canonical total order of the oracle.
// The exact comparison takes n_j from the key itself: fl(fl(c^2) / k) is n_j within n_j 2^-51 < 2^-20 for
// n_j, c < 2^31, so rounding it gives n_j exactly, without a global load in the sort.
struct SortOrder {
  u64 mask, M;
  int mode;
  __device__ __forceinline__ static u64 pop_of(u64 k, int c) {
    if (c == 0) return 1ull;  // padding
    return (u64)__double2ll_rn(__ddiv_rn((double)((u64)c * (u64)c), __longlong_as_double((long long)k)));
  }
  __device__ __forceinline__ int exact(u64 ka, int ca, u64 kb, int cb) const {
    if (mode != 0) return ka == kb ? 0 : (ka > kb ? 1 : -1);
    // c_a^2 / n_a  vs  c_b^2 / n_b   <=>   c_a^2 * n_b  vs  c_b^2 * n_a   (128-bit exact); padding: c = 0
    const u64 na = pop_of(ka, ca), nb = pop_of(kb, cb);
    const u64 ca2 = (u64)(unsigned)ca * (u64)(unsigned)ca, cb2 = (u64)(unsigned)cb * (u64)(unsigned)cb;
    const u64 l_lo = ca2 * nb, l_hi = __umul64hi(ca2, nb);
    const u64 r_lo = cb2 * na, r_hi = __umul64hi(cb2, na);
    if (l_hi != r_hi) return l_hi > r_hi ? 1 : -1;
    if (l_lo != r_lo) return l_lo > r_lo ? 1 : -1;
    return 0;
  }
  // true when a precedes b; keys are positive doubles (< 2^63 as patterns), so k + M does not wrap
  __device__ __forceinline__ bool before(u64 ka, int ia, int ca, u64 kb, int ib, int cb, unsigned& n_exact) const {
    const u64 a = ka & mask, b = kb & mask;
    if (a > b + M) return true;
    if (b > a + M) return false;
    ++n_exact;
    // the same key from the same count: the same n_j (cosine), the same value; padding against padding too
    if (ka == kb && ca == cb) return ia < ib;
    const int c3 = exact(ka, ca, kb, cb);
    return c3 != 0 ? c3 > 0 : ia < ib;
  }
};

// Group of GW threads: one warp, or a whole 256-thread block for the largest K.
template <int GW>
__device__ __forceinline__ void group_sync() {
  if (GW == 32) __syncwarp();
  else __syncthreads();
}
// Inclusive prefix sum over the group in thread order; *total = the group's sum.  wsum: GW / 32 ints of shared memory.
template <int GW>
__device__ __forceinline__ int group_scan(int v, int* wsum, int* total) {
  const int lane = threadIdx.x & 31;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (GW == 32) {
    *total = __shfl_sync(0xffffffffu, incl, 31);
    return incl;
  }
  const int w = (threadIdx.x % GW) >> 5;
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  int before = 0, tot = 0;
#pragma unroll
  for (int q = 0; q < GW / 32; ++q) {
    const int s = wsum[q];
    before += q < w ? s : 0;
    tot += s;
  }
  __syncthreads();
  *total = tot;
  return incl + before;
}
template <int GW>
__device__ __forceinline__ void group_min_max(u64& lo, u64& hi, u64* w64) {
  lo = warp_min_u64(lo);
  hi = warp_max_u64(hi);
  if (GW == 32) return;
  const int w = (threadIdx.x % GW) >> 5;
  if ((threadIdx.x & 31) == 0) {
    w64[w] = lo;
    w64[GW / 32 + w] = hi;
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < GW / 32; ++q) {
    lo = w64[q] < lo ? w64[q] : lo;
    hi = w64[GW / 32 + q] > hi ? w64[GW / 32 + q] : hi;
  }
  __syncthreads();
}

// One group per row, rows taken from a counter.  A deferred row (scr_len >= 0: its survivors, unsorted, written by
// k_fit_rows): keys into shared memory, a radix select of the K-th largest key tau, every survivor with key >= tau - M
// kept (one below is beaten by at least K others), a bitonic sort of those with the exact order, the first K written
// with their values.  A row already final (scr_len = -1): its values only.  GW = 32 for defer_max <= 1024 (K <= 512),
// 256 above.
template <int GW>
__global__ void __launch_bounds__(GW == 32 ? 64 : 256) k_fit_sort_rows(SortParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int D = p.defer_max, K = p.K;
  const int g = threadIdx.x % GW;
  unsigned char* base = smem + (size_t)(threadIdx.x / GW) * sort_group_bytes(D);
  u64* skey = reinterpret_cast<u64*>(base);
  int2* sic = reinterpret_cast<int2*>(skey + D);  // (index, count)
  int* hist = reinterpret_cast<int*>(sic + D);
  SortGroupShared* gs = reinterpret_cast<SortGroupShared*>(hist + SORT_BINS);
  const SortOrder ord{p.key_mask, p.margin, p.mode};
  unsigned n_exact = 0;
#ifdef RPK_PHASE_PROF
  unsigned long long n_sorted = 0, n_values = 0, cyc[5] = {0, 0, 0, 0, 0};
  long long t_prev = 0;
#endif
  for (;;) {
    if (g == 0) gs->row = atomicAdd(p.queue, 1);
    group_sync<GW>();
    const int64_t row = gs->row;
    group_sync<GW>();
    if (row >= p.nrows) break;
    const int m = p.scr_len[row];
    const int i = (int)(p.item_begin + row);
    const double f_i = row_factor(p.mode, p.n[i]);
    int* o_idx = p.out_idx + row * K;
    int* o_cnt = p.out_cnt + row * K;
    double* o_val = p.out_val ? p.out_val + row * K : nullptr;
    if (m < 0) {  // sorted by k_fit_rows or merged by k_fit_merge
      if (!o_val) continue;
      for (int t = g; t < K; t += GW) {
        const int j = o_idx[t];
        o_val[t] = j >= 0 ? sim_value(p.mode, f_i, p.n[j], o_cnt[t], p.pw, j) : 0.0;
      }
#ifdef RPK_PHASE_PROF
      n_values++;
#endif
      continue;
    }
#ifdef RPK_PHASE_PROF
    n_sorted++;
    if (g == 0) t_prev = clock64();
#endif
    const int* r_idx = p.scr_idx + row * D;
    const int* r_cnt = p.scr_cnt + row * D;
#pragma unroll 4
    for (int t = g; t < m; t += GW) sic[t] = make_int2(r_idx[t], r_cnt[t]);
    group_sync<GW>();
    u64 kmin = ~0ull, kmax = 0ull;
#pragma unroll 4
    for (int t = g; t < m; t += GW) {
      const int2 e = sic[t];
      u64 k;
      if (p.mode == 0) k = (u64)__double_as_longlong(__ddiv_rn((double)((u64)e.y * (u64)e.y), (double)p.n[e.x]));
      else if (p.mode == 1) k = (u64)__double_as_longlong((double)e.y);
      else k = (u64)__double_as_longlong(__dmul_rn((double)e.y, p.pw[e.x]));
      skey[t] = k;
      const u64 km = k & p.key_mask;
      kmin = km < kmin ? km : kmin;
      kmax = km > kmax ? km : kmax;
    }
    SORT_MARK(0);
    int kept = m;
    if (m > K) {
      // ---- radix select: narrow [lo, hi] to the bin of the K-th largest key until at most `room` keys lie at or
      //      above lo (or the bin is one key); g_above = keys above hi, n_in = keys in [lo, hi]
      group_min_max<GW>(kmin, kmax, gs->w64);
      int room = 1;
      while (room < K + K / 16 + 1) room <<= 1;
      u64 lo = kmin, hi = kmax;
      int g_above = 0, n_in = m;
      while (g_above + n_in > room && lo < hi) {
        int shift, nb;
        bin_geometry<8>(lo, hi, shift, nb);
        for (int b = g; b < nb; b += GW) hist[b] = 0;
        group_sync<GW>();
        for (int t = g; t < m; t += GW) {
          const u64 k = skey[t] & p.key_mask;
          if (k >= lo && k <= hi) atomicAdd(&hist[(int)((k - lo) >> shift)], 1);
        }
        group_sync<GW>();
        // the bin holding the K-th largest key, scanning from the top: thread g owns bins [b0, b1)
        const int per = (nb + GW - 1) / GW;
        const int b0 = min(nb, g * per), b1 = min(nb, b0 + per);
        int tsum = 0;
        for (int b = b0; b < b1; ++b) tsum += hist[b];
        int total;
        const int incl = group_scan<GW>(tsum, gs->wsum, &total);
        int above = g_above + total - incl;  // keys in bins of higher threads
        if (above < K && above + tsum >= K) {
          for (int b = b1 - 1; b >= b0; --b) {
            if (above + hist[b] >= K) {
              gs->lo = lo + ((u64)b << shift);
              gs->above = above;
              gs->n_in = hist[b];
              break;
            }
            above += hist[b];
          }
        }
        group_sync<GW>();
        const u64 nlo = gs->lo;
        g_above = gs->above;
        n_in = gs->n_in;
        group_sync<GW>();
        u64 nhi = nlo + ((1ull << shift) - 1);
        if (nhi > hi || nhi < nlo) nhi = hi;
        lo = nlo;
        hi = nhi;
      }
      const u64 thr = lo > p.margin ? lo - p.margin : 0ull;
      SORT_MARK(1);
      // ---- keep the survivors with key >= thr: stable compaction in place (a kept entry moves to a lower or its own
      //      position; each round reads its GW entries before any of them is overwritten)
      kept = 0;
      for (int r0 = 0; r0 < m; r0 += GW) {
        const int t = r0 + g;
        u64 k = 0;
        int2 e = make_int2(0, 0);
        bool keep = false;
        if (t < m) {
          k = skey[t];
          e = sic[t];
          keep = (k & p.key_mask) >= thr;
        }
        int total, pos;
        if (GW == 32) {
          const unsigned ball = __ballot_sync(0xffffffffu, keep);
          total = __popc(ball);
          pos = kept + __popc(ball & ((1u << g) - 1u));
        } else {
          pos = kept + group_scan<GW>(keep ? 1 : 0, gs->wsum, &total) - 1;
        }
        group_sync<GW>();
        if (keep) {
          skey[pos] = k;
          sic[pos] = e;
        }
        kept += total;
        group_sync<GW>();
      }
      SORT_MARK(2);
    }
    // ---- bitonic sort of the kept entries, best first; padding (key 0, count 0, index SENTINEL_IDX) sorts last
    int n2 = 1;
    while (n2 < kept) n2 <<= 1;
    for (int t = kept + g; t < n2; t += GW) {
      skey[t] = 0ull;
      sic[t] = make_int2(SENTINEL_IDX, 0);
    }
    group_sync<GW>();
    for (int k2 = 2; k2 <= n2; k2 <<= 1) {
      for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
#pragma unroll 4
        for (int q = g; q < (n2 >> 1); q += GW) {
          const int a = ((q & ~(j2 - 1)) << 1) | (q & (j2 - 1)), b = a + j2;
          const u64 ka = skey[a], kb = skey[b];
          const int2 ea = sic[a], eb = sic[b];
          const bool up = (a & k2) == 0;
          if (ord.before(kb, eb.x, eb.y, ka, ea.x, ea.y, n_exact) == up) {
            skey[a] = kb;
            skey[b] = ka;
            sic[a] = eb;
            sic[b] = ea;
          }
        }
        group_sync<GW>();
      }
    }
    SORT_MARK(3);
    const int keep = kept < K ? kept : K;
    // four entries per thread at a time, so that their popularity loads overlap
    for (int t0 = g; t0 < K; t0 += 4 * GW) {
      int2 e[4];
      int nj[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = t0 + u * GW;
        e[u] = t < keep ? sic[t] : make_int2(-1, 0);
        nj[u] = e[u].x >= 0 ? p.n[e[u].x] : 1;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = t0 + u * GW;
        if (t < K) {
          o_idx[t] = e[u].x;
          o_cnt[t] = e[u].y;
          if (o_val) o_val[t] = e[u].x >= 0 ? sim_value(p.mode, f_i, nj[u], e[u].y, p.pw, e[u].x) : 0.0;
        }
      }
    }
    if (g == 0) p.out_len[row] = keep;
    group_sync<GW>();
    SORT_MARK(4);
  }
#ifdef RPK_PHASE_PROF
  if (g == 0) {
    atomicAdd(&g_fit_sort[0], n_sorted);
    atomicAdd(&g_fit_sort[1], n_values);
    for (int k = 0; k < 5; ++k) atomicAdd(&g_fit_sort[3 + k], cyc[k]);
  }
  atomicAdd(&g_fit_sort[2], (unsigned long long)n_exact);
#else
  (void)n_exact;
#endif
}

// Stable split of the heaviest-first row order into rows whose counts fit 16 bits and the rest (one block).
__global__ void __launch_bounds__(1024) k_split_rows(const int* __restrict__ order, int nrows, const int* __restrict__ n,
                                                     int limit_in, const int* __restrict__ heavy_n, int* __restrict__ light,
                                                     int* __restrict__ heavy, int* __restrict__ counts) {
  // when the heavy items are few enough to be handled as exact "extra" columns, every row stays on the
  // 16-bit path; otherwise rows with >= limit users take the 32-bit path
  const int limit = (limit_in > 0 && heavy_n && heavy_n[0] <= HEAVY_CAP) ? 0x7fffffff : limit_in;
  __shared__ int wl[32], wh[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  int nl = 0, nh = 0;
  for (int base = 0; base < nrows; base += blockDim.x) {
    const int k = base + tid;
    const int row = k < nrows ? order[k] : -1;
    const bool is_l = row >= 0 && n[row] < limit;
    const bool is_h = row >= 0 && !is_l;
    const unsigned ml = __ballot_sync(0xffffffffu, is_l), mh = __ballot_sync(0xffffffffu, is_h);
    if (lane == 0) {
      wl[warp] = __popc(ml);
      wh[warp] = __popc(mh);
    }
    __syncthreads();
    int ol = 0, oh = 0, tl = 0, th = 0;
    for (int q = 0; q < nw; ++q) {
      if (q < warp) {
        ol += wl[q];
        oh += wh[q];
      }
      tl += wl[q];
      th += wh[q];
    }
    if (is_l) light[nl + ol + __popc(ml & ((1u << lane) - 1u))] = row;
    if (is_h) heavy[nh + oh + __popc(mh & ((1u << lane) - 1u))] = row;
    nl += tl;
    nh += th;
    __syncthreads();
  }
  if (tid == 0) {
    counts[0] = nl;
    counts[1] = nh;
  }
}

// ------------------------------------------------------------------------------------------
// Host driver
// ------------------------------------------------------------------------------------------
static int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// One contiguous block of item rows [item_begin, item_end).  `strip` > 0: a later strip of the same fit
// (run_fit cuts a large row range into strips so that only one strip of the dense-leg counts exists at a time):
// item counts, the dense/sparse split, the dense slots and the dense operand of strip 0 are reused.
// `rows_total` is the row count of the whole fit (the split is chosen for all of it).
static void fit_range(rpk_ctx* c, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
                      int similarity, const double* item_pow_u, int K, int64_t item_begin, int64_t item_end,
                      int32_t* out_idx_u, int32_t* out_cnt_u, double* out_val_u, int32_t* out_len_u, int strip,
                      int64_t rows_total) {
  RPK_REQUIRE(U >= 0 && I >= 0 && nnz >= 0, "negative dimension");
  RPK_REQUIRE(I < (int64_t)1 << 24, "more than 2^24 items are not supported");
  RPK_REQUIRE(U < (int64_t)1 << 31, "more than 2^31 users are not supported");
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(0 <= item_begin && item_begin <= item_end && item_end <= I, "bad item range");
  RPK_REQUIRE(similarity == RPK_SIM_COSINE || similarity == RPK_SIM_CONDPROB, "unknown similarity");
  RPK_REQUIRE(out_idx_u && out_len_u, "out_idx / out_len must not be null");
  cudaStream_t st = c->stream;
  const int64_t nrows = item_end - item_begin;
  const int mode = similarity == RPK_SIM_COSINE ? 0 : (item_pow_u ? 2 : 1);

  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "fit_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "fit_indices");
  const double* pw = item_pow_u ? stage_in(c, item_pow_u, (size_t)I, "fit_pw") : nullptr;

  // ---- preparation
  c->mark("fit: begin");
  int* n = c->buf<int>("fit_n", (size_t)I);
  int* cursor = c->buf<int>("fit_cursor", (size_t)I);
  u64* work = c->buf<u64>("fit_work", (size_t)I);
  int64_t* cscptr = c->buf<int64_t>("fit_cscptr", (size_t)I + 1);
  int* csc_users = c->buf<int>("fit_csc_users", (size_t)nnz);
  float* rnf = c->buf<float>("fit_rnf", (size_t)I);
  int* order = c->buf<int>("fit_order", (size_t)nrows);
  int* bcnt = c->buf<int>("fit_bcnt", 65 * 2 + 2);
  int* boff = bcnt + 65;
  (void)boff;
  c->fit_I = I;
  // ---- hybrid split (SURVEY.md 7, step 5): the users with the longest histories carry most of the
  //      sum of d_u^2; their Gram goes to the tensor cores, everybody else to the sparse kernel
  int hmax = c->dense_users;
  const int64_t rows_pad = (I + 255) / 256 * 256;
  const bool dense_auto = hmax < 0;
  if (dense_auto) hmax = (I >= 4096 && U >= 8192) ? 4096 : 0;
  if (hmax > U) hmax = (int)U;
  if (nnz == 0 || I < 2 || nrows == 0) hmax = 0;
  int dense_tau = 32;  // histories shorter than this are never worth a dense column
  int* lhist = nullptr;
  const bool decide = strip == 0 && hmax > 0;
  if (decide) {
    // the history-length histogram goes to the host first (pinned buffer, asynchronous copy); the item counts below
    // run while the host waits for it
    lhist = c->buf<int>("fit_len_hist", (size_t)I + 2);
    RPK_CUDA(cudaMemsetAsync(lhist, 0, sizeof(int) * ((size_t)I + 2), st));
    k_len_hist<<<ceil_div(U, 256), 256, 0, st>>>(indptr, U, I, lhist);
    RPK_LAUNCH_CHECK(c);
    RPK_CUDA(cudaMemcpyAsync(c->pinned_ints((size_t)I + 1), lhist, sizeof(int) * ((size_t)I + 1), cudaMemcpyDeviceToHost, st));
    if (!c->hist_ev) RPK_CUDA(cudaEventCreateWithFlags(&c->hist_ev, cudaEventDisableTiming));
    RPK_CUDA(cudaEventRecord(c->hist_ev, st));
  }
  if (strip == 0) RPK_CUDA(cudaMemsetAsync(n, 0, sizeof(int) * (size_t)I, st));
  RPK_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * (size_t)I, st));
  RPK_CUDA(cudaMemsetAsync(work, 0, sizeof(u64) * (size_t)I, st));
  RPK_CUDA(cudaMemsetAsync(bcnt, 0, sizeof(int) * (65 * 2 + 2), st));
  if (nnz > 0 && strip == 0) {
    int blocks = (int)std::min<int64_t>((nnz + 255) / 256, (int64_t)c->sm_count * 16);
    k_item_counts<<<blocks, 256, 0, st>>>(indices, nnz, n);
    RPK_LAUNCH_CHECK(c);
  }
  if (strip > 0) {
    hmax = c->strip_hmax;
    dense_tau = c->strip_tau;
  } else if (decide) {
    // The split is chosen per density on the host from the history-length histogram (one small copy):
    // moving the H longest histories to the tensor cores costs 2*H*rows*I int8 ops (+ the count matrix
    // traffic) and saves sum(d_u^2) * rows/I counter updates of the sparse kernel.
    RPK_CUDA(cudaEventSynchronize(c->hist_ev));
    const int* h = c->pinned_ints((size_t)I + 1);
    const double share = (double)rows_total / (double)I;
    // rates measured on B200 (profiles/r2_summary.md): the sparse kernel does 6-7e11 counter updates/s when the packed
    // counters of a row fit one pass, 1.8e11/s when the catalogue needs several item-range passes (I = 200,000: 3)
    const bool one_pass = (size_t)I * 2 + 49152 <= (size_t)c->smem_max;
    // The count strip costs its store: measured on B200 at ML-25M shape, Kd = 256 (profiles/r9_bench_before_after.txt),
    // the Gram writes the 7.0 GB uint16 strip at 2.3 TB/s (16 B per lane from registers) and the 3.5 GB uint8 strip at
    // 4.3 TB/s (TMA tensor stores).  Halving the bytes the row kernel reads back changed its time by 0.2 %, so the
    // read-back is not charged.  uint8 needs at most 255 dense users: the model weighs that against its best choice
    // at 16 bits.
    const double dense_rate = 1.6e15, sparse_rate = one_pass ? 7e11 : 1.8e11, store_u16 = 2.3e12, store_u8 = 4.3e12;
    double best_gain = 0.0, saved = 0.0;
    int best_h = 0, best_tau = 0;
    int64_t taken = 0;
    for (int64_t d = I; d >= dense_tau; --d) {
      const int cnt_d = h[(size_t)d];
      if (cnt_d == 0) continue;
      if (taken + cnt_d > hmax) break;
      taken += cnt_d;
      saved += (double)cnt_d * (double)d * (double)d * share / sparse_rate;
      const double kd = (double)((taken + 127) / 128 * 128);
      const double pairs = (double)rows_total * (double)rows_pad;
      const double strip = taken <= 255 ? pairs / store_u8 : 2.0 * pairs / store_u16;
      const double cost = 2.0 * kd * pairs / dense_rate + strip;
      const double gain = saved - cost;
      if (!dense_auto || gain > best_gain) {  // a fixed request takes as many users as allowed
        best_gain = gain;
        best_h = (int)taken;
        best_tau = (int)d;
      }
    }
    hmax = best_h;
    dense_tau = best_tau;
  }
  c->strip_hmax = hmax;
  c->strip_tau = dense_tau;
  c->mark("fit: item counts + split");
  const int* dense_slot = nullptr;
  const unsigned short* g16 = nullptr;
  const unsigned char* g8 = nullptr;
  const int* n_sparse = n;  // per-item user counts on the sparse path
  c->last_dense_users = hmax;
  c->last_dense_kd = hmax > 0 ? (int)(((int64_t)hmax + 127) / 128 * 128) : 0;
  if (hmax > 0) {
    const int64_t kd_pad = ((int64_t)hmax + 127) / 128 * 128;
    int* thr_cnt = c->buf<int>("fit_dense_thr", 4);
    int* slot = c->buf<int>("fit_dense_slot", (size_t)U);
    int* n_light = c->buf<int>("fit_n_light", (size_t)I);
    unsigned char* A = c->buf<unsigned char>("fit_dense_A", (size_t)rows_pad * kd_pad);
    // only this shard's item rows of the dense Gram are needed (row block aligned down to the 128-row tile)
    const int64_t g_row0 = item_begin / 128 * 128;
    // at most 255 dense users: every count fits 8 bits, and the strip is written and read at half the bytes
    const bool counts8 = hmax <= 255;
    unsigned char* G = c->buf<unsigned char>("fit_dense_G", (size_t)(item_end - g_row0 + 1) * rows_pad * (counts8 ? 1 : 2));
    if (strip == 0) {
      const int thr_init[2] = {dense_tau, 0};
      RPK_CUDA(cudaMemcpyAsync(thr_cnt, thr_init, sizeof(thr_init), cudaMemcpyHostToDevice, st));
      RPK_CUDA(cudaMemcpyAsync(n_light, n, sizeof(int) * (size_t)I, cudaMemcpyDeviceToDevice, st));
      RPK_CUDA(cudaMemsetAsync(A, 0, (size_t)rows_pad * kd_pad, st));
      int* dense_user = c->buf<int>("fit_dense_user", (size_t)hmax);
      k_assign_dense_slots<<<ceil_div(U, 256), 256, 0, st>>>(indptr, U, thr_cnt, hmax, slot, dense_user);
      RPK_LAUNCH_CHECK(c);
      k_fill_dense_users<<<hmax, 256, 0, st>>>(indptr, indices, dense_user, thr_cnt, kd_pad, A, n_light);
      RPK_LAUNCH_CHECK(c);
      c->mark("fit: dense operand");
    }
    c->span_begin(0);
    if (counts8) {
      run_gram_dense_tc(c, A, rows_pad, kd_pad, g_row0, item_end, G, rows_pad);
      g8 = G - g_row0 * rows_pad;  // indexed by absolute item row in the fit kernel
    } else {
      unsigned short* G16 = reinterpret_cast<unsigned short*>(G);
      run_gram_dense_tc(c, A, rows_pad, kd_pad, g_row0, item_end, G16, rows_pad);
      g16 = G16 - g_row0 * rows_pad;
    }
    c->span_end(0);
    c->mark("fit: tensor-core Gram");
    dense_slot = slot;
    n_sparse = n_light;
  }
  scan_i32_i64(c, n_sparse, cscptr, I);
  if (nnz > 0 && U > 0) {
    int blocks = (int)std::min<int64_t>((U * 32 + 255) / 256, (int64_t)c->sm_count * 16);
    k_fill_csc<<<blocks, 256, 0, st>>>(indptr, indices, U, dense_slot, cscptr, cursor, csc_users, work, (int)item_begin,
                                        (int)item_end);
    RPK_LAUNCH_CHECK(c);
  }
  unsigned* pref = c->buf<unsigned>("fit_pref", (size_t)nnz);
  if (nnz > 0 && I > 0) {
    int blocks = (int)std::min<int64_t>((nrows * 32 + 255) / 256, (int64_t)c->sm_count * 32);
    k_csc_prefix<<<std::max(blocks, 1), 256, 0, st>>>(cscptr, csc_users, indptr, item_begin, item_end, pref);
    RPK_LAUNCH_CHECK(c);
    k_csc_prefix_long<<<(int)std::min<int64_t>(nrows, (int64_t)c->sm_count * 2), 1024, 0, st>>>(cscptr, csc_users, indptr, item_begin,
                                                                                                  item_end, pref);
    RPK_LAUNCH_CHECK(c);
  }
  int* nmax = c->buf<int>("fit_nmax", 4);
  u64* pwmin = reinterpret_cast<u64*>(c->buf<double>("fit_pwmin", 2));
  RPK_CUDA(cudaMemsetAsync(nmax, 0, sizeof(int) * 4, st));
  RPK_CUDA(cudaMemsetAsync(pwmin, 0xff, sizeof(u64), st));
  if (I > 0) {
    k_item_extremes<<<ceil_div(I, 256), 256, 0, st>>>(n, pw, I, nmax, pwmin);
    RPK_LAUNCH_CHECK(c);
    k_recip_f32<<<ceil_div(I, 256), 256, 0, st>>>(n, rnf, I);
    RPK_LAUNCH_CHECK(c);
    k_pop_code<<<ceil_div(I, 256), 256, 0, st>>>(n, c->buf<unsigned char>("fit_pop_code", (size_t)I), I);
    RPK_LAUNCH_CHECK(c);
  }

  Out<int32_t> o_idx, o_cnt, o_len;
  Out<double> o_val;
  o_idx.init(c, out_idx_u, (size_t)nrows * K, "fit_out_idx");
  o_len.init(c, out_len_u, (size_t)nrows, "fit_out_len");
  int32_t* cnt_dev;  // counts are always produced (values need them)
  if (out_cnt_u) {
    o_cnt.init(c, out_cnt_u, (size_t)nrows * K, "fit_out_cnt");
    cnt_dev = o_cnt.dev;
  } else {
    cnt_dev = c->buf<int32_t>("fit_out_cnt", (size_t)nrows * K);
  }
  o_val.init(c, out_val_u, (size_t)nrows * K, "fit_out_val");

  if (nrows > 0) {
    k_bucket_count<<<ceil_div(nrows, 256), 256, 0, st>>>(work, item_begin, item_end, bcnt);
    RPK_LAUNCH_CHECK(c);
    k_bucket_offsets<<<1, 32, 0, st>>>(bcnt, boff);
    RPK_LAUNCH_CHECK(c);
    k_bucket_scatter<<<ceil_div(nrows, 256), 256, 0, st>>>(work, item_begin, item_end, boff, order);
    RPK_LAUNCH_CHECK(c);
    // rows with fewer than 65536 users -> 16-bit packed counters; the few heavier rows -> 32-bit counters
    int* order_l = c->buf<int>("fit_order_l", (size_t)nrows);
    int* order_h = c->buf<int>("fit_order_h", (size_t)nrows);
    int* split_cnt = c->buf<int>("fit_split_cnt", 4);
    int* queues = c->buf<int>("fit_queues", 4);
    RPK_CUDA(cudaMemsetAsync(queues, 0, sizeof(int) * 4, st));
    const bool force_wide = (c->flags & DBG_WIDE_ACC) != 0;  // test hook: every row through the 32-bit path
    int* heavy_ids = c->buf<int>("fit_heavy_ids", HEAVY_CAP + 4);
    int* heavy_n = heavy_ids + HEAVY_CAP;
    int* heavy_pair = c->buf<int>("fit_heavy_pair", HEAVY_CAP * HEAVY_CAP);
    RPK_CUDA(cudaMemsetAsync(heavy_ids, 0, sizeof(int) * (HEAVY_CAP + 4), st));
    RPK_CUDA(cudaMemsetAsync(heavy_pair, 0, sizeof(int) * HEAVY_CAP * HEAVY_CAP, st));
    if (!force_wide && U >= 65536) {
      k_find_heavy<<<ceil_div(I, 256), 256, 0, st>>>(n, I, heavy_ids, heavy_n);
      RPK_LAUNCH_CHECK(c);
      const int hb = (int)std::min<int64_t>((U * 32 + 255) / 256, (int64_t)c->sm_count * 16);
      k_heavy_pairs<<<hb, 256, 0, st>>>(indptr, indices, U, heavy_ids, heavy_n, heavy_pair);
      RPK_LAUNCH_CHECK(c);
    }
    k_split_rows<<<1, 1024, 0, st>>>(order, (int)nrows, n, force_wide ? 0 : 65536, force_wide ? nullptr : heavy_n, order_l,
                                     order_h, split_cnt);
    RPK_LAUNCH_CHECK(c);

    const bool tiny = c->flags & DBG_TINY_LIST;
    const int cap = std::max(tiny ? 64 : 1024, next_pow2(2 * K));
    const int direct_cap = tiny ? K : std::min(cap, std::max(2 * K, 64));
    const size_t fixed = sel_smem_bytes(cap);
    RPK_REQUIRE((size_t)c->smem_max > fixed + 1024 + 4096, "K too large for shared memory");
    const SimKey sk{n, rnf, pw, nmax, reinterpret_cast<const double*>(pwmin), nullptr, nullptr, mode};

    c->mark("fit: CSC + order + heavy");
    c->span_begin(1);
    const int defer_max = cap;
    int* scr_idx = c->buf<int>("fit_scr_idx", (size_t)nrows * defer_max);
    int* scr_cnt = c->buf<int>("fit_scr_cnt", (size_t)nrows * defer_max);
    int* scr_len = c->buf<int>("fit_scr_len", (size_t)nrows);
    RPK_CUDA(cudaMemsetAsync(scr_len, 0xff, sizeof(int) * (size_t)nrows, st));  // -1: nothing deferred
    bool any_deferred = false;
    // the handful of rows with >= 65536 users (32-bit counters) run on a side stream next to the main
    // launch: they occupy a few SMs for a long time and would otherwise serialise behind it
    if (!c->side) {
      RPK_CUDA(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
      RPK_CUDA(cudaEventCreateWithFlags(&c->side_ev[0], cudaEventDisableTiming));
      RPK_CUDA(cudaEventCreateWithFlags(&c->side_ev[1], cudaEventDisableTiming));
    }
#ifdef RPK_PHASE_PROF
    static const unsigned long long ev_zero[8] = {};
    RPK_CUDA(cudaMemcpyToSymbolAsync(g_fit_ev, ev_zero, sizeof(ev_zero), 0, cudaMemcpyHostToDevice, st));
    int geo_P = 0, geo_R = 0, geo_code = 0;
    size_t geo_smem = 0, geo_static = 0;
#endif
    RPK_CUDA(cudaEventRecord(c->side_ev[0], st));
    RPK_CUDA(cudaStreamWaitEvent(c->side, c->side_ev[0], 0));
    cudaStream_t main_st = st;
    for (int wide = 1; wide >= 0; --wide) {
      cudaStream_t st = wide ? c->side : main_st;  // shadows the outer stream inside this launch
      auto kern = wide ? (g8 ? k_fit_rows<false, true> : k_fit_rows<false, false>)
                       : (g8 ? k_fit_rows<true, true> : k_fit_rows<true, false>);
      // the kernel's static tables (popularity-code table, count floors, heavy columns) come out of the same
      // per-block limit as the dynamic shared memory
      cudaFuncAttributes fa;
      RPK_CUDA(cudaFuncGetAttributes(&fa, kern));
      const size_t static_smem = fa.sharedSizeBytes;
      RPK_REQUIRE((size_t)c->smem_max > fixed + static_smem + 4096, "K too large for shared memory");
      const size_t avail = (size_t)c->smem_max - fixed - static_smem;
      // coded reciprocals (1 B per item in shared memory) when the catalogue leaves room for them
      const bool use_code = mode == 0 && (size_t)I + 65536 < avail && U < ((int64_t)1 << 21);  // code 255 = 2.5M users
      // (the kernel keeps R * P >= I code bytes: R is rounded up to a multiple of 8 per range)
      const size_t code_bytes = use_code ? (((size_t)I + 8 * 64 + 15) & ~(size_t)15) : 0;
      // geometry: item-range passes so that the counters of one pass fit shared memory
      const int bytes_per_item = wide ? 4 : 2;
      int64_t Rmax = (int64_t)((avail - code_bytes) / bytes_per_item) & ~(int64_t)7;
      int P = (int)((I + Rmax - 1) / Rmax);
      if (P < 1) P = 1;
      if ((c->flags & DBG_MULTI_PASS) && P < 2 && I >= 16) P = 2;
      const int R = (int)(((I + P - 1) / P + 7) & ~(int64_t)7);
      const size_t smem = fixed + (size_t)R * bytes_per_item + code_bytes;
      RPK_REQUIRE(smem + static_smem <= (size_t)c->smem_max,
                  "fit geometry exceeds the shared memory of a block (dynamic + static)");
      const int nt = R >= 16384 ? 1024 : (R >= 4096 ? 512 : 256);
      const int64_t* usplit = nullptr;
      if (P > 1) {
        int64_t* us = c->buf<int64_t>(wide ? "fit_usplit32" : "fit_usplit16", (size_t)U * (P + 1));
        if (U > 0) {
          k_user_split<<<ceil_div(U * (P + 1), 256), 256, 0, st>>>(indptr, indices, U, P, R, us);
          RPK_LAUNCH_CHECK(c);
        }
        usplit = us;
      }
      int* part_idx = o_idx.dev;
      int* part_cnt = cnt_dev;
      int* part_len = o_len.dev;
      if (P > 1) {
        part_idx = c->buf<int>(wide ? "fit_part_idx32" : "fit_part_idx16", (size_t)nrows * P * K);
        part_cnt = c->buf<int>(wide ? "fit_part_cnt32" : "fit_part_cnt16", (size_t)nrows * P * K);
        part_len = c->buf<int>(wide ? "fit_part_len32" : "fit_part_len16", (size_t)nrows * P);
      }
      FitParams fp;
      fp.indptr = indptr;
      fp.indices = indices;
      fp.usplit = usplit;
      fp.cscptr = cscptr;
      fp.csc_users = csc_users;
      fp.pref = pref;
      fp.work = work;
      fp.g16 = g8 ? reinterpret_cast<const unsigned short*>(g8) : g16;
      fp.ldg = rows_pad;
      fp.sk = sk;
      fp.order = wide ? order_h : order_l;
      fp.nrows_dev = split_cnt + wide;
      fp.P = P;
      fp.R = R;
      fp.I = (int)I;
      fp.K = K;
      fp.item_begin = item_begin;
      fp.cap = cap;
      fp.direct_cap = direct_cap;
      fp.direct_out = P == 1;
      fp.queue = queues + wide;
      fp.out_idx = part_idx;
      fp.out_cnt = part_cnt;
      fp.out_len = part_len;
      // rows written directly to the final arrays may defer their sort to k_fit_sort_rows
      fp.pop_code = use_code ? c->get<unsigned char>("fit_pop_code") : nullptr;
      fp.heavy_ids = (!wide && !force_wide) ? heavy_ids : nullptr;
      fp.heavy_n = heavy_n;
      fp.heavy_pair = heavy_pair;
      fp.defer_max = (P == 1 && !tiny) ? defer_max : 0;
      fp.scr_idx = scr_idx;
      fp.scr_cnt = scr_cnt;
      fp.scr_len = scr_len;
      any_deferred = any_deferred || fp.defer_max > 0;
      fp.pre = nullptr;
      fp.hbuf = nullptr;
      fp.hstride = 0;
      fp.piece_tab = nullptr;
      fp.hcount = nullptr;
      fp.split_rows = nullptr;
      fp.hdone = nullptr;
      fp.hneed = nullptr;
      if (!wide && !force_wide && P == 1 && nrows > 0) {
        // rows too heavy for one CTA next to the others are counted in pieces (see k_heavy_plan)
        const int64_t hstride = (((I + 1) >> 1) + 3) & ~(int64_t)3;
        int4* piece_tab = c->buf<int4>("fit_heavy_pieces", HEAVY_ROWS * HEAVY_SPLITS);
        int* hmeta = c->buf<int>("fit_heavy_meta", 2 + 3 * HEAVY_ROWS);  // counts | split rows | done | need
        int* pre = c->buf<int>("fit_heavy_pre", (size_t)I);
        unsigned* hbuf = c->buf<unsigned>("fit_heavy_buf", (size_t)HEAVY_ROWS * hstride);
        RPK_CUDA(cudaMemsetAsync(pre, 0xff, sizeof(int) * (size_t)I, st));
        RPK_CUDA(cudaMemsetAsync(hmeta, 0, sizeof(int) * (2 + 3 * HEAVY_ROWS), st));
        RPK_CUDA(cudaMemsetAsync(hbuf, 0, sizeof(unsigned) * (size_t)HEAVY_ROWS * hstride, st));
        const u64 min_target = (c->flags & DBG_SPLIT_ROWS) ? 64ull : (1ull << 20);
        k_heavy_plan<<<1, 1024, 0, st>>>(fp.order, fp.nrows_dev, work, c->sm_count, min_target, piece_tab, hmeta, hmeta + 2,
                                         hmeta + 2 + 2 * HEAVY_ROWS, pre);
        RPK_LAUNCH_CHECK(c);
        fp.pre = pre;
        fp.hbuf = hbuf;
        fp.hstride = hstride;
        fp.piece_tab = piece_tab;
        fp.hcount = hmeta;
        fp.split_rows = hmeta + 2;
        fp.hdone = hmeta + 2 + HEAVY_ROWS;
        fp.hneed = hmeta + 2 + 2 * HEAVY_ROWS;
      }
      fp.prof = nullptr;
#ifdef RPK_PHASE_PROF
      if (!wide) {
        fp.prof = c->buf<unsigned long long>("fit_prof", 16);
        RPK_CUDA(cudaMemsetAsync(fp.prof, 0, 16 * sizeof(unsigned long long), st));
        geo_P = P;
        geo_R = R;
        geo_code = use_code;
        geo_smem = smem;
        geo_static = static_smem;
      }
#endif
      RPK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int occ = 0;
      RPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nt, smem));
      RPK_REQUIRE(occ >= 1, "fit kernel does not fit on an SM");
      // the heavy list is short (items seen by >= 65536 users): a small grid is enough for it
      const int64_t max_items = wide && !force_wide ? std::min<int64_t>(nrows * P, 64) : nrows * P;
      const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(max_items, (int64_t)c->sm_count * occ));
      kern<<<grid, nt, smem, st>>>(fp);
      RPK_LAUNCH_CHECK(c);
      if (P > 1) {
        MergeParams mp;
        mp.sk = sk;
        mp.part_idx = part_idx;
        mp.part_cnt = part_cnt;
        mp.order = fp.order;
        mp.nrows_dev = fp.nrows_dev;
        mp.item_begin = item_begin;
        mp.P = P;
        mp.K = K;
        mp.cap = cap;
        mp.direct_cap = direct_cap;
        mp.out_idx = o_idx.dev;
        mp.out_cnt = cnt_dev;
        mp.out_len = o_len.dev;
        RPK_CUDA(cudaFuncSetAttribute(k_fit_merge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fixed));
        const int mgrid = (int)std::min<int64_t>(max_items, (int64_t)c->sm_count * 8);
        k_fit_merge<<<std::max(1, mgrid), 256, fixed, st>>>(mp);
        RPK_LAUNCH_CHECK(c);
      }
    }
    RPK_CUDA(cudaEventRecord(c->side_ev[1], c->side));
    RPK_CUDA(cudaStreamWaitEvent(st, c->side_ev[1], 0));
#ifdef RPK_PHASE_PROF
    {
      unsigned long long h[16];
      RPK_CUDA(cudaMemcpyAsync(h, c->get<unsigned long long>("fit_prof"), sizeof(h), cudaMemcpyDeviceToHost, st));
      RPK_CUDA(cudaStreamSynchronize(st));
      unsigned long long sp[16];
      RPK_CUDA(cudaMemcpyFromSymbol(sp, g_sel_prof, sizeof(sp)));
      fprintf(stderr, "[select phases, all selection calls of the fit so far] stats %.3g  sampled histogram %.3g  boundary %.3g  copy %.3g  tail %.3g  (refinements entered: mark %.3g)\n",
              (double)sp[0], (double)sp[1], (double)sp[2], (double)sp[3], (double)sp[4], (double)sp[6]);
      static const char* nm[6] = {"queue", "init counters", "accumulate", "heavy + diagonal", "select", "survivors out"};
      unsigned long long tot = 0;
      for (int k = 0; k < 6; ++k) tot += h[k];
      fprintf(stderr, "[fit rows phases] rows=%llu survivors/row=%.0f cycles/row=%.0f\n", h[8], h[8] ? (double)h[9] / h[8] : 0.0,
              h[8] ? (double)tot / h[8] : 0.0);
      for (int k = 0; k < 6; ++k)
        fprintf(stderr, "  %-18s %5.1f%%  %8.0f cycles/row\n", nm[k], 100.0 * h[k] / (tot ? tot : 1), h[8] ? (double)h[k] / h[8] : 0.0);
      unsigned long long ev[8];
      RPK_CUDA(cudaMemcpyFromSymbol(ev, g_fit_ev, sizeof(ev)));
      fprintf(stderr, "[fit paths] guess_ok=%llu guess_rejected=%llu queue_overflow=%llu band=%llu index_radix=%llu deferred=%llu "
              "merged=%llu P=%d R=%d code=%d smem=%zu static=%zu\n",
              ev[SEL_EV_GUESS_OK], ev[SEL_EV_GUESS_REJECTED], ev[SEL_EV_QUEUE_OVERFLOW], ev[SEL_EV_BAND], ev[SEL_EV_INDEX_RADIX],
              ev[FIT_EV_DEFERRED], ev[FIT_EV_MERGED], geo_P, geo_R, geo_code, geo_smem, geo_static);
    }
#endif
    c->mark("fit: row kernels");
    c->span_end(1);  // the row kernels end here (rpk_last_timings); the deferred sort is timed with the rest of the fit
    if (any_deferred || o_val.dev) {
      // one finishing launch: the deferred rows are selected and sorted, every row gets its values
      const bool coarse = (c->flags & DBG_COARSE_SORT_KEY) != 0;  // test hook: nearly every order settled exactly
      int* queue = c->buf<int>("fit_sort_queue", 1);
      RPK_CUDA(cudaMemsetAsync(queue, 0, sizeof(int), st));
      SortParams sp;
      sp.n = n;
      sp.pw = pw;
      sp.scr_idx = scr_idx;
      sp.scr_cnt = scr_cnt;
      sp.scr_len = scr_len;
      sp.queue = queue;
      sp.defer_max = defer_max;
      sp.K = K;
      sp.mode = mode;
      sp.nrows = nrows;
      sp.item_begin = item_begin;
      sp.key_mask = coarse ? ~((1ull << 40) - 1) : ~0ull;
      sp.margin = coarse ? (1ull << 40) : (mode == 0 ? 4ull : 0ull);
      sp.out_idx = o_idx.dev;
      sp.out_cnt = cnt_dev;
      sp.out_len = o_len.dev;
      sp.out_val = o_val.dev;
#ifdef RPK_PHASE_PROF
      static const unsigned long long sort_zero[8] = {};
      RPK_CUDA(cudaMemcpyToSymbolAsync(g_fit_sort, sort_zero, sizeof(sort_zero), 0, cudaMemcpyHostToDevice, st));
#endif
      // one warp per row while the survivors fit 1,024 (K <= 512), a 256-thread block per row above
      const bool warp_rows = defer_max <= 1024;
      auto kern = warp_rows ? k_fit_sort_rows<32> : k_fit_sort_rows<256>;
      const int nt = warp_rows ? 64 : 256;
      const size_t ssm = sort_group_bytes(defer_max) * (nt / (warp_rows ? 32 : 256));
      RPK_REQUIRE(ssm <= (size_t)c->smem_max, "K too large for shared memory");
      RPK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm));
      int socc = 0;
      RPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&socc, kern, nt, ssm));
      const int rows_per_block = warp_rows ? nt / 32 : 1;
      const int sgrid = (int)std::max<int64_t>(1, std::min<int64_t>((nrows + rows_per_block - 1) / rows_per_block,
                                                                      (int64_t)c->sm_count * std::max(socc, 1)));
      kern<<<sgrid, nt, ssm, st>>>(sp);
      RPK_LAUNCH_CHECK(c);
#ifdef RPK_PHASE_PROF
      unsigned long long fs[8];
      RPK_CUDA(cudaMemcpyFromSymbolAsync(fs, g_fit_sort, sizeof(fs), 0, cudaMemcpyDeviceToHost, st));
      RPK_CUDA(cudaStreamSynchronize(st));
      const double rs = fs[0] ? (double)fs[0] : 1.0;
      fprintf(stderr, "[fit sort] sorted=%llu values_only=%llu exact_cmp=%llu coarse=%d  cycles/sorted row: load %.0f select %.0f "
              "compact %.0f sort %.0f out %.0f\n", fs[0], fs[1], fs[2], (int)coarse, fs[3] / rs, fs[4] / rs, fs[5] / rs, fs[6] / rs,
              fs[7] / rs);
#endif
    }
  }
  c->mark("fit: sort + values");
}

// The public fit: stages the inputs and outputs once and runs the row range in strips of at most `strip_rows` rows, so
// that only one strip of the dense-leg count matrix (uint16 or uint8, rows x I) exists at a time: the item x item matrix is
// never materialised as a whole (an 80 GB object at I = 200,000) and the tensor-core leg stays on for large catalogues.
void run_fit(rpk_ctx* c, int64_t U, int64_t I, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
             int similarity, const double* item_pow_u, int K, int64_t item_begin, int64_t item_end, int32_t* out_idx_u,
             int32_t* out_cnt_u, double* out_val_u, int32_t* out_len_u) {
  RPK_REQUIRE(U >= 0 && I >= 0 && nnz >= 0, "negative dimension");
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(0 <= item_begin && item_begin <= item_end && item_end <= I, "bad item range");
  RPK_REQUIRE(out_idx_u && out_len_u, "out_idx / out_len must not be null");
  const int64_t nrows = item_end - item_begin;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "fit_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "fit_indices");
  const double* pw = item_pow_u ? stage_in(c, item_pow_u, (size_t)I, "fit_pw") : nullptr;
  Out<int32_t> o_idx, o_cnt, o_len;
  Out<double> o_val;
  o_idx.init(c, out_idx_u, (size_t)nrows * K, "fit_out_idx");
  o_len.init(c, out_len_u, (size_t)nrows, "fit_out_len");
  if (out_cnt_u) o_cnt.init(c, out_cnt_u, (size_t)nrows * K, "fit_out_cnt");
  o_val.init(c, out_val_u, (size_t)nrows * K, "fit_out_val");
  c->span_reset();
  const int64_t rows_pad = (I + 255) / 256 * 256;
  int64_t strip_rows = c->strip_rows > 0 ? c->strip_rows : (int64_t)(8e9 / ((double)rows_pad * 2.0));
  strip_rows = std::max<int64_t>(128, strip_rows / 128 * 128);
  if (c->dense_users == 0 || nrows <= strip_rows) strip_rows = std::max<int64_t>(nrows, 1);  // no dense leg: nothing to bound
  int strip = 0;
  for (int64_t b = item_begin; b < item_end || strip == 0; b += strip_rows, ++strip) {
    const int64_t e = std::min(item_end, b + strip_rows);
    const int64_t off = b - item_begin;
    fit_range(c, U, I, nnz, indptr, indices, similarity, pw, K, b, e, o_idx.dev + off * K,
              o_cnt.dev ? o_cnt.dev + off * K : nullptr, o_val.dev ? o_val.dev + off * K : nullptr, o_len.dev + off, strip,
              nrows);
    if (e >= item_end) break;
  }
  // remember where the lists live on the device: predict can load its model from them without a round trip
  c->lf_token++;
  c->lf_idx = nullptr;
  if (item_begin == 0 && item_end == I && o_val.dev) {
    c->lf_idx = o_idx.dev;
    c->lf_val = o_val.dev;
    c->lf_len = o_len.dev;
    c->lf_I = I;
    c->lf_K = K;
  }
  o_idx.finish(c);
  o_cnt.finish(c);
  o_val.finish(c);
  o_len.finish(c);
  finish_call(c);
}

void run_fit_item_counts(rpk_ctx* c, int32_t* out_counts, int64_t I) {
  RPK_REQUIRE(c->fit_I == I && I >= 0, "rpk_fit_item_counts: no fit with this item count on the context");
  Out<int32_t> o;
  o.init(c, out_counts, (size_t)I, "fit_n_out");
  if (I > 0) RPK_CUDA(cudaMemcpyAsync(o.dev, c->get<int>("fit_n"), sizeof(int) * (size_t)I, cudaMemcpyDeviceToDevice, c->stream));
  o.finish(c);
  finish_call(c);
}

}  // namespace rpk
