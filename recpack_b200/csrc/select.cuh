// Block-wide exact top-K selection shared by the fit epilogue, the top-N of predict and the
// CSR row ranking.  Replaces np.argpartition + the Python row loop of
// recpack/util.py:50-77 (get_top_K_ranks) with a deterministic rule: best key first, ties by
// ascending index.
//
// A "source" owns the candidate slots and drives the iteration over them:
//   for_each(f)            calls f(slot, akey) for every candidate slot (any thread, any order; each
//                          candidate exactly once per block).  akey is a 64-bit SORTABLE key (larger =
//                          better) that may be approximate: it may mis-order two candidates only if
//                          their akeys differ by at most margin();
//   for_each_sampled(f)    the same for roughly one candidate in SEL_SAMPLE (a fixed subset);
//   set_floor(thr)         hint: until the next call the iteration may skip candidates with akey < thr;
//   stats(sh)              candidate count and key bounds into sh->count / kmin / kmax;
//   void entry(slot, e)    the Entry (16 B) of a candidate slot, carrying what cmp3 needs;
//   int cmp3(a, b)         exact three-way comparison of two entries' keys (index excluded).
//
// Algorithm (all control flow is block-uniform):
//   A. stats.  Few candidates -> copy them all, sort, done.
//   B0. many candidates: guess a threshold from a 1-in-16 sample; accept it when it leaves between
//       K and cap survivors (verified by the copy itself).
//   B. otherwise radix refinement on akey: 4096-bin histograms over [lo, hi], descending into the bin
//      that holds the K-th largest akey until the candidates with akey >= lo (minus margin) fit.
//   C. if they never fit (a huge group of equal / near-equal akeys straddles the K-th place): exact
//      quick-select inside that band with cmp3, and inside an exactly-tied class a second radix
//      refinement on the index picks the smallest indices.
//   D. exact sort of the (<= cap) survivors; the first K are the result.
#pragma once
#include <stdint.h>

namespace rpk {

typedef unsigned long long u64;

// Profiling hook (RPK_PHASE_PROF builds of fit.cu define it): cycles of thread 0 between the marks of
// block_select_topk.
#ifndef SEL_MARK
#define SEL_MARK(k) do {} while (0)
#define SEL_MARK_BEGIN() do {} while (0)
#endif
// Path counters (RPK_PHASE_PROF builds of fit.cu define it): called by thread 0 when block_select_topk takes a branch.
enum SelEvent { SEL_EV_GUESS_OK, SEL_EV_GUESS_REJECTED, SEL_EV_QUEUE_OVERFLOW, SEL_EV_BAND, SEL_EV_INDEX_RADIX, SEL_EV_COUNT };
#ifndef SEL_EVENT
#define SEL_EVENT(src, ev) do {} while (0)
#endif

struct __align__(16) Entry {
  u64 key;
  int idx;
  int aux;
};

constexpr int SEL_BINS = 4096;
constexpr int SENTINEL_IDX = 0x7fffffff;
constexpr int SEL_RANK_MAX = 64;     // up to this many survivors: rank by counting instead of bitonic
constexpr int SEL_SAMPLE = 16;       // the threshold guess looks at one slot in 16
constexpr int SEL_GUESS_MIN = 4096;  // below this many candidates the exact histogram is cheap enough

struct SelShared {
  u64 kmin, kmax;
  u64 lo, hi;
  Entry piv;
  int count;
  int count2;
  int bstar;
  int g_new;
  int n_in;
  int piv_slot;
  int warp_tot[33];
};

// Shared-memory layout of the selection workspace: [list: cap + SEL_RANK_MAX entries][hist][SelShared]
__host__ __device__ __forceinline__ size_t sel_list_bytes(int cap) { return (size_t)(cap + SEL_RANK_MAX) * sizeof(Entry); }
__host__ __device__ __forceinline__ size_t sel_smem_bytes(int cap, int bins = SEL_BINS) {
  return sel_list_bytes(cap) + bins * sizeof(int) + ((sizeof(SelShared) + 15) / 16) * 16;
}

__device__ __forceinline__ u64 warp_min_u64(u64 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    u64 t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t < v ? t : v;
  }
  return v;
}
__device__ __forceinline__ u64 warp_max_u64(u64 v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    u64 t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t > v ? t : v;
  }
  return v;
}

// Append one survivor (callable from divergent code; survivors are few, so one atomic each is fine).
// Every caller is counted, entries beyond `cap` are dropped -- the count tells.
__device__ __forceinline__ void append_one(const Entry& e, Entry* list, int cap, int* counter) {
  const int pos = atomicAdd(counter, 1);
  if (pos < cap) list[pos] = e;
}

// Exact total order used by the final sort: true when a must precede b.
template <class Src>
__device__ __forceinline__ bool entry_before(const Src& src, const Entry& a, const Entry& b) {
  if (a.idx == SENTINEL_IDX) return false;
  if (b.idx == SENTINEL_IDX) return true;
  int c = src.cmp3(a, b);
  if (c != 0) return c > 0;
  return a.idx < b.idx;
}

// Bitonic sort, best first.  Stages whose partner distance is below 32 only touch elements owned by
// one warp (element i belongs to thread i % blockDim.x), so they need a warp barrier, not a block barrier.
template <class Src>
__device__ void bitonic_sort_entries(const Src& src, Entry* list, int n_pow2) {
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int k = 2; k <= n_pow2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n_pow2; i += nt) {
        int ixj = i ^ j;
        if (ixj > i) {
          Entry a = list[i], b = list[ixj];
          bool up = (i & k) == 0;
          if (entry_before(src, b, a) == up) {
            list[i] = b;
            list[ixj] = a;
          }
        }
      }
      const bool next_is_wide = j > 1 ? (j >> 1) >= 32 : k >= 32;
      if (j >= 32 || next_is_wide || (j == 1 && k == n_pow2)) __syncthreads();
      else __syncwarp();
    }
  }
}

// Small lists (m <= SEL_RANK_MAX = 64): rank every element by counting the elements that precede it.
// 16 threads share one element (4 comparisons each, combined by shuffles), so the whole list is ranked
// in one short step by the first 16*m threads.  `tmp` must hold m entries and may not alias `list`.
template <class Src>
__device__ void rank_sort_entries(const Src& src, Entry* list, Entry* tmp, int m) {
  const int tid = threadIdx.x, nt = blockDim.x;
  if (nt >= 16 * SEL_RANK_MAX) {
    const int i = tid >> 4, part = tid & 15;
    int rank = 0;
    Entry a;
    if (i < m) {
      a = list[i];
      for (int f = part; f < m; f += 16) rank += (f != i) && entry_before(src, list[f], a);
    }
    rank += __shfl_xor_sync(0xffffffffu, rank, 8);
    rank += __shfl_xor_sync(0xffffffffu, rank, 4);
    rank += __shfl_xor_sync(0xffffffffu, rank, 2);
    rank += __shfl_xor_sync(0xffffffffu, rank, 1);
    if (i < m && part == 0) tmp[rank] = a;
  } else {
    for (int i = tid; i < m; i += nt) {
      const Entry a = list[i];
      int rank = 0;
      for (int f = 0; f < m; ++f) rank += (f != i) && entry_before(src, list[f], a);
      tmp[rank] = a;
    }
  }
  __syncthreads();
  for (int i = tid; i < m; i += nt) list[i] = tmp[i];
  __syncthreads();
}

// Finds the bin holding the need-th largest key of a histogram, scanning bins from the top:
// sh->bstar = that bin, sh->g_new = g + members of higher bins, sh->n_in = members of the bin.
// When fewer than `need` members exist in total, bstar = 0 and n_in / g_new describe bin 0.
__device__ __forceinline__ void find_boundary_bin(const int* hist, int nb, int g, int need, SelShared* sh) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  const int per = (nb + nt - 1) / nt;
  const int b0 = tid * per;
  const int b1 = min(nb, b0 + per);
  int tsum = 0;
  for (int b = b0; b < b1; ++b) tsum += hist[b];
  int incl = tsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) sh->warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = lane < nwarps ? sh->warp_tot[lane] : 0;
    int iv = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, iv, o);
      if (lane >= o) iv += t;
    }
    sh->warp_tot[lane] = iv - v;  // exclusive prefix of warp totals
    if (lane == 31) sh->warp_tot[32] = iv;
  }
  __syncthreads();
  const int total = sh->warp_tot[32];
  const int prefix_excl = sh->warp_tot[warp] + incl - tsum;
  int above = g + (total - prefix_excl - tsum);  // members in bins owned by higher threads
  if (g + total < need) {
    if (tid == 0) {
      sh->bstar = 0;
      sh->g_new = g + total - hist[0];
      sh->n_in = hist[0];
    }
  } else if (above < need && above + tsum >= need) {
    for (int b = b1 - 1; b >= b0; --b) {
      int h = hist[b];
      if (above + h >= need) {
        sh->bstar = b;
        sh->g_new = above;
        sh->n_in = h;
        break;
      }
      above += h;
    }
  }
  __syncthreads();
}

// Histogram geometry for keys in [lo, hi]: at most 2^BITS (<= SEL_BINS) bins of 2^shift consecutive keys.
template <int BITS = 12>
__device__ __forceinline__ void bin_geometry(u64 lo, u64 hi, int& shift, int& nb) {
  const u64 range = hi - lo;
  const int bits = range ? 64 - __clzll((long long)range) : 0;
  shift = bits > BITS ? bits - BITS : 0;
  nb = (int)(range >> shift) + 1;
}

// Step A for sources without a cheaper way: candidate count and smallest / largest key.
template <class Src>
__device__ void generic_stats(const Src& src, SelShared* sh) {
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) {
    sh->count = 0;
    sh->kmin = ~0ull;
    sh->kmax = 0ull;
  }
  __syncthreads();
  u64 lmin = ~0ull, lmax = 0ull;
  int cnt = 0;
  src.for_each([&](int, u64 k) {
    cnt++;
    lmin = k < lmin ? k : lmin;
    lmax = k > lmax ? k : lmax;
  });
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  lmin = warp_min_u64(lmin);
  lmax = warp_max_u64(lmax);
  if (lane == 0 && cnt) {
    atomicAdd(&sh->count, cnt);
    atomicMin(&sh->kmin, lmin);
    atomicMax(&sh->kmax, lmax);
  }
  __syncthreads();
}

// One refinement run over the candidates of `src`.  On entry [lo, hi] bounds the keys of interest,
// n_in = candidates inside, g = candidates known to be above hi.  Descends while g + n_in > room and
// lo < hi.  Results in sh->lo / sh->hi / sh->g_new / sh->n_in.
template <int BITS = 12, class Src>
__device__ void refine_keys(Src& src, int need, int room, u64 lo, u64 hi, int g, int n_in, int* hist, SelShared* sh) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const u64 M = src.margin();
  while (g + n_in > room && lo < hi) {
    int shift, nb;
    bin_geometry<BITS>(lo, hi, shift, nb);
    for (int b = tid; b < nb; b += nt) hist[b] = 0;
    src.set_floor(lo > M ? lo - M : 0ull);
    __syncthreads();
    src.for_each([&](int, u64 k) {
      if (k >= lo && k <= hi) atomicAdd(&hist[(int)((k - lo) >> shift)], 1);
    });
    __syncthreads();
    find_boundary_bin(hist, nb, g, need, sh);
    const int bstar = sh->bstar;
    g = sh->g_new;
    n_in = sh->n_in;
    const u64 nlo = lo + ((u64)bstar << shift);
    const u64 span = (((u64)1) << shift) - 1;
    u64 nhi = nlo + span;
    if (nhi > hi || nhi < nlo) nhi = hi;
    lo = nlo;
    hi = nhi;
    __syncthreads();
  }
  if (tid == 0) {
    sh->lo = lo;
    sh->hi = hi;
    sh->g_new = g;
    sh->n_in = n_in;
  }
  __syncthreads();
}

// Copies every candidate with key >= thr to list; returns how many there were (may exceed cap).
// With `certain` set, *certain is also incremented for every candidate with key >= edge (edge >= thr).
// Sources with a cheap pre-filter (has_queue()) are visited in two steps when `scratch` is given: a dense pass queues
// the slots that pass the pre-filter, then the queue is worked off one candidate per thread -- so the expensive part
// (exact key, the entry's global loads, the append) runs with full warps instead of once per warp for every lane
// that happens to hold a candidate.
template <class Src>
__device__ int compact_above(Src& src, u64 thr, Entry* list, int cap, SelShared* sh, u64 edge = 0ull,
                             int* certain = nullptr, int* scratch = nullptr, int scratch_cap = 0) {
  if (threadIdx.x == 0) sh->count = 0;
  src.set_floor(thr);
  __syncthreads();
  auto take = [&](int slot, u64 k) {
    if (k >= thr) {
      Entry e;
      src.entry(slot, e);
      append_one(e, list, cap, &sh->count);
      if (certain && k >= edge) atomicAdd(certain, 1);
    }
  };
  if (scratch && src.has_queue()) {
    if (src.for_each_queued(take, scratch, scratch_cap, &sh->n_in)) {
      __syncthreads();
      return sh->count;
    }
    // the queue overflowed: nothing was taken yet, visit directly
    if (threadIdx.x == 0) {
      sh->count = 0;
      SEL_EVENT(src, SEL_EV_QUEUE_OVERFLOW);
    }
    __syncthreads();
  }
  src.for_each([&](int slot, u64 k) {
    if (k >= thr) {
      Entry e;
      src.entry(slot, e);
      append_one(e, list, cap, &sh->count);
      if (certain && k >= edge) atomicAdd(certain, 1);
    }
  });
  __syncthreads();
  return sh->count;
}

// Returns m = number of selected entries (<= K); list[0..m) holds them best-first.
// defer_max > 0: when at most defer_max survivors remain they are returned UNSORTED (*sorted = false,
// return value = their number, possibly > K) so that the caller can sort them elsewhere.
// SURVIVORS_ONLY: the source cannot compare exactly (cmp3 unusable).  The call then returns every candidate
// that could belong to the top K -- unsorted, their number (possibly > K, at most cap) as the result --
// or -1 when they do not fit the list; the caller settles the order by other means.
template <bool SURVIVORS_ONLY = false, int BITS = 12, class Src>
__device__ int block_select_topk(Src& src, int K, Entry* list, int cap, int direct_cap, int* hist, SelShared* sh,
                                 int defer_max = 0, bool* sorted = nullptr) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const u64 M = src.margin();
  if (K > cap) K = cap;
  if (direct_cap < K) direct_cap = K;  // the refinement needs at least K candidates
  if (direct_cap > cap) direct_cap = cap;

  // ---- A: count candidates and bound their keys
  SEL_MARK_BEGIN();
  src.set_floor(0ull);
  src.stats(sh);
  SEL_MARK(0);
  const int n_c = sh->count;
  const u64 kmin = sh->kmin, kmax = sh->kmax;
  __syncthreads();
  int m = -1;
  if (n_c <= direct_cap) {
    m = compact_above(src, 0ull, list, cap, sh);
  } else {
    // keep the survivor list (and the final sort) close to K
    int room = K + (K / 4 > 32 ? K / 4 : 32);
    if (room > cap) room = cap;
    // ---- B0: cheap threshold guess from a 1-in-16 sample; accepted when it leaves between K and cap
    //          candidates, which the copy itself verifies
    if (n_c >= SEL_GUESS_MIN && kmax > kmin) {
      int shift, nb;
      bin_geometry<BITS>(kmin, kmax, shift, nb);
      for (int b = tid; b < nb; b += nt) hist[b] = 0;
      __syncthreads();
      src.for_each_sampled([&](int, u64 k) {
        if (k >= kmin && k <= kmax) atomicAdd(&hist[(int)((k - kmin) >> shift)], 1);
      });
      __syncthreads();
      SEL_MARK(1);
      const int ks = (K + SEL_SAMPLE - 1) / SEL_SAMPLE;
      int sd = 1;
      while (sd * sd < ks) ++sd;
      find_boundary_bin(hist, nb, 0, ks + 3 * sd + 3, sh);
      const u64 edge = kmin + ((u64)sh->bstar << shift);
      const u64 thr = edge > M ? edge - M : 0;
      __syncthreads();
      SEL_MARK(2);
      // the guess stands when at least K candidates lie at or above the edge (they certainly beat everything
      // below edge - M) and the copy fitted
      if (tid == 0) sh->count2 = 0;
      const int got = compact_above(src, thr, list, cap, sh, edge, &sh->count2, hist, 1 << BITS);
      if (sh->count2 >= K && got <= cap) m = got;
      if (tid == 0) SEL_EVENT(src, m >= 0 ? SEL_EV_GUESS_OK : SEL_EV_GUESS_REJECTED);
      __syncthreads();
      SEL_MARK(3);
    }
    if (m < 0) {
      SEL_MARK(6);
      // ---- B: exact radix refinement on the (approximate) key until the survivors fit
      refine_keys<BITS>(src, K, room, kmin, kmax, 0, n_c, hist, sh);
      u64 lo = sh->lo, hi = sh->hi;
      int g = sh->g_new, n_in = sh->n_in;
      u64 thr = lo > M ? lo - M : 0;
      __syncthreads();
      m = compact_above(src, thr, list, cap, sh);
      if (SURVIVORS_ONLY && m > cap) {
        src.set_floor(0ull);
        __syncthreads();
        return -1;
      }
      if (m > cap) {
        // ---- C: a band of (near-)equal keys is too large.  Pin tau = the K-th largest akey.
        if (tid == 0) SEL_EVENT(src, SEL_EV_BAND);
        __syncthreads();
        refine_keys<BITS>(src, K, -1, lo, hi, g, n_in, hist, sh);
        const u64 tau = sh->lo;
        const u64 band_lo = tau > M ? tau - M : 0;
        const u64 band_hi = tau + M < tau ? ~0ull : tau + M;
        src.set_floor(band_lo);
        // certain members: akey above the band (fewer than K of them)
        if (tid == 0) sh->count = 0;
        __syncthreads();
        src.for_each([&](int slot, u64 k) {
          if (k > band_hi) {
            Entry e;
            src.entry(slot, e);
            append_one(e, list, cap, &sh->count);
          }
        });
        __syncthreads();
        int have = sh->count;  // entries in list so far (all certain)
        int need = K - have;   // still to take from the band, by exact order
        bool has_lb = false, has_ub = false;
        Entry lb = {0, 0, 0}, ub = {0, 0, 0};
        // group = band members with exact key strictly between lb and ub
        auto in_group = [&](int slot, u64 k, Entry& e) -> bool {
          if (k < band_lo || k > band_hi) return false;
          src.entry(slot, e);
          if (has_ub && src.cmp3(e, ub) >= 0) return false;
          if (has_lb && src.cmp3(e, lb) <= 0) return false;
          return true;
        };
        while (need > 0) {
          // pivot: the group member in the lowest slot
          if (tid == 0) sh->piv_slot = 0x7fffffff;
          __syncthreads();
          {
            int best = 0x7fffffff;
            src.for_each([&](int slot, u64 k) {
              Entry e;
              if (slot < best && in_group(slot, k, e)) best = slot;
            });
            if (best != 0x7fffffff) atomicMin(&sh->piv_slot, best);
          }
          __syncthreads();
          const int ps = sh->piv_slot;
          if (ps == 0x7fffffff) break;  // group exhausted (cannot happen while need > 0)
          if (tid == 0) {
            Entry e;
            src.entry(ps, e);
            sh->piv = e;
            sh->count = 0;   // greater than pivot
            sh->count2 = 0;  // equal to pivot
          }
          __syncthreads();
          const Entry piv = sh->piv;
          {
            int gt = 0, eq = 0;
            src.for_each([&](int slot, u64 k) {
              Entry e;
              if (in_group(slot, k, e)) {
                int c = src.cmp3(e, piv);
                gt += c > 0;
                eq += c == 0;
              }
            });
            gt = __reduce_add_sync(0xffffffffu, gt);
            eq = __reduce_add_sync(0xffffffffu, eq);
            if ((tid & 31) == 0) {
              if (gt) atomicAdd(&sh->count, gt);
              if (eq) atomicAdd(&sh->count2, eq);
            }
          }
          __syncthreads();
          const int gt = sh->count, eq = sh->count2;
          __syncthreads();
          if (gt >= need) {  // the need-th best is above the pivot
            has_lb = true;
            lb = piv;
            continue;
          }
          // everything above the pivot is in
          if (tid == 0) sh->count = have;
          __syncthreads();
          const bool take_eq = gt + eq <= need || eq <= cap - have - gt;
          src.for_each([&](int slot, u64 k) {
            Entry e;
            if (in_group(slot, k, e)) {
              int c3 = src.cmp3(e, piv);
              if (c3 > 0 || (c3 == 0 && take_eq)) append_one(e, list, cap, &sh->count);
            }
          });
          __syncthreads();
          have = sh->count;
          if (gt + eq < need) {  // pivot class fully in, continue below the pivot
            need -= gt + eq;
            has_ub = true;
            ub = piv;
            continue;
          }
          if (take_eq) break;  // the class fitted as a whole; the final sort trims it
          // ---- exact tie class larger than the list: take the (need - gt) smallest indices by a radix
          //      refinement on the index
          if (tid == 0) SEL_EVENT(src, SEL_EV_INDEX_RADIX);
          const int need_idx = need - gt;
          u64 ilo = 0, ihi = (u64)SENTINEL_IDX;
          int ig = 0, iin = eq;
          const int iroom = cap - have;
          while (ig + iin > iroom && ilo < ihi) {
            int shift, nb;
            bin_geometry<BITS>(ilo, ihi, shift, nb);
            for (int b = tid; b < nb; b += nt) hist[b] = 0;
            __syncthreads();
            src.for_each([&](int slot, u64 k) {
              Entry e;
              if (in_group(slot, k, e) && src.cmp3(e, piv) == 0) {
                const u64 ik = (u64)(unsigned)(SENTINEL_IDX - e.idx);
                if (ik >= ilo && ik <= ihi) atomicAdd(&hist[(int)((ik - ilo) >> shift)], 1);
              }
            });
            __syncthreads();
            find_boundary_bin(hist, nb, ig, need_idx, sh);
            const int bstar = sh->bstar;
            ig = sh->g_new;
            iin = sh->n_in;
            const u64 nlo = ilo + ((u64)bstar << shift);
            u64 nhi = nlo + ((((u64)1) << shift) - 1);
            if (nhi > ihi || nhi < nlo) nhi = ihi;
            ilo = nlo;
            ihi = nhi;
            __syncthreads();
          }
          if (tid == 0) sh->count = have;
          __syncthreads();
          src.for_each([&](int slot, u64 k) {
            Entry e;
            if (in_group(slot, k, e) && src.cmp3(e, piv) == 0 && (u64)(unsigned)(SENTINEL_IDX - e.idx) >= ilo)
              append_one(e, list, cap, &sh->count);
          });
          __syncthreads();
          have = sh->count;
          break;
        }
        m = have < cap ? have : cap;
      }
    }
  }
  // ---- D: exact sort of the survivors
  SEL_MARK(4);
  src.set_floor(0ull);
  if (SURVIVORS_ONLY) {
    __syncthreads();
    return m > cap ? -1 : m;
  }
  if (m > cap) m = cap;
  if (sorted) *sorted = true;
  if (defer_max > 0 && m <= defer_max) {
    *sorted = false;
    __syncthreads();
    return m;
  }
  if (m <= SEL_RANK_MAX) {
    rank_sort_entries(src, list, list + cap, m);
  } else {
    int n2 = 1;
    while (n2 < m) n2 <<= 1;
    for (int i = m + tid; i < n2; i += nt) {
      Entry s;
      s.key = 0;
      s.idx = SENTINEL_IDX;
      s.aux = 0;
      list[i] = s;
    }
    __syncthreads();
    bitonic_sort_entries(src, list, n2);
  }
  return m < K ? m : K;
}

}  // namespace rpk
