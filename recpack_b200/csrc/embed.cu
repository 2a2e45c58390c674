// Item neighbours of a dense embedding matrix E [I x D] (float64): per item row i the K largest stored values of
// s_ij over the columns j != i, where s is the float64 dot product (RPK_SIM_DOT) or the dot product of the
// L2-normalised rows (RPK_SIM_COSINE), each the left fold over d of fl(x_id * x_jd) without FMA contraction
// (DESIGN.md 2, "Embedding neighbours").  This is what Prod2Vec builds from cosine_similarity + get_top_K_values, and
// what users build from any item-factor matrix.
//
// The I x I product never reaches HBM:
//   1. k_embed_norms / k_embed_prep   canonical norms and normalised rows (float64, kept for step 4); the screen
//                                     operand: rows scaled by one power of two (largest row norm in [1, 2)), rounded
//                                     to tf32, K-major, padded to the TMA box; per-row norms r_i of the scaled rows
//   2. k_embed_screen                 tcgen05.mma kind::tf32 (M 128, N 256, K 8), fp32 accumulators double-buffered in
//                                     TMEM, warp roles as in gram_tc.cu.  The epilogue compares every element against
//                                     its row's threshold and appends the rare survivor (column, s^) to the row's
//                                     candidate buffer.
//   3. k_embed_compact                columns are screened in chunks of doubling width; after each chunk the row's
//                                     threshold tau'_i rises to the K-th largest certain lower bound s^ - delta in the
//                                     buffer and the buffer is cut to the entries that can still reach it
//   4. k_embed_exact                  the survivors are rescored in the canonical float64 fold and selected with
//                                     block_select_topk; rows whose buffer overflowed, or whose stored values do not
//                                     prove the cut (exact zeros), go to k_embed_exact_rows, which scores the whole row
//                                     in float64.
// The screen bound |s^_ij - s_ij| <= delta_ij = eps_D r_i r_j + beta (scaled units) is derived in DESIGN.md 4.9.
//
// Factor models (DESIGN.md 2, "Factor models"; 4.10) run the same pipeline with two operands: the screened rows are
// the user factors P of the users with history (a row map compacted on the device from indptr), the columns the item
// factors Q, each with its own scale.  Instead of j != i a column must be eligible: not in the user's history (when
// masked) and allowed by the item filter.  The screen epilogue never appends an ineligible column, so it never counts
// toward tau' and never reaches a list; k_embed_exact_rows zeroes the same columns.  The mode is a template argument
// of the two kernels that test eligibility, so the embedding instantiations are the code they were.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "internal.h"
#include "select.cuh"
#include "tc.cuh"

namespace rpk {

constexpr int EB_BM = 128;          // UMMA M
constexpr int EB_BN = 256;          // UMMA N
constexpr int EB_BK = 32;           // tf32 elements per k-block: one 128 B swizzle atom row
constexpr int EB_UMMA_K = 8;        // tf32 elements per tcgen05.mma
constexpr int EB_STAGES = 4;
constexpr int EB_A_BYTES = EB_BM * EB_BK * 4;  // 16 KB
constexpr int EB_B_BYTES = EB_BN * EB_BK * 4;  // 32 KB
constexpr int EB_STAGE_BYTES = EB_A_BYTES + EB_B_BYTES;
constexpr uint32_t EB_TMEM_COLS = 512;
constexpr int EB_THREADS = 192;     // TMA warp, MMA warp, 4 epilogue warps
constexpr size_t EB_SMEM = (size_t)EB_STAGES * EB_STAGE_BYTES + 1024 + 256;
constexpr int EB_SEL_NT = 256;
constexpr int64_t EB_BUF_BYTES = (int64_t)1 << 30;  // candidate buffers of one row group

enum { EC_CAND, EC_COMPACT, EC_OVERFLOW, EC_ZERO, EC_EXACT, EC_MASKED, EC_N };

// Instruction descriptor: dense, D = F32, A = B = TF32, both K-major, N, M.
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Larger key = larger value (no NaN reaches these).
__device__ __forceinline__ u64 okey_f64(double v) {
  const u64 b = (u64)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double from_okey_f64(u64 k) {
  const u64 b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}
__device__ __forceinline__ uint32_t okey_f32(float v) {
  const uint32_t b = __float_as_uint(v);
  return (b >> 31) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float from_okey_f32(uint32_t k) { return __uint_as_float((k >> 31) ? (k & 0x7fffffffu) : ~k); }

// The canonical value: left fold over d of fl(a_d * b_d), separate multiply and add.
__device__ __forceinline__ double dot_fold(const double* a, const double* __restrict__ b, int D) {
  double s = __dmul_rn(a[0], b[0]);
  for (int d = 1; d < D; ++d) s = __dadd_rn(s, __dmul_rn(a[d], b[d]));
  return s;
}

// ------------------------------------------------------------------------------------------
// 1. Prep
// ------------------------------------------------------------------------------------------
// One thread per row: the fold of squares; cosine rows are normalised into xhat (n_i == 0 leaves the row as it is,
// which is all zeros).  flags[0] = 1 on a non-finite value; stats[0] / stats[1] = bit patterns of the largest
// squared norm of the rows used by the screen and of the largest |x_id|.
__global__ void k_embed_norms(const double* __restrict__ E, int64_t I, int D, int cosine, double* __restrict__ xhat,
                              int* __restrict__ flags, u64* __restrict__ stats) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < I; i += (int64_t)gridDim.x * blockDim.x) {
    const double* e = E + i * D;
    bool finite = true;
    double ss = __dmul_rn(e[0], e[0]);
    finite &= isfinite(e[0]);
    for (int d = 1; d < D; ++d) {
      finite &= isfinite(e[d]);
      ss = __dadd_rn(ss, __dmul_rn(e[d], e[d]));
    }
    if (!finite) {
      flags[0] = 1;
      continue;
    }
    double q = ss, amax = 0.0;
    if (cosine) {
      const double n = __dsqrt_rn(ss);
      double* o = xhat + i * D;
      q = 0.0;
      for (int d = 0; d < D; ++d) {
        const double v = n != 0.0 ? __ddiv_rn(e[d], n) : e[d];
        o[d] = v;
        q = __dadd_rn(q, __dmul_rn(v, v));
        amax = fmax(amax, fabs(v));
      }
    } else {
      for (int d = 0; d < D; ++d) amax = fmax(amax, fabs(e[d]));
    }
    atomicMax(&stats[0], (u64)__double_as_longlong(q));  // non-negative doubles order as their bit patterns
    atomicMax(&stats[1], (u64)__double_as_longlong(amax));
  }
}

// One thread per row: the tf32 screen row of 2^sigma x_i (values below the fp32 normal range flushed to 0, which the
// bound's absolute term covers), r_i >= ||2^sigma x_i|| and c_i >= eps_D r_i, both rounded up.  Row i of the operand is
// row rows[i] of X (rows null: row i); cr null: not needed (the column operand of a factor model).
__global__ void k_embed_prep(const double* __restrict__ X, const int* __restrict__ rows, int64_t I, int D, int sigma,
                             double eps, int kd_pad, float* __restrict__ A, float* __restrict__ r, float* __restrict__ cr) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < I; i += (int64_t)gridDim.x * blockDim.x) {
    const double* x = X + (rows ? (int64_t)rows[i] : i) * D;
    float* a = A + i * kd_pad;
    double q = 0.0;
    for (int d = 0; d < D; ++d) {
      const double u = ldexp(x[d], sigma);
      q = __dadd_ru(q, __dmul_ru(u, u));
      float f = __double2float_rn(u);
      if (fabsf(f) < 1.17549435e-38f) f = 0.f;
      uint32_t t;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(f));
      a[d] = __uint_as_float(t);
    }
    const double rr = __dmul_ru(__dsqrt_ru(q), 1.0 + 0x1p-40);
    r[i] = __double2float_ru(rr);
    if (cr) cr[i] = __double2float_ru(__dmul_ru(eps, (double)r[i]));
  }
}

// One warp per user of a factor model's X: checks the CSR row (ascending unique columns in [0, I)) -> flags[1], and
// appends every user with history to row_map (null: not wanted) through the counter flags[2].  The order of row_map
// does not matter: a screened row writes its list to its own user's row.
__global__ void k_factor_rows(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, int64_t U, int64_t I,
                              int64_t nnz, int* __restrict__ row_map, int* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < U; u += warps) {
    const int64_t a = indptr[u], b = indptr[u + 1];
    if (a < 0 || b < a || b > nnz) {
      if (lane == 0) flags[1] = 1;
      continue;
    }
    bool bad = false;
    for (int64_t k = a + lane; k < b; k += 32) {
      const int j = indices[k];
      bad |= j < 0 || j >= I || (k > a && indices[k - 1] >= j);
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) flags[1] = 1;
    if (row_map && b > a && lane == 0) row_map[atomicAdd(&flags[2], 1)] = (int)u;
  }
}

// ------------------------------------------------------------------------------------------
// 2. Screen GEMM
// ------------------------------------------------------------------------------------------
struct ScreenParams {
  int m_tiles, n_tiles, k_blocks;
  int row0;          // first screened row (any value; tiles of 128 rows from here)
  int row_end;       // rows >= row_end are not screened
  int col0;          // first column of the chunk (multiple of 256)
  int col_end;       // columns >= col_end are not screened
  const float* r;    // [column rows_alloc] scaled norms of the column operand, zero past I
  const float* cr;   // [screened rows] eps_D * r_i of the row operand
  const float* tau_e;  // [group rows] epilogue threshold
  int* cnt;          // [group rows] appends (may exceed cap: overflow)
  int2* buf;         // [group rows x cap] (column, float bits of s^)
  int cap;
  float* S;          // verification: every s^ * unscale, [row_end - row0 x lds]; null in the screen
  int64_t lds;
  float unscale;
};

// Factor models: screened row l is user row_map[l]; a column is screened only when it is eligible.
struct FactorScreenParams : ScreenParams {
  const int* row_map;
  const int64_t* hist_ptr;        // the users' sorted histories (CSR of X); null: the history is not masked
  const int32_t* hist_idx;
  const unsigned char* allowed;   // item filter (1 = may be recommended); null: none
  u64* prof;                      // RPK_PHASE_PROF builds: EC_* counters
};

template <bool FACTOR>
using ScreenParamsOf = typename std::conditional<FACTOR, FactorScreenParams, ScreenParams>::type;

template <bool FACTOR>
__global__ void __launch_bounds__(EB_THREADS, 1)
k_embed_screen(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, ScreenParamsOf<FACTOR> p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* smem_a = smem;
  unsigned char* smem_b = smem + (size_t)EB_STAGES * EB_A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)EB_STAGES * EB_STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + EB_STAGES;
  uint64_t* tmem_full = bars + 2 * EB_STAGES;
  uint64_t* tmem_empty = bars + 2 * EB_STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * EB_STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles_total = p.m_tiles * p.n_tiles;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    for (int s = 0; s < EB_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(EB_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // TMA producer
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < n_tiles_total; t += gridDim.x) {
        const int m_blk = t / p.n_tiles, n_blk = t % p.n_tiles;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], EB_STAGE_BYTES);
          tma_load_2d(smem_a + (size_t)stage * EB_A_BYTES, &map_a, &full_bar[stage], kb * EB_BK, p.row0 + m_blk * EB_BM);
          tma_load_2d(smem_b + (size_t)stage * EB_B_BYTES, &map_b, &full_bar[stage], kb * EB_BK, p.col0 + n_blk * EB_BN);
          if (++stage == EB_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // MMA issuer
      constexpr uint32_t idesc = umma_idesc_tf32(EB_BM, EB_BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < n_tiles_total; t += gridDim.x) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)acc * EB_BN;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t da = umma_desc_kmajor_sw128(smem_u32(smem_a + (size_t)stage * EB_A_BYTES));
          const uint64_t db = umma_desc_kmajor_sw128(smem_u32(smem_b + (size_t)stage * EB_B_BYTES));
#pragma unroll
          for (int k = 0; k < EB_BK / EB_UMMA_K; ++k)  // 32 B along K per MMA: +2 in 16 B units
            umma_tf32(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          if (++stage == EB_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&tmem_full[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // epilogue: lane = one row of the tile, 32 columns per tcgen05.ld
    const int quarter = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = blockIdx.x; t < n_tiles_total; t += gridDim.x) {
      const int m_blk = t / p.n_tiles, n_blk = t % p.n_tiles;
      const int row = p.row0 + m_blk * EB_BM + quarter * 32 + lane;
      const bool valid = row < p.row_end;
      const int l = row - p.row0;
      float te = INFINITY, ci = 0.f;
      if (valid && !p.S) {
        te = p.tau_e[l];
        ci = p.cr[row];
      }
      // factor models: the lane's cursor into its user's history, at the first item of this tile (binary search)
      int64_t hc = 0, he = 0;
      if constexpr (FACTOR) {
        if (valid && p.hist_ptr) {
          const int u = p.row_map[row];
          int64_t lo = p.hist_ptr[u], hi = p.hist_ptr[u + 1];
          he = hi;
          const int c0 = p.col0 + n_blk * EB_BN;
          while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (p.hist_idx[mid] < c0) lo = mid + 1;
            else hi = mid;
          }
          hc = lo;
        }
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < EB_BN / 32; ++c) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * EB_BN + c * 32);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
              "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
              "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
              "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const int colbase = p.col0 + n_blk * EB_BN + c * 32;
        if (p.S) {
          if (valid) {
            float* o = p.S + (int64_t)l * p.lds + colbase;
#pragma unroll
            for (int k = 0; k < 32; ++k)
              if (colbase + k < p.col_end) o[k] = __uint_as_float(v[k]) * p.unscale;
          }
          continue;
        }
        const float rj = p.r[colbase + lane];
        uint32_t mask = 0;
        if constexpr (FACTOR) {
          // eligible columns of this group of 32: in range and allowed (one byte per column, as r_j), minus the history
          const int colj = colbase + lane;
          const uint32_t in_range = __ballot_sync(0xffffffffu, colj < p.col_end);
          uint32_t ok = __ballot_sync(0xffffffffu, colj < p.col_end && (!p.allowed || p.allowed[colj]));
          for (; hc < he; ++hc) {
            const int j = p.hist_idx[hc];
            if (j >= colbase + 32) break;
            ok &= ~(1u << (j - colbase));
          }
#pragma unroll
          for (int k = 0; k < 32; ++k) {
            const float rk = __shfl_sync(0xffffffffu, rj, k);
            mask |= (uint32_t)(__fmaf_ru(ci, rk, __uint_as_float(v[k])) >= te) << k;
          }
#ifdef RPK_PHASE_PROF
          const uint32_t skipped = mask & in_range & ~ok;
          if (skipped) atomicAdd(&p.prof[EC_MASKED], (u64)__popc(skipped));
#endif
          (void)in_range;
          mask &= ok;
        } else {
#pragma unroll
          for (int k = 0; k < 32; ++k) {
            const float rk = __shfl_sync(0xffffffffu, rj, k);
            const int col = colbase + k;
            const bool pass = __fmaf_ru(ci, rk, __uint_as_float(v[k])) >= te && col < p.col_end && col != row;
            mask |= (uint32_t)pass << k;
          }
        }
        if (mask) {  // rare after the first chunk: one atomic per (row, 32 columns)
          int pos = atomicAdd(&p.cnt[l], __popc(mask));
          int2* dst = p.buf + (int64_t)l * p.cap;
#pragma unroll
          for (int k = 0; k < 32; ++k) {  // static indices keep v[] in registers
            if ((mask >> k) & 1u) {
              if (pos < p.cap) dst[pos] = make_int2(colbase + k, (int)v[k]);
              ++pos;
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(EB_TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------
// 3. Compaction: raise tau'_i, cut the buffer
// ------------------------------------------------------------------------------------------
struct RowState {
  int row0, rows;     // the row group: global rows row0 .. row0 + rows - 1
  int K, cap;
  float beta;         // absolute term of the bound (scaled units), rounded up; may be +inf
  const float* r;     // column operand's scaled norms
  const float* cr;    // row operand's eps_D * r_i, by screened row
  float* tau_p;       // tau'_i: K columns of the row certainly have scaled s >= tau'_i (-inf: none known)
  float* tau_e;       // tau'_i - beta rounded down, the threshold of the screen's test (+inf: row overflowed)
  int* cnt;
  int2* buf;
  int* over;          // 1: the buffer overflowed, the row is scored by k_embed_exact_rows
  u64* prof;          // RPK_PHASE_PROF builds: EC_* counters
};

__global__ void k_embed_init(RowState s) {
  for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < s.rows; l += gridDim.x * blockDim.x) {
    s.tau_p[l] = -INFINITY;
    s.tau_e[l] = -INFINITY;
    s.cnt[l] = 0;
    s.over[l] = 0;
  }
}

// One CTA per row.  The K-th largest lower bound L_k = s^_k - delta_ik (rounded down) by a 4 x 8-bit radix select.
__global__ void __launch_bounds__(EB_SEL_NT) k_embed_compact(RowState s) {
  extern __shared__ __align__(16) unsigned char smem[];
  int2* ent = reinterpret_cast<int2*>(smem);
  uint32_t* keys = reinterpret_cast<uint32_t*>(ent + s.cap);
  __shared__ int hist[256];
  __shared__ int sh_need, sh_kept;
  __shared__ uint32_t sh_prefix;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int l = blockIdx.x; l < s.rows; l += gridDim.x) {
    if (s.over[l]) continue;
    const int n = s.cnt[l];
    if (n > s.cap) {
      if (tid == 0) {
        s.over[l] = 1;
        s.tau_e[l] = INFINITY;
#ifdef RPK_PHASE_PROF
        atomicAdd(&s.prof[EC_OVERFLOW], 1ull);
#endif
      }
      continue;
    }
    const int row = s.row0 + l;
    const float ci = s.cr[row];
    const int2* b = s.buf + (int64_t)l * s.cap;
    for (int k = tid; k < n; k += nt) {
      const int2 e = b[k];
      ent[k] = e;
      keys[k] = okey_f32(__fsub_rd(__int_as_float(e.y), __fadd_ru(__fmul_ru(ci, s.r[e.x]), s.beta)));
    }
    __syncthreads();
    float tp = s.tau_p[l];
    if (n >= s.K) {
      uint32_t prefix = 0, pmask = 0;
      if (tid == 0) sh_need = s.K;
      for (int shift = 24; shift >= 0; shift -= 8) {
        for (int q = tid; q < 256; q += nt) hist[q] = 0;
        __syncthreads();
        for (int k = tid; k < n; k += nt)
          if ((keys[k] & pmask) == prefix) atomicAdd(&hist[(keys[k] >> shift) & 255], 1);
        __syncthreads();
        if (tid < 32) {  // lane q holds bins 255 - 8q .. 248 - 8q (from the top)
          int sum = 0;
          for (int t = 0; t < 8; ++t) sum += hist[255 - 8 * tid - t];
          int incl = sum;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, o);
            if (tid >= o) incl += y;
          }
          const int need = sh_need;
          const unsigned hit = __ballot_sync(0xffffffffu, incl >= need);
          const int q = __ffs(hit) - 1;
          if (tid == q) {
            int acc = incl - sum;
            for (int t = 0; t < 8; ++t) {
              const int bin = 255 - 8 * q - t;
              if (acc + hist[bin] >= need) {
                sh_need = need - acc;
                sh_prefix = prefix | ((uint32_t)bin << shift);
                break;
              }
              acc += hist[bin];
            }
          }
        }
        __syncthreads();
        prefix = sh_prefix;
        pmask |= 255u << shift;
      }
      tp = fmaxf(tp, from_okey_f32(prefix));
    }
    const float te = __fsub_rd(tp, s.beta);
    if (tid == 0) sh_kept = 0;
    __syncthreads();
    int2* bw = s.buf + (int64_t)l * s.cap;
    for (int k = tid; k < n; k += nt) {
      const int2 e = ent[k];
      if (__fmaf_ru(ci, s.r[e.x], __int_as_float(e.y)) >= te) bw[atomicAdd(&sh_kept, 1)] = e;
    }
    __syncthreads();
    if (tid == 0) {
      s.cnt[l] = sh_kept;
      s.tau_p[l] = tp;
      s.tau_e[l] = te;
#ifdef RPK_PHASE_PROF
      atomicAdd(&s.prof[EC_COMPACT], 1ull);
#endif
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// 4. Exact pass
// ------------------------------------------------------------------------------------------
// Candidates: float64 values of slots 0..ns-1 (column = col[slot], or the slot itself); exact zeros are not stored.
struct EmbedSrc {
  const double* val;
  const int* col;
  int ns;
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
      const double v = val[slot];
      if (v != 0.0) f(slot, okey_f64(v));
    }
  }
  template <class F>
  __device__ __forceinline__ void for_each(F f) const { visit(f, 1); }
  template <class F>
  __device__ __forceinline__ void for_each_sampled(F f) const { visit(f, SEL_SAMPLE); }
  __device__ __forceinline__ void entry(int slot, Entry& e) const {
    e.key = okey_f64(val[slot]);
    e.idx = col ? col[slot] : slot;
    e.aux = 0;
  }
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const {
    if (a.key != b.key) return a.key > b.key ? 1 : -1;
    return 0;
  }
};

struct ExactParams {
  RowState s;
  const double* X;    // [I x D] the rows of the definition (xhat or E); factor models: P [U x D]
  int64_t I;
  int D, sigma2;      // sigma_row + sigma_col: scaled s = s * 2^sigma2
  int sel_cap, direct_cap;
  int64_t out_row0;   // output row of group row 0 (embeddings)
  int* out_idx;
  double* out_val;
  int* out_len;
  int* handoff;       // [group rows] rows for k_embed_exact_rows
  int* n_handoff;
  double* scratch;    // k_embed_exact_rows: [gridDim.x x I]
};

// Factor models: the columns are Q, screened row l is user row_map[l] (its row of P and its output row).
struct FactorExactParams : ExactParams {
  const double* Xc;   // [I x D] Q
  const int* row_map;
  const int64_t* hist_ptr;        // as in FactorScreenParams
  const int32_t* hist_idx;
  const unsigned char* allowed;
};

template <bool FACTOR>
using ExactParamsOf = typename std::conditional<FACTOR, FactorExactParams, ExactParams>::type;

template <bool FACTOR>
__device__ __forceinline__ const double* exact_cols(const ExactParamsOf<FACTOR>& p) {
  if constexpr (FACTOR) return p.Xc;
  else return p.X;
}

__device__ __forceinline__ void write_list(const ExactParams& p, int l, const Entry* list, int m) {
  const int64_t o = (p.out_row0 + l) * (int64_t)p.s.K;
  for (int t = threadIdx.x; t < p.s.K; t += blockDim.x) {
    p.out_idx[o + t] = t < m ? list[t].idx : -1;
    if (p.out_val) p.out_val[o + t] = t < m ? from_okey_f64(list[t].key) : 0.0;
  }
  if (threadIdx.x == 0) p.out_len[p.out_row0 + l] = m;
}

// Factor models: the list of group row l goes to its user's row.
__device__ __forceinline__ void write_list(const FactorExactParams& p, int l, const Entry* list, int m) {
  const int64_t u = p.row_map[p.s.row0 + l];
  const int64_t o = u * (int64_t)p.s.K;
  for (int t = threadIdx.x; t < p.s.K; t += blockDim.x) {
    p.out_idx[o + t] = t < m ? list[t].idx : -1;
    if (p.out_val) p.out_val[o + t] = t < m ? from_okey_f64(list[t].key) : 0.0;
  }
  if (threadIdx.x == 0) p.out_len[u] = m;
}

template <bool FACTOR>
__global__ void __launch_bounds__(EB_SEL_NT) k_embed_exact(ExactParamsOf<FACTOR> p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.sel_cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + SEL_BINS);
  double* xi = reinterpret_cast<double*>(smem + sel_smem_bytes(p.sel_cap));
  double* val = xi + p.D;
  int* col = reinterpret_cast<int*>(val + p.s.cap);
  const int tid = threadIdx.x, nt = blockDim.x;
  const RowState& s = p.s;
  for (int l = blockIdx.x; l < s.rows; l += gridDim.x) {
    bool handoff = s.over[l] != 0;
    if (!handoff) {
      const int row = s.row0 + l;
      const int n = s.cnt[l];
      if constexpr (FACTOR) {
        for (int d = tid; d < p.D; d += nt) xi[d] = p.X[(int64_t)p.row_map[row] * p.D + d];
      } else {
        for (int d = tid; d < p.D; d += nt) xi[d] = p.X[(int64_t)row * p.D + d];
      }
      __syncthreads();
      const int2* b = s.buf + (int64_t)l * s.cap;
      for (int k = tid; k < n; k += nt) {
        const int j = b[k].x;
        col[k] = j;
        val[k] = dot_fold(xi, exact_cols<FACTOR>(p) + (int64_t)j * p.D, p.D);
      }
      __syncthreads();
#ifdef RPK_PHASE_PROF
      if (tid == 0) atomicAdd(&s.prof[EC_CAND], (u64)n);
#endif
      EmbedSrc src{val, col, n};
      const int m = block_select_topk(src, s.K, list, p.sel_cap, p.direct_cap, hist, sh);
      // Every column outside the buffer has scaled s < tau'.  The lists are final when K stored values reach it.
      const float tp = s.tau_p[l];
      handoff = tp != -INFINITY && (m < s.K || !(ldexp(from_okey_f64(list[s.K - 1].key), p.sigma2) > (double)tp));
      if (!handoff) write_list(p, l, list, m);
#ifdef RPK_PHASE_PROF
      if (handoff && tid == 0) atomicAdd(&s.prof[EC_ZERO], 1ull);
#endif
    }
    if (handoff && tid == 0) p.handoff[atomicAdd(p.n_handoff, 1)] = l;
    __syncthreads();
  }
}

// One CTA per handed-over row: every column in the canonical fold, then the same selection.  A column that is not
// eligible (j == i for embeddings; history or filtered item for factor models) gets 0.0, which is never listed.
template <bool FACTOR>
__global__ void __launch_bounds__(EB_SEL_NT) k_embed_exact_rows(ExactParamsOf<FACTOR> p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.sel_cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + SEL_BINS);
  double* xi = reinterpret_cast<double*>(smem + sel_smem_bytes(p.sel_cap));
  double* acc = p.scratch + (int64_t)blockIdx.x * p.I;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int nh = *p.n_handoff;
  for (int h = blockIdx.x; h < nh; h += gridDim.x) {
    const int l = p.handoff[h];
    const int row = p.s.row0 + l;
    if constexpr (FACTOR) {
      const int64_t u = p.row_map[row];
      for (int d = tid; d < p.D; d += nt) xi[d] = p.X[u * p.D + d];
      __syncthreads();
      for (int64_t j = tid; j < p.I; j += nt) acc[j] = (!p.allowed || p.allowed[j]) ? dot_fold(xi, p.Xc + j * p.D, p.D) : 0.0;
      __syncthreads();
      if (p.hist_ptr)
        for (int64_t k = p.hist_ptr[u] + tid; k < p.hist_ptr[u + 1]; k += nt) acc[p.hist_idx[k]] = 0.0;
    } else {
      for (int d = tid; d < p.D; d += nt) xi[d] = p.X[(int64_t)row * p.D + d];
      __syncthreads();
      for (int64_t j = tid; j < p.I; j += nt) acc[j] = j == row ? 0.0 : dot_fold(xi, p.X + j * p.D, p.D);
    }
    __syncthreads();
    EmbedSrc src{acc, nullptr, (int)p.I};
    const int m = block_select_topk(src, p.s.K, list, p.sel_cap, p.direct_cap, hist, sh);
    write_list(p, l, list, m);
#ifdef RPK_PHASE_PROF
    if (tid == 0) atomicAdd(&p.s.prof[EC_EXACT], 1ull);
#endif
    __syncthreads();
  }
}


// ------------------------------------------------------------------------------------------
// 5. Full scores of a factor model (rpk_factor_full)
// ------------------------------------------------------------------------------------------
// One 64 x 64 tile of (user, item) per CTA, 256 threads with 4 x 4 scores each; the fold runs over d in order through
// shared-memory slices of 16.  Users without history and filtered items get 0.0.
constexpr int FF_T = 64, FF_DK = 16;

__global__ void __launch_bounds__(256) k_factor_full(const double* __restrict__ P, const double* __restrict__ Q,
                                                     const int64_t* __restrict__ indptr, int64_t U, int64_t I, int D,
                                                     const unsigned char* __restrict__ allowed, double* __restrict__ out) {
  __shared__ double ps[FF_DK][FF_T + 1], qs[FF_DK][FF_T + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t j0 = (int64_t)blockIdx.x * FF_T;
  for (int64_t ub = blockIdx.y; ub * FF_T < U; ub += gridDim.y) {
    const int64_t u0 = ub * FF_T;
    double acc[4][4];
    for (int d0 = 0; d0 < D; d0 += FF_DK) {
      for (int t = threadIdx.x; t < FF_DK * FF_T; t += blockDim.x) {
        const int r = t / FF_DK, dd = t % FF_DK;
        const int64_t u = u0 + r, j = j0 + r;
        const bool din = d0 + dd < D;
        ps[dd][r] = (u < U && din) ? P[u * D + d0 + dd] : 0.0;
        qs[dd][r] = (j < I && din) ? Q[j * D + d0 + dd] : 0.0;
      }
      __syncthreads();
      const int dn = min(FF_DK, D - d0);
      for (int dd = 0; dd < dn; ++dd) {
        double a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          a[i] = ps[dd][ty + 16 * i];
          b[i] = qs[dd][tx + 16 * i];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const double pr = __dmul_rn(a[i], b[k]);
            acc[i][k] = d0 + dd == 0 ? pr : __dadd_rn(acc[i][k], pr);
          }
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t u = u0 + ty + 16 * i;
      if (u >= U) continue;
      const bool has = indptr[u + 1] > indptr[u];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int64_t j = j0 + tx + 16 * k;
        if (j < I) out[u * I + j] = has && (!allowed || allowed[j]) ? acc[i][k] : 0.0;
      }
    }
  }
}

// One warp per user: the history columns of the full scores become 0.0.
__global__ void k_factor_mask_history(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, int64_t U,
                                      int64_t I, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < U; u += warps)
    for (int64_t k = indptr[u] + lane; k < indptr[u + 1]; k += 32) out[u * I + indices[k]] = 0.0;
}

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
struct ScreenOperand {
  const double* X;   // rows of the definition
  float* A;          // screen operand [rows_alloc x kd_pad]
  float* r;          // [rows_alloc]
  float* cr;         // [rows_alloc]; null for a column operand of its own
  int sigma;
  int64_t rows_alloc;
};

struct EmbedPrep {
  ScreenOperand row, col;  // one operand twice for embeddings
  int kd_pad;
  double eps, beta;
};

static int next_pow2_(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// sigma from the largest squared row norm and the largest |x_id| (bit patterns as k_embed_norms leaves them): the
// largest row norm of 2^sigma x in [1, 2); from the largest |x_id| when the squared norms underflow
static int screen_sigma(const int* stats) {
  u64 b0, b1;
  memcpy(&b0, stats, 8);
  memcpy(&b1, stats + 2, 8);
  double maxq, maxabs;
  memcpy(&maxq, &b0, 8);
  memcpy(&maxabs, &b1, 8);
  int ex = 0;
  if (maxq >= 0x1p-1000) {
    frexp(sqrt(maxq), &ex);
    return 1 - ex;
  }
  if (maxabs > 0.0) {
    frexp(maxabs, &ex);
    return 1 - ex;
  }
  return 0;
}

static double stat_maxq(const int* stats) {
  double q;
  memcpy(&q, stats, 8);
  return q;
}

// The tf32 screen operand of n rows of X (row i = X row rows[i], or i when rows is null).
static ScreenOperand build_operand(rpk_ctx* c, const double* X, const int* rows, int64_t n, int D, int sigma, double eps,
                                   int kd_pad, bool want_cr, const char* a_name, const char* r_name, const char* cr_name) {
  cudaStream_t st = c->stream;
  ScreenOperand o;
  o.X = X;
  o.sigma = sigma;
  o.rows_alloc = (n + EB_BN - 1) / EB_BN * EB_BN + EB_BN;  // every TMA box lies inside the operand
  o.A = c->buf<float>(a_name, (size_t)o.rows_alloc * kd_pad);
  o.r = c->buf<float>(r_name, (size_t)o.rows_alloc);
  o.cr = want_cr ? c->buf<float>(cr_name, (size_t)o.rows_alloc) : nullptr;
  RPK_CUDA(cudaMemsetAsync(o.A, 0, sizeof(float) * (size_t)o.rows_alloc * kd_pad, st));
  RPK_CUDA(cudaMemsetAsync(o.r, 0, sizeof(float) * (size_t)o.rows_alloc, st));
  if (n > 0) {
    const int grid = (int)std::min<int64_t>((n + 127) / 128, (int64_t)c->sm_count * 8);
    k_embed_prep<<<grid, 128, 0, st>>>(X, rows, n, D, sigma, eps, kd_pad, o.A, o.r, o.cr);
    RPK_LAUNCH_CHECK(c);
  }
  return o;
}

// DESIGN.md 4.9 / 4.10: tf32 operands (2^-11 + 2^-23 relative each), exact products, D truncating fp32 additions and
// the float64 fold of the definition; beta: flushed operands, products and sums below 2^-126 (scaled units, where
// every element is below 2), and the fold's underflow, (2D + 2) 2^-1074 in the units of s, times 2^(sigma_r + sigma_c)
static void set_bound(EmbedPrep& q, int D) {
  q.eps = 0x1p-10 + (double)(D + 2) * 0x1p-22;
  q.beta = 0x1p-100 + ldexp((double)(2 * D + 2), q.row.sigma + q.col.sigma - 1074);
}

static void launch_norms(rpk_ctx* c, const double* X, int64_t n, int D, int cosine, double* xhat, int* flags, int* stats) {
  if (n == 0) return;
  const int grid = (int)std::min<int64_t>((n + 127) / 128, (int64_t)c->sm_count * 8);
  k_embed_norms<<<grid, 128, 0, c->stream>>>(X, n, D, cosine, xhat, flags, reinterpret_cast<u64*>(stats));
  RPK_LAUNCH_CHECK(c);
}

// Validates E (synchronises once: NaN / inf and the range checks are reported by this call) and builds the operand.
static EmbedPrep embed_prep(rpk_ctx* c, int64_t I, int D, const double* E_u, int similarity) {
  RPK_REQUIRE(I >= 1 && I < ((int64_t)1 << 24), "embedding: I must be in [1, 2^24)");
  RPK_REQUIRE(D >= 1 && D <= 1024, "embedding: D must be in [1, 1024]");
  RPK_REQUIRE(similarity == RPK_SIM_COSINE || similarity == RPK_SIM_DOT, "embedding: similarity must be cosine or dot");
  cudaStream_t st = c->stream;
  const double* E = stage_in(c, E_u, (size_t)I * D, "eb_E_in");
  const bool cosine = similarity == RPK_SIM_COSINE;
  double* xhat = cosine ? c->buf<double>("eb_xhat", (size_t)I * D) : nullptr;
  int* flags = c->buf<int>("eb_flags", 8);
  RPK_CUDA(cudaMemsetAsync(flags, 0, 8 * sizeof(int), st));
  c->mark("embed: start");
  launch_norms(c, E, I, D, cosine ? 1 : 0, xhat, flags, flags + 2);
  int h[6];
  RPK_CUDA(cudaMemcpyAsync(h, flags, sizeof(h), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaStreamSynchronize(st));
  RPK_REQUIRE(h[0] == 0, "embedding: E contains NaN or inf");
  // dot: |partial sums| <= ||e_i|| ||e_j|| (up to rounding) stay finite
  RPK_REQUIRE(cosine || stat_maxq(h + 2) < 0x1p1020, "embedding: dot similarity needs every squared row norm below 2^1020");
  EmbedPrep q;
  q.kd_pad = (D + EB_BK - 1) / EB_BK * EB_BK;
  const int sigma = screen_sigma(h + 2);
  q.eps = 0x1p-10 + (double)(D + 2) * 0x1p-22;
  q.row = build_operand(c, cosine ? xhat : E, nullptr, I, D, sigma, q.eps, q.kd_pad, true, "eb_A", "eb_r", "eb_cr");
  q.col = q.row;
  set_bound(q, D);
  c->mark("embed: prep");
  return q;
}

static void encode_maps(const EmbedPrep& q, CUtensorMap* map_a, CUtensorMap* map_b) {
  const cuuint64_t dims_a[2] = {(cuuint64_t)q.kd_pad, (cuuint64_t)q.row.rows_alloc};
  const cuuint64_t dims_b[2] = {(cuuint64_t)q.kd_pad, (cuuint64_t)q.col.rows_alloc};
  const cuuint64_t strides[1] = {(cuuint64_t)q.kd_pad * 4};
  const cuuint32_t box_a[2] = {EB_BK, EB_BM}, box_b[2] = {EB_BK, EB_BN}, estr[2] = {1, 1};
  EncodeTiledFn enc = get_encode_tiled();
  CUresult r1 = enc(map_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, q.row.A, dims_a, strides, box_a, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CUresult r2 = enc(map_b, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, q.col.A, dims_b, strides, box_b, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RPK_REQUIRE(r1 == CUDA_SUCCESS && r2 == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed");
}

template <bool FACTOR>
static void launch_screen(rpk_ctx* c, const CUtensorMap& map_a, const CUtensorMap& map_b, const ScreenParamsOf<FACTOR>& sp) {
  RPK_REQUIRE(EB_SMEM <= (size_t)c->smem_max, "embedding screen: shared memory ring does not fit");
  RPK_CUDA(cudaFuncSetAttribute(k_embed_screen<FACTOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EB_SMEM));
  const int grid = std::max(1, std::min(c->sm_count, sp.m_tiles * sp.n_tiles));
  k_embed_screen<FACTOR><<<grid, EB_THREADS, EB_SMEM, c->stream>>>(map_a, map_b, sp);
  RPK_LAUNCH_CHECK(c);
}

template <bool FACTOR>
static ScreenParamsOf<FACTOR> screen_params() {
  ScreenParamsOf<FACTOR> sp;
  memset(&sp, 0, sizeof(sp));
  sp.unscale = 1.f;
  return sp;
}

// What a top-K call screens and where its lists go.
struct TopkJob {
  int64_t I;                      // columns
  int D, K;
  int64_t row_begin, row_end;     // screened rows
  int64_t out_row0;               // embeddings: output row of screened row row_begin
  const int* row_map;             // factor models: the user of each screened row
  const int64_t* hist_ptr;        // factor models: histories to mask (null: none)
  const int32_t* hist_idx;
  const unsigned char* allowed;   // factor models: item filter (null: none)
  int32_t* out_idx;               // device outputs
  double* out_val;
  int32_t* out_len;
  int64_t n_users;                // factor models: rows of the outputs (for the counters line)
};

// Steps 2-4 of the file comment for the rows [row_begin, row_end) of the row operand against every column.
template <bool FACTOR>
static void screen_topk(rpk_ctx* c, const EmbedPrep& q, const TopkJob& job) {
  cudaStream_t st = c->stream;
  const int64_t I = job.I;
  const int D = job.D, K = job.K;
  const int64_t rows = job.row_end - job.row_begin;
  const char* m_chunk = FACTOR ? "factor: screen chunk" : "embed: screen chunk";
  const char* m_compact = FACTOR ? "factor: compaction" : "embed: compaction";
  const char* m_exact = FACTOR ? "factor: exact pass" : "embed: exact pass";
  const char* m_rows = FACTOR ? "factor: exact rows" : "embed: exact rows";
  CUtensorMap map_a, map_b;
  encode_maps(q, &map_a, &map_b);
  const int64_t cols_pad = (I + EB_BN - 1) / EB_BN * EB_BN;
  // first chunk: about 4K columns, all appended; then doubling widths.  cap: the first chunk plus two lists' worth.
  const int64_t c0 = std::min<int64_t>(cols_pad, (std::max(4 * K, EB_BN) + EB_BN - 1) / EB_BN * EB_BN);
  const int cap = (int)(c0 + (std::max(2 * K, EB_BN) + EB_BN - 1) / EB_BN * EB_BN);
  int64_t rg = std::max<int64_t>(EB_BM, EB_BUF_BYTES / ((int64_t)cap * 8) / EB_BM * EB_BM);
  rg = std::min(rg, rows);

  RowState s;
  s.K = K;
  s.cap = cap;
  s.beta = (float)q.beta;
  if ((double)s.beta < q.beta) s.beta = nextafterf(s.beta, INFINITY);
  s.r = q.col.r;
  s.cr = q.row.cr;
  s.tau_p = c->buf<float>("eb_tau_p", (size_t)rg);
  s.tau_e = c->buf<float>("eb_tau_e", (size_t)rg);
  s.cnt = c->buf<int>("eb_cnt", (size_t)rg);
  s.over = c->buf<int>("eb_over", (size_t)rg);
  s.buf = c->buf<int2>("eb_buf", (size_t)rg * cap);
  s.prof = nullptr;
#ifdef RPK_PHASE_PROF
  s.prof = c->buf<u64>("eb_prof", EC_N);
  RPK_CUDA(cudaMemsetAsync(s.prof, 0, EC_N * sizeof(u64), st));
#endif
  ExactParamsOf<FACTOR> ep;
  memset(&ep, 0, sizeof(ep));
  ep.X = q.row.X;
  ep.I = I;
  ep.D = D;
  ep.sigma2 = q.row.sigma + q.col.sigma;
  ep.sel_cap = std::max(256, next_pow2_(2 * K));
  ep.direct_cap = std::min(ep.sel_cap, std::max(64, 2 * K));
  if constexpr (FACTOR) {
    ep.Xc = q.col.X;
    ep.row_map = job.row_map;
    ep.hist_ptr = job.hist_ptr;
    ep.hist_idx = job.hist_idx;
    ep.allowed = job.allowed;
  }
  ep.out_idx = job.out_idx;
  ep.out_val = job.out_val;
  ep.out_len = job.out_len;
  ep.handoff = c->buf<int>("eb_handoff", (size_t)rg);
  ep.n_handoff = c->buf<int>("eb_nhandoff", 1);
  const int rows_grid = (int)std::min<int64_t>(I, std::max<int64_t>(1, std::min<int64_t>(c->sm_count, EB_BUF_BYTES / (I * 8))));
  ep.scratch = c->buf<double>("eb_scratch", (size_t)rows_grid * I);
  const size_t sel_bytes = sel_smem_bytes(ep.sel_cap);
  const size_t exact_smem = sel_bytes + (size_t)D * 8 + (size_t)cap * 12;
  const size_t rows_smem = sel_bytes + (size_t)D * 8;
  const size_t compact_smem = (size_t)cap * 12;
  RPK_REQUIRE(exact_smem <= (size_t)c->smem_max, "embedding: K too large for shared memory");
  RPK_CUDA(cudaFuncSetAttribute(k_embed_exact<FACTOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)exact_smem));
  RPK_CUDA(cudaFuncSetAttribute(k_embed_exact_rows<FACTOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem));
  RPK_CUDA(cudaFuncSetAttribute(k_embed_compact, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)compact_smem));
  int n_chunks = 0;
  for (int64_t g0 = job.row_begin; g0 < job.row_end; g0 += rg) {
    const int64_t g1 = std::min(job.row_end, g0 + rg);
    s.row0 = (int)g0;
    s.rows = (int)(g1 - g0);
    const int sgrid = (int)std::min<int64_t>(s.rows, (int64_t)c->sm_count * 8);
    k_embed_init<<<(s.rows + 255) / 256, 256, 0, st>>>(s);
    RPK_LAUNCH_CHECK(c);
    ScreenParamsOf<FACTOR> sp = screen_params<FACTOR>();
    sp.m_tiles = ceil_div(s.rows, EB_BM);
    sp.k_blocks = q.kd_pad / EB_BK;
    sp.row0 = s.row0;
    sp.row_end = (int)g1;
    sp.r = q.col.r;
    sp.cr = q.row.cr;
    sp.tau_e = s.tau_e;
    sp.cnt = s.cnt;
    sp.buf = s.buf;
    sp.cap = cap;
    if constexpr (FACTOR) {
      sp.row_map = job.row_map;
      sp.hist_ptr = job.hist_ptr;
      sp.hist_idx = job.hist_idx;
      sp.allowed = job.allowed;
      sp.prof = s.prof;
    }
    n_chunks = 0;
    for (int64_t a = 0, w = c0; a < cols_pad; a += w, w = a) {
      const int64_t b = std::min(cols_pad, a + w);
      sp.col0 = (int)a;
      sp.col_end = (int)std::min<int64_t>(b, I);
      sp.n_tiles = (int)((b - a) / EB_BN);
      launch_screen<FACTOR>(c, map_a, map_b, sp);
      c->mark(m_chunk);
      k_embed_compact<<<sgrid, EB_SEL_NT, compact_smem, st>>>(s);
      RPK_LAUNCH_CHECK(c);
      c->mark(m_compact);
      ++n_chunks;
    }
    ep.s = s;
    ep.out_row0 = job.out_row0 + (g0 - job.row_begin);
    RPK_CUDA(cudaMemsetAsync(ep.n_handoff, 0, sizeof(int), st));
    k_embed_exact<FACTOR><<<sgrid, EB_SEL_NT, exact_smem, st>>>(ep);
    RPK_LAUNCH_CHECK(c);
    c->mark(m_exact);
    k_embed_exact_rows<FACTOR><<<rows_grid, EB_SEL_NT, rows_smem, st>>>(ep);
    RPK_LAUNCH_CHECK(c);
    c->mark(m_rows);
  }
#ifdef RPK_PHASE_PROF
  {
    u64 h[EC_N];
    RPK_CUDA(cudaMemcpyAsync(h, s.prof, sizeof(h), cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));
    if (FACTOR)
      fprintf(stderr, "[factor paths] users=%lld scored=%lld D=%d N=%d sigma_p=%d sigma_q=%d chunks=%d cap=%d group rows=%lld "
              "candidates=%llu compactions=%llu overflow rows=%llu zero handoffs=%llu exact rows=%llu masked skips=%llu\n",
              (long long)job.n_users, (long long)rows, D, K, q.row.sigma, q.col.sigma, n_chunks, cap, (long long)rg, h[EC_CAND],
              h[EC_COMPACT], h[EC_OVERFLOW], h[EC_ZERO], h[EC_EXACT], h[EC_MASKED]);
    else
      fprintf(stderr, "[embed paths] rows=%lld D=%d K=%d sigma=%d chunks=%d cap=%d group rows=%lld candidates=%llu "
              "compactions=%llu overflow rows=%llu zero handoffs=%llu exact rows=%llu\n",
              (long long)rows, D, K, q.row.sigma, n_chunks, cap, (long long)rg, h[EC_CAND], h[EC_COMPACT], h[EC_OVERFLOW],
              h[EC_ZERO], h[EC_EXACT]);
  }
#endif
}

void run_embed_topk(rpk_ctx* c, int64_t I, int D, const double* E_u, int similarity, int K, int64_t item_begin,
                    int64_t item_end, int32_t* out_idx_u, double* out_val_u, int32_t* out_len_u) {
  RPK_REQUIRE(K >= 1 && K <= 1024, "embedding: K must be in [1, 1024]");
  RPK_REQUIRE(0 <= item_begin && item_begin <= item_end && item_end <= I, "embedding: bad item range");
  RPK_REQUIRE(out_idx_u && out_len_u, "out_idx / out_len must not be null");
  const EmbedPrep q = embed_prep(c, I, D, E_u, similarity);
  const int64_t rows = item_end - item_begin;
  Out<int32_t> o_idx, o_len;
  Out<double> o_val;
  o_idx.init(c, out_idx_u, (size_t)rows * K, "eb_out_idx");
  o_val.init(c, out_val_u, (size_t)rows * K, "eb_out_val");
  o_len.init(c, out_len_u, (size_t)rows, "eb_out_len");
  if (rows > 0) {
    TopkJob job;
    memset(&job, 0, sizeof(job));
    job.I = I;
    job.D = D;
    job.K = K;
    job.row_begin = item_begin;
    job.row_end = item_end;
    job.out_row0 = 0;
    job.out_idx = o_idx.dev;
    job.out_val = o_val.dev;
    job.out_len = o_len.dev;
    screen_topk<false>(c, q, job);
  }
  o_idx.finish(c);
  o_val.finish(c);
  o_len.finish(c);
  finish_call(c);
}

void run_embed_screen_f32(rpk_ctx* c, int64_t I, int D, const double* E_u, int similarity, float* out_S_u) {
  RPK_REQUIRE(out_S_u, "out_S must not be null");
  RPK_REQUIRE(I <= 65536, "embedding screen: the verification matrix is limited to I <= 65536");
  const EmbedPrep q = embed_prep(c, I, D, E_u, similarity);
  Out<float> o;
  o.init(c, out_S_u, (size_t)I * I, "eb_S_out");
  CUtensorMap map_a, map_b;
  encode_maps(q, &map_a, &map_b);
  ScreenParams sp = screen_params<false>();
  sp.m_tiles = ceil_div(I, EB_BM);
  sp.n_tiles = ceil_div(I, EB_BN);
  sp.k_blocks = q.kd_pad / EB_BK;
  sp.row_end = (int)I;
  sp.col_end = (int)I;
  sp.r = q.col.r;
  sp.cr = q.row.cr;
  sp.S = o.dev;
  sp.lds = I;
  sp.unscale = (float)ldexp(1.0, -(q.row.sigma + q.col.sigma));
  launch_screen<false>(c, map_a, map_b, sp);
  o.finish(c);
  finish_call(c);
}

// ------------------------------------------------------------------------------------------
// Factor models: s_uj = fold over d of fl(p_ud * q_jd) for the users with history
// ------------------------------------------------------------------------------------------
struct FactorIn {
  const double* P;       // device [U x D]
  const double* Q;       // device [I x D]
  const int64_t* indptr; // device CSR of X (null without one)
  const int32_t* indices;
  int* row_map;          // users with history (topn), in any order
  int64_t n_scored;
  EmbedPrep q;           // screen operands (topn, screen)
};

enum { FP_TOPN, FP_FULL, FP_SCREEN };

static const unsigned char* factor_item_filter(rpk_ctx* c, int64_t I) {
  if (c->filter_I < 0) return nullptr;
  RPK_REQUIRE(c->filter_I == I, "factor model: the item filter was set for a different number of items");
  return c->get<unsigned char>("p_item_ok");
}

// Validates P, Q and X (synchronises once: NaN / inf, the norm limit and a malformed X are reported by this call),
// compacts the users with history (FP_TOPN) and builds the screen operands (FP_TOPN: those users; FP_SCREEN: all).
static FactorIn factor_prep(rpk_ctx* c, int64_t U, int64_t I, int D, const double* P_u, const double* Q_u, int64_t nnz,
                            const int64_t* indptr_u, const int32_t* indices_u, int mode) {
  RPK_REQUIRE(U >= 0 && U < ((int64_t)1 << 31), "factor model: U must be in [0, 2^31)");
  RPK_REQUIRE(I >= 1 && I < ((int64_t)1 << 24), "factor model: I must be in [1, 2^24)");
  RPK_REQUIRE(D >= 1 && D <= 1024, "factor model: D must be in [1, 1024]");
  RPK_REQUIRE(nnz >= 0, "factor model: negative nnz");
  cudaStream_t st = c->stream;
  FactorIn f;
  memset(&f, 0, sizeof(f));
  f.P = stage_in(c, P_u, (size_t)U * D, "fc_P_in");
  f.Q = stage_in(c, Q_u, (size_t)I * D, "fc_Q_in");
  int* flags = c->buf<int>("fc_flags", 12);  // [0] non-finite, [1] bad X, [2] users with history, [4..7] P, [8..11] Q stats
  RPK_CUDA(cudaMemsetAsync(flags, 0, 12 * sizeof(int), st));
  c->mark("factor: start");
  launch_norms(c, f.P, U, D, 0, nullptr, flags, flags + 4);
  launch_norms(c, f.Q, I, D, 0, nullptr, flags, flags + 8);
  if (mode != FP_SCREEN) {
    f.indptr = stage_in(c, indptr_u, (size_t)U + 1, "fc_indptr_in");
    f.indices = stage_in(c, indices_u, (size_t)nnz, "fc_indices_in");
    if (mode == FP_TOPN) f.row_map = c->buf<int>("fc_row_map", (size_t)std::max<int64_t>(U, 1));
    if (U > 0) {
      const int grid = (int)std::min<int64_t>((U + 7) / 8, (int64_t)c->sm_count * 16);
      k_factor_rows<<<grid, 256, 0, st>>>(f.indptr, f.indices, U, I, nnz, f.row_map, flags);
      RPK_LAUNCH_CHECK(c);
    }
  }
  int h[12];
  RPK_CUDA(cudaMemcpyAsync(h, flags, sizeof(h), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaStreamSynchronize(st));
  RPK_REQUIRE(h[0] == 0, "factor model: P or Q contains NaN or inf");
  RPK_REQUIRE(h[1] == 0, "factor model: X must be a CSR with ascending unique columns in [0, I) per row");
  // |partial sums| <= ||p_u|| ||q_j|| (up to rounding) stay finite
  RPK_REQUIRE(stat_maxq(h + 4) < 0x1p1020 && stat_maxq(h + 8) < 0x1p1020,
              "factor model: every squared row norm of P and Q must be below 2^1020");
  f.n_scored = mode == FP_TOPN ? h[2] : U;
  if (mode != FP_FULL) {
    f.q.kd_pad = (D + EB_BK - 1) / EB_BK * EB_BK;
    f.q.eps = 0x1p-10 + (double)(D + 2) * 0x1p-22;
    f.q.row = build_operand(c, f.P, f.row_map, f.n_scored, D, screen_sigma(h + 4), f.q.eps, f.q.kd_pad, true, "fc_A_p",
                            "fc_r_p", "fc_cr_p");
    f.q.col = build_operand(c, f.Q, nullptr, I, D, screen_sigma(h + 8), f.q.eps, f.q.kd_pad, false, "fc_A_q", "fc_r_q", "");
    set_bound(f.q, D);
  }
  c->mark("factor: prep");
  return f;
}

void run_factor_topn(rpk_ctx* c, int64_t U, int64_t I, int D, const double* P_u, const double* Q_u, int64_t nnz,
                     const int64_t* indptr_u, const int32_t* indices_u, int N, int mask_history, int32_t* out_idx_u,
                     double* out_val_u, int32_t* out_len_u) {
  RPK_REQUIRE(N >= 1 && N <= 1024, "factor model: N must be in [1, 1024]");
  RPK_REQUIRE(out_idx_u && out_len_u, "out_idx / out_len must not be null");
  const unsigned char* allowed = factor_item_filter(c, I);
  const FactorIn f = factor_prep(c, U, I, D, P_u, Q_u, nnz, indptr_u, indices_u, FP_TOPN);
  cudaStream_t st = c->stream;
  Out<int32_t> o_idx, o_len;
  Out<double> o_val;
  o_idx.init(c, out_idx_u, (size_t)U * N, "fc_out_idx");
  o_val.init(c, out_val_u, (size_t)U * N, "fc_out_val");
  o_len.init(c, out_len_u, (size_t)U, "fc_out_len");
  if (U > 0) {  // users without history: empty rows
    RPK_CUDA(cudaMemsetAsync(o_idx.dev, 0xff, sizeof(int32_t) * (size_t)U * N, st));
    if (o_val.dev) RPK_CUDA(cudaMemsetAsync(o_val.dev, 0, sizeof(double) * (size_t)U * N, st));
    RPK_CUDA(cudaMemsetAsync(o_len.dev, 0, sizeof(int32_t) * (size_t)U, st));
  }
  if (f.n_scored > 0) {
    TopkJob job;
    memset(&job, 0, sizeof(job));
    job.I = I;
    job.D = D;
    job.K = N;
    job.row_begin = 0;
    job.row_end = f.n_scored;
    job.row_map = f.row_map;
    job.hist_ptr = mask_history ? f.indptr : nullptr;
    job.hist_idx = mask_history ? f.indices : nullptr;
    job.allowed = allowed;
    job.out_idx = o_idx.dev;
    job.out_val = o_val.dev;
    job.out_len = o_len.dev;
    job.n_users = U;
    screen_topk<true>(c, f.q, job);
  }
  o_idx.finish(c);
  o_val.finish(c);
  o_len.finish(c);
  finish_call(c);
}

void run_factor_full(rpk_ctx* c, int64_t U, int64_t I, int D, const double* P_u, const double* Q_u, int64_t nnz,
                     const int64_t* indptr_u, const int32_t* indices_u, int mask_history, double* out_u) {
  RPK_REQUIRE(out_u, "out_scores must not be null");
  const unsigned char* allowed = factor_item_filter(c, I);
  const FactorIn f = factor_prep(c, U, I, D, P_u, Q_u, nnz, indptr_u, indices_u, FP_FULL);
  Out<double> o;
  o.init(c, out_u, (size_t)U * I, "fc_full_out");
  if (U > 0) {
    const dim3 grid((unsigned)ceil_div(I, FF_T), (unsigned)std::min(ceil_div(U, FF_T), 65535));
    k_factor_full<<<grid, 256, 0, c->stream>>>(f.P, f.Q, f.indptr, U, I, D, allowed, o.dev);
    RPK_LAUNCH_CHECK(c);
    if (mask_history) {
      const int g = (int)std::min<int64_t>((U + 7) / 8, (int64_t)c->sm_count * 16);
      k_factor_mask_history<<<g, 256, 0, c->stream>>>(f.indptr, f.indices, U, I, o.dev);
      RPK_LAUNCH_CHECK(c);
    }
    c->mark("factor: full scores");
  }
  o.finish(c);
  finish_call(c);
}

void run_factor_screen_f32(rpk_ctx* c, int64_t U, int64_t I, int D, const double* P_u, const double* Q_u, float* out_S_u) {
  RPK_REQUIRE(out_S_u, "out_S must not be null");
  RPK_REQUIRE(U >= 1 && U <= 65536 && I <= 65536, "factor screen: the verification matrix is limited to U, I <= 65536");
  const FactorIn f = factor_prep(c, U, I, D, P_u, Q_u, 0, nullptr, nullptr, FP_SCREEN);
  Out<float> o;
  o.init(c, out_S_u, (size_t)U * I, "fc_S_out");
  CUtensorMap map_a, map_b;
  encode_maps(f.q, &map_a, &map_b);
  ScreenParams sp = screen_params<false>();
  sp.m_tiles = ceil_div(U, EB_BM);
  sp.n_tiles = ceil_div(I, EB_BN);
  sp.k_blocks = f.q.kd_pad / EB_BK;
  sp.row_end = (int)U;
  sp.col_end = (int)I;
  sp.r = f.q.col.r;
  sp.cr = f.q.row.cr;
  sp.S = o.dev;
  sp.lds = I;
  sp.unscale = (float)ldexp(1.0, -(f.q.row.sigma + f.q.col.sigma));
  launch_screen<false>(c, map_a, map_b, sp);
  o.finish(c);
  finish_call(c);
}

}  // namespace rpk
