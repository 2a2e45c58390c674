// Scoring on the GPU: score_uj = sum_{i in hist(u)} S_ij for a K-sparse S, history masking and
// top-N fused in shared memory; optional full CSR output for drop-in predict().
//
// Replaces (reference, /root/reference):
//   recpack/algorithms/base.py:237-255     ItemSimilarityMatrixAlgorithm._predict  (X @ similarity_matrix_)
//   recpack/pipelines/pipeline.py:174-175  history removal
//   recpack/metrics/base.py:189            get_top_K_ranks(y_pred, K) on the prediction rows
//
// Scores are exact integers: every similarity value is stored as q = max(rint(v * 2^e), 1) (40 bits), with the
// power of two 2^e chosen per model so that the largest similarity lands in [2^39, 2^40) -- the resolution is
// relative to the model's largest value (2^-40 of it), whatever its magnitude.  A score is the integer sum of q
// over the history, reported as sum * 2^-e.  Integer sums make the result independent of the order in which the
// atomics land, so the top-N lists are deterministic.  Two kernels:
//   k_predict_a32  top-N: 32-bit approximate sums with one native shared-memory atomic (ATOMS.ADD) per
//                  entry pick the few items that can be in the top N, a second sweep adds their exact q;
//   k_predict      full CSR output, and the exact path for users k_predict_a32 hands over: one CTA per user runs
//                  its item ranges in order, the sum is kept in two 32-bit limbs (q & 0xFFFFF, q >> 20), 64-bit
//                  accumulators when a limb could overflow.
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "internal.h"
#include "prims.cuh"
#include "select.cuh"

namespace rpk {

constexpr u64 Q_MASK40 = (((u64)1) << 40) - 1;
constexpr int LIMB_BITS = 20;
constexpr unsigned LIMB_MASK = (1u << LIMB_BITS) - 1;
constexpr int LIMB_CHUNK = 4095;  // rows that can be added before the low limb must be normalised

// ------------------------------------------------------------------------------------------
// Model construction
// ------------------------------------------------------------------------------------------
// Scale of the loaded model: q = rint(v * 2^e), scores come back as sum * inv (inv = 2^-e).
struct ModelScale {
  double inv;
  int e;
  int pad;
};

__device__ __forceinline__ bool quantize(double v, int e, u64& q) {
  if (!(v >= 0.0) || !(v <= 1.7e308)) return false;  // negative, NaN or infinite
  const double sv = scalbn(v, e);                   // exact power-of-two scaling
  if (!(sv < 1099511627776.0)) return false;        // does not fit 40 bits (cannot happen with the model's own scale)
  long long r = __double2ll_rn(sv);                 // round half to even like np.rint
  q = r < 1 ? 1ull : (u64)r;                        // a stored entry never vanishes
  if (q > Q_MASK40) q = Q_MASK40;                   // a value within half a step of 2^40 rounds up to it: clamp
  return true;
}

// Largest value of the lists / CSR about to be loaded (bit pattern of a non-negative double orders like an integer).
__global__ void k_model_vmax_lists(const double* __restrict__ val, const int* __restrict__ len, const int64_t* __restrict__ row_src,
                                   int K, int64_t nrows, u64* __restrict__ vmax_bits, int* __restrict__ flag) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  u64 best = 0;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nrows * K; t += stride) {
    const int64_t src = row_src ? row_src[t / K] : t / K;
    int m = len[src];
    m = m > K ? K : m;
    if ((int)(t % K) < m) {
      const double v = val[src * K + t % K];
      if (!(v >= 0.0) || !(v <= 1.7e308)) atomicOr(flag, 1);
      else best = max(best, (u64)__double_as_longlong(v));
    }
  }
  best = warp_max_u64(best);
  if ((threadIdx.x & 31) == 0 && best) atomicMax(vmax_bits, best);
}

__global__ void k_model_vmax_flat(const double* __restrict__ val, int64_t n, u64* __restrict__ vmax_bits, int* __restrict__ flag) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  u64 best = 0;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    const double v = val[t];
    if (!(v >= 0.0) || !(v <= 1.7e308)) atomicOr(flag, 1);
    else best = max(best, (u64)__double_as_longlong(v));
  }
  best = warp_max_u64(best);
  if ((threadIdx.x & 31) == 0 && best) atomicMax(vmax_bits, best);
}

// e = 39 - floor(log2(vmax)): vmax * 2^e lies in [2^39, 2^40).  An empty (or all-zero) model gets e = 39.
// (vmax_bits: bit pattern of a non-negative double, which is also how a device-resident double is passed in.)
__global__ void k_model_scale(const u64* __restrict__ vmax_bits, ModelScale* __restrict__ sc, int forced_e, int use_forced) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int e = 39;
    if (use_forced) {
      e = forced_e;
    } else {
      const double vmax = __longlong_as_double((long long)vmax_bits[0]);
      if (vmax > 0.0) e = 39 - ilogb(vmax);
    }
    sc->e = e;
    sc->inv = scalbn(1.0, -e);
    sc->pad = 0;
  }
}

// One CTA per row: pack (idx, q), sort by idx, write the row.
__global__ void __launch_bounds__(256) k_model_from_topk(const int* __restrict__ idx, const double* __restrict__ val,
                                                         const int* __restrict__ len, const int64_t* __restrict__ row_src,
                                                         int K, int I, int nrows,
                                                         const int64_t* __restrict__ m_ptr, u64* __restrict__ m_ent,
                                                         unsigned* __restrict__ m_rowmax, int* __restrict__ flag,
                                                         const ModelScale* __restrict__ scale) {
  extern __shared__ __align__(16) unsigned char smem[];
  u64* buf = reinterpret_cast<u64*>(smem);
  __shared__ unsigned s_max;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int sc_e = scale->e;
  int n2 = 2;
  while (n2 < K) n2 <<= 1;
  for (int i = blockIdx.x; i < nrows; i += gridDim.x) {
    const int64_t src = row_src ? row_src[i] : (int64_t)i;  // where row i lives in the (gathered) input
    int m = len[src];
    if (m > K) m = K;
    if (m < 0) m = 0;
    if (tid == 0) s_max = 0;
    __syncthreads();
    unsigned lmax = 0;
    for (int t = tid; t < n2; t += nt) {
      u64 packed = ~0ull;
      if (t < m) {
        int j = idx[src * K + t];
        u64 q = 1;
        bool ok = quantize(val[src * K + t], sc_e, q);
        if (!ok || j < 0 || j >= I) atomicOr(flag, 1);
        packed = ((u64)(unsigned)j << 40) | (q & Q_MASK40);
        lmax = max(lmax, (unsigned)(q >> LIMB_BITS) + 1u);
      }
      buf[t] = packed;
    }
    atomicMax(&s_max, lmax);
    __syncthreads();
    for (int k = 2; k <= n2; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int t = tid; t < n2; t += nt) {
          int x = t ^ j;
          if (x > t) {
            u64 a = buf[t], b = buf[x];
            bool up = (t & k) == 0;
            if ((a > b) == up) {
              buf[t] = b;
              buf[x] = a;
            }
          }
        }
        __syncthreads();
      }
    if (m_ptr) {
      const int64_t base = m_ptr[i];
      for (int t = tid; t < m; t += nt) m_ent[base + t] = buf[t];
      if (tid == 0) m_rowmax[i] = s_max;
    } else {  // packed rows of K places each, all-ones after the row's entries (they sort last)
      for (int t = tid; t < K; t += nt) m_ent[(int64_t)i * K + t] = buf[t];
    }
    for (int t = tid + 1; t < m; t += nt)
      if ((buf[t] >> 40) == (buf[t - 1] >> 40)) atomicOr(flag, 2);  // duplicate column
    __syncthreads();
  }
}

// One warp per row of a CSR with ascending unique columns.
__global__ void k_model_from_csr(const int64_t* __restrict__ indptr, const int* __restrict__ indices,
                                 const double* __restrict__ values, int64_t I, u64* __restrict__ m_ent,
                                 unsigned* __restrict__ m_rowmax, int* __restrict__ m_len, int* __restrict__ flag,
                                 const ModelScale* __restrict__ scale) {
  const int lane = threadIdx.x & 31;
  const int sc_e = scale->e;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < I; i += nwarps) {
    int64_t b = indptr[i], e = indptr[i + 1];
    unsigned lmax = 0;
    for (int64_t k = b + lane; k < e; k += 32) {
      int j = indices[k];
      u64 q = 1;
      bool ok = quantize(values[k], sc_e, q);
      if (!ok || j < 0 || j >= I) atomicOr(flag, 1);
      if (k > b && indices[k - 1] >= j) atomicOr(flag, 2);
      m_ent[k] = ((u64)(unsigned)j << 40) | (q & Q_MASK40);
      lmax = max(lmax, (unsigned)(q >> LIMB_BITS) + 1u);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    if (lane == 0) {
      m_rowmax[i] = lmax;
      m_len[i] = (int)(e - b);
    }
  }
}

// seg[i*(P+1)+p] = offset inside row i of the first entry with column >= p*R
__global__ void k_model_seg(const int64_t* __restrict__ m_ptr, const u64* __restrict__ m_ent, int64_t I, int P, int R,
                            int* __restrict__ seg) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= I * (P + 1)) return;
  int64_t i = t / (P + 1);
  int p = (int)(t % (P + 1));
  int64_t b = m_ptr[i], lo = b, hi = m_ptr[i + 1];
  if (p == P) {
    seg[t] = (int)(hi - b);
    return;
  }
  u64 target = (u64)p * (u64)R;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if ((m_ent[mid] >> 40) < target) lo = mid + 1;
    else hi = mid;
  }
  seg[t] = (int)(lo - b);
}

// ---- block layout for the 32-bit scoring kernel, built per geometry (P item ranges of R items).  The entries of
// every (row, item range) segment are copied out on their own, padded to a multiple of 4 entries (32 bytes, one
// sector), and re-packed as (q << 24) | 4 * slot with slot = column - p*R, the accumulator the kernel adds to (as a
// byte offset): one AND and one shift per entry, no range test -- which bounds R to 2^22 slots, far beyond what
// shared memory holds.  Padding entries have q = 0 and slot = R + (position in the segment & 31):
// they land in 32 scratch accumulators behind the range, a different bank for every lane of the warp that reads them.
// seg[t] = {offset of the segment inside its model row, entries}, t = row * P + range
__global__ void k_model_seg_len(const int64_t* __restrict__ m_ptr, const u64* __restrict__ m_ent, int64_t I, int P, int R,
                                int2* __restrict__ seg, int* __restrict__ len4) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= I * P) return;
  const int64_t i = t / P;
  const int p = (int)(t % P);
  const int64_t b = m_ptr[i], e = m_ptr[i + 1];
  auto lower = [&](u64 target) {
    int64_t lo = b, hi = e;
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if ((m_ent[mid] >> 40) < target) lo = mid + 1;
      else hi = mid;
    }
    return lo - b;
  };
  const int64_t s0 = lower((u64)p * (u64)R), s1 = lower((u64)(p + 1) * (u64)R);
  seg[t] = make_int2((int)s0, (int)(s1 - s0));
  len4[t] = (int)((s1 - s0 + 3) & ~(int64_t)3);
}

// One warp per segment: copy + re-pack + pad; blk[t] = {first 4-entry block, number of blocks, ceil(largest q / 2^20), 0}.
// The third field bounds every term of the segment: the kernel sums it over a user's rows to choose the shift of
// its 32-bit sums.
__global__ void k_model_pad(const int64_t* __restrict__ m_ptr, const u64* __restrict__ m_ent, const int2* __restrict__ seg,
                            const int64_t* __restrict__ ptr4, int64_t I, int P, int R, u64* __restrict__ ent4,
                            int4* __restrict__ blk) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t t = warp; t < I * P; t += nwarps) {
    const int64_t i = t / P;
    const int p = (int)(t % P);
    const int2 sg = seg[t];
    const int64_t src = m_ptr[i] + sg.x, o = ptr4[t], n4 = ptr4[t + 1] - o;
    u64 qmax = 0;
    for (int64_t k = lane; k < n4; k += 32) {
      u64 v = (u64)(unsigned)(R + (int)(k & 31)) << 2;  // padding: q = 0, a scratch slot of this lane's own
      if (k < sg.y) {
        const u64 e = m_ent[src + k];
        const u64 q = e & Q_MASK40;
        v = (q << 24) | ((u64)((unsigned)(e >> 40) - (unsigned)p * (unsigned)R) << 2);
        qmax = max(qmax, q);
      }
      ent4[o + k] = v;
    }
    qmax = warp_max_u64(qmax);
    if (lane == 0) blk[t] = make_int4((int)(o >> 2), (int)(n4 >> 2), (int)(unsigned)((qmax + 0xfffffull) >> 20), 0);
  }
}

__global__ void k_gather_len(const int* __restrict__ len, const int64_t* __restrict__ row_src, int64_t I, int* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < I) out[i] = len[row_src[i]];
}

static void model_common_begin(rpk_ctx* c, int64_t I) {
  c->mark("model: begin");
  RPK_REQUIRE(I >= 0 && I < ((int64_t)1 << 24), "item count must be below 2^24");
  c->m_I = I;
  c->m_P = 0;  // segment tables must be rebuilt
  c->m_P2 = 0;
  c->m_pad = false;
  c->m_signed = false;
  int* flag = c->buf<int>("m_flag", 1);
  RPK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), c->stream));
  RPK_CUDA(cudaMemsetAsync(c->buf<u64>("m_vmax", 1), 0, sizeof(u64), c->stream));
  c->buf<ModelScale>("m_scale", 1);
}

// Scale of the model about to be loaded: from the largest value (forced < 0 ... use_forced = false) or as given.
static const ModelScale* model_set_scale(rpk_ctx* c, bool use_forced, int forced_e) {
  ModelScale* sc = c->get<ModelScale>("m_scale");
  k_model_scale<<<1, 32, 0, c->stream>>>(c->get<u64>("m_vmax"), sc, forced_e, use_forced ? 1 : 0);
  RPK_LAUNCH_CHECK(c);
  return sc;
}

static void model_check_flag(rpk_ctx* c) {
  int h = 0, hp = 0;
  ModelScale hs;
  if (c->pack_flag_pending) RPK_CUDA(cudaMemcpyAsync(&hp, c->get<int>("pk_flag"), sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  RPK_CUDA(cudaMemcpyAsync(&h, c->get<int>("m_flag"), sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  RPK_CUDA(cudaMemcpyAsync(&hs, c->get<ModelScale>("m_scale"), sizeof(ModelScale), cudaMemcpyDeviceToHost, c->stream));
  RPK_CUDA(cudaStreamSynchronize(c->stream));
  c->m_exp = hs.e;
  c->mark("model: loaded (sync)");
  if (c->pack_flag_pending) {
    c->pack_flag_pending = false;
    h |= hp;  // what the (stream-ordered) packing of this rank's rows found
  }
  if (h & 1) {
    c->m_I = 0;
    throw Error("similarity model: values must be finite and non-negative, columns in [0, I)");
  }
  if (h & 2) {
    c->m_I = 0;
    throw Error("similarity model: column indices must be unique (and ascending for CSR input) within a row");
  }
}

// rows_in: number of rows of the input arrays (>= I when row_src maps model rows into a larger, e.g.
// all-gathered, array); row_src: int64[I] source row of every model row, or null for the identity.
void run_model_load_topk_rows(rpk_ctx* c, int64_t I, int K, int64_t rows_in, const int32_t* idx_u, const double* val_u,
                              const int32_t* len_u, const int64_t* row_src_u) {
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(rows_in >= I || row_src_u, "fewer input rows than items");
  model_common_begin(c, I);
  cudaStream_t st = c->stream;
  const int32_t* idx = stage_in(c, idx_u, (size_t)rows_in * K, "m_in_idx");
  const double* val = stage_in(c, val_u, (size_t)rows_in * K, "m_in_val");
  const int32_t* len = stage_in(c, len_u, (size_t)rows_in, "m_in_len");
  const int64_t* row_src = row_src_u ? stage_in(c, row_src_u, (size_t)I, "m_in_rowsrc") : nullptr;
  int64_t* m_ptr = c->buf<int64_t>("m_ptr", (size_t)I + 1);
  int* m_len = c->buf<int>("m_len", (size_t)I);
  if (I > 0) {
    if (row_src) {
      k_gather_len<<<ceil_div(I, 256), 256, 0, st>>>(len, row_src, I, m_len);
      RPK_LAUNCH_CHECK(c);
    } else {
      RPK_CUDA(cudaMemcpyAsync(m_len, len, sizeof(int) * (size_t)I, cudaMemcpyDeviceToDevice, st));
    }
  }
  scan_i32_i64(c, m_len, m_ptr, I);
  u64* m_ent = c->buf<u64>("m_ent", (size_t)I * K);
  unsigned* m_rowmax = c->buf<unsigned>("m_rowmax", (size_t)I);
  if (I > 0) {
    k_model_vmax_lists<<<(int)std::min<int64_t>(ceil_div(I * K, 256), (int64_t)c->sm_count * 16), 256, 0, st>>>(
        val, len, row_src, K, I, c->get<u64>("m_vmax"), c->get<int>("m_flag"));
    RPK_LAUNCH_CHECK(c);
  }
  const ModelScale* scale = model_set_scale(c, false, 0);
  if (I > 0) {
    int n2 = 2;
    while (n2 < K) n2 <<= 1;
    const int grid = (int)std::min<int64_t>(I, (int64_t)c->sm_count * 16);
    k_model_from_topk<<<grid, 128, (size_t)n2 * sizeof(u64), st>>>(idx, val, len, row_src, K, (int)I, (int)I, m_ptr, m_ent, m_rowmax,
                                                                  c->get<int>("m_flag"), scale);
    RPK_LAUNCH_CHECK(c);
  }
  int64_t total = 0;
  RPK_CUDA(cudaMemcpyAsync(&total, m_ptr + I, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  model_check_flag(c);
  RPK_REQUIRE(total >= 0 && total <= I * (int64_t)K, "similarity model: row lengths exceed K");
  c->m_nnz = total;
  c->m_max_len = K;
}

// One warp per model row: copy its entries out of the packed input rows, check them, record the row maximum.
__global__ void k_model_from_packed(const u64* __restrict__ ent, const int64_t* __restrict__ row_src, int K, int64_t I,
                                    const int64_t* __restrict__ m_ptr, const int* __restrict__ m_len,
                                    u64* __restrict__ m_ent, unsigned* __restrict__ m_rowmax, int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < I; i += nwarps) {
    const int64_t src = row_src ? row_src[i] : i;
    const u64* row = ent + src * K;
    const int64_t base = m_ptr[i];
    const int n = m_len[i];
    unsigned lmax = 0;
    for (int t = lane; t < n; t += 32) {
      const u64 e = row[t];
      const u64 col = e >> 40, q = e & Q_MASK40;
      if (col >= (u64)I || q == 0ull) atomicOr(flag, 1);
      if (t > 0 && (row[t - 1] >> 40) >= col) atomicOr(flag, 2);
      m_ent[base + t] = e;
      lmax = max(lmax, (unsigned)(q >> LIMB_BITS) + 1u);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    if (lane == 0) m_rowmax[i] = lmax;
  }
}

// Exponent e of the scale 2^e these lists would get as a model of their own (39 - floor(log2(largest value))).
void run_model_scale_exp(rpk_ctx* c, int K, int64_t rows, const double* val_u, const int32_t* len_u, int32_t* out_exp) {
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(rows >= 0 && out_exp, "bad arguments");
  cudaStream_t st = c->stream;
  const double* val = stage_in(c, val_u, (size_t)rows * K, "pk_in_val");
  const int32_t* len = stage_in(c, len_u, (size_t)rows, "pk_in_len");
  u64* vmax = c->buf<u64>("pk_vmax", 1);
  int* flag = c->buf<int>("pk_flag", 1);
  ModelScale* sc = c->buf<ModelScale>("pk_scale", 1);
  RPK_CUDA(cudaMemsetAsync(vmax, 0, sizeof(u64), st));
  RPK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
  if (rows > 0) {
    k_model_vmax_lists<<<(int)std::min<int64_t>(ceil_div(rows * K, 256), (int64_t)c->sm_count * 16), 256, 0, st>>>(val, len, nullptr, K, rows,
                                                                                                                  vmax, flag);
    RPK_LAUNCH_CHECK(c);
  }
  k_model_scale<<<1, 32, 0, st>>>(vmax, sc, 0, 0);
  RPK_LAUNCH_CHECK(c);
  ModelScale hs;
  int h = 0;
  RPK_CUDA(cudaMemcpyAsync(&hs, sc, sizeof(ModelScale), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaStreamSynchronize(st));
  RPK_REQUIRE(!(h & 1), "similarity lists: values must be finite and non-negative");
  *out_exp = hs.e;
}

// Largest value of the lists as a double in device (or host) memory -- the stream-ordered form of
// rpk_model_scale_exp: no synchronisation when out_vmax is device memory.
void run_model_vmax(rpk_ctx* c, int K, int64_t rows, const double* val_u, const int32_t* len_u, double* out_vmax_u) {
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(rows >= 0 && out_vmax_u, "bad arguments");
  cudaStream_t st = c->stream;
  const double* val = stage_in(c, val_u, (size_t)rows * K, "pk_in_val");
  const int32_t* len = stage_in(c, len_u, (size_t)rows, "pk_in_len");
  Out<double> o;
  o.init(c, out_vmax_u, 1, "pk_vmax_out");
  int* flag = c->buf<int>("pk_flag", 1);
  RPK_CUDA(cudaMemsetAsync(o.dev, 0, sizeof(double), st));
  RPK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
  if (rows > 0) {
    k_model_vmax_lists<<<(int)std::min<int64_t>(ceil_div(rows * K, 256), (int64_t)c->sm_count * 16), 256, 0, st>>>(
        val, len, nullptr, K, rows, reinterpret_cast<u64*>(o.dev), flag);
    RPK_LAUNCH_CHECK(c);
  }
  o.finish(c);
  finish_call(c);
}

void run_model_pack_rows(rpk_ctx* c, int64_t I, int K, int64_t rows, const int32_t* idx_u, const double* val_u,
                         const int32_t* len_u, int scale_exp, const double* vmax_u, uint64_t* out_u) {
  c->mark("pack: begin");
  RPK_REQUIRE(vmax_u || (scale_exp > -1000 && scale_exp < 1100), "scale exponent out of range");
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(I >= 0 && I < ((int64_t)1 << 24), "item count must be below 2^24");
  RPK_REQUIRE(rows >= 0, "negative row count");
  RPK_REQUIRE(out_u != nullptr, "out_ent must not be null");
  cudaStream_t st = c->stream;
  const int32_t* idx = stage_in(c, idx_u, (size_t)rows * K, "pk_in_idx");
  const double* val = stage_in(c, val_u, (size_t)rows * K, "pk_in_val");
  const int32_t* len = stage_in(c, len_u, (size_t)rows, "pk_in_len");
  Out<u64> o;
  o.init(c, reinterpret_cast<u64*>(out_u), (size_t)rows * K, "pk_out");
  int* flag = c->buf<int>("pk_flag", 1);
  RPK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
  ModelScale* sc = c->buf<ModelScale>("pk_scale", 1);
  const bool deferred = vmax_u != nullptr && is_device_ptr(vmax_u) && !o.host;  // everything stays on the stream
  if (vmax_u) {
    const double* vm = stage_in(c, vmax_u, 1, "pk_vmax_in");
    k_model_scale<<<1, 32, 0, st>>>(reinterpret_cast<const u64*>(vm), sc, 0, 0);
  } else {
    k_model_scale<<<1, 32, 0, st>>>(nullptr, sc, scale_exp, 1);
  }
  RPK_LAUNCH_CHECK(c);
  if (rows > 0) {
    int n2 = 2;
    while (n2 < K) n2 <<= 1;
    const int grid = (int)std::min<int64_t>(rows, (int64_t)c->sm_count * 16);
    k_model_from_topk<<<grid, 128, (size_t)n2 * sizeof(u64), st>>>(idx, val, len, nullptr, K, (int)I, (int)rows, nullptr, o.dev, nullptr, flag, sc);
    RPK_LAUNCH_CHECK(c);
  }
  if (deferred) {
    c->pack_flag_pending = true;  // checked together with the flags of the next model load (no synchronisation here)
    c->mark("pack: rows packed");
    return;
  }
  int h = 0;
  RPK_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaStreamSynchronize(st));
  RPK_REQUIRE(!(h & 1), "similarity lists: values must be finite, non-negative and below 2^(40 - scale_exp); columns in [0, I)");
  RPK_REQUIRE(!(h & 2), "similarity lists: column indices must be unique within a row");
  c->mark("pack: rows packed (sync)");
  o.finish(c);
  finish_call(c);
}

void run_model_load_packed_rows(rpk_ctx* c, int64_t I, int K, int64_t rows_in, const uint64_t* ent_u, const int32_t* len_u,
                                const int64_t* row_src_u, int scale_exp, const double* vmax_u) {
  RPK_REQUIRE(K >= 1 && K <= 4096, "K must be in [1, 4096]");
  RPK_REQUIRE(rows_in >= I || row_src_u, "fewer input rows than items");
  RPK_REQUIRE(vmax_u || (scale_exp > -1000 && scale_exp < 1100), "scale exponent out of range");
  model_common_begin(c, I);
  if (vmax_u) {
    const double* vm = stage_in(c, vmax_u, 1, "pk_vmax_in");
    k_model_scale<<<1, 32, 0, c->stream>>>(reinterpret_cast<const u64*>(vm), c->get<ModelScale>("m_scale"), 0, 0);
    RPK_LAUNCH_CHECK(c);
  } else {
    model_set_scale(c, true, scale_exp);
  }
  cudaStream_t st = c->stream;
  const u64* ent = stage_in(c, reinterpret_cast<const u64*>(ent_u), (size_t)rows_in * K, "m_in_ent");
  const int32_t* len = stage_in(c, len_u, (size_t)rows_in, "m_in_len");
  const int64_t* row_src = row_src_u ? stage_in(c, row_src_u, (size_t)I, "m_in_rowsrc") : nullptr;
  int64_t* m_ptr = c->buf<int64_t>("m_ptr", (size_t)I + 1);
  int* m_len = c->buf<int>("m_len", (size_t)I);
  if (I > 0) {
    if (row_src) {
      k_gather_len<<<ceil_div(I, 256), 256, 0, st>>>(len, row_src, I, m_len);
      RPK_LAUNCH_CHECK(c);
    } else {
      RPK_CUDA(cudaMemcpyAsync(m_len, len, sizeof(int) * (size_t)I, cudaMemcpyDeviceToDevice, st));
    }
  }
  scan_i32_i64(c, m_len, m_ptr, I);
  u64* m_ent = c->buf<u64>("m_ent", (size_t)I * K);
  unsigned* m_rowmax = c->buf<unsigned>("m_rowmax", (size_t)I);
  if (I > 0) {
    const int grid = (int)std::min<int64_t>((I * 32 + 255) / 256, (int64_t)c->sm_count * 16);
    k_model_from_packed<<<grid, 256, 0, st>>>(ent, row_src, K, I, m_ptr, m_len, m_ent, m_rowmax, c->get<int>("m_flag"));
    RPK_LAUNCH_CHECK(c);
  }
  int64_t total = 0;
  RPK_CUDA(cudaMemcpyAsync(&total, m_ptr + I, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  model_check_flag(c);
  RPK_REQUIRE(total >= 0 && total <= I * (int64_t)K, "similarity model: row lengths exceed K");
  c->m_nnz = total;
  c->m_max_len = K;
}

void run_model_load_topk(rpk_ctx* c, int64_t I, int K, const int32_t* idx_u, const double* val_u, const int32_t* len_u) {
  run_model_load_topk_rows(c, I, K, I, idx_u, val_u, len_u, nullptr);
}

void run_model_load_last_fit(rpk_ctx* c, int64_t token) {
  RPK_REQUIRE(c->lf_idx != nullptr && token == c->lf_token, "no complete fit result of that token is resident on the device");
  run_model_load_topk(c, c->lf_I, c->lf_K, c->lf_idx, c->lf_val, c->lf_len);
}

void run_model_load_csr(rpk_ctx* c, int64_t I, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
                        const double* values_u) {
  model_common_begin(c, I);
  cudaStream_t st = c->stream;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)I + 1, "m_in_ptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "m_in_idx");
  const double* values = stage_in(c, values_u, (size_t)nnz, "m_in_val");
  int64_t* m_ptr = c->buf<int64_t>("m_ptr", (size_t)I + 1);
  RPK_CUDA(cudaMemcpyAsync(m_ptr, indptr, sizeof(int64_t) * ((size_t)I + 1), cudaMemcpyDeviceToDevice, st));
  u64* m_ent = c->buf<u64>("m_ent", (size_t)nnz);
  unsigned* m_rowmax = c->buf<unsigned>("m_rowmax", (size_t)I);
  int* m_len = c->buf<int>("m_len", (size_t)I);
  if (nnz > 0) {
    k_model_vmax_flat<<<(int)std::min<int64_t>(ceil_div(nnz, 256), (int64_t)c->sm_count * 16), 256, 0, st>>>(
        values, nnz, c->get<u64>("m_vmax"), c->get<int>("m_flag"));
    RPK_LAUNCH_CHECK(c);
  }
  const ModelScale* scale = model_set_scale(c, false, 0);
  if (I > 0) {
    const int grid = (int)std::min<int64_t>((I * 32 + 255) / 256, (int64_t)c->sm_count * 16);
    k_model_from_csr<<<grid, 256, 0, st>>>(indptr, indices, values, I, m_ent, m_rowmax, m_len, c->get<int>("m_flag"), scale);
    RPK_LAUNCH_CHECK(c);
  }
  int64_t ends[2] = {0, 0};
  RPK_CUDA(cudaMemcpyAsync(&ends[0], m_ptr, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaMemcpyAsync(&ends[1], m_ptr + I, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  model_check_flag(c);
  RPK_REQUIRE(ends[0] == 0 && ends[1] == nnz, "similarity model: indptr does not match nnz");
  c->m_nnz = nnz;
  c->m_max_len = 0;
}

// ------------------------------------------------------------------------------------------
// Scoring kernel
// ------------------------------------------------------------------------------------------
// Candidate source of the two-limb kernel: slots [0, ns) are the accumulators of the item range, slots
// [ns, ns + nc) the user's running list carried from the earlier ranges (exact keys).
struct ScoreSrc {
  __device__ __forceinline__ bool has_queue() const { return false; }
  template <class F>
  __device__ __forceinline__ bool for_each_queued(F, int*, int, int*) const { return false; }
  const unsigned* lo;
  const unsigned* hi;
  const u64* wide;     // non-null: 64-bit accumulators
  const Entry* carry;  // the running list
  int r0, ns, nc;
  u64 floor_;
  __device__ __forceinline__ u64 score_at(int j) const {
    return wide ? wide[j] : (((u64)hi[j] << LIMB_BITS) + (u64)lo[j]);
  }
  __device__ __forceinline__ int nslots() const { return ns + nc; }
  __device__ __forceinline__ u64 margin() const { return 0ull; }
  __device__ __forceinline__ void set_floor(u64 thr) { floor_ = thr; }
  // Selection key: the score rounded toward zero to float, as a bit pattern.  The map is monotone
  // (a <= b => key(a) <= key(b)), so margin() = 0 is right: equal keys are told apart by cmp3 on the exact
  // score.  Scores lie in [1, 2^53), which gives constant key bounds -- no pass over the slots is needed.
  __device__ __forceinline__ static u64 key_of(u64 score) { return (u64)__float_as_uint(__ull2float_rz(score)); }
  __device__ __forceinline__ void stats(SelShared* sh) const {
    if (threadIdx.x == 0) {
      sh->count = ns + nc;  // upper bound of the candidate count (slots can be empty or masked)
      sh->kmin = (u64)__float_as_uint(1.0f);
      sh->kmax = (u64)__float_as_uint(9007199254740992.0f);
    }
    __syncthreads();
  }
  template <class F>
  __device__ __forceinline__ void visit(F f, int stride) const {
    for (int slot = threadIdx.x * stride; slot < ns; slot += blockDim.x * stride) {
      const u64 sc = score_at(slot);
      if (sc != 0) {
        const u64 k = key_of(sc);
        if (k >= floor_) f(slot, k);
      }
    }
    for (int t = threadIdx.x * stride; t < nc; t += blockDim.x * stride) {
      const u64 k = key_of(carry[t].key);
      if (k >= floor_) f(ns + t, k);
    }
  }
  template <class F>
  __device__ __forceinline__ void for_each(F f) const { visit(f, 1); }
  template <class F>
  __device__ __forceinline__ void for_each_sampled(F f) const { visit(f, SEL_SAMPLE); }
  __device__ __forceinline__ void entry(int slot, Entry& e) const {
    if (slot >= ns) {
      e = carry[slot - ns];
      return;
    }
    e.key = score_at(slot);
    e.idx = r0 + slot;
    e.aux = 0;
  }
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const {
    if (a.key != b.key) return a.key > b.key ? 1 : -1;
    return 0;
  }
};

enum { PRED_TOPN = 0, PRED_COUNT = 1, PRED_FILL = 2 };

struct PredParams {
  const int64_t* indptr;
  const int* indices;
  const int64_t* m_ptr;
  const u64* m_ent;
  const int* m_seg;
  const unsigned* m_rowmax;
  const int4* work_tab;  // {user, history length, row start lo, hi} in processing order
  const int* n_work;     // non-null: number of work_tab records (device side), replaces U
  int U, P, R, I, N, mask, mode, force_wide;
  int cap, direct_cap;
  int* queue;
  int* out_idx;          // top-N: [U x N] lists, [U x N] scores or null, [U] lengths
  double* out_val;
  int* out_len;
  int64_t* out_row_nnz;  // count: [U] non-empty scores of every user
  const int64_t* out_indptr;  // fill: the CSR the count sized
  int* out_indices;
  double* out_values;
  const ModelScale* scale;   // scores are reported as sum * scale->inv
  const unsigned char* item_ok;  // non-null: item filter, 1 = may be recommended
};

#ifdef RPK_PHASE_PROF
#define PROF_MARK(k)                                         \
  do {                                                       \
    if (tid == 0) {                                          \
      const long long t_now = clock64();                     \
      atomicAdd(p.prof + (k), (unsigned long long)(t_now - t_prev)); \
      t_prev = t_now;                                        \
    }                                                        \
  } while (0)
#else
#define PROF_MARK(k) do {} while (0)
#endif

// One work item is a user: its P item ranges run one after the other on the same accumulators.  Invariant: the
// accumulators of a CTA are all zero between ranges.  Top-N: the user's running list (at most N entries, exact
// keys) is kept behind the accumulators and offered to the next range's selection as extra candidates, so that
// the selection of the last range gives the user's final list.
__global__ void __launch_bounds__(1024, 1) k_predict(PredParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + SEL_BINS);
  u64* acc64 = reinterpret_cast<u64*>(smem + sel_smem_bytes(p.cap));
  unsigned* acc_lo = reinterpret_cast<unsigned*>(acc64);
  unsigned* acc_hi = acc_lo + p.R;
  Entry* carry = reinterpret_cast<Entry*>(acc64 + p.R);
  __shared__ int s_work;
  __shared__ int s_next;      // work item fetched ahead (its record is warmed in L2 on the way)
  __shared__ u64 s_bound;
  __shared__ int s_cnt;

  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  const int total = p.n_work ? *p.n_work : p.U;
  if (total == 0) return;
  for (int s = tid; s < p.R; s += nt) acc64[s] = 0ull;
  if (tid == 0) s_next = atomicAdd(p.queue, 1);
  for (;;) {
    if (tid == 0) {
      s_work = s_next;
      const int nx = atomicAdd(p.queue, 1);
      s_next = nx;
      if (nx < total) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.work_tab + nx) : "memory");
      s_bound = 0;
      s_cnt = 0;
    }
    __syncthreads();
    const int w = s_work;
    __syncthreads();
    if (w >= total) break;
    const int4 rec = p.work_tab[w];
    const int u = rec.x;
    const int64_t xb = ((int64_t)(unsigned)rec.z) | ((int64_t)rec.w << 32);
    const int d = rec.y;
    if (d == 0) {  // user without history: empty prediction row (algorithms/base.py:123-127)
      if (p.mode == PRED_TOPN) {
        for (int t = tid; t < p.N; t += nt) {
          p.out_idx[(int64_t)u * p.N + t] = -1;
          if (p.out_val) p.out_val[(int64_t)u * p.N + t] = 0.0;
        }
        if (tid == 0) p.out_len[u] = 0;
      } else if (p.mode == PRED_COUNT) {
        if (tid == 0) p.out_row_nnz[u] = 0;
      }
      continue;
    }
    // ---- can the high limb overflow?  sum of per-row maxima bounds every score's high limb
    bool wide = p.force_wide != 0;
    if (!wide && d > LIMB_CHUNK) {
      u64 b = 0;
      for (int r = tid; r < d; r += nt) b += (u64)p.m_rowmax[p.indices[xb + r]];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
      if (lane == 0) atomicAdd(&s_bound, b);
      __syncthreads();
      wide = s_bound >= (((u64)1) << 32);
    }
    int nc = 0;       // top-N: entries of the running list
    int running = 0;  // fill: entries written for this user so far
    for (int pass = 0; pass < p.P; ++pass) {
      const int r0 = pass * p.R;
      const int ns = min(p.R, p.I - r0);
      // ---- accumulate: history rows are dealt to the warps in chunks (<= 32 rows, one per lane, so that the
      //      segment bounds are fetched in parallel); rows are added in groups of LIMB_CHUNK so that the low
      //      limb (20 bits per term) cannot overflow 32 bits between normalisations
      // the loop is instantiated for both accumulator modes so that the hot path carries no mode tests
      auto accumulate = [&](auto wide_c) {
        constexpr bool WIDE = decltype(wide_c)::value;
        for (int c0 = 0; c0 < d; c0 += LIMB_CHUNK) {
          const int c1 = min(d, c0 + LIMB_CHUNK);
          int chunk = (c1 - c0 + nwarps - 1) / nwarps;
          chunk = chunk < 1 ? 1 : (chunk > 32 ? 32 : chunk);
          for (int base = c0 + warp * chunk; base < c1; base += nwarps * chunk) {
            const int nvalid = min(chunk, c1 - base);
            int64_t beg = 0;
            int len = 0;
            if (lane < nvalid) {
              const int i = p.indices[xb + base + lane];
              const int* sg = p.m_seg + (int64_t)i * (p.P + 1) + pass;
              const int s0 = sg[0];
              beg = p.m_ptr[i] + s0;
              len = sg[1] - s0;
            }
            auto add_entry = [&](u64 ent) {
              if (ent != 0ull) {
                const int j = (int)(ent >> 40) - r0;
                const u64 q = ent & Q_MASK40;
                if (WIDE) {
                  atomicAdd(&acc64[j], q);
                } else {
                  atomicAdd(&acc_lo[j], (unsigned)q & LIMB_MASK);
                  atomicAdd(&acc_hi[j], (unsigned)(q >> LIMB_BITS));
                }
              }
            };
            // rows are taken four at a time: the first 96 entries of each (a row segment rarely has more) are
            // loaded up front -- 12 independent loads in flight per lane -- and only then added
            for (int l0 = 0; l0 < nvalid; l0 += 4) {
              u64 ent[4][3];
              int64_t bq[4];
              int nq[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int l = l0 + q;  // lanes >= nvalid hold len = 0
                bq[q] = __shfl_sync(0xffffffffu, beg, l & 31);
                nq[q] = l < nvalid ? __shfl_sync(0xffffffffu, len, l & 31) : 0;
#pragma unroll
                for (int it = 0; it < 3; ++it) {
                  const int e = it * 32 + lane;
                  ent[q][it] = e < nq[q] ? p.m_ent[bq[q] + e] : 0ull;
                }
              }
#pragma unroll
              for (int q = 0; q < 4; ++q) {
#pragma unroll
                for (int it = 0; it < 3; ++it)
                  if (it * 32 < nq[q]) add_entry(ent[q][it]);
                for (int e0 = 96; e0 < nq[q]; e0 += 32) {
                  const int e = e0 + lane;
                  add_entry(e < nq[q] ? p.m_ent[bq[q] + e] : 0ull);
                }
              }
            }
          }
          __syncthreads();
          if (!WIDE && c1 < d) {  // carry the low limb into the high limb before the next chunk
            for (int s = tid; s < ns; s += nt) {
              unsigned l = acc_lo[s];
              acc_hi[s] += l >> LIMB_BITS;
              acc_lo[s] = l & LIMB_MASK;
            }
            __syncthreads();
          }
        }
      };
      if (wide) accumulate(std::true_type{});
      else accumulate(std::false_type{});
      if (p.mask) {  // pipelines/pipeline.py:174-175 -- before the truncation to N
        for (int r = tid; r < d; r += nt) {
          const int j = p.indices[xb + r] - r0;
          if (j >= 0 && j < ns) {
            if (wide) acc64[j] = 0ull;
            else {
              acc_lo[j] = 0u;
              acc_hi[j] = 0u;
            }
          }
        }
        __syncthreads();
      }
      if (p.item_ok) {  // postprocessing/filters.py:58-101: filtered items are never recommended
        for (int s = tid; s < ns; s += nt)
          if (!p.item_ok[r0 + s]) {
            if (wide) acc64[s] = 0ull;
            else {
              acc_lo[s] = 0u;
              acc_hi[s] = 0u;
            }
          }
        __syncthreads();
      }
      ScoreSrc src{acc_lo, acc_hi, wide ? acc64 : nullptr, carry, r0, ns, nc, 0ull};
      if (p.mode == PRED_TOPN) {
        // top N of this range and the earlier ones: the carried keys are exact sums and key_of is monotone, so
        // margin() = 0 holds for them too, and ties still go to the lower index
        const int m = block_select_topk(src, p.N, list, p.cap, p.direct_cap, hist, sh);
        if (pass + 1 == p.P) {
          const double inv_scale = p.scale->inv;
          for (int t = tid; t < p.N; t += nt) {
            p.out_idx[(int64_t)u * p.N + t] = t < m ? list[t].idx : -1;
            if (p.out_val) p.out_val[(int64_t)u * p.N + t] = t < m ? (double)list[t].key * inv_scale : 0.0;
          }
          if (tid == 0) p.out_len[u] = m;
        } else {
          for (int t = tid; t < m; t += nt) carry[t] = list[t];
          nc = m;
        }
      } else if (p.mode == PRED_COUNT) {
        int cnt = 0;
        for (int s = tid; s < ns; s += nt) cnt += src.score_at(s) != 0;
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0 && cnt) atomicAdd(&s_cnt, cnt);
      } else {
        const int64_t out = p.out_indptr[u];
        const double inv_scale = p.scale->inv;
        for (int base = 0; base < ns; base += nt) {
          const int s = base + tid;
          const u64 sc = s < ns ? src.score_at(s) : 0ull;
          const unsigned bal = __ballot_sync(0xffffffffu, sc != 0);
          if (lane == 0) sh->warp_tot[warp] = __popc(bal);
          __syncthreads();
          int off = 0, tot = 0;
          for (int q = 0; q < nwarps; ++q) {
            int v = sh->warp_tot[q];
            if (q < warp) off += v;
            tot += v;
          }
          if (sc != 0) {
            const int pos = running + off + __popc(bal & ((1u << lane) - 1u));
            p.out_indices[out + pos] = r0 + s;
            p.out_values[out + pos] = (double)sc * inv_scale;
          }
          running += tot;
          __syncthreads();
        }
      }
      __syncthreads();
      // ---- restore the all-zero invariant
      for (int s = tid; s < ns; s += nt) acc64[s] = 0ull;
      if (ns < p.R)
        for (int s = tid; s < ns; s += nt) acc_hi[s] = 0u;
      __syncthreads();
    }
    if (p.mode == PRED_COUNT && tid == 0) p.out_row_nnz[u] = s_cnt;
  }
}


// ------------------------------------------------------------------------------------------
// Scoring kernel, top-N mode: 32-bit approximate sums, exact scores only where the order needs them
// ------------------------------------------------------------------------------------------
// The two-limb kernel above pays two shared-memory atomics per similarity entry and 8 bytes per item slot.
// For top-N only a handful of scores per user matter, so this kernel works on approximations:
//   1. sweep: a_j += (q >> s) | 1 with ONE fire-and-forget 32-bit atomic per entry.  s is the smallest shift that
//      keeps every sum below 2^32, taken from a bound on the user's terms (sum over the history rows of the largest
//      q of the row's segment).  Each term is within 1 of q / 2^s, so |a_j - score_j / 2^s| <= d (d = history
//      length): a_x - a_y > 2d proves score_x > score_y.
//   2. history items are zeroed, then the survivor threshold: either the range's own bound (the N-th largest of the
//      per-thread maxima, two small histogram rounds) or, once the user's running list holds N entries, the bound
//      carried from the earlier ranges (the N-th entry's lower end).  One dense pass copies every item at or above
//      the threshold to the list and clears the accumulators.
//   3. the survivors are merged into the running list.  Every key is an interval of the exact score: an approximate
//      sum a stands for [(a - d) * 2^s, (a + d) * 2^s], an exact one for itself.  The list is ordered by upper end;
//      when every neighbour pair down to the (N+1)-th is separated (or exact), its order is the exact order.
//      Otherwise a second sweep over the rows adds the exact q of this range's survivors (two 20-bit limbs, native
//      atomics) while their accumulators are still live.  Scores requested: every survivor takes the second sweep.
// One work item is a whole user: the P ranges run one after the other on the same accumulators, the history is
// fetched once, and the list is written out after the last range.  All ranges share one shift s (from the bound
// over whole rows), so their approximate sums compare as plain integers.  A user whose order the approximate sums
// of an earlier range (their accumulators are gone) leave open is run again with exact sums throughout.  4 bytes
// per slot let two CTAs share an SM, so one CTA's latency-bound steps hide behind the other's atomics.  A user whose
// survivors do not fit the list (huge groups of near-equal scores) is handed to the two-limb kernel.
struct ExactOrder {
  __device__ __forceinline__ int cmp3(const Entry& a, const Entry& b) const {
    if (a.key != b.key) return a.key > b.key ? 1 : -1;
    return 0;
  }
};

struct Pred32Params {
  const int* indices;
  const u64* ent;        // model rows in 4-entry blocks, entries (q << 24) | column
  const int4* blk;       // {first block, blocks, bound of q >> 20, 0} per (row, item range), at row * P + range
  const int4* work_tab;  // {user, history length, row start lo, hi} in processing order
  int U, P, R, I, N, mask;
  int exact;             // 1: exact scores for every list (scores requested)
  int cap;
  int* queue;
  int* out_idx;          // [U x N] final lists
  double* out_val;       // [U x N] scores (exact mode), or null
  int* out_len;          // [U]
  const ModelScale* scale;
  const unsigned char* item_ok;  // non-null: item filter (1 = may be recommended), padded to a multiple of 4 items
  int* ovf_count;        // number of users handed to the two-limb kernel
  int4* ovf_tab;         // their work records
  unsigned long long* prof;
};

constexpr int A32_BITS = 10;            // selection histogram: 1024 bins
constexpr int A32_BINS = 1 << A32_BITS;
constexpr int A32_ROWS = 512;           // history rows staged per chunk (= threads per CTA)
constexpr int A32_NT = 512;

// Row table of one chunk of the user's history: {first block, number of blocks} of every row's segment, and the
// history item itself (for the history mask).
struct RowTab {
  int2 seg[A32_ROWS];
  int item[A32_ROWS];
};

// Histogram bin of a 32-bit sum: 32 bins per octave (bit pattern of the sum as a float, top 13 bits), so that bins
// are ~2.2 % wide at every magnitude -- the bin of the N-th largest value holds few items whatever the scale of the
// scores.
__device__ __forceinline__ int a32_bin(unsigned a) {
  const int b = (int)(__float_as_uint((float)a) >> 18) - (127 << 5);
  return b > A32_BINS - 1 ? A32_BINS - 1 : b;
}
// A value that every sum of bin b and above certainly reaches: the lower edge of bin b - 1 (the float conversion
// rounds by at most 2^-24, far less than a bin).
__device__ __forceinline__ unsigned a32_bin_floor(int b) {
  if (b <= 1) return 1u;
  return (unsigned)__uint_as_float((unsigned)(b - 1 + (127 << 5)) << 18);
}

// Loads of two history rows in flight: the first 96 entries of each (a row segment rarely has more).
struct RowPair {
  u64 e1[3], e2[3];
};

__device__ __forceinline__ void pair_load(RowPair& rp, const u64* __restrict__ ent, const RowTab* rt, int r, int n, int lane, int nwarps,
                                          u64 idle) {
  const int r2 = r + nwarps;
  const int2 s1 = rt->seg[r];
  const int2 s2 = r2 < n ? rt->seg[r2] : make_int2(0, 0);
  const u64* b1 = ent + ((int64_t)s1.x << 2) + lane;
  const u64* b2 = ent + ((int64_t)s2.x << 2) + lane;
  const int n1 = (s1.y << 2) - lane, n2 = (s2.y << 2) - lane;  // entries left from this lane's first one
#pragma unroll
  for (int it = 0; it < 3; ++it) {
    rp.e1[it] = 32 * it < n1 ? __ldg(b1 + 32 * it) : idle;
    rp.e2[it] = 32 * it < n2 ? __ldg(b2 + 32 * it) : idle;
  }
}

template <class F>
__device__ __forceinline__ void pair_apply(const RowPair& rp, F f) {
#pragma unroll
  for (int it = 0; it < 3; ++it) {
    f(rp.e1[it]);
    f(rp.e2[it]);
  }
}

// Calls f(entry) for every entry of the staged segments, padding included, and for `idle` in the places of a load
// slot that a short segment leaves empty (idle = a padding entry: q = 0, a scratch slot of the lane's own).  One
// warp per row, a lane per entry, so that a load covers 256 contiguous bytes.  Software pipeline: the loads of the
// next two rows of the warp are issued before the entries of the current two are added, so that a warp always has
// loads in flight.  Segments longer than 96 entries (rare: K / P entries on average) get their tail in a second loop.
template <class F>
__device__ __forceinline__ void sweep_rows(const u64* __restrict__ ent, const RowTab* rt, int n, u64 idle, F f) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int nwarps = A32_NT / 32;
  constexpr int step = 2 * nwarps;
  int r = warp;
  if (r >= n) return;
  RowPair A, B;
  pair_load(A, ent, rt, r, n, lane, nwarps, idle);
  for (;;) {
    r += step;
    const bool more_b = r < n;
    if (more_b) pair_load(B, ent, rt, r, n, lane, nwarps, idle);
    pair_apply(A, f);
    if (!more_b) break;
    r += step;
    const bool more_a = r < n;
    if (more_a) pair_load(A, ent, rt, r, n, lane, nwarps, idle);
    pair_apply(B, f);
    if (!more_a) break;
  }
  for (int q = warp; q < n; q += nwarps) {
    const int2 sg = rt->seg[q];
    if (sg.y > 24) {
      const u64* b = ent + ((int64_t)sg.x << 2);
      for (int e = 96 + lane; e < (sg.y << 2); e += 32) f(__ldg(b + e));
    }
  }
}

// m <= 32 entries: warp w ranks entries w, w + nwarps, ... by (key desc, index asc) -- lane f holds opponent f, one
// ballot counts the opponents that come first -- and writes them to their places in `dst`.  Barrier afterwards.
__device__ __forceinline__ void rank_by_warps(const Entry* src, Entry* dst, int m) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  u64 kf = 0ull;
  int jf = SENTINEL_IDX, af = 0;
  if (lane < m) {
    kf = src[lane].key;
    jf = src[lane].idx;
    af = src[lane].aux;
  }
  for (int i = warp; i < m; i += nwarps) {
    const u64 ki = __shfl_sync(0xffffffffu, kf, i);
    const int ji = __shfl_sync(0xffffffffu, jf, i);
    const int ai = __shfl_sync(0xffffffffu, af, i);
    const unsigned first = __ballot_sync(0xffffffffu, lane < m && (kf > ki || (kf == ki && jf < ji)));
    if (lane == 0) {
      Entry e;
      e.key = ki;
      e.idx = ji;
      e.aux = ai;
      dst[__popc(first)] = e;
    }
  }
}

// Orders m entries best first by (key desc, index asc).  Up to SEL_RANK_MAX entries are ranked by counting
// (nt / 64 threads per entry) from `src` into `other`; more are sorted in place.  Returns where the result is.
__device__ __forceinline__ Entry* a32_sort(Entry* src, Entry* other, int m) {
  ExactOrder ord;
  const int tid = threadIdx.x, nt = blockDim.x;
  if (m <= SEL_RANK_MAX) {
    const int tpe = nt / SEL_RANK_MAX, i = tid / tpe, part = tid % tpe;
    int rank = 0;
    Entry a;
    a.key = 0;
    a.idx = 0;
    a.aux = 0;
    if (i < m) {
      a = src[i];
      for (int f = part; f < m; f += tpe) rank += (f != i) && entry_before(ord, src[f], a);
    }
    for (int o = tpe >> 1; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
    if (i < m && part == 0) other[rank] = a;
    __syncthreads();
    return other;
  }
  int n2 = 1;
  while (n2 < m) n2 <<= 1;
  for (int i = m + tid; i < n2; i += nt) {
    Entry s;
    s.key = 0;
    s.idx = SENTINEL_IDX;
    s.aux = 0;
    src[i] = s;
  }
  __syncthreads();
  bitonic_sort_entries(ord, src, n2);
  return src;
}

#ifdef RPK_PHASE_PROF
#define PROF32_MARK(k) PROF_MARK(k)
#else
#define PROF32_MARK(k) do {} while (0)
#endif

__host__ __device__ __forceinline__ size_t a32_fixed_bytes(int cap) {
  return sel_smem_bytes(cap, A32_BINS) + 2 * ((sizeof(RowTab) + 15) / 16) * 16;
}

// Lower end of a key's interval (aux = 1: approximate key = upper end, the interval is W wide; aux = 0: exact).
__device__ __forceinline__ u64 a32_lo(const Entry& e, u64 W) { return e.aux ? (e.key > W ? e.key - W : 0ull) : e.key; }

// Orders list[0..m) best first by (upper end desc, index asc); returns where the result is (list or list2).
// Barrier before (the entries are in place) and after.
__device__ __forceinline__ Entry* a32_order(Entry* list, Entry* list2, int m) {
  if (m <= 32) {
    rank_by_warps(list, list2, m);
    __syncthreads();
    return list2;
  }
  return a32_sort(list, list2, m);
}

// True (in every thread) unless each neighbour pair of the first min(m - 1, N) places is proven: the first one's
// interval lies strictly above the second one's, or both are exact (then the order by index decides ties).
__device__ __forceinline__ bool a32_unproven(const Entry* s, int m, int N, u64 W) {
  const int pairs = (m - 1) < N ? (m - 1) : N;
  bool bad = false;
  for (int k = threadIdx.x; k < pairs; k += blockDim.x)
    if (s[k].aux | s[k + 1].aux) bad |= a32_lo(s[k], W) <= s[k + 1].key;
  return __syncthreads_or(bad) != 0;
}

// Work distribution: the users are sorted heaviest first; CTA b starts with user b and takes every further user
// from a shared counter (longest-processing-time scheduling: the few users with five-digit histories then cost
// their CTAs other users instead of coming on top of an equal share of everything -- that tail bounded the kernel
// once a rank's shard became small).  The counter is read TWO users ahead by thread 0, so the atomic's latency
// hides behind a whole user and the next user can still be staged while the current one is swept.  Users with histories of at least A32_EXACT_D rows get exact sums from the start: the margin 2 d of their
// approximate sums never proves a list.
constexpr int A32_EXACT_D = 2048;

__global__ void __launch_bounds__(A32_NT, 2) k_predict_a32(Pred32Params p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);  // the user's running list, then this range's survivors
  Entry* list2 = list + p.cap;  // SEL_RANK_MAX entries
  int* hist = reinterpret_cast<int*>(smem + sel_list_bytes(p.cap));
  SelShared* sh = reinterpret_cast<SelShared*>(hist + A32_BINS);
  RowTab* rtab = reinterpret_cast<RowTab*>(smem + sel_smem_bytes(p.cap, A32_BINS));
  unsigned* acc = reinterpret_cast<unsigned*>(smem + a32_fixed_bytes(p.cap));
  __shared__ int4 s_rec[2];
  __shared__ int s_w[2];
  __shared__ u64 s_bsum[2];       // bound of the sums, in units of 2^20: rows beyond the first chunk ...
  __shared__ unsigned s_bsum32[2];  // ... and the first chunk
  __shared__ int s_pend;            // the user after the next one (thread 0 asks for it one user ahead of its use)

  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
  const int total = p.U, P = p.P, N = p.N;
  const int G = gridDim.x, bid = blockIdx.x;
  if (bid >= total) return;
  uint4* acc4 = reinterpret_cast<uint4*>(acc);
  const unsigned acc_s = (unsigned)__cvta_generic_to_shared(acc);
  const int nvec = p.R >> 2;  // R is a multiple of 4
  for (int v = tid; v < nvec; v += nt) acc4[v] = make_uint4(0u, 0u, 0u, 0u);
  for (int b = tid; b < A32_BINS; b += nt) hist[b] = 0;
  if (tid == 0) {
    const int w0 = bid;
    s_pend = G + atomicAdd(p.queue, 1);
    s_w[0] = w0;
    s_rec[0] = p.work_tab[w0];
    s_bsum[0] = 0ull;
    s_bsum[1] = 0ull;
    s_bsum32[0] = 0u;
    s_bsum32[1] = 0u;
  }
  __syncthreads();
  // ---- staging of a user, in three parts so that its two dependent global loads (history item -> block table
  //      entries) hide behind other work: part 1 issues the load of this thread's history item, part 2 the loads of
  //      that row's table entries (all P ranges, adjacent), part 3 writes the row table of range 0 and adds up the
  //      bound of the sums (largest q of each whole row)
  int st_item = -1;
  int2 st_seg = make_int2(0, 0);
  unsigned st_bnd = 0;
  auto row_bound = [&](int item, int2* seg0) {
    const int4* b = p.blk + (int64_t)item * P;
    const int4 b0 = __ldg(b);
    unsigned z = (unsigned)b0.z;
    for (int q = 1; q < P; ++q) z = max(z, (unsigned)__ldg(b + q).z);
    if (seg0) *seg0 = make_int2(b0.x, b0.y);
    return z;
  };
  auto stage1 = [&](int buf) {
    st_item = -1;
    if (s_w[buf] < total) {
      const int4 rc = s_rec[buf];
      const int64_t xb2 = ((int64_t)(unsigned)rc.z) | ((int64_t)rc.w << 32);
      if (tid < rc.y) st_item = p.indices[xb2 + tid];
    }
  };
  auto stage2 = [&](int buf) {
    st_seg = make_int2(0, 0);
    st_bnd = 0;
    if (st_item >= 0) st_bnd = row_bound(st_item, &st_seg);
  };
  auto stage3 = [&](int buf) {
    if (s_w[buf] >= total) return;
    const int4 rc = s_rec[buf];
    const int d2 = rc.y;
    const int64_t xb2 = ((int64_t)(unsigned)rc.z) | ((int64_t)rc.w << 32);
    RowTab* rt2 = rtab + buf;
    unsigned b32 = 0;  // first chunk: at most 512 terms of at most 2^20 each
    if (tid < d2) {
      rt2->seg[tid] = st_seg;
      rt2->item[tid] = st_item;
      b32 = st_bnd;
    }
    b32 = __reduce_add_sync(0xffffffffu, b32);
    if (lane == 0 && b32) atomicAdd(&s_bsum32[buf], b32);
    if (d2 > nt) {  // long histories: the rows beyond the first chunk only add to the bound
      u64 bsum = 0;
      for (int r = tid + nt; r < d2; r += nt) bsum += (u64)row_bound(p.indices[xb2 + r], nullptr);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) bsum += __shfl_xor_sync(0xffffffffu, bsum, o);
      if (lane == 0 && bsum) atomicAdd(&s_bsum[buf], bsum);
    }
  };
  stage1(0);
  stage2(0);
  stage3(0);
  __syncthreads();
#ifdef RPK_PHASE_PROF
  long long t_prev = clock64();
#endif
  for (int k = 0;; ++k) {
    const int cur = k & 1, nxt = cur ^ 1;
    const int w = s_w[cur];
    if (w >= total) break;
    const int4 rec = s_rec[cur];
    RowTab* rt = rtab + cur;
    // the next user: its record is copied into shared memory asynchronously while this one's first range is
    // swept; its bound is reset here too (every thread has left the previous user, nobody reads these before the
    // barrier after the sweep)
    if (tid == 0) {
      int w_n = s_pend;                    // asked for while the previous user was processed
      s_pend = G + atomicAdd(p.queue, 1);  // used at the top of the next user
      if (w_n < total) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(&s_rec[nxt])),
                     "l"(p.work_tab + w_n)
                     : "memory");
      } else {
        w_n = total;
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      s_w[nxt] = w_n;
      s_bsum[nxt] = 0ull;
      s_bsum32[nxt] = 0u;
    }
    const int u = rec.x;
    const int64_t xb = ((int64_t)(unsigned)rec.z) | ((int64_t)rec.w << 32);
    const int d = rec.y;
    PROF32_MARK(0);
    if (d == 0) {  // user without history: empty prediction row (algorithms/base.py:123-127)
      if (tid == 0) asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
      stage1(nxt);
      for (int t = tid; t < N; t += nt) {
        p.out_idx[(int64_t)u * N + t] = -1;
        if (p.out_val) p.out_val[(int64_t)u * N + t] = 0.0;
      }
      if (tid == 0) p.out_len[u] = 0;
      stage2(nxt);
      stage3(nxt);
      __syncthreads();
      continue;
    }
    // ---- shift of the 32-bit sums from the bound staged with the user
    // B = b20 * 2^20 >= sum over the rows of their largest q; the smallest shift with (B >> sft) + d < 2^32
    const u64 b20 = s_bsum[cur] + (u64)s_bsum32[cur];  // < 2^45 (d < 2^24 rows of at most 2^20 each)
    int sft = 0;
    {
      const u64 room = 0xffffffffull - (u64)d;
      auto fits = [&](int sf) { return sf >= 20 ? (b20 >> (sf - 20)) <= room : b20 <= (room >> (20 - sf)); };
      if (!fits(0)) {
        sft = 64 - __clzll((long long)b20) - 12;  // bits(B) - 32
        sft = sft < 1 ? 1 : sft;
        while (!fits(sft)) ++sft;
      }
    }
    const int sh_a = 24 + sft;
    const unsigned margin = 2u * (unsigned)d;
    const u64 idle = (u64)(unsigned)(p.R + lane) << 2;
    bool uexact = p.exact != 0 || d >= A32_EXACT_D;
    bool first = true;   // the user's first range: the next user is staged alongside
    bool staged = true;  // the row table holds chunk 0 of the current range
    bool own = false;    // the range takes its own bound even when a carried one exists
    int r = 0;           // entries of the running list (list[0..r), best first, proven order)
    for (int pass = 0; pass < P; ++pass) {
      const int r0 = pass * p.R;
      const int ns = min(p.R, p.I - r0);
      if (tid == 0) sh->count = 0;
      // ---- sweep 1: approximate sums, one fire-and-forget atomic per entry
      for (int c0 = 0; c0 < d; c0 += A32_ROWS) {
        const int n = min(A32_ROWS, d - c0);
        if (c0 > 0 || !staged) {
          __syncthreads();  // the previous table is still being read
          for (int rr = tid; rr < n; rr += nt) {
            const int i = p.indices[xb + c0 + rr];
            const int4 b = __ldg(p.blk + (int64_t)i * P + pass);
            rt->seg[rr] = make_int2(b.x, b.y);
            rt->item[rr] = i;
          }
          __syncthreads();
        }
        // no test per entry: real entries carry their slot, padding lands in the scratch slots behind the range
        sweep_rows(p.ent, rt, n, idle, [&](u64 e) {
          asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(acc_s + ((unsigned)e & 0xffffffu)), "r"((unsigned)(e >> sh_a) | 1u) : "memory");
        });
      }
      staged = d <= A32_ROWS;
      if (tid == 0) asm volatile("cp.async.wait_group 0;" ::: "memory");  // the next user's record has landed
      __syncthreads();
      PROF32_MARK(1);
      if (first) stage1(nxt);
      // the next range's table entry of this thread's row, written to the table once this range is done
      const bool pre = d <= A32_ROWS && pass + 1 < P && tid < d;
      if (pre) asm volatile("prefetch.global.L1 [%0];" ::"l"(p.blk + (int64_t)rt->item[tid] * P + pass + 1));
      if (p.mask) {  // pipelines/pipeline.py:174-175 -- before the truncation to N
        if (d <= A32_ROWS) {
          if (tid < d) {
            const int j = rt->item[tid] - r0;
            if (j >= 0 && j < ns) acc[j] = 0u;
          }
        } else {
          for (int rr = tid; rr < d; rr += nt) {
            const int j = p.indices[xb + rr] - r0;
            if (j >= 0 && j < ns) acc[j] = 0u;
          }
        }
        __syncthreads();
      }
      if (p.item_ok) {  // postprocessing/filters.py:58-101: filtered items are never recommended (4 items per word)
        const unsigned* ok4 = reinterpret_cast<const unsigned*>(p.item_ok + r0);
        for (int v = tid; v < nvec; v += nt) {
          const unsigned okw = 4 * v < ns ? __ldg(ok4 + v) : 0x01010101u;
          if (okw != 0x01010101u) {
            uint4 x = acc4[v];
            if (!(okw & 0xffu)) x.x = 0u;
            if (!(okw & 0xff00u)) x.y = 0u;
            if (!(okw & 0xff0000u)) x.z = 0u;
            if (!(okw & 0xff000000u)) x.w = 0u;
            acc4[v] = x;
          }
        }
        __syncthreads();
      }
      PROF32_MARK(2);
      // ---- survivor threshold.  Carried: with N entries in the list, an item can only reach the top N when its
      //      upper end (a + d) * 2^s reaches the N-th entry's lower end L (the order of the list is proven, so the
      //      lower ends decrease along it): a >= ceil(L / 2^s) - d.  With an approximate N-th entry a_N that is
      //      a_N - 2d, the rule of a range's own bound.
      unsigned thr_c = 1u;
      if (r >= N) {
        const u64 need = (a32_lo(list[N - 1], (u64)margin << sft) + ((1ull << sft) - 1)) >> sft;
        thr_c = need > (u64)d + 1 ? (unsigned)min(need - (u64)d, 0xffffffffull) : 1u;
      }
      const bool carried = r >= N && !own;
      unsigned thr = thr_c;
      if (!carried) {
        // own bound.  A dense pass costs a warp its full instruction stream whenever any of its lanes has work, so
        // the per-range work is kept out of it: every thread takes the maximum of its own slots (no branches, no
        // atomics), and the N-th largest of these per-thread maxima -- found with one histogram entry per thread,
        // 32 bins per octave -- is a lower bound of the N-th largest sum (N distinct items reach it).  Everything
        // within the margin below that bin survives.
        unsigned mymax = 0u;
        for (int v = tid; v < nvec; v += nt) {
          const uint4 x = acc4[v];
          mymax = max(mymax, max(max(x.x, x.y), max(x.z, x.w)));
        }
        // N-th largest of the 512 per-thread maxima, in two rounds of a 32-bin histogram (octave, then 32 bins
        // inside the octave).  Every warp scans the 32 bins by itself (one bin per lane), so no warp waits for
        // another one beyond the two barriers.
        const int mybin = mymax ? a32_bin(mymax) : -1;  // (octave << 5) | bin inside the octave
        if (mybin >= 0) atomicAdd(&hist[mybin >> 5], 1);
        __syncthreads();
        PROF32_MARK(12);
        if (first) stage2(nxt);
        int bstar = 0;
        {
          const int h1 = hist[lane];
          int incl = h1;  // maxima in my octave and the higher ones
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_down_sync(0xffffffffu, incl, o);
            if (lane + o < 32) incl += t;
          }
          const unsigned hit = __ballot_sync(0xffffffffu, incl >= N);  // lanes whose octave-and-above hold N maxima
          if (hit) {
            const int oct = 31 - __clz(hit);  // the highest such octave holds the N-th largest
            const int above = __shfl_sync(0xffffffffu, incl - h1, oct);
            if (mybin >= 0 && (mybin >> 5) == oct) atomicAdd(&hist[32 + (mybin & 31)], 1);
            __syncthreads();
            const int h2 = hist[32 + lane];
            int incl2 = h2;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const int t = __shfl_down_sync(0xffffffffu, incl2, o);
              if (lane + o < 32) incl2 += t;
            }
            const unsigned hit2 = __ballot_sync(0xffffffffu, above + incl2 >= N);
            bstar = (oct << 5) | (hit2 ? 31 - __clz(hit2) : 0);
          } else {
            __syncthreads();  // fewer than N non-empty threads: everything survives (bstar = 0)
          }
        }
        __syncthreads();  // every warp has read both histograms
        if (mybin >= 0) {
          hist[mybin >> 5] = 0;
          hist[32 + (mybin & 31)] = 0;
        }
        const unsigned edge = a32_bin_floor(bstar);
        thr = max(thr, edge > margin + 1u ? edge - margin : 1u);
      } else if (first) {
        stage2(nxt);
      }
      PROF32_MARK(13);
      // copy the survivors behind the running list, clear the accumulators: one compare per vector, the rest only
      // for the few that pass
      const int room = p.cap - r;
      for (int v = tid; v < nvec; v += nt) {
        const uint4 x = acc4[v];
        acc4[v] = make_uint4(0u, 0u, 0u, 0u);
        if (max(max(x.x, x.y), max(x.z, x.w)) < thr) continue;
        const unsigned xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (xs[q] >= thr) {
            const int pos = atomicAdd(&sh->count, 1);
            if (pos < room) {
              Entry e;
              e.key = ((u64)xs[q] + (u64)d) << sft;
              e.idx = r0 + 4 * v + q;
              e.aux = 1;
              list[r + pos] = e;
            }
          }
      }
      PROF32_MARK(14);
      if (first) stage3(nxt);
      first = false;
      __syncthreads();
      const int m = sh->count;
      const int tot = r + m;
      __syncthreads();  // every thread has read the count (thread 0 resets it at the next range)
      PROF32_MARK(3);
#ifdef RPK_PHASE_PROF
      if (tid == 0) {
        atomicAdd(p.prof + 10, 1ull);
        atomicAdd(p.prof + 11, (unsigned long long)(m > room ? 0 : m));
        if (carried) atomicAdd(p.prof + 17, 1ull);
      }
#endif
      if (m > room) {
        if (carried) {  // the carried bound is too loose for this range: sweep it again and take its own bound
#ifdef RPK_PHASE_PROF
          if (tid == 0) atomicAdd(p.prof + 16, 1ull);
#endif
          own = true;
          --pass;
          continue;
        }
        // survivors do not fit: the exact kernel takes the whole user
        if (tid == 0) p.ovf_tab[atomicAdd(p.ovf_count, 1)] = s_rec[cur];
        break;
      }
      own = false;
      // ---- sweep 2: exact scores of the entries of this range in s[0..tot) (slot -> place + 1, key -> exact sum);
      //      the accumulators are all zero again afterwards
      auto exact_pass = [&](Entry* s) {
#ifdef RPK_PHASE_PROF
        if (tid == 0) atomicAdd(p.prof + 9, 1ull);
#endif
        auto mine = [&](const Entry& e) { return e.aux && (unsigned)(e.idx - r0) < (unsigned)ns; };
        for (int t = tid; t < tot; t += nt)
          if (mine(s[t])) {
            acc[s[t].idx - r0] = (unsigned)t + 1u;
            s[t].key = 0ull;
          }
        __syncthreads();
        PROF32_MARK(4);
        const bool limbs = d <= LIMB_CHUNK;  // two 32-bit adds (20-bit limbs) cannot overflow
        for (int c0 = 0; c0 < d; c0 += A32_ROWS) {
          const int n = min(A32_ROWS, d - c0);
          if (d > A32_ROWS) {  // a single chunk is still staged from sweep 1
            if (c0 > 0) __syncthreads();
            for (int rr = tid; rr < n; rr += nt) {
              const int i = p.indices[xb + c0 + rr];
              const int4 b = __ldg(p.blk + (int64_t)i * P + pass);
              rt->seg[rr] = make_int2(b.x, b.y);
              rt->item[rr] = i;
            }
            __syncthreads();
          }
          sweep_rows(p.ent, rt, n, idle, [&](u64 e) {
            const unsigned j = ((unsigned)e & 0xffffffu) >> 2;
            if (j < (unsigned)ns) {
              const unsigned cn = acc[j];
              if (cn) {
                const u64 q = e >> 24;
                if (limbs) {
                  unsigned* wd = reinterpret_cast<unsigned*>(&s[cn - 1u].key);
                  atomicAdd(wd, (unsigned)q & LIMB_MASK);
                  atomicAdd(wd + 1, (unsigned)(q >> LIMB_BITS));
                } else {
                  atomicAdd(&s[cn - 1u].key, q);
                }
              }
            }
          });
        }
        __syncthreads();
        PROF32_MARK(5);
        for (int t = tid; t < tot; t += nt)
          if (mine(s[t])) {
            acc[s[t].idx - r0] = 0u;
            if (limbs) {
              const u64 kv = s[t].key;
              s[t].key = ((kv >> 32) << LIMB_BITS) + (kv & 0xffffffffull);
            }
            s[t].aux = 0;
          }
        __syncthreads();
      };
      // order the list; approximate keys that leave the order open take the exact pass (scores requested: all
      // of them, before the first ordering)
      Entry* s = list;
      bool restart = false;
      if (m > 0) {
        bool due = uexact, done = false;
        for (;;) {
          if (due) {
            exact_pass(s);
            done = true;
          }
          s = a32_order(s, s == list ? list2 : list, tot);
          if (uexact || !a32_unproven(s, tot, N, (u64)margin << sft)) break;
          if (done) {  // an approximate key of an earlier range is too close to call
            restart = true;
            break;
          }
          due = true;
        }
      }
      if (restart) {  // the user again, exact throughout
#ifdef RPK_PHASE_PROF
        if (tid == 0) atomicAdd(p.prof + 15, 1ull);
#endif
        uexact = true;
        staged = false;
        r = 0;
        pass = -1;
        continue;
      }
      const int keep = tot < N ? tot : N;
      if (pass + 1 == P) {  // the user's list is final
        const double inv = p.scale->inv;
        for (int t = tid; t < N; t += nt) {
          p.out_idx[(int64_t)u * N + t] = t < keep ? s[t].idx : -1;
          if (p.out_val) p.out_val[(int64_t)u * N + t] = t < keep ? (double)s[t].key * inv : 0.0;
        }
        if (tid == 0) p.out_len[u] = keep;
      } else {
        if (s != list)
          for (int t = tid; t < keep; t += nt) list[t] = s[t];
        if (pre) {
          const int4 b = __ldg(p.blk + (int64_t)rt->item[tid] * P + pass + 1);
          rt->seg[tid] = make_int2(b.x, b.y);
        }
      }
      r = keep;
      __syncthreads();
      PROF32_MARK(6);
    }
#ifdef RPK_PHASE_PROF
    if (tid == 0) atomicAdd(p.prof + 8, 1ull);
#endif
    __syncthreads();
  }
}

// Work table in processing order: one 16-byte record per user {user, history length, row start}, so that a
// CTA needs a single load (prefetched one item ahead) to start on a user.
__global__ void k_build_work_tab(const int* __restrict__ order, const int64_t* __restrict__ indptr, int64_t U,
                                 int4* __restrict__ tab) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= U) return;
  const int u = order[k];
  const int64_t xb = indptr[u];
  const int64_t d = indptr[u + 1] - xb;
  tab[k] = make_int4(u, (int)d, (int)(xb & 0xffffffffll), (int)(xb >> 32));
}

__global__ void k_row_lengths(const int64_t* __restrict__ indptr, int64_t U, u64* __restrict__ work) {
  int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u < U) work[u] = (u64)(indptr[u + 1] - indptr[u]);
}

// ------------------------------------------------------------------------------------------
// Host driver
// ------------------------------------------------------------------------------------------
static int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

struct PredGeom {
  int cap, direct_cap, P, R, nt;
  size_t fixed, smem;
};

static PredGeom predict_geometry(rpk_ctx* c, int N) {
  PredGeom g;
  const bool tiny = c->flags & DBG_TINY_LIST;
  g.cap = std::max(tiny ? 64 : 256, next_pow2(2 * std::max(N, 1)));
  g.direct_cap = tiny ? std::max(N, 1) : std::min(g.cap, std::max(64, 2 * N));
  // the user's running list (top-N), carried from range to range behind the accumulators
  g.fixed = sel_smem_bytes(g.cap) + (size_t)N * sizeof(Entry);
  RPK_REQUIRE((size_t)c->smem_max > g.fixed + 1024 + 8192, "N too large for shared memory");
  const size_t avail = (size_t)c->smem_max - g.fixed - 1024;
  const int64_t I = c->m_I;
  // 8 B of accumulator per item of a range
  int P = 1;
  int64_t R = 0;
  for (;; ++P) {
    R = ((I + P - 1) / P + 3) & ~(int64_t)3;
    if (R < 4) R = 4;
    if ((size_t)R * 8 <= avail) break;
  }
  const int p_min = (c->flags & DBG_MANY_PASS) ? 4 : ((c->flags & DBG_MULTI_PASS) ? 2 : 1);
  if (P < p_min && I >= 4 * p_min) {
    P = p_min;
    R = ((I + P - 1) / P + 3) & ~(int64_t)3;
  }
  g.P = P;
  g.R = (int)R;
  g.smem = g.fixed + (size_t)R * sizeof(u64);
  g.nt = g.R >= 8192 ? 1024 : (g.R >= 2048 ? 512 : 256);
  return g;
}

// Segment table of the two-limb kernel: offset of each item range inside every model row.
static void ensure_segments(rpk_ctx* c, const PredGeom& g) {
  if (c->m_P == g.P && c->m_R == g.R) return;
  const int64_t I = c->m_I;
  int* seg = c->buf<int>("m_seg", (size_t)I * (g.P + 1));
  if (I > 0) {
    k_model_seg<<<ceil_div(I * (g.P + 1), 256), 256, 0, c->stream>>>(c->get<int64_t>("m_ptr"), c->get<u64>("m_ent"), I, g.P,
                                                                      g.R, seg);
    RPK_LAUNCH_CHECK(c);
  }
  c->m_P = g.P;
  c->m_R = g.R;
}

// Block layout of the model for one geometry of the 32-bit kernel (rebuilt when the model or the geometry changes).
static void ensure_blocks(rpk_ctx* c, int P, int R) {
  if (c->m_pad && c->m_P2 == P && c->m_R2 == R) return;
  const int64_t I = c->m_I;
  cudaStream_t st = c->stream;
  const int64_t* m_ptr = c->get<int64_t>("m_ptr");
  const u64* m_ent = c->get<u64>("m_ent");
  const int64_t nseg = I * P;
  int2* seg = c->buf<int2>("m_seg2", (size_t)nseg);
  int* len4 = c->buf<int>("m_len4", (size_t)nseg);
  int64_t* ptr4 = c->buf<int64_t>("m_ptr4", (size_t)nseg + 1);
  int4* blk = c->buf<int4>("m_blk", (size_t)nseg);
  // every segment is padded by at most 3 entries
  u64* ent4 = c->buf<u64>("m_ent4", (size_t)c->m_nnz + 3 * (size_t)nseg + 4);
  if (nseg > 0) {
    k_model_seg_len<<<ceil_div(nseg, 256), 256, 0, st>>>(m_ptr, m_ent, I, P, R, seg, len4);
    RPK_LAUNCH_CHECK(c);
  }
  scan_i32_i64(c, len4, ptr4, nseg);
  if (nseg > 0) {
    k_model_pad<<<(int)std::min<int64_t>(ceil_div(nseg * 32, 256), (int64_t)c->sm_count * 32), 256, 0, st>>>(m_ptr, m_ent, seg, ptr4, I, P, R,
                                                                                                          ent4, blk);
    RPK_LAUNCH_CHECK(c);
  }
  c->m_pad = true;
  c->m_P2 = P;
  c->m_R2 = R;
}

// Geometry of the 32-bit kernel: two CTAs per SM when that costs at most one more item range than one CTA
// per SM would need (or at most three ranges), else one.
struct Pred32Geom {
  int cap, P, R, nt, ctas;
  size_t smem;
};

static Pred32Geom predict32_geometry(rpk_ctx* c, int N) {
  Pred32Geom g;
  const bool tiny = c->flags & DBG_TINY_LIST;
  g.cap = std::max(tiny ? 64 : 256, next_pow2(2 * std::max(N, 1)));
  const size_t fixed = a32_fixed_bytes(g.cap);
  const int64_t I = c->m_I;
  auto solve = [&](int ctas, int& P, int64_t& R) -> bool {
    const size_t per_cta = std::min<size_t>((size_t)c->smem_max, (size_t)c->smem_per_sm / ctas - 1024);
    if (per_cta < fixed + 1024 + 4096) return false;
    const size_t avail = per_cta - fixed - 256;
    for (P = 1;; ++P) {
      R = ((I + P - 1) / P + 3) & ~(int64_t)3;
      if (R < 4) R = 4;
      if ((size_t)R * 4 + 128 <= avail) return true;  // + 32 scratch slots for padding entries
      if (R <= 4) return false;
    }
  };
  int P1 = 0, P2 = 0;
  int64_t R1 = 0, R2 = 0;
  const bool ok1 = solve(1, P1, R1);
  const bool ok2 = solve(2, P2, R2);
  RPK_REQUIRE(ok1, "N too large for shared memory");
  bool two = ok2 && (P2 <= 3 || P2 <= P1 + 1);
  if (const char* e = getenv("RPK_PRED_CTAS")) {  // tuning hook
    const int v = atoi(e);
    if (v == 1) two = false;
    if (v == 2 && ok2) two = true;
  }
  g.ctas = two ? 2 : 1;
  g.P = two ? P2 : P1;
  int64_t R = two ? R2 : R1;
  const int p_min = (c->flags & DBG_MANY_PASS) ? 4 : ((c->flags & DBG_MULTI_PASS) ? 2 : 1);
  if (g.P < p_min && I >= 4 * p_min) {
    g.P = p_min;
    R = ((I + g.P - 1) / g.P + 3) & ~(int64_t)3;
  }
  g.R = (int)R;
  g.smem = fixed + (size_t)R * 4 + 128;
  g.nt = A32_NT;  // the kernel stages one history row per thread
  return g;
}

// Users in processing order (heaviest first) as 16-byte work records, plus the zeroed work counters.
struct PredWork {
  int4* tab;
  int* queue;   // [0]: two-limb kernel, [1]: 32-bit kernel
};

static PredWork prepare_work(rpk_ctx* c, int64_t U, const int64_t* indptr) {
  cudaStream_t st = c->stream;
  u64* work = c->buf<u64>("p_work", (size_t)U);
  int* order = c->buf<int>("p_order", (size_t)U);
  int* bcnt = c->buf<int>("p_bcnt", 65 * 2 + 4);
  int* boff = bcnt + 65;
  int* queue = boff + 65;  // [0] two-limb kernel, [1] 32-bit kernel
  RPK_CUDA(cudaMemsetAsync(bcnt, 0, sizeof(int) * (65 * 2 + 4), st));
  k_row_lengths<<<ceil_div(U, 256), 256, 0, st>>>(indptr, U, work);
  RPK_LAUNCH_CHECK(c);
  k_bucket_count<<<ceil_div(U, 256), 256, 0, st>>>(work, 0, U, bcnt);
  RPK_LAUNCH_CHECK(c);
  k_bucket_offsets<<<1, 32, 0, st>>>(bcnt, boff);
  RPK_LAUNCH_CHECK(c);
  k_bucket_scatter<<<ceil_div(U, 256), 256, 0, st>>>(work, 0, U, boff, order);
  RPK_LAUNCH_CHECK(c);
  int4* tab = c->buf<int4>("p_work_tab", (size_t)U);
  k_build_work_tab<<<ceil_div(U, 256), 256, 0, st>>>(order, indptr, U, tab);
  RPK_LAUNCH_CHECK(c);
  return PredWork{tab, queue};
}

// Launches the two-limb kernel on the records of pp.work_tab (pp.n_work: device-side count, or null = U).
static void launch_predict_kernel(rpk_ctx* c, PredParams& pp, const PredGeom& g, int64_t U) {
  RPK_CUDA(cudaFuncSetAttribute(k_predict, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
  int occ = 0;
  RPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_predict, g.nt, g.smem));
  RPK_REQUIRE(occ >= 1, "predict kernel does not fit on an SM");
  const int grid = (int)std::min<int64_t>(U, (int64_t)c->sm_count * occ);
  k_predict<<<grid, g.nt, g.smem, c->stream>>>(pp);
  RPK_LAUNCH_CHECK(c);
}

static void launch_predict(rpk_ctx* c, PredParams& pp, const PredGeom& g, int64_t U, const int64_t* indptr) {
  const PredWork w = prepare_work(c, U, indptr);
  pp.work_tab = w.tab;
  pp.n_work = nullptr;
  pp.queue = w.queue;
  c->ev_record(4);
  launch_predict_kernel(c, pp, g, U);
  c->ev_record(5);
  c->ev_valid[2] = true;
}

static const unsigned char* item_filter_ptr(rpk_ctx* c);

static void fill_common(rpk_ctx* c, PredParams& pp, const PredGeom& g, int64_t U, const int64_t* indptr,
                        const int32_t* indices, int N, int mask, int mode) {
  pp.indptr = indptr;
  pp.indices = indices;
  pp.m_ptr = c->get<int64_t>("m_ptr");
  pp.m_ent = c->get<u64>("m_ent");
  pp.m_seg = c->get<int>("m_seg");
  pp.n_work = nullptr;
  pp.m_rowmax = c->get<unsigned>("m_rowmax");
  pp.U = (int)U;
  pp.P = g.P;
  pp.R = g.R;
  pp.I = (int)c->m_I;
  pp.N = N;
  pp.mask = mask;
  pp.mode = mode;
  pp.force_wide = (c->flags & DBG_WIDE_ACC) ? 1 : 0;
  pp.cap = g.cap;
  pp.direct_cap = g.direct_cap;
  pp.out_idx = nullptr;
  pp.out_val = nullptr;
  pp.out_len = nullptr;
  pp.out_row_nnz = nullptr;
  pp.out_indptr = nullptr;
  pp.out_indices = nullptr;
  pp.out_values = nullptr;
  pp.scale = c->get<ModelScale>("m_scale");
  pp.item_ok = item_filter_ptr(c);
}

// Item filter of the predict calls: a copy of the caller's mask, normalised to 0 / 1 bytes and padded (with 1 = allowed)
// so that the kernels can read it four items at a time up to the end of the last item range.
__global__ void k_filter_copy(const unsigned char* __restrict__ in, int64_t I, int64_t padded, unsigned char* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < padded) out[j] = j < I ? (in[j] ? 1 : 0) : 1;
}

void run_predict_item_filter(rpk_ctx* c, const uint8_t* allowed_u, int64_t I) {
  if (!allowed_u) {
    c->filter_I = -1;
    return;
  }
  RPK_REQUIRE(I >= 0, "negative item count");
  const unsigned char* in = stage_in(c, allowed_u, (size_t)I, "p_item_ok_in");
  const int64_t padded = I + 4096;
  unsigned char* ok = c->buf<unsigned char>("p_item_ok", (size_t)padded);
  k_filter_copy<<<ceil_div(padded, 256), 256, 0, c->stream>>>(in, I, padded, ok);
  RPK_LAUNCH_CHECK(c);
  c->filter_I = I;
  if (!is_device_ptr(allowed_u)) RPK_CUDA(cudaStreamSynchronize(c->stream));  // the caller may reuse its buffer
}

static const unsigned char* item_filter_ptr(rpk_ctx* c) {
  if (c->filter_I < 0) return nullptr;
  RPK_REQUIRE(c->filter_I == c->m_I, "the item filter was set for a different number of items than the model has");
  return c->get<unsigned char>("p_item_ok");
}

static void check_predict_args(rpk_ctx* c, int64_t U, int64_t nnz) {
  RPK_REQUIRE(c->m_I > 0 || c->m_nnz == 0, "no similarity model loaded");
  RPK_REQUIRE(c->bufs.count("m_ptr") != 0, "no similarity model loaded (call rpk_model_load_* first)");
  RPK_REQUIRE(U >= 0 && nnz >= 0, "negative dimension");
  RPK_REQUIRE(U < ((int64_t)1 << 27), "too many users in one call; split the batch");
  RPK_REQUIRE(c->bufs.count("m_scale") != 0, "no similarity model loaded (call rpk_model_load_* first)");
}

static void predict_signed_topn(rpk_ctx* c, int64_t U, const int64_t* indptr, const int32_t* indices, int N, int mask_history,
                                int32_t* out_idx, double* out_val, int32_t* out_len);

void run_predict_topn(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u, int N,
                      int mask_history, int32_t* out_idx_u, double* out_val_u, int32_t* out_len_u) {
  check_predict_args(c, U, nnz);
  RPK_REQUIRE(N >= 1 && N <= 2048, "N must be in [1, 2048]");
  RPK_REQUIRE(out_idx_u && out_len_u, "out_idx / out_len must not be null");
  cudaStream_t st = c->stream;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "p_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "p_indices");
  Out<int32_t> o_idx, o_len;
  Out<double> o_val;
  o_idx.init(c, out_idx_u, (size_t)U * N, "p_out_idx");
  o_val.init(c, out_val_u, (size_t)U * N, "p_out_val");
  o_len.init(c, out_len_u, (size_t)U, "p_out_len");
  if (U > 0 && c->m_signed) {
    // exact float64 scores are computed for every list either way; without out_val they go to a scratch buffer
    double* val = o_val.dev ? o_val.dev : c->buf<double>("ps_val", (size_t)U * N);
    predict_signed_topn(c, U, indptr, indices, N, mask_history, o_idx.dev, val, o_len.dev);
  } else if (U > 0) {
    c->mark("predict: begin");
    PredGeom g = predict_geometry(c, N);
    ensure_segments(c, g);
    PredParams pp;
    fill_common(c, pp, g, U, indptr, indices, N, mask_history, PRED_TOPN);
    pp.out_idx = o_idx.dev;
    pp.out_val = o_val.dev;
    pp.out_len = o_len.dev;
    const ModelScale* scale = c->get<ModelScale>("m_scale");
    // the block table of the 32-bit kernel indexes 4-entry blocks with 32 bits
    const Pred32Geom g2 = predict32_geometry(c, N);
    const bool blocks_fit = (c->m_nnz + 3 * c->m_I * g2.P) / 4 < (int64_t)0x7fffffff;
    if ((c->flags & DBG_WIDE_ACC) || !blocks_fit) {  // debug flag / giant models: every user through the two-limb kernel
      launch_predict(c, pp, g, U, indptr);
    } else {
      ensure_blocks(c, g2.P, g2.R);
      Pred32Params qp;
      qp.indices = indices;
      qp.ent = c->get<u64>("m_ent4");
      qp.blk = c->get<int4>("m_blk");
      qp.U = (int)U;
      qp.P = g2.P;
      qp.R = g2.R;
      qp.I = (int)c->m_I;
      qp.N = N;
      qp.mask = mask_history;
      // lists only (no scores wanted): the approximate sums settle most lists, exact sums only where they do not
      qp.exact = (o_val.dev != nullptr || (c->flags & DBG_EXACT_SCORES)) ? 1 : 0;
      qp.item_ok = item_filter_ptr(c);
      qp.cap = g2.cap;
      qp.out_idx = o_idx.dev;
      qp.out_val = o_val.dev;
      qp.out_len = o_len.dev;
      qp.scale = scale;
      // users handed to the two-limb kernel (each at most once: the handoff leaves the user's range loop)
      qp.ovf_count = c->buf<int>("p_ovf_count", 1);
      qp.ovf_tab = c->buf<int4>("p_ovf_tab", (size_t)U);
      RPK_CUDA(cudaMemsetAsync(qp.ovf_count, 0, sizeof(int), st));
      const PredWork w = prepare_work(c, U, indptr);
      qp.work_tab = w.tab;
      qp.queue = w.queue + 1;
      qp.prof = nullptr;
#ifdef RPK_PHASE_PROF
      qp.prof = c->buf<unsigned long long>("p_prof32", 24);
      RPK_CUDA(cudaMemsetAsync(qp.prof, 0, 24 * sizeof(unsigned long long), st));  // 0-6 phases, 8-11 and 15-17 counters, 12-14 inside select
#endif
      RPK_CUDA(cudaFuncSetAttribute(k_predict_a32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g2.smem));
      int occ = 0;
      RPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_predict_a32, g2.nt, g2.smem));
      RPK_REQUIRE(occ >= 1, "predict kernel does not fit on an SM");
      const int grid = (int)std::min<int64_t>(U, (int64_t)c->sm_count * occ);
      c->mark("predict: layout + work table");
      c->ev_record(4);
      k_predict_a32<<<grid, g2.nt, g2.smem, st>>>(qp);
      RPK_LAUNCH_CHECK(c);
      c->mark("predict: scoring kernel");
      // users whose survivors overflowed the list: exact two-limb kernel, which writes their final lists (normally
      // none; the kernel then exits)
      pp.work_tab = qp.ovf_tab;
      pp.n_work = qp.ovf_count;
      pp.queue = w.queue;
      launch_predict_kernel(c, pp, g, U);
      c->ev_record(5);
      c->ev_valid[2] = true;
      c->mark("predict: exact passes");
#ifdef RPK_PHASE_PROF
      {
        unsigned long long h[24];
        int novf = 0;
        RPK_CUDA(cudaMemcpyAsync(h, qp.prof, sizeof(h), cudaMemcpyDeviceToHost, st));
        RPK_CUDA(cudaMemcpyAsync(&novf, qp.ovf_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        RPK_CUDA(cudaStreamSynchronize(st));
        static const char* nm[7] = {"fetch", "bound+sweep1", "mask", "select", "tag", "sweep2", "sort+out"};
        unsigned long long tot = 0;
        for (int k = 0; k < 7; ++k) tot += h[k];
        tot += h[12] + h[13] + h[14];
        const double us = h[8] ? (double)h[8] : 1.0;
        fprintf(stderr, "[predict32 phases] grid=%d nt=%d P=%d R=%d smem=%zu occ=%d exact=%d users=%llu ranges=%llu carried ranges=%llu "
                "carried retries=%llu exact range passes=%llu exact restarts=%llu survivors/user=%.1f overflow users=%d cycles/user=%.0f\n",
                grid, g2.nt, g2.P, g2.R, g2.smem, occ, qp.exact, h[8], h[10], h[17], h[16], h[9], h[15], (double)h[11] / us, novf,
                (double)tot / us);
        for (int k = 0; k < 7; ++k)
          fprintf(stderr, "  %-12s %5.1f%%  %8.0f cycles/user\n", nm[k], 100.0 * h[k] / (tot ? tot : 1), (double)h[k] / us);
        fprintf(stderr, "  select = thread maxima %.0f + boundary bin %.0f + copy/clear %.0f + staging of the next user %.0f cycles/user\n",
                (double)h[12] / us, (double)h[13] / us, (double)h[14] / us, (double)h[3] / us);
      }
#endif
    }
  }
  c->mark("predict: final lists");
  o_idx.finish(c);
  o_val.finish(c);
  o_len.finish(c);
  finish_call(c);
}

void run_predict_csr_count(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
                           int mask_history, int64_t* out_row_nnz_u) {
  check_predict_args(c, U, nnz);
  RPK_REQUIRE(out_row_nnz_u, "out_row_nnz must not be null");
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "p_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "p_indices");
  Out<int64_t> o;
  o.init(c, out_row_nnz_u, (size_t)U, "p_row_nnz");
  if (U > 0 && c->m_signed) {
    spgemm_rows_device(c, U, indptr, indices, nullptr, c->m_I, c->get<int64_t>("m_ptr"), c->get<int>("ms_idx"),
                       c->get<double>("ms_val"), nullptr, nullptr, 1, mask_history, item_filter_ptr(c), PRED_COUNT, nullptr,
                       nullptr, nullptr, o.dev, nullptr, nullptr, nullptr);
    c->pc_U = U;
  } else if (U > 0) {
    PredGeom g = predict_geometry(c, 1);
    ensure_segments(c, g);
    PredParams pp;
    fill_common(c, pp, g, U, indptr, indices, 1, mask_history, PRED_COUNT);
    pp.out_row_nnz = o.dev;
    launch_predict(c, pp, g, U, indptr);
    c->pc_U = U;
  }
  o.finish(c);
  finish_call(c);
}

void run_predict_csr_fill(rpk_ctx* c, int64_t U, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
                          int mask_history, const int64_t* out_indptr_u, int32_t* out_indices_u, double* out_values_u) {
  check_predict_args(c, U, nnz);
  RPK_REQUIRE(out_indptr_u && out_indices_u && out_values_u, "output pointers must not be null");
  if (U == 0) return;
  RPK_REQUIRE(c->pc_U == U, "rpk_predict_csr_fill must follow rpk_predict_csr_count on the same input");
  cudaStream_t st = c->stream;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)U + 1, "p_indptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "p_indices");
  const int64_t* out_indptr = stage_in(c, out_indptr_u, (size_t)U + 1, "p_out_indptr");
  int64_t total = 0;
  if (is_device_ptr(out_indptr_u)) {
    RPK_CUDA(cudaMemcpyAsync(&total, out_indptr + U, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));
  } else {
    total = out_indptr_u[U];
  }
  Out<int32_t> o_i;
  Out<double> o_v;
  o_i.init(c, out_indices_u, (size_t)total, "p_csr_idx");
  o_v.init(c, out_values_u, (size_t)total, "p_csr_val");
  if (c->m_signed) {
    spgemm_rows_device(c, U, indptr, indices, nullptr, c->m_I, c->get<int64_t>("m_ptr"), c->get<int>("ms_idx"),
                       c->get<double>("ms_val"), nullptr, nullptr, 1, mask_history, item_filter_ptr(c), PRED_FILL, nullptr,
                       nullptr, nullptr, nullptr, out_indptr, o_i.dev, o_v.dev);
    o_i.finish(c);
    o_v.finish(c);
    finish_call(c);
    return;
  }
  PredGeom g = predict_geometry(c, 1);
  ensure_segments(c, g);
  PredParams pp;
  fill_common(c, pp, g, U, indptr, indices, 1, mask_history, PRED_FILL);
  pp.out_indptr = out_indptr;
  pp.out_indices = o_i.dev;
  pp.out_values = o_v.dev;
  launch_predict(c, pp, g, U, indptr);
  o_i.finish(c);
  o_v.finish(c);
  finish_call(c);
}


// ------------------------------------------------------------------------------------------
// Signed models: float64 scores, bit-identical to scipy's X @ S
// ------------------------------------------------------------------------------------------
// A model with negative values is scored in float64: score_uj is the left fold of s_ij over the user's history rows in
// their stored (ascending) order, exactly scipy's csr_matmat, and a sum of exactly 0.0 is not stored.  k_predict_signed
// screens with signed fixed-point sums and folds in float64 only the items that can reach the list:
//   model    every entry is kept as (q << 24) | column, q = rint(v * 2^e) signed (|q| <= 2^38, e from max |v|), next to
//            its float64 value and column; rowmax = ceil(max |q| / 2^20) per row.
//   screen   the accumulator of item j is x = (sum of t_ij) * 2^c + (rows that touched j), t_ij = floor(q_ij / 2^sft),
//            c = bits of d (the history length), so x != 0 exactly when j was touched and a = x >> c is the signed sum.
//            sft is the smallest shift with (sum of rowmax * 2^20 >> sft + d) * 2^c + d < 2^31: no int32 overflow.
//            With unit = 2^(sft - e), each term satisfies v / unit in [t - 1/2, t + 3/2) (floor plus rint), and the
//            float64 fold differs from the real sum by at most gamma_{d-1} * sum |v| < unit (d < 2048), so the
//            float64 score lies in unit * [a - W, a + W], W = 2d + 2.
//   bound    L = the larger of (a_N - W) * unit, a_N the N-th largest of the per-thread maxima of a (N distinct items
//            reach it), and the N-th exact score carried from the earlier item ranges.  Survivors: the touched items
//            with (a + W) * unit >= L; every other item of the range scores strictly below L.
//   exact    the survivors' scores are folded in float64 in history order (their s_ij gathered into shared memory a
//            chunk of rows at a time), exact zeros dropped, merged with the carried list, ordered by (score desc,
//            column asc).  The list is proven when no touched item was screened out, or when its N-th score >= L.
//   fallback the user goes to the float64 row kernel (k_real_rows) when the survivors do not fit the list, when the
//            list is not proven (exact zeros left fewer than N scores >= L), and for histories of >= 2048 rows.
constexpr int SG_NT = 512;
constexpr int SG_EXACT_D = 2048;
#ifdef RPK_PHASE_PROF
constexpr int SG_LONG_SEG = 1024;  // counted: model row segments longer than this
#endif

__global__ void k_signed_vmax(const double* __restrict__ val, int64_t n, u64* __restrict__ vmax_bits, int* __restrict__ flag) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  u64 best = 0;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    const double v = fabs(val[t]);
    if (!(v <= 1.7976931348623157e308)) atomicOr(flag, 1);  // NaN or infinite
    else best = max(best, (u64)__double_as_longlong(v));
  }
  best = warp_max_u64(best);
  if ((threadIdx.x & 31) == 0 && best) atomicMax(vmax_bits, best);
}

// One warp per row of a CSR with ascending unique columns.
__global__ void k_model_from_signed_csr(const int64_t* __restrict__ indptr, const int* __restrict__ indices,
                                        const double* __restrict__ values, int64_t I, int e, u64* __restrict__ ent,
                                        unsigned* __restrict__ rowmax, int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < I; i += nwarps) {
    const int64_t b = indptr[i], en = indptr[i + 1];
    u64 qmax = 0;
    for (int64_t k = b + lane; k < en; k += 32) {
      const int j = indices[k];
      if (j < 0 || j >= I) atomicOr(flag, 1);
      if (k > b && indices[k - 1] >= j) atomicOr(flag, 2);
      const long long q = __double2ll_rn(scalbn(values[k], e));  // |q| <= 2^38
      qmax = max(qmax, (u64)(q < 0 ? -q : q));
      ent[k] = ((u64)q << 24) | (u64)(unsigned)(j & 0xffffff);
    }
    qmax = warp_max_u64(qmax);
    if (lane == 0) rowmax[i] = (unsigned)((qmax + 0xfffffull) >> 20);
  }
}

void run_model_load_signed_csr(rpk_ctx* c, int64_t I, int64_t nnz, const int64_t* indptr_u, const int32_t* indices_u,
                               const double* values_u) {
  model_common_begin(c, I);
  RPK_REQUIRE(nnz >= 0, "negative nnz");
  cudaStream_t st = c->stream;
  const int64_t* indptr = stage_in(c, indptr_u, (size_t)I + 1, "m_in_ptr");
  const int32_t* indices = stage_in(c, indices_u, (size_t)nnz, "m_in_idx");
  const double* values = stage_in(c, values_u, (size_t)nnz, "m_in_val");
  int64_t* m_ptr = c->buf<int64_t>("m_ptr", (size_t)I + 1);
  int32_t* m_idx = c->buf<int32_t>("ms_idx", (size_t)nnz);
  double* m_val = c->buf<double>("ms_val", (size_t)nnz);
  RPK_CUDA(cudaMemcpyAsync(m_ptr, indptr, sizeof(int64_t) * ((size_t)I + 1), cudaMemcpyDeviceToDevice, st));
  RPK_CUDA(cudaMemcpyAsync(m_idx, indices, sizeof(int32_t) * (size_t)nnz, cudaMemcpyDeviceToDevice, st));
  RPK_CUDA(cudaMemcpyAsync(m_val, values, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToDevice, st));
  u64* vmax = c->get<u64>("m_vmax");
  int* flag = c->get<int>("m_flag");
  if (nnz > 0) {
    k_signed_vmax<<<(int)std::min<int64_t>(ceil_div(nnz, 256), (int64_t)c->sm_count * 16), 256, 0, st>>>(values, nnz, vmax, flag);
    RPK_LAUNCH_CHECK(c);
  }
  u64 vb = 0;
  int64_t ends[2] = {0, 0};
  RPK_CUDA(cudaMemcpyAsync(&vb, vmax, sizeof(u64), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaMemcpyAsync(&ends[0], m_ptr, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaMemcpyAsync(&ends[1], m_ptr + I, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaStreamSynchronize(st));
  if (!(ends[0] == 0 && ends[1] == nnz)) {
    c->m_I = 0;
    throw Error("similarity model: indptr does not match nnz");
  }
  double vm = 0.0;
  memcpy(&vm, &vb, sizeof(vm));
  const int e = vm > 0.0 ? 37 - ilogb(vm) : 37;  // max |v| * 2^e in [2^37, 2^38)
  u64* ent = c->buf<u64>("ms_ent", (size_t)nnz);
  unsigned* rowmax = c->buf<unsigned>("ms_rowmax", (size_t)I);
  if (I > 0) {
    const int grid = (int)std::min<int64_t>((I * 32 + 255) / 256, (int64_t)c->sm_count * 16);
    k_model_from_signed_csr<<<grid, 256, 0, st>>>(indptr, indices, values, I, e, ent, rowmax, flag);
    RPK_LAUNCH_CHECK(c);
  }
  int h = 0;
  RPK_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  RPK_CUDA(cudaStreamSynchronize(st));
  if (h & 1) {
    c->m_I = 0;
    throw Error("similarity model: values must be finite, columns in [0, I)");
  }
  if (h & 2) {
    c->m_I = 0;
    throw Error("similarity model: column indices must be unique and ascending within a row");
  }
  ModelScale hs;
  hs.e = e;
  hs.inv = ldexp(1.0, -e);
  hs.pad = 0;
  RPK_CUDA(cudaMemcpyAsync(c->get<ModelScale>("m_scale"), &hs, sizeof(hs), cudaMemcpyHostToDevice, st));
  RPK_CUDA(cudaStreamSynchronize(st));
  c->m_exp = e;
  c->m_nnz = nnz;
  c->m_max_len = 0;
  c->m_signed = true;
  c->mark("model: signed CSR loaded (sync)");
}

// seg[i * (P + 1) + p] = offset inside row i of the first entry with column >= p * R
__global__ void k_signed_seg(const int64_t* __restrict__ m_ptr, const int* __restrict__ m_idx, int64_t I, int P, int R,
                             int* __restrict__ seg) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= I * (P + 1)) return;
  const int64_t i = t / (P + 1);
  const int p = (int)(t % (P + 1));
  const int64_t b = m_ptr[i];
  int lo = 0, hi = (int)(m_ptr[i + 1] - b);
  const int64_t target = (int64_t)p * R;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (m_idx[b + mid] < target) lo = mid + 1;
    else hi = mid;
  }
  seg[t] = lo;
}

struct SignedParams {
  const int* indices;    // histories (CSR columns of the users)
  const int4* work_tab;  // {user, history length, row start lo, hi} in processing order
  const int64_t* m_ptr;
  const int* seg;        // [I x (P + 1)] offset of every item range inside every model row
  const u64* ent;        // (q << 24) | column
  const double* val;     // float64 values of the entries
  const unsigned* rowmax;
  int U, P, R, N, mask, cap, gbuf, e;
  int* queue;
  int* out_idx;
  double* out_val;
  int* out_len;
  const unsigned char* item_ok;  // non-null: item filter (1 = may be recommended)
  int* ovf_count;                // users handed to the float64 row kernel ...
  int* ovf_users;                // ... and their ids
  unsigned long long* prof;      // instrumented build: path counters
};

__host__ __device__ __forceinline__ size_t sg_fixed_bytes(int cap, int gbuf) {
  return (size_t)(cap + SEL_RANK_MAX) * sizeof(Entry) + (size_t)cap * sizeof(double) + (size_t)gbuf * sizeof(double) +
         (size_t)SG_NT * (sizeof(int64_t) + sizeof(int));
}

__device__ __forceinline__ u64 sg_key(double v) {  // orders like v (v is never NaN)
  const u64 b = (u64)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double sg_value(u64 k) {
  const u64 b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

#ifdef RPK_PHASE_PROF
#define SG_COUNT(k, v) \
  do {                 \
    if (tid == 0) atomicAdd(p.prof + (k), (unsigned long long)(v)); \
  } while (0)
#else
#define SG_COUNT(k, v) do {} while (0)
#endif
enum { SGC_USERS, SGC_RANGES, SGC_SURVIVORS, SGC_OVERLAP, SGC_OVERFLOW, SGC_ZEROS, SGC_HEAVY, SGC_LONG, SGC_N };

// One CTA per user (heaviest first from a shared counter); the user's item ranges run in order on the same
// accumulators, which are all zero between ranges.
__global__ void __launch_bounds__(SG_NT) k_predict_signed(SignedParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  Entry* list = reinterpret_cast<Entry*>(smem);  // the user's running list, then this range's survivors behind it
  Entry* list2 = list + p.cap;                   // SEL_RANK_MAX entries
  double* fsum = reinterpret_cast<double*>(list2 + SEL_RANK_MAX);  // float64 folds of the survivors
  double* gbuf = fsum + p.cap;                   // gathered s_ij: [rows of a chunk x survivors]
  int64_t* tab_b = reinterpret_cast<int64_t*>(gbuf + p.gbuf);  // staged rows: first entry of the range's segment ...
  int* tab_n = reinterpret_cast<int*>(tab_b + SG_NT);          // ... and its length
  int* acc = tab_n + SG_NT;
  __shared__ int s_w, s_cnt, s_out, s_keep;
  __shared__ unsigned long long s_b20;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  const int N = p.N, P = p.P;
  for (int t = tid; t < p.R; t += nt) acc[t] = 0;
  for (;;) {
    __syncthreads();
    if (tid == 0) {
      s_w = atomicAdd(p.queue, 1);
      s_b20 = 0ull;
    }
    __syncthreads();
    const int w = s_w;
    if (w >= p.U) break;
    const int4 rec = p.work_tab[w];
    const int u = rec.x, d = rec.y;
    const int64_t xb = ((int64_t)(unsigned)rec.z) | ((int64_t)rec.w << 32);
    SG_COUNT(SGC_USERS, 1);
    if (d == 0) {  // user without history: empty prediction row
      for (int t = tid; t < N; t += nt) {
        p.out_idx[(int64_t)u * N + t] = -1;
        p.out_val[(int64_t)u * N + t] = 0.0;
      }
      if (tid == 0) p.out_len[u] = 0;
      continue;
    }
    if (d >= SG_EXACT_D) {  // the margin 2d + 2 would let too much through: float64 row kernel
      if (tid == 0) p.ovf_users[atomicAdd(p.ovf_count, 1)] = u;
      SG_COUNT(SGC_HEAVY, 1);
      continue;
    }
    // ---- shift of the fixed-point sums from the bound of the user's rows
    {
      u64 b = 0;
      for (int r = tid; r < d; r += nt) b += p.rowmax[p.indices[xb + r]];
      b = __reduce_add_sync(0xffffffffu, (unsigned)b);  // d < 2048 rows of at most 2^18 + 1 each: fits 32 bits
      if (lane == 0 && b) atomicAdd(&s_b20, b);
    }
    __syncthreads();
    const u64 B = s_b20 << 20;
    const int cb = 32 - __clz(d);  // count field: d < 2^cb
    int sft = 0;
    while ((((B >> sft) + (u64)d) << cb) + (u64)d > 0x7fffffffull) ++sft;
    const int sh = 24 + sft;
    const long long W = 2ll * d + 2;
    const int uexp = sft - p.e;  // unit = 2^uexp
    int r = 0;                   // entries of the running list (best first, exact)
    bool handed = false;
    for (int pass = 0; pass < P && !handed; ++pass) {
      const int r0 = pass * p.R;
      // ---- screen: one shared-memory reduction per model entry
      for (int c0 = 0; c0 < d; c0 += SG_NT) {
        const int n = min(SG_NT, d - c0);
        __syncthreads();
        if (tid < n) {
          const int i = p.indices[xb + c0 + tid];
          const int* sg = p.seg + (int64_t)i * (P + 1) + pass;
          const int s0 = sg[0], s1 = sg[1];
          tab_b[tid] = p.m_ptr[i] + s0;
          tab_n[tid] = s1 - s0;
#ifdef RPK_PHASE_PROF
          if (s1 - s0 > SG_LONG_SEG) atomicAdd(p.prof + SGC_LONG, 1ull);
#endif
        }
        __syncthreads();
        for (int rr = warp; rr < n; rr += nwarps) {
          const u64* row = p.ent + tab_b[rr];
          const int len = tab_n[rr];
          for (int k = lane; k < len; k += 32) {
            const u64 e = __ldg(row + k);
            const unsigned add = ((unsigned)(int)((long long)e >> sh) << cb) + 1u;
            asm volatile("red.shared.add.u32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(acc + ((int)(e & 0xffffff) - r0))),
                         "r"(add)
                         : "memory");
          }
        }
      }
      __syncthreads();
      const int ns = p.R;  // slots of this range (those beyond the last item are never touched)
      if (p.mask) {  // pipelines/pipeline.py:174-175, before the truncation to N
        for (int rr = tid; rr < d; rr += nt) {
          const int j = p.indices[xb + rr] - r0;
          if (j >= 0 && j < ns) acc[j] = 0;
        }
      }
      if (p.item_ok) {  // postprocessing/filters.py:58-101
        for (int t = tid; t < ns; t += nt)
          if (acc[t] && !p.item_ok[r0 + t]) acc[t] = 0;
      }
      __syncthreads();
      // ---- bound: the N-th largest of the per-thread maxima of a (bit by bit, one block count per bit)
      unsigned mykey = 0u;  // 0: no touched slot; else a ^ 2^31 (orders like a)
      for (int t = tid; t < ns; t += nt) {
        const int x = acc[t];
        if (x) mykey = max(mykey, (unsigned)(x >> cb) ^ 0x80000000u);
      }
      if (tid == 0) {
        s_cnt = 0;
        s_out = 0;
        s_keep = 0;
      }
      long long thr = LLONG_MIN;  // survivors: a >= thr
      double L = -INFINITY;       // the N-th stored score is at least L (when the list is proven)
      if (__syncthreads_count(mykey != 0u) >= N) {
        unsigned pre = 0u;
        for (int bit = 31; bit >= 0; --bit) {
          const unsigned cand = pre | (1u << bit);
          if (__syncthreads_count(mykey >= cand) >= N) pre = cand;
        }
        const long long aN = (long long)(int)(pre ^ 0x80000000u);
        thr = aN - 2 * W;
        L = scalbn((double)(aN - W), uexp);
      }
      if (r >= N) {  // the carried N-th exact score
        const double EN = sg_value(list[N - 1].key);
        const double up = ceil(scalbn(EN, -uexp));
        const long long tc = up > 4.0e18 ? LLONG_MAX / 2 : (up < -4.0e18 ? LLONG_MIN / 2 : (long long)up - W);
        thr = max(thr, tc);
        L = fmax(L, EN);
      }
      // ---- survivors behind the running list; every touched slot is cleared
      const int room = p.cap - r;
      for (int t = tid; t < ns; t += nt) {
        const int x = acc[t];
        if (!x) continue;
        acc[t] = 0;
        if ((long long)(x >> cb) >= thr) {
          const int pos = atomicAdd(&s_cnt, 1);
          if (pos < room) {
            Entry en;
            en.key = 0ull;
            en.idx = r0 + t;
            en.aux = 0;
            list[r + pos] = en;
          }
        } else {
          s_out = 1;
        }
      }
      __syncthreads();
      const int m = s_cnt;
      const bool screened_out = s_out != 0;
      SG_COUNT(SGC_RANGES, 1);
      SG_COUNT(SGC_SURVIVORS, m);
      if (m > N) SG_COUNT(SGC_OVERLAP, 1);
      if (m > room) {  // the survivors do not fit the list
        if (tid == 0) p.ovf_users[atomicAdd(p.ovf_count, 1)] = u;
        SG_COUNT(SGC_OVERFLOW, 1);
        handed = true;
        break;
      }
      // ---- exact pass: float64 left folds of the survivors, rows in history order
      if (m > 0) {
        Entry* sv = list + r;
        for (int t = tid; t < m; t += nt) {
          acc[sv[t].idx - r0] = t + 1;
          fsum[t] = 0.0;
        }
        const int dc = min(SG_NT, max(1, p.gbuf / m));  // rows per gathered chunk
        int tc0 = 0, tn = min(SG_NT, d);                // rows staged in the table (the last screen chunk)
        if (d > SG_NT) tc0 = ((d - 1) / SG_NT) * SG_NT, tn = d - tc0;
        for (int g0 = 0; g0 < d; g0 += dc) {
          const int gn = min(dc, d - g0);
          __syncthreads();  // the previous chunk is folded
          if (g0 < tc0 || g0 + gn > tc0 + tn) {
            tc0 = g0;
            tn = min(SG_NT, d - g0);
            if (tid < tn) {
              const int i = p.indices[xb + tc0 + tid];
              const int* sg = p.seg + (int64_t)i * (P + 1) + pass;
              tab_b[tid] = p.m_ptr[i] + sg[0];
              tab_n[tid] = sg[1] - sg[0];
            }
          }
          for (int t = tid; t < gn * m; t += nt) gbuf[t] = 0.0;
          __syncthreads();
          for (int rr = warp; rr < gn; rr += nwarps) {
            const int64_t b = tab_b[g0 - tc0 + rr];
            const int len = tab_n[g0 - tc0 + rr];
            for (int k = lane; k < len; k += 32) {
              const int sidx = acc[(int)(__ldg(p.ent + b + k) & 0xffffff) - r0];
              if (sidx) gbuf[rr * m + sidx - 1] = __ldg(p.val + b + k);
            }
          }
          __syncthreads();
          for (int t = tid; t < m; t += nt) {
            double f = fsum[t];
            for (int k = 0; k < gn; ++k) f = __dadd_rn(f, gbuf[k * m + t]);  // + 0.0 where row k has no entry j
            fsum[t] = f;
          }
        }
        __syncthreads();
        // stored survivors (non-zero folds) -> gbuf as entries, then back behind the running list
        Entry* tmp = reinterpret_cast<Entry*>(gbuf);
        for (int t = tid; t < m; t += nt) {
          Entry en = sv[t];
          acc[en.idx - r0] = 0;
          const double v = fsum[t];
          if (v != 0.0) {
            en.key = sg_key(v);
            tmp[atomicAdd(&s_keep, 1)] = en;
          }
        }
        __syncthreads();
        const int kept = s_keep;
        for (int t = tid; t < kept; t += nt) sv[t] = tmp[t];
        __syncthreads();
        const int tot = r + kept;
        Entry* s = tot > 1 ? a32_order(list, list2, tot) : list;
        const int keep = min(tot, N);
        if (s != list) {
          for (int t = tid; t < keep; t += nt) list[t] = s[t];
          __syncthreads();
        }
        r = keep;
      }
      // the list is proven when nothing was screened out, or when its N-th score reaches L
      if (screened_out && (r < N || sg_value(list[N - 1].key) < L)) {
        if (tid == 0) p.ovf_users[atomicAdd(p.ovf_count, 1)] = u;
        SG_COUNT(SGC_ZEROS, 1);
        handed = true;
        break;
      }
      __syncthreads();
    }
    if (handed) continue;
    for (int t = tid; t < N; t += nt) {
      p.out_idx[(int64_t)u * N + t] = t < r ? list[t].idx : -1;
      p.out_val[(int64_t)u * N + t] = t < r ? sg_value(list[t].key) : 0.0;
    }
    if (tid == 0) p.out_len[u] = r;
  }
}

static void predict_signed_topn(rpk_ctx* c, int64_t U, const int64_t* indptr, const int32_t* indices, int N, int mask_history,
                                int32_t* out_idx, double* out_val, int32_t* out_len) {
  cudaStream_t st = c->stream;
  const int64_t I = c->m_I;
  const bool tiny = c->flags & DBG_TINY_LIST;
  const int cap = std::max(tiny ? 64 : 256, next_pow2(2 * N));
  const int gbuf = std::max(2048, 2 * cap);  // also holds cap entries (16 B) while the survivors are compacted
  const size_t fixed = sg_fixed_bytes(cap, gbuf);
  // two CTAs per SM when the accumulators of the item ranges still fit, else one
  auto ranges = [&](int ctas, int64_t& R) -> int {
    const size_t per_cta = std::min<size_t>((size_t)c->smem_max, (size_t)c->smem_per_sm / ctas - 1024);
    if (per_cta < fixed + 4096) return 0;
    const int64_t Rmax = (int64_t)((per_cta - fixed) / sizeof(int)) & ~(int64_t)3;
    const int P = (int)std::max<int64_t>(1, (I + Rmax - 1) / Rmax);
    R = ((I + P - 1) / P + 3) & ~(int64_t)3;
    return P;
  };
  int64_t R1 = 0, R2 = 0;
  const int P1 = ranges(1, R1), P2 = ranges(2, R2);
  RPK_REQUIRE(P1 > 0, "N too large for shared memory");
  const bool two = P2 > 0 && (P2 <= 3 || P2 <= P1 + 1);
  int P = two ? P2 : P1;
  int64_t R = std::max<int64_t>(4, two ? R2 : R1);
  const int p_min = (c->flags & DBG_MANY_PASS) ? 4 : ((c->flags & DBG_MULTI_PASS) ? 2 : 1);
  if (P < p_min && I >= 4 * p_min) {
    P = p_min;
    R = ((I + P - 1) / P + 3) & ~(int64_t)3;
  }
  const size_t smem = fixed + (size_t)R * sizeof(int);
  if (c->m_P != P || c->m_R != (int)R) {
    int* seg = c->buf<int>("ms_seg", (size_t)I * (P + 1));
    if (I > 0) {
      k_signed_seg<<<ceil_div(I * (P + 1), 256), 256, 0, st>>>(c->get<int64_t>("m_ptr"), c->get<int>("ms_idx"), I, P, (int)R, seg);
      RPK_LAUNCH_CHECK(c);
    }
    c->m_P = P;
    c->m_R = (int)R;
  }
  SignedParams sp;
  sp.indices = indices;
  sp.m_ptr = c->get<int64_t>("m_ptr");
  sp.seg = c->get<int>("ms_seg");
  sp.ent = c->get<u64>("ms_ent");
  sp.val = c->get<double>("ms_val");
  sp.rowmax = c->get<unsigned>("ms_rowmax");
  sp.U = (int)U;
  sp.P = P;
  sp.R = (int)R;
  sp.N = N;
  sp.mask = mask_history;
  sp.cap = cap;
  sp.gbuf = gbuf;
  sp.e = c->m_exp;
  sp.out_idx = out_idx;
  sp.out_val = out_val;
  sp.out_len = out_len;
  sp.item_ok = item_filter_ptr(c);
  sp.ovf_count = c->buf<int>("ps_ovf_count", 1);
  sp.ovf_users = c->buf<int>("ps_ovf_users", (size_t)U);
  RPK_CUDA(cudaMemsetAsync(sp.ovf_count, 0, sizeof(int), st));
  const PredWork w = prepare_work(c, U, indptr);
  sp.work_tab = w.tab;
  sp.queue = w.queue + 1;
  sp.prof = nullptr;
#ifdef RPK_PHASE_PROF
  sp.prof = c->buf<unsigned long long>("ps_prof", SGC_N);
  RPK_CUDA(cudaMemsetAsync(sp.prof, 0, SGC_N * sizeof(unsigned long long), st));
#endif
  RPK_CUDA(cudaFuncSetAttribute(k_predict_signed, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  RPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_predict_signed, SG_NT, smem));
  RPK_REQUIRE(occ >= 1, "predict kernel does not fit on an SM");
  const int grid = (int)std::min<int64_t>(U, (int64_t)c->sm_count * occ);
  c->mark("predict signed: work table");
  c->ev_record(4);
  k_predict_signed<<<grid, SG_NT, smem, st>>>(sp);
  RPK_LAUNCH_CHECK(c);
  // the users handed over: float64 rows of X @ S with unit left values (normally few; the kernel then exits)
  spgemm_rows_device(c, U, indptr, indices, nullptr, I, sp.m_ptr, c->get<int>("ms_idx"), sp.val, sp.ovf_users, sp.ovf_count, N,
                     mask_history, sp.item_ok, 0, out_idx, out_val, out_len, nullptr, nullptr, nullptr, nullptr);
  c->ev_record(5);
  c->ev_valid[2] = true;
  c->mark("predict signed: scoring");
#ifdef RPK_PHASE_PROF
  {
    unsigned long long h[SGC_N];
    RPK_CUDA(cudaMemcpyAsync(h, sp.prof, sizeof(h), cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));
    fprintf(stderr, "[predict signed paths] grid=%d P=%d R=%lld smem=%zu occ=%d users=%llu ranges=%llu survivors=%llu "
            "overlap ranges=%llu overflow users=%llu zero users=%llu heavy users=%llu long segments=%llu\n",
            grid, P, (long long)R, smem, occ, h[SGC_USERS], h[SGC_RANGES], h[SGC_SURVIVORS], h[SGC_OVERLAP], h[SGC_OVERFLOW],
            h[SGC_ZEROS], h[SGC_HEAVY], h[SGC_LONG]);
  }
#endif
}

}  // namespace rpk
