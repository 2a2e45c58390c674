// Dense co-occurrence Gram on the 5th-generation tensor cores:  G = A * A^T  for a 0/1 int8 matrix
// A [items x users] (users contiguous = K-major for both operands), exact int32 accumulation in TMEM,
// written out as uint16 counts, or as uint8 counts when A has at most 255 user columns.  This is the dense leg of ItemKNN.fit for the densest user columns of
// the interaction matrix (the reference computes the same counts with scipy's csr_matmat,
// recpack/algorithms/nearest_neighbour.py:48,80); the sparse leg (fit.cu) adds the remaining users on
// top of these counts and runs the fused epilogue.
//
// Kernel shape (one CTA per SM, persistent over output tiles, warp-specialised):
//   warp 0      TMA producer: cp.async.bulk.tensor 128 B-swizzled boxes of A into a 4-stage smem ring
//   warp 1      MMA issuer:   tcgen05.mma.cta_group::1.kind::i8, M=128 N=256 K=32, SS operands,
//                             accumulators double-buffered in TMEM (2 x 256 columns)
//   warps 2..5  epilogue:     tcgen05.ld 32x32b.x32 -> pack to uint16 -> 64 B row segments to global, or
//                             (uint8) -> 128 B-swizzled 32 x 128 staging boxes in smem -> TMA tensor stores
//
// The uint8 output halves the bytes of the count strip, and the TMA store writes whole 128 B row runs of the
// tile instead of 16 B pieces of 32 different rows per warp store (that store pattern bounds the uint16 kernel
// at small Kd, DESIGN.md 7).
#include <cuda.h>

#include "common.cuh"
#include "internal.h"
#include "tc.cuh"

namespace rpk {

constexpr int TC_BM = 128;       // UMMA M (cta_group::1)
constexpr int TC_BN = 256;       // UMMA N
constexpr int TC_BK = 128;       // bytes (= int8 elements) per k-block: one 128 B swizzle atom row
constexpr int TC_UMMA_K = 32;    // int8 elements per tcgen05.mma
constexpr int TC_STAGES = 4;
constexpr int TC_A_BYTES = TC_BM * TC_BK;  // 16 KB
constexpr int TC_B_BYTES = TC_BN * TC_BK;  // 32 KB
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr uint32_t TC_TMEM_COLS = 512;
constexpr int TC_THREADS = 192;  // 6 warps
// uint8 epilogue: each epilogue warp stages its 32 rows x 256 columns as two 32 x 128 B boxes
constexpr int TC_STG_BOX_ROWS = 32, TC_STG_BOX_COLS = 128;
constexpr int TC_STG_WARP_BYTES = 2 * TC_STG_BOX_ROWS * TC_STG_BOX_COLS;  // 8 KB
constexpr int TC_STG_BYTES = 4 * TC_STG_WARP_BYTES;                         // 32 KB
template <class OutT>
constexpr size_t tc_smem_bytes() {
  return (size_t)TC_STAGES * TC_STAGE_BYTES + (sizeof(OutT) == 1 ? TC_STG_BYTES : 0) + 1024 /*alignment slack*/ +
         256 /*barriers*/;
}

// D[tmem] (+)= A[smem] * B[smem]^T, int8 x int8 -> int32
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Instruction descriptor: dense, no saturation, D = S32, A = B = unsigned 8 bit, both K-major, N, M.
__host__ __device__ constexpr uint32_t umma_idesc_i8(int M, int N) {
  return (2u << 4) | (0u << 7) | (0u << 10) | (0u << 15) | (0u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

struct GramParams {
  int m_tiles, n_tiles, k_blocks;
  int row_begin;    // first row of G that is computed (multiple of 128); G points at it
  int rows_valid;   // rows of A / columns of G that exist; rows >= row_end are not written
  int row_end;
  int64_t ldg;      // leading dimension of G in elements (multiple of 32)
  void* G;          // OutT [(row_end - row_begin) x ldg]; the uint8 kernel writes it through map_g
};

template <class OutT>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_gram_i8_tc(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
             const __grid_constant__ CUtensorMap map_g, GramParams p) {
  constexpr bool U8 = sizeof(OutT) == 1;
  extern __shared__ unsigned char smem_raw[];
  // 128 B swizzle needs 1024 B aligned tiles
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* smem_a = smem;
  unsigned char* smem_b = smem + (size_t)TC_STAGES * TC_A_BYTES;
  unsigned char* smem_stg = smem + (size_t)TC_STAGES * TC_STAGE_BYTES;  // uint8 only
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_stg + (U8 ? TC_STG_BYTES : 0));
  uint64_t* full_bar = bars;                      // [TC_STAGES]
  uint64_t* empty_bar = bars + TC_STAGES;         // [TC_STAGES]
  uint64_t* tmem_full = bars + 2 * TC_STAGES;     // [2]
  uint64_t* tmem_empty = bars + 2 * TC_STAGES + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles_total = p.m_tiles * p.n_tiles;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    if (U8) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_g) : "memory");
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // one full warp allocates all 512 TMEM columns (two 256-column accumulators)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TC_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < n_tiles_total; t += gridDim.x) {
        const int m_blk = t / p.n_tiles, n_blk = t % p.n_tiles;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], TC_STAGE_BYTES);
          tma_load_2d(smem_a + (size_t)stage * TC_A_BYTES, &map_a, &full_bar[stage], kb * TC_BK, p.row_begin + m_blk * TC_BM);
          tma_load_2d(smem_b + (size_t)stage * TC_B_BYTES, &map_b, &full_bar[stage], kb * TC_BK, n_blk * TC_BN);
          if (++stage == TC_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_i8(TC_BM, TC_BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int t = blockIdx.x; t < n_tiles_total; t += gridDim.x) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)acc * TC_BN;
        for (int kb = 0; kb < p.k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);  // TMA bytes have landed
          tc_fence_after();
          const uint64_t da = umma_desc_kmajor_sw128(smem_u32(smem_a + (size_t)stage * TC_A_BYTES));
          const uint64_t db = umma_desc_kmajor_sw128(smem_u32(smem_b + (size_t)stage * TC_B_BYTES));
#pragma unroll
          for (int k = 0; k < TC_BK / TC_UMMA_K; ++k) {
            // advance 32 B along K inside the 128 B swizzle atom: +2 in 16 B units on the start address
            umma_i8(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // frees the smem slot when these MMAs have read it
          if (++stage == TC_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&tmem_full[acc]);  // accumulator complete -> epilogue
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // ===================== epilogue: TMEM -> registers -> OutT -> global =====================
    const int quarter = warp & 3;  // a warp may only touch TMEM lanes 32*(warp%4) .. +31
    unsigned char* stg = smem_stg + quarter * TC_STG_WARP_BYTES;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = blockIdx.x; t < n_tiles_total; t += gridDim.x) {
      const int m_blk = t / p.n_tiles, n_blk = t % p.n_tiles;
      if (U8) {  // the staging boxes are free again once the previous tile's stores have read them
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const int row = p.row_begin + m_blk * TC_BM + quarter * 32 + lane;
      unsigned short* grow = reinterpret_cast<unsigned short*>(p.G) + (int64_t)(row - p.row_begin) * p.ldg + (int64_t)n_blk * TC_BN;
#pragma unroll 1
      for (int c = 0; c < TC_BN / 32; ++c) {
        uint32_t v[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * TC_BN + c * 32);
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
        if (U8) {
          // every count is <= 255: 32 counts = 32 B of this lane's row, two 16 B chunks of a 128 B swizzled box row
          // (chunk k of row r sits at chunk k ^ (r & 7): the 8 lanes of a quarter-warp hit 8 different bank groups)
          uint32_t w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) w[q] = v[4 * q] | (v[4 * q + 1] << 8) | (v[4 * q + 2] << 16) | (v[4 * q + 3] << 24);
          unsigned char* brow = stg + (c >> 2) * (TC_STG_BOX_ROWS * TC_STG_BOX_COLS) + lane * TC_STG_BOX_COLS;
          const int k0 = (c & 3) * 2;
          *reinterpret_cast<uint4*>(brow + ((k0 ^ (lane & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
          *reinterpret_cast<uint4*>(brow + (((k0 + 1) ^ (lane & 7)) << 4)) = make_uint4(w[4], w[5], w[6], w[7]);
        } else if (row < p.row_end) {
          uint4* dst = reinterpret_cast<uint4*>(grow + c * 32);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint4 o;
            o.x = (v[8 * q + 0] & 0xffffu) | (v[8 * q + 1] << 16);
            o.y = (v[8 * q + 2] & 0xffffu) | (v[8 * q + 3] << 16);
            o.z = (v[8 * q + 4] & 0xffffu) | (v[8 * q + 5] << 16);
            o.w = (v[8 * q + 6] & 0xffffu) | (v[8 * q + 7] << 16);
            dst[q] = o;
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);  // 128 arrivals release the accumulator
      if (U8) {
        // generic-proxy smem writes -> visible to the async proxy, then one lane stores the warp's two boxes
        // (rows past the tensor map's row count, i.e. >= row_end, are not written)
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          const int r = m_blk * TC_BM + quarter * 32;
          tma_store_2d(&map_g, stg, n_blk * TC_BN, r);
          tma_store_2d(&map_g, stg + TC_STG_BOX_ROWS * TC_STG_BOX_COLS, n_blk * TC_BN + TC_STG_BOX_COLS, r);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (U8 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // smem must outlive the stores
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
// A: device, [rows_pad x kd_pad] uint8 row-major, rows_pad % 256 == 0, kd_pad % 128 == 0.
// Computes rows [row_begin, row_end) of G = A A^T (row_begin % 128 == 0) against all columns.
// G: device, [(row_end - row_begin) x ldg] OutT, ldg >= rows_pad.  OutT = uint8 needs at most 255 ones in every row
// of A (the caller's dense-user count), so that no count exceeds 255.
template <class OutT>
static void gram_dense_tc(rpk_ctx* c, const unsigned char* A, int64_t rows_pad, int64_t kd_pad, int64_t row_begin,
                          int64_t row_end, OutT* G, int64_t ldg) {
  constexpr bool U8 = sizeof(OutT) == 1;
  RPK_REQUIRE(rows_pad % TC_BN == 0 && kd_pad % TC_BK == 0 && kd_pad >= TC_BK, "dense Gram: operand is not tile aligned");
  RPK_REQUIRE(kd_pad <= 65535, "dense Gram: counts must fit 16 bits");
  RPK_REQUIRE(ldg >= rows_pad && ldg % 32 == 0, "dense Gram: bad output stride");
  RPK_REQUIRE(row_begin % TC_BM == 0 && row_begin <= row_end && row_end <= rows_pad, "dense Gram: bad row range");
  if (row_end == row_begin) return;
  CUtensorMap map_a, map_b, map_g;
  const cuuint64_t dims[2] = {(cuuint64_t)kd_pad, (cuuint64_t)rows_pad};
  const cuuint64_t strides[1] = {(cuuint64_t)kd_pad};
  const cuuint32_t box_a[2] = {TC_BK, TC_BM}, box_b[2] = {TC_BK, TC_BN}, estr[2] = {1, 1};
  EncodeTiledFn enc = get_encode_tiled();
  CUresult r1 = enc(&map_a, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<unsigned char*>(A), dims, strides, box_a, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CUresult r2 = enc(&map_b, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<unsigned char*>(A), dims, strides, box_b, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CUresult r3 = CUDA_SUCCESS;
  memset(&map_g, 0, sizeof(map_g));
  if (U8) {
    // the output strip: ldg columns x (row_end - row_begin) rows, written in 128 B x 32-row swizzled boxes
    const cuuint64_t gdims[2] = {(cuuint64_t)ldg, (cuuint64_t)(row_end - row_begin)};
    const cuuint64_t gstrides[1] = {(cuuint64_t)ldg};
    const cuuint32_t box_g[2] = {TC_STG_BOX_COLS, TC_STG_BOX_ROWS};
    r3 = enc(&map_g, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, G, gdims, gstrides, box_g, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  RPK_REQUIRE(r1 == CUDA_SUCCESS && r2 == CUDA_SUCCESS && r3 == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed");
  GramParams p;
  p.m_tiles = (int)(rows_pad / TC_BM);
  p.n_tiles = (int)(rows_pad / TC_BN);
  p.k_blocks = (int)(kd_pad / TC_BK);
  p.row_begin = (int)row_begin;
  p.row_end = (int)row_end;
  p.rows_valid = (int)row_end;
  p.ldg = ldg;
  p.G = G;
  p.m_tiles = (int)((row_end - row_begin + TC_BM - 1) / TC_BM);
  constexpr size_t smem = tc_smem_bytes<OutT>();
  RPK_REQUIRE(smem <= (size_t)c->smem_max, "dense Gram: shared memory ring does not fit");
  RPK_CUDA(cudaFuncSetAttribute(k_gram_i8_tc<OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = std::min(c->sm_count, p.m_tiles * p.n_tiles);
  k_gram_i8_tc<OutT><<<std::max(grid, 1), TC_THREADS, smem, c->stream>>>(map_a, map_b, map_g, p);
  RPK_LAUNCH_CHECK(c);
}

void run_gram_dense_tc(rpk_ctx* c, const unsigned char* A, int64_t rows_pad, int64_t kd_pad, int64_t row_begin,
                       int64_t row_end, unsigned short* G, int64_t ldg) {
  gram_dense_tc(c, A, rows_pad, kd_pad, row_begin, row_end, G, ldg);
}

void run_gram_dense_tc(rpk_ctx* c, const unsigned char* A, int64_t rows_pad, int64_t kd_pad, int64_t row_begin,
                       int64_t row_end, unsigned char* G, int64_t ldg) {
  RPK_REQUIRE(ldg % 16 == 0, "dense Gram: uint8 output stride must be a multiple of 16 B");
  gram_dense_tc(c, A, rows_pad, kd_pad, row_begin, row_end, G, ldg);
}

// Test / bring-up entry: G = A A^T for a caller-provided 0/1 matrix.
void run_gram_dense_u16(rpk_ctx* c, int64_t I, int64_t Kd, const unsigned char* A_u, unsigned short* G_u) {
  RPK_REQUIRE(I >= 1 && Kd >= 1 && Kd <= 32768, "bad dense Gram shape");
  cudaStream_t st = c->stream;
  const int64_t rows_pad = (I + TC_BN - 1) / TC_BN * TC_BN, kd_pad = (Kd + TC_BK - 1) / TC_BK * TC_BK;
  const unsigned char* A_in = stage_in(c, A_u, (size_t)I * Kd, "tc_A_in");
  unsigned char* A = c->buf<unsigned char>("tc_A", (size_t)rows_pad * kd_pad);
  RPK_CUDA(cudaMemsetAsync(A, 0, (size_t)rows_pad * kd_pad, st));
  RPK_CUDA(cudaMemcpy2DAsync(A, (size_t)kd_pad, A_in, (size_t)Kd, (size_t)Kd, (size_t)I, cudaMemcpyDeviceToDevice, st));
  unsigned short* G = c->buf<unsigned short>("tc_G", (size_t)I * rows_pad);
  run_gram_dense_tc(c, A, rows_pad, kd_pad, 0, I, G, rows_pad);
  Out<unsigned short> o;
  o.init(c, G_u, (size_t)I * I, "tc_G_out");
  RPK_CUDA(cudaMemcpy2DAsync(o.dev, (size_t)I * 2, G, (size_t)rows_pad * 2, (size_t)I * 2, (size_t)I, cudaMemcpyDeviceToDevice, st));
  o.finish(c);
  finish_call(c);
}

}  // namespace rpk
