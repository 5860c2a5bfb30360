// topk_common.cuh — pieces of the top-K selection shared by topk.cu and topk_condensed.cu: the 64-bit selection key,
// the CTA bitonic sort, and the host launchers of the exact path that the condensed path reuses.
#pragma once
#include "common.cuh"

namespace gdr {

constexpr uint32_t TK_EXCLUDED = 0xFFFFFFFFu;    // NaN pattern fmaf never produces: marks an excluded item

static inline int64_t next_pow2(int64_t x) {
  int64_t p = 1;
  while (p < x) p <<= 1;
  return p;
}
__device__ __forceinline__ int64_t next_pow2_dev(int64_t x) {
  int64_t p = 1;
  while (p < x) p <<= 1;
  return p;
}

// 64-bit selection key: larger = better.  -0 is ordered (and reported) as +0; 0 = excluded.
__device__ __forceinline__ uint64_t tk_key(uint32_t bits, int64_t j) {
  if (bits == TK_EXCLUDED) return 0ull;
  uint32_t b = __float_as_uint(__uint_as_float(bits) + 0.f);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((uint64_t)b << 32) | (uint32_t)(0xFFFFFFFFu - (uint32_t)j);
}
__device__ __forceinline__ float tk_key_score(uint64_t key) {
  uint32_t b = (uint32_t)(key >> 32);
  b = (b & 0x80000000u) ? (b & 0x7FFFFFFFu) : ~b;
  return __uint_as_float(b);
}

// descending bitonic sort of n (power of two) keys held in shared or global memory by the whole CTA
__device__ inline void tk_bitonic_desc(uint64_t* a, int64_t n) {
  for (int64_t len = 2; len <= n; len <<= 1) {
    for (int64_t j = len >> 1; j > 0; j >>= 1) {
      for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const int64_t p = i ^ j;
        if (p > i) {
          const uint64_t x = a[i], y = a[p];
          const bool desc = (i & len) == 0;
          if (desc ? x < y : x > y) {
            a[i] = y;
            a[p] = x;
          }
        }
      }
      __syncthreads();
    }
  }
}

// topk.cu: S[r][j] = fp32 fmaf chain of U row rows[r0 + r] (nullable: r0 + r) with I row j, r < nr, j < n_items
// (k_topk_score); lds a multiple of 4, S 16-byte aligned
int topk_score_rows(int64_t nr, int64_t r0, int64_t n_users, int64_t n_items, int64_t d, const float* U, int64_t ldu,
                    const int64_t* rows, const float* I, int64_t ldi, float* S, int64_t lds, cudaStream_t s);
// topk.cu: the exact path over n_rows output rows (out_rows: their indices, nullable = 0..n_rows-1)
int64_t topk_exact_ws_bytes(int64_t n_rows, int64_t n_items, int64_t k);
int topk_exact(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t d, int64_t k, const float* U, int64_t ldu,
               const int64_t* rows, const int32_t* out_rows, const float* I, int64_t ldi, const int32_t* ex_rowptr,
               const int32_t* ex_colidx, float* scores_out, int64_t lds, int32_t* items_out, int64_t ldit,
               int32_t* status, void* ws, int64_t ws_bytes, cudaStream_t s);

}  // namespace gdr
