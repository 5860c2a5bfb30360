// topk.cu — full-ranking top-K recommendation and its Recall / Precision / NDCG@K.
//
//   s(u, j) = fp32 chain  acc = 0; for t < d: acc = fmaf(U[u, t], I[j, t], acc)
//   items[r] = the k non-excluded items of user rows[r] by (score desc, item asc), padded with (-1, -inf)
//
// The reference scores every user against every item, masks the training items and keeps the K best
// (distill_recsys.py:446-497 recall_at_k; Rankformer/code/model.py:27-53), i.e. an n_users x n_items fp32
// product.  Two paths, chosen from d, k and the size of the product (gdr_debug_set("topk_path") forces one); both give
// the same bytes.  Exact path, one row slab at a time (bounded scratch, never n_users x n_items):
//   k_topk_check    non-finite operands / out-of-range user ids -> status word (one pass over U rows and I)
//   k_topk_score    register-tiled SIMT product of the slab; every output is ONE fmaf chain in t order, so the
//                   scores are bit-identical to the chain above (and to tests/topk_ref.c: glibc's fmaf rounds correctly)
//   k_topk_select   one CTA per row: exclusion row -> sentinel, radix select of the k-th largest 64-bit key
//                   (ordered score bits << 32 | ~item), compaction, bitonic sort, output
// Keys are unique (the item index is part of the key), so the selected set is exactly the top k and the
// output does not depend on thread scheduling.
// Tensor-core path (d <= 128, k <= 256): k_topk_split (hi/lo TF32 operands, norms, the non-finite check), k_topk_tc
// (3xTF32 tcgen05 + TMA screen whose epilogue keeps a bounded candidate list per user row), k_topk_tc_finish (exact
// re-score of the candidates, sort); rows whose list overflows (ties) are finished by the exact path.
#include "tc_common.cuh"
#include "topk_common.cuh"

namespace gdr {

constexpr int TK_BM = 128;          // users per score tile
constexpr int TK_BN = 128;          // items per score tile
constexpr int TK_BK = 16;           // contraction step held in shared memory
constexpr int TK_SEL_THREADS = 512;
constexpr int TK_SMEM_K = 2048;     // k up to this sorts in shared memory; larger k sorts in workspace
constexpr int64_t TK_SLAB_BYTES = 384ll << 20;   // score scratch of one row slab
constexpr int TK_MAX_KS = 32;

static inline int64_t tk_ld(int64_t n_items) { return align_up(n_items, 4); }
static inline int64_t tk_kbuf(int64_t k) { return k > TK_SMEM_K ? next_pow2(k) * 8 : 0; }
// rows per slab: as many as the scratch budget holds, a multiple of the score tile when more than one tile fits
static int64_t tk_slab_rows(int64_t n_rows, int64_t n_items, int64_t k) {
  const int64_t per_row = tk_ld(n_items) * 4 + tk_kbuf(k);
  int64_t r = TK_SLAB_BYTES / per_row;
  if (r >= TK_BM) r = r / TK_BM * TK_BM;
  if (r < 1) r = 1;
  return r < n_rows ? r : n_rows;
}

// status bit 0: a non-finite value in U (rows used) or I; bit 1: a user id outside [0, n_users)
__global__ void __launch_bounds__(256) k_topk_check(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t d,
                                                    const float* __restrict__ U, int64_t ldu,
                                                    const int64_t* __restrict__ rows, const float* __restrict__ I,
                                                    int64_t ldi, int32_t* __restrict__ status) {
  // one warp per row: rows of U first, then the items
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= n_rows + n_items) return;
  const float* p;
  if (w < n_rows) {
    const int64_t u = rows ? rows[w] : w;
    if (u < 0 || u >= n_users) {
      if (lane_id() == 0) atomicOr(status, 2);
      return;
    }
    p = U + u * ldu;
  } else {
    p = I + (w - n_rows) * ldi;
  }
  bool bad = false;
  for (int64_t t = lane_id(); t < d; t += 32) bad |= !isfinite(p[t]);
  if (__any_sync(0xffffffffu, bad) && lane_id() == 0) atomicOr(status, 1);
}

// S[r][j] = s(user of output row g, j) for the slab's nr rows, g = out_rows[r0 + r] (or r0 + r), user = rows[g] (or g).  256 threads, 8 x 8 outputs each (rows ty*4 + {0..3} and
// 64 + ty*4 + {0..3}, items tx*4 + {0..3} and 64 + tx*4 + {0..3}); each accumulator sees its fmaf terms in t order.
__global__ void __launch_bounds__(256) k_topk_score(int64_t nr, int64_t r0, int64_t n_users, int64_t n_items, int64_t d,
                                                    const float* __restrict__ U, int64_t ldu,
                                                    const int64_t* __restrict__ rows,
                                                    const int32_t* __restrict__ out_rows, const float* __restrict__ I,
                                                    int64_t ldi, float* __restrict__ S, int64_t lds) {
  __shared__ __align__(16) float As[TK_BK][TK_BM + 4];   // +4: the transposed stores spread over the banks
  __shared__ __align__(16) float Bs[TK_BK][TK_BN + 4];
  __shared__ int64_t urow[TK_BM];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t rbase = (int64_t)blockIdx.y * TK_BM, jbase = (int64_t)blockIdx.x * TK_BN;
  if (tid < TK_BM) {
    const int64_t r = rbase + tid;
    int64_t u = -1;
    if (r < nr) {
      const int64_t g = out_rows ? (int64_t)out_rows[r0 + r] : r0 + r;
      u = rows ? rows[g] : g;
      if (u < 0 || u >= n_users) u = -1;   // reported by k_topk_check; scored as a zero row here
    }
    urow[tid] = u;
  }
  float acc[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
  __syncthreads();
  for (int64_t t0 = 0; t0 < d; t0 += TK_BK) {
    // 128 rows x 16 t per operand, 8 elements per thread, stored transposed ([t][row])
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int idx = e * 256 + tid;
      const int row = idx >> 4, tt = idx & 15;
      const int64_t t = t0 + tt;
      const int64_t u = urow[row];
      const int64_t j = jbase + row;
      As[tt][row] = (u >= 0 && t < d) ? U[u * ldu + t] : 0.f;
      Bs[tt][row] = (j < n_items && t < d) ? I[j * ldi + t] : 0.f;
    }
    __syncthreads();
    const int tmax = (int)(d - t0 < TK_BK ? d - t0 : TK_BK);   // no padding terms enter the chain
    for (int tt = 0; tt < tmax; ++tt) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[tt][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[tt][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[tt][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[tt][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(av[a], bv[b], acc[a][b]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 8; ++a) {
    const int64_t r = rbase + (a < 4 ? ty * 4 + a : 64 + ty * 4 + a - 4);
    if (r >= nr) continue;
    float* out = S + r * lds;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t j = jbase + h * 64 + tx * 4;
      if (j + 3 < n_items) {
        *reinterpret_cast<float4*>(out + j) =
            make_float4(acc[a][h * 4], acc[a][h * 4 + 1], acc[a][h * 4 + 2], acc[a][h * 4 + 3]);
      } else {
        for (int b = 0; b < 4; ++b)
          if (j + b < n_items) out[j + b] = acc[a][h * 4 + b];
      }
    }
  }
}

__global__ void __launch_bounds__(TK_SEL_THREADS) k_topk_select(int64_t nr, int64_t r0, int64_t n_users,
                                                                int64_t n_items, int64_t k,
                                                                const int64_t* __restrict__ rows,
                                                                const int32_t* __restrict__ out_rows,
                                                                const int32_t* __restrict__ ex_rowptr,
                                                                const int32_t* __restrict__ ex_colidx,
                                                                float* __restrict__ S, int64_t lds,
                                                                uint64_t* __restrict__ kbuf_g, int64_t kbuf_n,
                                                                float* __restrict__ scores_out, int64_t ldso,
                                                                int32_t* __restrict__ items_out, int64_t ldit) {
  __shared__ uint32_t hist[256];
  __shared__ uint64_t s_prefix;
  __shared__ int64_t s_need;
  __shared__ int s_done;
  __shared__ unsigned long long s_cnt;   // eligible items (read by every thread, never reused)
  __shared__ unsigned long long s_pos;   // compaction cursor
  __shared__ uint64_t kbuf_s[TK_SMEM_K];
  const int64_t r = blockIdx.x;
  if (r >= nr) return;
  const int64_t g = out_rows ? (int64_t)out_rows[r0 + r] : r0 + r;   // output row
  float* Srow = S + r * lds;
  const uint32_t* Sb = reinterpret_cast<const uint32_t*>(Srow);
  const int64_t u = rows ? rows[g] : g;

  // 1. exclusion row -> sentinel (a user id out of range has no exclusions; the call reports it)
  if (ex_rowptr && u >= 0 && u < n_users) {
    for (int64_t e = (int64_t)ex_rowptr[u] + threadIdx.x; e < ex_rowptr[u + 1]; e += blockDim.x) {
      const int32_t j = ex_colidx[e];
      if (j >= 0 && j < n_items) reinterpret_cast<uint32_t*>(Srow)[j] = TK_EXCLUDED;
    }
  }
  if (threadIdx.x == 0) {
    s_cnt = 0;
    s_pos = 0;
  }
  __syncthreads();
  // 2. eligible count
  {
    unsigned long long c = 0;
    for (int64_t j = threadIdx.x; j < n_items; j += blockDim.x) c += Sb[j] != TK_EXCLUDED;
    atomicAdd(&s_cnt, c);
  }
  __syncthreads();
  const int64_t eligible = (int64_t)s_cnt;
  uint64_t thresh;   // selected = keys >= thresh (exactly min(k, eligible) of them)
  if (eligible <= k) {
    thresh = 1;
  } else {
    // 3. radix select of the k-th largest key, 8 bits per pass from the top; stops as soon as the bin holding
    //    the k-th key is taken whole
    if (threadIdx.x == 0) {
      s_prefix = 0;
      s_need = k;
      s_done = 0;
    }
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
      __syncthreads();
      const uint64_t prefix = s_prefix;
      const uint64_t hmask = shift == 56 ? 0ull : (~0ull << (shift + 8));
      // warp-aggregated histogram: the early passes put most keys of a row into a handful of bins
      for (int64_t j0 = 0; j0 < n_items; j0 += blockDim.x) {
        const int64_t j = j0 + threadIdx.x;
        int bin = -1;
        if (j < n_items) {
          const uint64_t key = tk_key(Sb[j], j);
          if ((key & hmask) == prefix) bin = (int)((key >> shift) & 255);
        }
        if (!__any_sync(0xffffffffu, bin >= 0)) continue;
        const uint32_t same = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0 && lane_id() == __ffs(same) - 1) atomicAdd(&hist[bin], (uint32_t)__popc(same));
      }
      __syncthreads();
      if (threadIdx.x < 32) {
        // lane l holds bins [8l, 8l + 8); suffix sums from the top bin down
        const int l = threadIdx.x;
        uint32_t c8[8], tot = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          c8[q] = hist[8 * l + q];
          tot += c8[q];
        }
        uint32_t suf = tot;   // sum over lanes >= l
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t v = __shfl_down_sync(0xffffffffu, suf, o);
          if (l + o < 32) suf += v;
        }
        const int64_t need = s_need;
        const uint32_t ball = __ballot_sync(0xffffffffu, (int64_t)suf >= need);
        const int lw = 31 - __clz(ball);   // the highest lane whose suffix still reaches the k-th key
        if (l == lw) {
          int64_t above = (int64_t)(suf - tot);   // keys in higher lanes
          int b = 7;
          for (; b > 0; --b) {
            if (above + c8[b] >= need) break;
            above += c8[b];
          }
          const int bin = 8 * l + b;
          const int64_t rem = need - above;
          s_prefix = prefix | ((uint64_t)bin << shift);
          s_need = rem;
          s_done = (rem == (int64_t)c8[b]) ? 1 : 0;
        }
      }
      __syncthreads();
      if (s_done) break;
    }
    thresh = s_prefix;
  }
  // 4. compaction of the selected keys, sort, output
  const int64_t m = eligible < k ? eligible : k;
  const int64_t mp = next_pow2_dev(m);
  uint64_t* buf = k <= TK_SMEM_K ? kbuf_s : kbuf_g + r * kbuf_n;
  for (int64_t j = threadIdx.x; j < n_items; j += blockDim.x) {
    const uint64_t key = tk_key(Sb[j], j);
    if (key >= thresh && key != 0ull) buf[atomicAdd(&s_pos, 1ull)] = key;
  }
  for (int64_t i = m + threadIdx.x; i < mp; i += blockDim.x) buf[i] = 0ull;
  __syncthreads();
  tk_bitonic_desc(buf, mp);
  for (int64_t i = threadIdx.x; i < k; i += blockDim.x) {
    if (i < m) {
      const uint64_t key = buf[i];
      items_out[g * ldit + i] = (int32_t)(0xFFFFFFFFu - (uint32_t)key);
      scores_out[g * ldso + i] = tk_key_score(key);
    } else {
      items_out[g * ldit + i] = -1;
      scores_out[g * ldso + i] = -INFINITY;
    }
  }
}

int64_t topk_exact_ws_bytes(int64_t n_rows, int64_t n_items, int64_t k) {
  const int64_t sr = tk_slab_rows(n_rows, n_items, k);
  return ws_need(sr * tk_ld(n_items), 4) + ws_need(sr * tk_kbuf(k), 1) + 256;
}

int topk_score_rows(int64_t nr, int64_t r0, int64_t n_users, int64_t n_items, int64_t d, const float* U, int64_t ldu,
                    const int64_t* rows, const float* I, int64_t ldi, float* S, int64_t lds, cudaStream_t s) {
  dim3 grid((unsigned)cdiv(n_items, TK_BN), (unsigned)cdiv(nr, TK_BM));
  k_topk_score<<<grid, 256, 0, s>>>(nr, r0, n_users, n_items, d, U, ldu, rows, nullptr, I, ldi, S, lds);
  GDR_LAUNCHED();
  return GDR_OK;
}

// exact path over n_rows output rows (out_rows: their indices, nullable = 0..n_rows-1)
int topk_exact(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t d, int64_t k, const float* U, int64_t ldu,
               const int64_t* rows, const int32_t* out_rows, const float* I, int64_t ldi, const int32_t* ex_rowptr,
               const int32_t* ex_colidx, float* scores_out, int64_t lds, int32_t* items_out, int64_t ldit,
               int32_t* status, void* ws, int64_t ws_bytes, cudaStream_t s) {
  const int64_t sr = tk_slab_rows(n_rows, n_items, k), ld = tk_ld(n_items);
  const int64_t kbuf_n = tk_kbuf(k) / 8;
  Workspace W(ws, ws_bytes);
  float* S = W.take<float>(sr * ld);
  uint64_t* kbuf = kbuf_n ? W.take<uint64_t>(sr * kbuf_n) : nullptr;
  if (!W.ok()) {
    set_error("topk_scores: workspace too small");
    return GDR_EWORKSPACE;
  }
  if (status) {
    k_topk_check<<<(unsigned)cdiv((n_rows + n_items) * 32, 256), 256, 0, s>>>(n_rows, n_users, n_items, d, U, ldu, rows,
                                                                              I, ldi, status);
    GDR_LAUNCHED();
  }
  for (int64_t r0 = 0; r0 < n_rows; r0 += sr) {
    const int64_t nr = n_rows - r0 < sr ? n_rows - r0 : sr;
    dim3 grid((unsigned)cdiv(n_items, TK_BN), (unsigned)cdiv(nr, TK_BM));
    k_topk_score<<<grid, 256, 0, s>>>(nr, r0, n_users, n_items, d, U, ldu, rows, out_rows, I, ldi, S, ld);
    GDR_LAUNCHED();
    k_topk_select<<<(unsigned)nr, TK_SEL_THREADS, 0, s>>>(nr, r0, n_users, n_items, k, rows, out_rows, ex_rowptr, ex_colidx, S, ld,
                                                          kbuf, kbuf_n, scores_out, lds, items_out, ldit);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}


// ---------------------------------------------------------------------------------
// tensor-core screen (d <= 128): 3xTF32 tcgen05 product with a per-row candidate epilogue, exact finish
// ---------------------------------------------------------------------------------
// Error bound.  hi = tf32(x), lo = tf32(x - hi): |x - hi - lo| <= 2^-22 |x|, and the screen drops lo_u.lo_i and the
// residuals, <= 3 2^-22 |u||i| by Cauchy-Schwarz.  The tensor core sums the 3d products into an fp32 accumulator: at most
// 3d roundings of a partial sum bounded by sum_t |u_t i_t| <= |u||i|, unit <= 2^-23 even for a truncating adder, so
// <= 384 2^-23 |u||i| for d <= 128.  The exact chain itself is within d 2^-24 |u||i| <= 128 2^-24 |u||i| of the real dot.
// Together |s~ - s| <= (12 + 768 + 128) 2^-24 |u||i| < 2^-14 |u| max_j |i_j|.  tol_u = 2^-13 |u| max_j |i_j| doubles
// that, which also covers the fp32 rounding of |u|, max |i|, tol_u and tau - 2 tol_u.
// Candidate rule.  tau~ is always <= the k-th largest screened score of the row's non-excluded items (it is the max of
// k-th largest screened scores of subsets of them), and item j is kept iff s~_j >= tau~ - 2 tol_u.  For an exact top-k
// item j*: s~_j* >= s_j* - tol >= s_k - tol >= (k-th largest s~) - 2 tol >= tau~ - 2 tol, at any time: j* is never
// dropped, so the candidates are a superset of the exact top k and the exact re-score + sort reproduces the exact path.
constexpr int TK_TC_BN = 128;             // items per accumulator tile (UMMA N)
constexpr int TK_TC_MAX_KB = 4;           // d padded <= 128
constexpr int TK_TC_THREADS = 192;        // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue (one row per thread)
constexpr int TK_TC_STAGE_BYTES = 2 * TK_TC_BN * TC_BK * 4;   // one item K-block, hi + lo
constexpr int TK_TC_MAX_STAGES = 8;
constexpr int TK_TC_SMEM = 227 * 1024;
constexpr int TK_TC_MAX_K = 256;          // larger k runs on the exact path
constexpr float TK_TOL = 1.220703125e-04f;   // 2^-13
int g_topk_path = 0;                      // gdr_debug_set("topk_path"): 0 auto, 1 exact, 2 tensor core
int64_t g_topk_last_overflow = -1;        // rows the last tensor-core run handed to the exact path

__host__ __device__ inline int tk_tc_stages(int nkb) {
  const int n = (TK_TC_SMEM - 1024 - 512 - 2 * nkb * TC_KBLK_BYTES) / TK_TC_STAGE_BYTES;
  return n > TK_TC_MAX_STAGES ? TK_TC_MAX_STAGES : n;
}
static inline int tk_tc_smem(int nkb) { return 2 * nkb * TC_KBLK_BYTES + tk_tc_stages(nkb) * TK_TC_STAGE_BYTES + 512 + 1024; }
static inline int64_t tk_cap(int64_t k) {
  int64_t c = next_pow2(4 * k);
  return c < 128 ? 128 : c;
}

// hi / lo TF32 split of the used U rows (rows 0..n_rows) and of I, zero-padded to Dp; |u| per row, max |i| (atomicMax on
// the bits of a non-negative float); status bits as k_topk_check.  One warp per row.
__global__ void __launch_bounds__(256) k_topk_split(int64_t n_rows, int64_t n_users, int64_t n_items, int d, int Dp,
                                                    const float* __restrict__ U, int64_t ldu,
                                                    const int64_t* __restrict__ rows, const float* __restrict__ I,
                                                    int64_t ldi, float* __restrict__ u_hi, float* __restrict__ u_lo,
                                                    float* __restrict__ i_hi, float* __restrict__ i_lo,
                                                    float* __restrict__ unorm, uint32_t* __restrict__ imax_bits,
                                                    int32_t* __restrict__ status) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= n_rows + n_items) return;
  const bool is_u = w < n_rows;
  const int64_t r = is_u ? w : w - n_rows;
  const float* p = nullptr;
  if (is_u) {
    const int64_t u = rows ? rows[r] : r;
    if (u >= 0 && u < n_users) p = U + u * ldu;
    else if (lane_id() == 0) atomicOr(status, 2);
  } else {
    p = I + r * ldi;
  }
  float* hi = (is_u ? u_hi : i_hi) + r * Dp;
  float* lo = (is_u ? u_lo : i_lo) + r * Dp;
  float ss = 0.f;
  bool bad = false;
  for (int c = lane_id(); c < Dp; c += 32) {
    const float x = (p && c < d) ? p[c] : 0.f;
    bad |= !isfinite(x);
    const float h = to_tf32(x);
    hi[c] = h;
    lo[c] = to_tf32(__fsub_rn(x, h));
    ss = fmaf(x, x, ss);
  }
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if (__any_sync(0xffffffffu, bad) && lane_id() == 0) atomicOr(status, 1);
  if (lane_id() == 0) {
    if (is_u) unorm[r] = sqrtf(ss);
    else atomicMax(imax_bits, __float_as_uint(sqrtf(ss)));
  }
}

__device__ __forceinline__ uint32_t tk_ord(float s) {
  const uint32_t b = __float_as_uint(s);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// full candidate list: tau = max(tau, k-th largest screened score of the list) (bisection on the order-preserving
// bits), then keep only the entries >= tau - 2 tol.  Returns the new length.
__device__ __noinline__ int tk_refresh(uint64_t* __restrict__ list, int cnt, int k, float tol, float& tau) {
  uint32_t lo = 0, hi = 0xFFFFFFFFu;
  while (lo < hi) {
    const uint32_t mid = lo + (uint32_t)(((uint64_t)hi - lo + 1) >> 1);
    int c = 0;
    for (int i = 0; i < cnt; ++i) c += tk_ord(__uint_as_float((uint32_t)(list[i] >> 32))) >= mid;
    if (c >= k) lo = mid;
    else hi = mid - 1;
  }
  const uint32_t b = (lo & 0x80000000u) ? (lo & 0x7FFFFFFFu) : ~lo;
  tau = fmaxf(tau, __uint_as_float(b));
  const float lim = tau - 2.f * tol;
  int n = 0;
  for (int i = 0; i < cnt; ++i)
    if (__uint_as_float((uint32_t)(list[i] >> 32)) >= lim) list[n++] = list[i];
  return n;
}

// Persistent CTA per SM; a resident 128-row user tile (hi + lo) while the item tiles stream through an mbarrier ring;
// two 128-column TMEM accumulators; epilogue thread = one user row, items in ascending order.
__global__ void __launch_bounds__(TK_TC_THREADS, 1)
k_topk_tc(const __grid_constant__ CUtensorMap map_uhi, const __grid_constant__ CUtensorMap map_ulo,
          const __grid_constant__ CUtensorMap map_ihi, const __grid_constant__ CUtensorMap map_ilo, int64_t n_rows,
          int64_t n_users, int64_t n_items, int d, int nkb, int k, int cap, const int64_t* __restrict__ rows,
          const int32_t* __restrict__ ex_rowptr, const int32_t* __restrict__ ex_colidx,
          const float* __restrict__ unorm, const uint32_t* __restrict__ imax_bits, uint64_t* __restrict__ cand,
          int32_t* __restrict__ cand_cnt, int32_t* __restrict__ ovf_list, int32_t* __restrict__ ovf_count) {
  const int S = tk_tc_stages(nkb);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int x_bytes = 2 * nkb * TC_KBLK_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + x_bytes + S * TK_TC_STAGE_BYTES);
  uint64_t* x_full = bars;                              // [TK_TC_MAX_KB]
  uint64_t* x_empty = bars + TK_TC_MAX_KB;
  uint64_t* c_full = bars + 2 * TK_TC_MAX_KB;           // [TK_TC_MAX_STAGES]
  uint64_t* c_empty = c_full + TK_TC_MAX_STAGES;
  uint64_t* t_full = c_empty + TK_TC_MAX_STAGES;        // [2]
  uint64_t* t_empty = t_full + 2;
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(t_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_row_tiles = (int)((n_rows + TC_BM - 1) / TC_BM);
  const int n_col_tiles = (int)((n_items + TK_TC_BN - 1) / TK_TC_BN);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < TK_TC_MAX_KB; ++i) {
      mbar_init(&x_full[i], 1);
      mbar_init(&x_empty[i], 1);
    }
    for (int i = 0; i < TK_TC_MAX_STAGES; ++i) {
      mbar_init(&c_full[i], 1);
      mbar_init(&c_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&t_full[i], 1);
      mbar_init(&t_empty[i], 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_smem)),
                 "r"(2 * TK_TC_BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;

  if (warp == 0) {
    // ================= TMA producer =================
    uint32_t tile_it = 0, ph = 0;
    int s = 0;
    for (int rt = blockIdx.x; rt < n_row_tiles; rt += gridDim.x, ++tile_it) {
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&x_empty[kb], (tile_it & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&x_full[kb], 2 * TC_KBLK_BYTES);
          tma_load_2d(smem + kb * TC_KBLK_BYTES, &map_uhi, kb * TC_BK, rt * TC_BM, &x_full[kb]);
          tma_load_2d(smem + (nkb + kb) * TC_KBLK_BYTES, &map_ulo, kb * TC_BK, rt * TC_BM, &x_full[kb]);
        }
        __syncwarp();
      }
      for (int ct = 0; ct < n_col_tiles; ++ct) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&c_empty[s], ph ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&c_full[s], TK_TC_STAGE_BYTES);
            uint8_t* dst = smem + x_bytes + s * TK_TC_STAGE_BYTES;
            tma_load_2d(dst, &map_ihi, kb * TC_BK, ct * TK_TC_BN, &c_full[s]);
            tma_load_2d(dst + TK_TC_BN * TC_BK * 4, &map_ilo, kb * TC_BK, ct * TK_TC_BN, &c_full[s]);
          }
          __syncwarp();
          if (++s == S) {
            s = 0;
            ph ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer: x_lo.i_hi + x_hi.i_lo + x_hi.i_hi per K = 8 step =================
    constexpr uint32_t idesc = umma_idesc_tf32(TC_BM, TK_TC_BN);
    uint32_t tile_it = 0, g = 0, ph = 0;
    int s = 0;
    const uint64_t dx0 = umma_desc_sw128(smem_u32(smem));
    const uint64_t dc0 = umma_desc_sw128(smem_u32(smem + x_bytes));
    constexpr uint64_t kKb = TC_KBLK_BYTES >> 4, kStage = TK_TC_STAGE_BYTES >> 4, kLo = (uint64_t)(TK_TC_BN * TC_BK * 4) >> 4;
    for (int rt = blockIdx.x; rt < n_row_tiles; rt += gridDim.x, ++tile_it) {
      for (int ct = 0; ct < n_col_tiles; ++ct, ++g) {
        const uint32_t a = g & 1, aph = (g >> 1) & 1;
        mbar_wait(&t_empty[a], aph ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + a * TK_TC_BN;
        const bool last_ct = ct == n_col_tiles - 1;
        for (int kb = 0; kb < nkb; ++kb) {
          if (ct == 0) mbar_wait(&x_full[kb], tile_it & 1);
          mbar_wait(&c_full[s], ph);
          tc_fence_after();
          const uint64_t d_chi = dc0 + (uint64_t)s * kStage, d_clo = d_chi + kLo;
          const uint64_t d_xhi = dx0 + (uint64_t)kb * kKb, d_xlo = dx0 + (uint64_t)(nkb + kb) * kKb;
          const int ksteps = min(TC_BK / 8, (d - kb * TC_BK + 7) >> 3);
          if (elect_one()) {
            for (int kk = 0; kk < ksteps; ++kk) {
              const uint64_t adv = (uint64_t)((kk * 8 * 4) >> 4);
              tc_mma_tf32(tmem_d, d_xlo + adv, d_chi + adv, idesc, (kb | kk) != 0);
              tc_mma_tf32(tmem_d, d_xhi + adv, d_clo + adv, idesc, 1);
              tc_mma_tf32(tmem_d, d_xhi + adv, d_chi + adv, idesc, 1);
            }
            tc_commit(&c_empty[s]);
            if (last_ct) tc_commit(&x_empty[kb]);
            if (kb == nkb - 1) tc_commit(&t_full[a]);
          }
          __syncwarp();
          if (++s == S) {
            s = 0;
            ph ^= 1;
          }
        }
      }
    }
  } else {
    // ================= epilogue: warp w reads TMEM lanes [32 (w % 4), +32); thread = user row =================
    const int quarter = warp & 3;
    const int rl = quarter * 32 + lane;
    const float imax = __uint_as_float(*imax_bits);
    uint32_t g = 0;
    for (int rt = blockIdx.x; rt < n_row_tiles; rt += gridDim.x) {
      const int64_t row = (int64_t)rt * TC_BM + rl;
      const bool valid = row < n_rows;
      int64_t u = valid ? (rows ? rows[row] : row) : -1;
      if (u >= n_users) u = -1;   // reported by the split pass
      const float tol = valid ? TK_TOL * unorm[row] * imax : 0.f;
      float tau = -INFINITY, lim = -INFINITY;
      int cnt = 0;
      bool live = valid && u >= 0;   // false: padding row, bad user id, or overflowed list
      bool ovf = false;
      int32_t ep = 0, ee = 0;
      if (live && ex_rowptr) {
        ep = ex_rowptr[u];
        ee = ex_rowptr[u + 1];
      }
      uint64_t* list = cand + (valid ? row : 0) * (int64_t)cap;
      for (int ct = 0; ct < n_col_tiles; ++ct, ++g) {
        const uint32_t a = g & 1, aph = (g >> 1) & 1;
        mbar_wait(&t_full[a], aph);
        tc_fence_after();
#pragma unroll 1
        for (int h = 0; h < TK_TC_BN / 32; ++h) {
          uint32_t v[32];
          tc_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + a * TK_TC_BN + h * 32, v);
          tc_wait_ld();
          float m = __uint_as_float(v[0]);
#pragma unroll
          for (int q = 1; q < 32; ++q) m = fmaxf(m, __uint_as_float(v[q]));
          if (!__any_sync(0xffffffffu, live && m >= lim)) continue;
          const int64_t jbase = (int64_t)ct * TK_TC_BN + h * 32;
#pragma unroll
          for (int q = 0; q < 32; ++q) {
            const float sv = __uint_as_float(v[q]);
            const int64_t j = jbase + q;
            if (live && sv >= lim && j < n_items) {
              while (ep < ee && ex_colidx[ep] < j) ++ep;   // exclusion row walked in step with the ascending items
              if (!(ep < ee && ex_colidx[ep] == j)) {
                list[cnt++] = ((uint64_t)__float_as_uint(sv) << 32) | (uint32_t)j;
                if (cnt == cap) {
                  cnt = tk_refresh(list, cnt, k, tol, tau);
                  lim = tau - 2.f * tol;
                  if (cnt > cap / 2) {   // ties: the band keeps most of the row; the exact path finishes it
                    live = false;
                    ovf = true;
                  }
                }
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(&t_empty[a]);
      }
      if (valid) {
        cand_cnt[row] = ovf ? -1 : cnt;
        if (ovf) ovf_list[atomicAdd(ovf_count, 1)] = (int32_t)row;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * TK_TC_BN) : "memory");
  }
}

// exact finish of a row whose candidate list held: re-score every candidate with the exact chain, sort, keep k
__global__ void __launch_bounds__(256) k_topk_tc_finish(int64_t n_rows, int64_t n_users, int d, int64_t k, int cap,
                                                        const float* __restrict__ U, int64_t ldu,
                                                        const int64_t* __restrict__ rows, const float* __restrict__ I,
                                                        int64_t ldi, const uint64_t* __restrict__ cand,
                                                        const int32_t* __restrict__ cand_cnt,
                                                        float* __restrict__ scores_out, int64_t ldso,
                                                        int32_t* __restrict__ items_out, int64_t ldit) {
  __shared__ uint64_t buf[1024];
  const int64_t r = blockIdx.x;
  const int c = cand_cnt[r];
  if (c < 0) return;   // overflowed: the exact path writes this row
  const int64_t u = rows ? rows[r] : r;
  if (u < 0 || u >= n_users) return;   // the call reports the bad id
  const int64_t cp = next_pow2_dev(c > 0 ? c : 1);
  for (int i = threadIdx.x; i < cp; i += blockDim.x) {
    uint64_t key = 0ull;
    if (i < c) {
      const int64_t j = (int64_t)(uint32_t)cand[r * cap + i];
      const float* pu = U + u * ldu;
      const float* pi = I + j * ldi;
      float acc = 0.f;
      for (int t = 0; t < d; ++t) acc = fmaf(pu[t], pi[t], acc);
      key = tk_key(__float_as_uint(acc), j);
    }
    buf[i] = key;
  }
  __syncthreads();
  tk_bitonic_desc(buf, cp);
  const int64_t m = c < k ? c : k;
  for (int64_t i = threadIdx.x; i < k; i += blockDim.x) {
    if (i < m) {
      items_out[r * ldit + i] = (int32_t)(0xFFFFFFFFu - (uint32_t)buf[i]);
      scores_out[r * ldso + i] = tk_key_score(buf[i]);
    } else {
      items_out[r * ldit + i] = -1;
      scores_out[r * ldso + i] = -INFINITY;
    }
  }
}

static bool tk_tc_supported(int64_t d, int64_t k) { return d <= TK_TC_MAX_KB * TC_BK && k <= TK_TC_MAX_K; }
// automatic choice from the size of the product (tools/topk_bench.py, one B200, d = 64, k = 20): 1.2 G scores
// (Yelp2018 shape) exact 16.2 ms vs screen 25.4 ms; 4.8 G scores (Amazon-book shape) exact 72.5 ms vs screen 50.8 ms
static bool tk_use_tc(int64_t n_rows, int64_t n_items, int64_t d, int64_t k) {
  if (g_topk_path == 1 || !tk_tc_supported(d, k)) return false;
  if (g_topk_path == 2) return true;
  return n_rows >= TC_BM && n_rows * n_items >= (1ll << 32);
}

static int64_t topk_tc_ws_bytes(int64_t n_rows, int64_t n_items, int64_t d, int64_t k) {
  const int64_t Dp = align_up(d, TC_BK);
  return 2 * ws_need(n_rows * Dp, 4) + 2 * ws_need(n_items * Dp, 4) + ws_need(n_rows, 4) + 256 +
         ws_need(n_rows * tk_cap(k), 8) + 2 * ws_need(n_rows, 4) + 256;
}

int64_t topk_scores_ws_bytes(int64_t n_rows, int64_t n_items, int64_t d, int64_t k) {
  int64_t b = topk_exact_ws_bytes(n_rows, n_items, k);
  if (tk_tc_supported(d, k)) b += topk_tc_ws_bytes(n_rows, n_items, d, k);
  return b;
}

int topk_scores(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t d, int64_t k, const float* U, int64_t ldu,
                const int64_t* rows, const float* I, int64_t ldi, const int32_t* ex_rowptr, const int32_t* ex_colidx,
                float* scores_out, int64_t lds, int32_t* items_out, int64_t ldit, int32_t* status, void* ws,
                int64_t ws_bytes, cudaStream_t s) {
  const int64_t exact_ws = topk_exact_ws_bytes(n_rows, n_items, k);
  if (g_topk_path == 2 && !tk_tc_supported(d, k)) {
    set_error("topk_scores: the tensor-core path needs d <= 128 and k <= %d", TK_TC_MAX_K);
    return GDR_EUNSUPPORTED;
  }
  if (!tk_use_tc(n_rows, n_items, d, k))
    return topk_exact(n_rows, n_users, n_items, d, k, U, ldu, rows, nullptr, I, ldi, ex_rowptr, ex_colidx, scores_out,
                      lds, items_out, ldit, status, ws, ws_bytes, s);
  if (n_rows >= (1ll << 31) - TC_BM || n_items >= (1ll << 31) - TK_TC_BN) {
    set_error("topk_scores: sizes exceed int32 tile coordinates");
    return GDR_ERANGE;
  }
  const int Dp = (int)align_up(d, TC_BK), nkb = Dp / TC_BK;
  const int cap = (int)tk_cap(k);
  Workspace W((char*)ws + exact_ws, ws_bytes - exact_ws);
  float* u_hi = W.take<float>(n_rows * Dp);
  float* u_lo = W.take<float>(n_rows * Dp);
  float* i_hi = W.take<float>(n_items * Dp);
  float* i_lo = W.take<float>(n_items * Dp);
  float* unorm = W.take<float>(n_rows);
  uint32_t* imax = W.take<uint32_t>(1);
  uint64_t* cand = W.take<uint64_t>(n_rows * cap);
  int32_t* cand_cnt = W.take<int32_t>(n_rows);
  int32_t* ovf_list = W.take<int32_t>(n_rows);
  int32_t* ovf_count = W.take<int32_t>(1);
  if (!W.ok()) {
    set_error("topk_scores: workspace too small");
    return GDR_EWORKSPACE;
  }
  GDR_CUDA(cudaMemsetAsync(imax, 0, 4, s));
  GDR_CUDA(cudaMemsetAsync(ovf_count, 0, 4, s));
  k_topk_split<<<(unsigned)cdiv((n_rows + n_items) * 32, 256), 256, 0, s>>>(n_rows, n_users, n_items, (int)d, Dp, U, ldu,
                                                                            rows, I, ldi, u_hi, u_lo, i_hi, i_lo, unorm,
                                                                            imax, status);
  GDR_LAUNCHED();
  CUtensorMap m_uhi, m_ulo, m_ihi, m_ilo;
  int rc;
  if ((rc = make_map(&m_uhi, u_hi, n_rows, Dp, TC_BM))) return rc;
  if ((rc = make_map(&m_ulo, u_lo, n_rows, Dp, TC_BM))) return rc;
  if ((rc = make_map(&m_ihi, i_hi, n_items, Dp, TK_TC_BN))) return rc;
  if ((rc = make_map(&m_ilo, i_lo, n_items, Dp, TK_TC_BN))) return rc;
  static PerDevice<bool> attr_set_dev;
  bool& attr_set = attr_set_dev.get();
  if (!attr_set) {
    GDR_CUDA(cudaFuncSetAttribute(k_topk_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, TK_TC_SMEM));
    attr_set = true;
  }
  int sms = kSMs, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t tiles = cdiv(n_rows, TC_BM);
  k_topk_tc<<<(unsigned)(tiles < sms ? tiles : sms), TK_TC_THREADS, tk_tc_smem(nkb), s>>>(
      m_uhi, m_ulo, m_ihi, m_ilo, n_rows, n_users, n_items, (int)d, nkb, (int)k, cap, rows, ex_rowptr, ex_colidx, unorm,
      imax, cand, cand_cnt, ovf_list, ovf_count);
  GDR_LAUNCHED();
  k_topk_tc_finish<<<(unsigned)n_rows, 256, 0, s>>>(n_rows, n_users, (int)d, k, cap, U, ldu, rows, I, ldi, cand, cand_cnt,
                                                    scores_out, lds, items_out, ldit);
  GDR_LAUNCHED();
  // rows whose list overflowed (tie-heavy rows) are finished by the exact path; their count decides its launches
  int32_t n_ovf = 0;
  GDR_CUDA(cudaMemcpyAsync(&n_ovf, ovf_count, 4, cudaMemcpyDeviceToHost, s));
  GDR_CUDA(cudaStreamSynchronize(s));
  g_topk_last_overflow = n_ovf;
  if (n_ovf == 0) return GDR_OK;
  return topk_exact(n_ovf, n_users, n_items, d, k, U, ldu, rows, ovf_list, I, ldi, ex_rowptr, ex_colidx, scores_out, lds,
                    items_out, ldit, nullptr, ws, exact_ws, s);
}

// ---------------------------------------------------------------------------------
// ranking metrics: one warp per evaluated row, per-row fp64 values, then fixed-order sums
// ---------------------------------------------------------------------------------
struct TkKs {
  int n;
  int32_t k[TK_MAX_KS];
};

// per_row[(q * 3 + m) * n_rows + r] (fp64, 0 for a row without test items); valid[r] = |test_u| > 0
__global__ void __launch_bounds__(256) k_rank_metrics(int64_t n_rows, int64_t n_users, const int32_t* __restrict__ items,
                                                      int64_t ldit, const int64_t* __restrict__ rows,
                                                      const int32_t* __restrict__ tp, const int32_t* __restrict__ tc,
                                                      TkKs ks, double* __restrict__ per_row,
                                                      float* __restrict__ per_row_out, int32_t* __restrict__ valid) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_rows) return;
  const int lane = lane_id();
  const int64_t u = rows ? rows[r] : r;
  const bool in_range = u >= 0 && u < n_users;
  const int32_t t0 = in_range ? tp[u] : 0, t1 = in_range ? tp[u + 1] : 0;
  const int64_t nt = t1 - t0;
  if (lane == 0) valid[r] = nt > 0;
  for (int q = 0; q < ks.n; ++q) {
    const int K = ks.k[q];
    double hits = 0.0, dcg = 0.0, idcg = 0.0;
    if (nt > 0) {
      for (int base = 0; base < K; base += 32) {
        const int rank = base + lane;
        bool hit = false;
        if (rank < K) {
          const int32_t it = items[r * ldit + rank];
          if (it >= 0) {   // binary search in the sorted test row
            int32_t lo = t0, hi = t1;
            while (lo < hi) {
              const int32_t mid = (lo + hi) >> 1;
              if (tc[mid] < it) lo = mid + 1;
              else hi = mid;
            }
            hit = lo < t1 && tc[lo] == it;
          }
        }
        uint32_t mask = __ballot_sync(0xffffffffu, hit);
        hits += __popc(mask);
        while (mask) {   // rank order
          const int b = __ffs(mask) - 1;
          mask &= mask - 1;
          dcg += 1.0 / log2((double)(base + b + 2));
        }
      }
      const int64_t ni = nt < K ? nt : K;
      for (int64_t i = 0; i < ni; ++i) idcg += 1.0 / log2((double)(i + 2));
    }
    const double v[3] = {nt > 0 ? hits / (double)nt : 0.0, nt > 0 ? hits / (double)K : 0.0, nt > 0 ? dcg / idcg : 0.0};
    if (lane < 3) {
      per_row[((int64_t)q * 3 + lane) * n_rows + r] = v[lane];
      if (per_row_out) per_row_out[((int64_t)q * 3 + lane) * n_rows + r] = nt > 0 ? (float)v[lane] : NAN;
    }
  }
}

// warp w sums series w of per_row (w < 3 n_ks) in ascending row order; warp 3 n_ks counts the evaluated rows
__global__ void __launch_bounds__(32) k_rank_sums(int64_t n_rows, int n_series, const double* __restrict__ per_row,
                                                  const int32_t* __restrict__ valid, double* __restrict__ sums,
                                                  int64_t* __restrict__ n_eval) {
  const int w = blockIdx.x, lane = lane_id();
  if (w == n_series) {
    long long c = 0;
    for (int64_t i = lane; i < n_rows; i += 32) c += valid[i];
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) *n_eval = c;
    return;
  }
  const double* p = per_row + (int64_t)w * n_rows;
  double acc = 0.0;
  for (int64_t base = 0; base < n_rows; base += 32) {
    const double v = base + lane < n_rows ? p[base + lane] : 0.0;
    for (int l = 0; l < 32 && base + l < n_rows; ++l) acc += __shfl_sync(0xffffffffu, v, l);
  }
  if (lane == 0) sums[w] = acc;
}

int64_t ranking_metrics_ws_bytes(int64_t n_rows, int n_ks) {
  return ws_need((int64_t)n_ks * 3 * n_rows, 8) + ws_need(n_rows, 4) + 256;
}

}  // namespace gdr

extern "C" {

int64_t gdr_topk_scores_ws_bytes(int64_t n_rows, int64_t n_items, int64_t d, int64_t k) {
  if (n_rows <= 0 || n_items <= 0 || k <= 0) return 256;
  return gdr::topk_scores_ws_bytes(n_rows, n_items, d, k);
}

int gdr_topk_scores(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t d, int64_t k, const float* U, int64_t ldu,
                    const int64_t* rows, const float* I, int64_t ldi, const int32_t* ex_rowptr, const int32_t* ex_colidx,
                    float* scores_out, int64_t lds, int32_t* items_out, int64_t ldit, int32_t* status_dev, void* ws,
                    int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows > 0 && n_users > 0 && n_items > 0 && d > 0, "topk_scores: sizes must be positive");
  GDR_CHECK_ARG(k >= 1 && k <= n_items, "topk_scores: k=%lld outside [1, n_items=%lld]", (long long)k,
                (long long)n_items);
  GDR_CHECK_ARG(n_items < INT32_MAX && n_users < INT32_MAX, "topk_scores: item / user ids must fit int32");
  GDR_CHECK_ARG(U && I && scores_out && items_out && status_dev && ws, "topk_scores: null pointer");
  GDR_CHECK_ARG((ex_rowptr == nullptr) == (ex_colidx == nullptr), "topk_scores: exclusion CSR needs both arrays");
  GDR_CHECK_ARG(ldu >= d && ldi >= d && lds >= k && ldit >= k, "topk_scores: leading dimension too small");
  GDR_CHECK_ARG(rows || n_rows <= n_users, "topk_scores: n_rows > n_users without a rows list");
  if (ws_bytes < gdr::topk_scores_ws_bytes(n_rows, n_items, d, k)) {
    gdr::set_error("topk_scores: workspace too small");
    return GDR_EWORKSPACE;
  }
  return gdr::topk_scores(n_rows, n_users, n_items, d, k, U, ldu, rows, I, ldi, ex_rowptr, ex_colidx, scores_out, lds,
                          items_out, ldit, status_dev, ws, ws_bytes, (cudaStream_t)stream);
}

int64_t gdr_ranking_metrics_ws_bytes(int64_t n_rows, int n_ks) {
  if (n_rows <= 0 || n_ks <= 0) return 256;
  return gdr::ranking_metrics_ws_bytes(n_rows, n_ks);
}

int gdr_ranking_metrics(int64_t n_rows, int64_t n_users, int64_t k, const int32_t* items, int64_t ldit,
                        const int64_t* rows, const int32_t* test_rowptr, const int32_t* test_colidx, int n_ks,
                        const int32_t* ks_host, double* sums_out_dev, int64_t* n_eval_dev, float* per_row_out,
                        void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows > 0 && n_users > 0 && k >= 1 && ldit >= k, "ranking_metrics: bad sizes");
  GDR_CHECK_ARG(items && test_rowptr && test_colidx && ks_host && sums_out_dev && n_eval_dev && ws,
                "ranking_metrics: null pointer");
  GDR_CHECK_ARG(n_ks >= 1 && n_ks <= gdr::TK_MAX_KS, "ranking_metrics: n_ks must be in [1, %d]", gdr::TK_MAX_KS);
  GDR_CHECK_ARG(rows || n_rows <= n_users, "ranking_metrics: n_rows > n_users without a rows list");
  gdr::TkKs ks;
  ks.n = n_ks;
  for (int q = 0; q < n_ks; ++q) {
    GDR_CHECK_ARG(ks_host[q] >= 1 && ks_host[q] <= k, "ranking_metrics: K=%d outside [1, k=%lld]", ks_host[q],
                  (long long)k);
    ks.k[q] = ks_host[q];
  }
  if (ws_bytes < gdr::ranking_metrics_ws_bytes(n_rows, n_ks)) {
    gdr::set_error("ranking_metrics: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  gdr::Workspace W(ws, ws_bytes);
  double* per_row = W.take<double>((int64_t)n_ks * 3 * n_rows);
  int32_t* valid = W.take<int32_t>(n_rows);
  gdr::k_rank_metrics<<<(unsigned)gdr::cdiv(n_rows * 32, 256), 256, 0, s>>>(
      n_rows, n_users, items, ldit, rows, test_rowptr, test_colidx, ks, per_row, per_row_out, valid);
  GDR_LAUNCHED();
  gdr::k_rank_sums<<<3 * n_ks + 1, 32, 0, s>>>(n_rows, 3 * n_ks, per_row, valid, sums_out_dev, n_eval_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

}  // extern "C"
