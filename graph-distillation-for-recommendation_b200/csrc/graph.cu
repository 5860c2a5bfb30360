// graph.cu — stage 1 (CSR construction, degrees, D^-1/2 A D^-1/2, bipartite
// normalisation, transpose) and stage 4 (cluster-coarsened graph by segmented
// edge counting).  All of it is integer / streaming work bound by HBM: packed
// 64-bit keys, the stable radix sort of primitives.cu, head flags + scan, and
// fixed-order run reductions — so integer outputs are bit-exact and float sums
// are deterministic.
//
// Reference semantics followed (paths relative to /root/reference/ClustGDD):
//   utils.py:66-67, distill_recsys.py:110-117   COO -> CSR, duplicates summed
//   utils_graphsaint.py:20-22                   A + A^T ; A[A>1] = 1
//   deep_robust_utils.py:180-207, 245-265       normalize_adj / normalize_adj_tensor
//   distill_recsys.py:184-201                   build_condensed_bipartite
//   clustgdd_agent_transduct.py:234-250         graph_compress
//   distill_recsys.py:329-335                   bipartite degree normalisation
#include "common.cuh"

namespace gdr {

static inline int bits_for(int64_t n) {  // bits needed to store values in [0, n)
  int b = 1;
  while ((1ll << b) < n) ++b;
  return b;
}

// ----------------------------------------------------------------------------
// reduce-by-key over SORTED (key, float payload) pairs
// ----------------------------------------------------------------------------
constexpr int RUN_SEQ_MAX = 64;  // runs up to this length are summed by one thread

__global__ void k_head_flags(int64_t n, const uint64_t* __restrict__ keys, int32_t* __restrict__ flags) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
}

// pos = exclusive scan of head flags (pos[n] = #runs).  For every head i write
// head_index[pos[i]] = i ; head_index[m] = n is written by the thread owning i = n-1.
__global__ void k_head_index(int64_t n, const uint64_t* __restrict__ keys,
                             const int32_t* __restrict__ pos, int32_t* __restrict__ head_index) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    if (i == 0 || keys[i] != keys[i - 1]) head_index[pos[i]] = (int32_t)i;
    if (i == n - 1) head_index[pos[n]] = (int32_t)n;
  }
}

// One thread per run: unique key, run length, and (short runs) the sequential
// fp32 sum in input order.  Long runs are queued for k_long_runs.
__global__ void k_run_reduce(const int32_t* __restrict__ n_runs_dev, const uint64_t* __restrict__ keys,
                             const uint32_t* __restrict__ payload,
                             const int32_t* __restrict__ head_index, uint64_t* __restrict__ ukeys,
                             int32_t* __restrict__ run_len, float* __restrict__ run_sum,
                             int32_t* __restrict__ long_list, int32_t* __restrict__ long_count) {
  int64_t m = *n_runs_dev;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m;
       p += (int64_t)gridDim.x * blockDim.x) {
    int b = head_index[p], e = head_index[p + 1];
    ukeys[p] = keys[b];
    run_len[p] = e - b;
    if (run_sum) {
      if (e - b <= RUN_SEQ_MAX) {
        float s = 0.f;
        for (int j = b; j < e; ++j) s = __fadd_rn(s, __uint_as_float(payload[j]));
        run_sum[p] = s;
      } else {
        int slot = atomicAdd(long_count, 1);
        long_list[slot] = (int32_t)p;
      }
    }
  }
}

// One CTA per long run (grid-strided over the queue); fixed summation shape:
// thread t adds elements t, t+256, ... in order, then a fixed tree.
__global__ void __launch_bounds__(256) k_long_runs(const int32_t* __restrict__ long_list,
                                                   const int32_t* __restrict__ long_count,
                                                   const uint32_t* __restrict__ payload,
                                                   const int32_t* __restrict__ head_index,
                                                   float* __restrict__ run_sum) {
  __shared__ float s_f[256];
  int cnt = *long_count;
  for (int q = blockIdx.x; q < cnt; q += gridDim.x) {
    int p = long_list[q];
    int b = head_index[p], e = head_index[p + 1];
    float s = 0.f;
    for (int j = b + threadIdx.x; j < e; j += 256) s = __fadd_rn(s, __uint_as_float(payload[j]));
    s_f[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (threadIdx.x < o) s_f[threadIdx.x] = __fadd_rn(s_f[threadIdx.x], s_f[threadIdx.x + o]);
      __syncthreads();
    }
    if (threadIdx.x == 0) run_sum[p] = s_f[0];
    __syncthreads();
  }
}

struct RunBuffers {
  int32_t* pos;         // n+1  (flags, scanned in place); pos[n] = #runs
  int32_t* head_index;  // n+1
  uint64_t* ukeys;      // n
  int32_t* run_len;     // n
  float* run_sum;       // n (or null)
  int32_t* long_list;   // n / RUN_SEQ_MAX + 1
  int32_t* long_count;  // 1
  void* scan_ws;
  int64_t scan_ws_b;
};

static int64_t runs_ws_bytes(int64_t n, bool with_sum) {
  return 2 * ws_need(n + 1, 4) + ws_need(n, 8) + ws_need(n, 4) + (with_sum ? ws_need(n, 4) : 0) +
         ws_need(n / RUN_SEQ_MAX + 2, 4) + 256 + scan_ws_bytes(n) + 256;
}

static RunBuffers carve_runs(Workspace& W, int64_t n, bool with_sum) {
  RunBuffers R;
  R.pos = W.take<int32_t>(n + 1);
  R.head_index = W.take<int32_t>(n + 1);
  R.ukeys = W.take<uint64_t>(n);
  R.run_len = W.take<int32_t>(n);
  R.run_sum = with_sum ? W.take<float>(n) : nullptr;
  R.long_list = W.take<int32_t>(n / RUN_SEQ_MAX + 2);
  R.long_count = W.take<int32_t>(1);
  R.scan_ws_b = scan_ws_bytes(n);
  R.scan_ws = W.take<char>(R.scan_ws_b);
  return R;
}

static unsigned grid_for(int64_t n, int threads = 256) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(n, threads), kSMs * 32));
}

// keys sorted ascending, payload (float bits) optional.
static int reduce_runs(int64_t n, const uint64_t* keys, const uint32_t* payload, RunBuffers& R,
                       cudaStream_t s) {
  k_head_flags<<<grid_for(n), 256, 0, s>>>(n, keys, R.pos);
  GDR_LAUNCHED();
  int rc = exclusive_scan_i32(R.pos, R.pos, n, R.scan_ws, R.scan_ws_b, s);
  if (rc) return rc;
  k_head_index<<<grid_for(n), 256, 0, s>>>(n, keys, R.pos, R.head_index);
  GDR_LAUNCHED();
  GDR_CUDA(cudaMemsetAsync(R.long_count, 0, 4, s));
  k_run_reduce<<<grid_for(n), 256, 0, s>>>(R.pos + n, keys, payload, R.head_index, R.ukeys, R.run_len,
                                           payload ? R.run_sum : nullptr, R.long_list, R.long_count);
  GDR_LAUNCHED();
  if (payload) {
    k_long_runs<<<kSMs * 2, 256, 0, s>>>(R.long_list, R.long_count, payload, R.head_index, R.run_sum);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

// rowptr[r] = first run whose (ukey >> shift) >= r, for r in [0, n_rows]
__global__ void k_rowptr_from_ukeys(const int32_t* __restrict__ n_runs_dev, int64_t n_rows, int shift,
                                    uint64_t valid_limit, const uint64_t* __restrict__ ukeys,
                                    int32_t* __restrict__ rowptr, int64_t* __restrict__ nnz_out) {
  int64_t m = *n_runs_dev;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= m;
       i += (int64_t)gridDim.x * blockDim.x) {
    // keys >= valid_limit are sentinels (dropped entries): they sort last
    int64_t lo = i == 0 ? -1 : (ukeys[i - 1] >= valid_limit ? n_rows : (int64_t)(ukeys[i - 1] >> shift));
    int64_t hi = i == m ? n_rows : (ukeys[i] >= valid_limit ? n_rows : (int64_t)(ukeys[i] >> shift));
    if (hi > n_rows) hi = n_rows;
    for (int64_t r = lo + 1; r <= hi; ++r) rowptr[r] = (int32_t)i;
    // all sentinel keys are equal, so they form at most one (the last) run
    if (i == m) *nnz_out = (m > 0 && ukeys[m - 1] >= valid_limit) ? m - 1 : m;
  }
}

// ----------------------------------------------------------------------------
// COO -> CSR
// ----------------------------------------------------------------------------
__global__ void k_pack_coo(int64_t nnz, int64_t n_rows, int64_t n_cols, const int64_t* __restrict__ row,
                           const int64_t* __restrict__ col, const float* __restrict__ val,
                           int symmetrize, int cbits, uint64_t* __restrict__ keys,
                           uint32_t* __restrict__ payload, int32_t* __restrict__ status) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz;
       e += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = row[e], c = col[e];
    float v = val ? val[e] : 1.0f;
    if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) {
      atomicOr(status, 1);
      r = 0;
      c = 0;
      v = 0.f;
    }
    if (symmetrize) {
      keys[2 * e] = ((uint64_t)r << cbits) | (uint64_t)c;
      keys[2 * e + 1] = ((uint64_t)c << cbits) | (uint64_t)r;
      if (payload) {
        payload[2 * e] = __float_as_uint(v);
        payload[2 * e + 1] = __float_as_uint(v);
      }
    } else {
      keys[e] = ((uint64_t)r << cbits) | (uint64_t)c;
      if (payload) payload[e] = __float_as_uint(v);
    }
  }
}

__global__ void k_emit_csr_entries(const int32_t* __restrict__ n_runs_dev,
                                   const uint64_t* __restrict__ ukeys, const float* __restrict__ run_sum,
                                   const int32_t* __restrict__ run_len,
                                   uint64_t cmask, int binarize, int32_t* __restrict__ colidx,
                                   float* __restrict__ vals) {
  int64_t m = *n_runs_dev;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m;
       p += (int64_t)gridDim.x * blockDim.x) {
    colidx[p] = (int32_t)(ukeys[p] & cmask);
    vals[p] = binarize ? 1.0f : (run_sum ? run_sum[p] : (float)run_len[p]);
  }
}

// ----------------------------------------------------------------------------
// sorted unique keys -> binarised CSR in two passes over the keys (the keys-only build of stage 1):
// count the heads of every 2048-key tile, scan the tile counts, then emit (colidx, 1.0) per head and fill rowptr on the
// fly.  Replaces head flags + scan + head index + run reduce + emit + rowptr (six passes) when no values are carried.
// ----------------------------------------------------------------------------
constexpr int UQ_THREADS = 256;
constexpr int UQ_ITEMS = 8;
constexpr int UQ_TILE = UQ_THREADS * UQ_ITEMS;

__global__ void __launch_bounds__(UQ_THREADS) k_unique_count(int64_t n, const uint64_t* __restrict__ keys,
                                                             int32_t* __restrict__ tile_count) {
  __shared__ int s_w[UQ_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * UQ_TILE;
  int c = 0;
#pragma unroll
  for (int q = 0; q < UQ_ITEMS; ++q) {
    const int64_t i = base + q * UQ_THREADS + threadIdx.x;
    if (i < n) c += (i == 0 || keys[i] != keys[i - 1]) ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane_id() == 0) s_w[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
#pragma unroll
    for (int w = 0; w < UQ_THREADS / 32; ++w) t += s_w[w];
    tile_count[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(UQ_THREADS) k_unique_emit_csr(int64_t n, int64_t n_rows, int cbits,
                                                                const uint64_t* __restrict__ keys,
                                                                const int32_t* __restrict__ tile_off /*[tiles + 1]*/,
                                                                int32_t* __restrict__ rowptr, int32_t* __restrict__ colidx,
                                                                float* __restrict__ vals, int64_t* __restrict__ nnz_out,
                                                                int32_t* __restrict__ head_pos /*nullable: sorted index of every head*/) {
  __shared__ int s_w[UQ_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * UQ_TILE;
  const uint64_t cmask = (1ull << cbits) - 1ull;
  int run = tile_off[blockIdx.x];
  const int w = threadIdx.x >> 5;
  // items are taken round by round (q * UQ_THREADS + thread): positions inside a round are consecutive over the threads
  for (int q = 0; q < UQ_ITEMS; ++q) {
    const int64_t i = base + q * UQ_THREADS + threadIdx.x;
    uint64_t k = 0, kp = 0;
    bool head = false;
    if (i < n) {
      k = keys[i];
      kp = i > 0 ? keys[i - 1] : 0;
      head = i == 0 || k != kp;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, head);
    if (lane_id() == 0) s_w[w] = __popc(bal);
    __syncthreads();
    int woff = 0, tot = 0;
#pragma unroll
    for (int ww = 0; ww < UQ_THREADS / 32; ++ww) {
      const int c = s_w[ww];
      woff += ww < w ? c : 0;
      tot += c;
    }
    if (head) {
      const int pos = run + woff + __popc(bal & ((1u << lane_id()) - 1u));
      colidx[pos] = (int32_t)(k & cmask);
      if (head_pos) head_pos[pos] = (int32_t)i;
      else vals[pos] = 1.0f;
      // rows (previous row, this row] start at this entry
      const int64_t r = (int64_t)(k >> cbits), rp = i == 0 ? -1 : (int64_t)(kp >> cbits);
      for (int64_t rr = rp + 1; rr <= r; ++rr) rowptr[rr] = pos;
    }
    if (i == n - 1) {   // rows after the last key, and the total
      const int total = run + tot;
      for (int64_t rr = (int64_t)(k >> cbits) + 1; rr <= n_rows; ++rr) rowptr[rr] = total;
      *nnz_out = total;
      if (head_pos) head_pos[total] = (int32_t)n;
    }
    run += tot;
    __syncthreads();
  }
}

// ----------------------------------------------------------------------------
// CSR transpose
// ----------------------------------------------------------------------------
__global__ void k_pack_transpose(int64_t n_rows, const int32_t* __restrict__ rowptr,
                                 const int32_t* __restrict__ colidx, int rbits,
                                 uint64_t* __restrict__ keys, uint32_t* __restrict__ payload) {
  // one warp per row
  int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = w; r < n_rows; r += nw) {
    int b = rowptr[r], e = rowptr[r + 1];
    for (int j = b + lane_id(); j < e; j += 32) {
      keys[j] = ((uint64_t)(uint32_t)colidx[j] << rbits) | (uint64_t)r;
      payload[j] = (uint32_t)j;
    }
  }
}

__global__ void k_unpack_transpose(int64_t nnz, int64_t n_cols, int rbits, const uint64_t* __restrict__ keys,
                                   const uint32_t* __restrict__ payload, int32_t* __restrict__ t_rowptr,
                                   int32_t* __restrict__ t_colidx, int32_t* __restrict__ t_perm) {
  uint64_t rmask = (1ull << rbits) - 1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= nnz;
       i += (int64_t)gridDim.x * blockDim.x) {
    if (i < nnz) {
      t_colidx[i] = (int32_t)(keys[i] & rmask);
      t_perm[i] = (int32_t)payload[i];
    }
    int64_t lo = i == 0 ? -1 : (int64_t)(keys[i - 1] >> rbits);
    int64_t hi = i == nnz ? n_cols : (int64_t)(keys[i] >> rbits);
    for (int64_t c = lo + 1; c <= hi; ++c) t_rowptr[c] = (int32_t)i;
  }
}

// ----------------------------------------------------------------------------
// symmetric normalisation
// ----------------------------------------------------------------------------
// flag[0] = 1 when the identity has to be added.
__global__ void k_selfloop_flag(int64_t nnz, const int32_t* __restrict__ rowptr,
                                const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                                int mode, int32_t* __restrict__ flag) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (mode == 0) {
    flag[0] = 0;
  } else if (mode == 1) {
    flag[0] = 1;
  } else {
    // reference quirk: `if mx[0, 0] == 0: mx = mx + I`  (deep_robust_utils.py:199-200)
    float a00 = 0.f;
    int b = rowptr[0], e = rowptr[1];
    for (int j = b; j < e; ++j)
      if (colidx[j] == 0) a00 += vals[j];
    flag[0] = (a00 == 0.f) ? 1 : 0;
  }
}

// one warp per row: degree (fp64 or fp32 chain, see k_norm_fill), diagonal presence, output length
__global__ void __launch_bounds__(256) k_row_degree(int64_t n, const int32_t* __restrict__ rowptr,
                                                    const int32_t* __restrict__ colidx,
                                                    const float* __restrict__ vals,
                                                    const int32_t* __restrict__ flag,
                                                    double* __restrict__ deg, int32_t* __restrict__ out_len,
                                                    int64_t row_offset /*global id of local row 0 (row-block mode)*/) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const int add = flag[0];
  const int32_t diag = (int32_t)(r + row_offset);
  int b = rowptr[r], e = rowptr[r + 1];
  double s = 0.0;
  float sf = 0.f;
  int has_diag = 0;
  for (int j = b + lane_id(); j < e; j += 32) {
    float v = vals[j];
    s += (double)v;
    sf += v;
    has_diag |= (colidx[j] == diag);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    sf += __shfl_xor_sync(0xffffffffu, sf, o);
    has_diag |= __shfl_xor_sync(0xffffffffu, has_diag, o);
  }
  if (lane_id() == 0) {
    // with +I the reference sums an fp64 matrix; without it the matrix (and the row sum) stay fp32
    deg[r] = add ? s + 1.0 : (double)sf;
    out_len[r] = (e - b) + ((add && !has_diag) ? 1 : 0);
  }
}

__global__ void __launch_bounds__(256) k_norm_fill(int64_t n, const int32_t* __restrict__ rowptr,
                                                   const int32_t* __restrict__ colidx,
                                                   const float* __restrict__ vals,
                                                   const int32_t* __restrict__ flag,
                                                   const double* __restrict__ deg_row /*by local row*/,
                                                   const double* __restrict__ deg /*by (global) column*/,
                                                   const int32_t* __restrict__ rowptr_out,
                                                   int32_t* __restrict__ colidx_out,
                                                   float* __restrict__ vals_out,
                                                   int64_t* __restrict__ nnz_out, int64_t row_offset) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const int add = flag[0];
  const int32_t diag = (int32_t)(r + row_offset);
  const int b = rowptr[r], e = rowptr[r + 1];
  const int ob = rowptr_out[r];
  const bool inserts = add && (rowptr_out[r + 1] - ob) > (e - b);
  if (r == n - 1 && lane_id() == 0) *nnz_out = rowptr_out[n];
  // r_i = deg^-1/2 ; inf -> 0   (deep_robust_utils.py:202-203)
  const double di = deg_row[r];
  if (add) {
    const double ri = di == 0.0 ? 0.0 : 1.0 / sqrt(di);
    // entries left of the diagonal keep their slot; the rest shift by one when I inserts
    for (int j = b + lane_id(); j < e; j += 32) {
      int c = colidx[j];
      double a = (double)vals[j] + (c == diag ? 1.0 : 0.0);
      double dj = deg[c];
      double rj = dj == 0.0 ? 0.0 : 1.0 / sqrt(dj);
      int o = ob + (j - b) + ((inserts && c > diag) ? 1 : 0);
      colidx_out[o] = c;
      vals_out[o] = (float)((ri * a) * rj);
    }
    if (inserts) {
      // position of the new diagonal entry = #entries with col < r (one lane finds it)
      int cnt = 0;
      for (int j = b + lane_id(); j < e; j += 32) cnt += (colidx[j] < diag);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      if (lane_id() == 0) {
        colidx_out[ob + cnt] = diag;
        vals_out[ob + cnt] = (float)((ri * 1.0) * ri);
      }
    }
  } else {
    // fp32 path of the reference when no identity is added: r = fp32 deg ^ -1/2
    const float dfi = (float)di;
    const float ri = dfi == 0.f ? 0.f : (float)(1.0 / sqrt((double)dfi));
    for (int j = b + lane_id(); j < e; j += 32) {
      int c = colidx[j];
      float dfj = (float)deg[c];
      float rj = dfj == 0.f ? 0.f : (float)(1.0 / sqrt((double)dfj));
      colidx_out[ob + (j - b)] = c;
      vals_out[ob + (j - b)] = __fmul_rn(__fmul_rn(ri, vals[j]), rj);
    }
  }
}

// dense n x n:  mx = A + I ; r = rowsum^-1/2 ; out = r_i * mx_ij * r_j  (fp32)
__global__ void __launch_bounds__(256) k_dense_rowsum(int64_t n, const float* __restrict__ A, int64_t lda,
                                                      float* __restrict__ rinv) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  float s = 0.f;
  for (int64_t c = lane_id(); c < n; c += 32) s += A[r * lda + c] + (c == r ? 1.f : 0.f);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane_id() == 0) {
    // torch CPU evaluates pow(x, -0.5) as 1 / sqrt(x) in fp32 (two roundings)
    float ri = __fdiv_rn(1.f, __fsqrt_rn(s));
    if (isinf(ri)) ri = 0.f;
    rinv[r] = ri;
  }
}

__global__ void k_dense_scale(int64_t n, const float* __restrict__ A, int64_t lda,
                              const float* __restrict__ rinv, float* __restrict__ out, int64_t ldo) {
  int64_t total = n * n;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / n, c = i - r * n;
    float m = A[r * lda + c] + (c == r ? 1.f : 0.f);
    out[r * ldo + c] = __fmul_rn(__fmul_rn(rinv[r], m), rinv[c]);
  }
}

// ----------------------------------------------------------------------------
// bipartite normalisation
// ----------------------------------------------------------------------------
// sequential fp32 row sums (index_add_ order on the CPU reference), one thread per row
__global__ void k_rowsum_seq(int64_t n, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ perm,
                             const float* __restrict__ w, float* __restrict__ deg) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n;
       r += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j) s = __fadd_rn(s, w[perm ? perm[j] : j]);
    deg[r] = s;
  }
}

__global__ void __launch_bounds__(256) k_bip_norm(int64_t n_u, const int32_t* __restrict__ rowptr,
                                                  const int32_t* __restrict__ colidx,
                                                  const float* __restrict__ w, const float* __restrict__ deg_u,
                                                  const float* __restrict__ deg_i, float eps,
                                                  float* __restrict__ norm_out) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_u) return;
  float su = __fsqrt_rn(__fadd_rn(deg_u[r], eps));
  for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
    float si = __fsqrt_rn(__fadd_rn(deg_i[colidx[j]], eps));
    norm_out[j] = __fdiv_rn(w[j], __fmul_rn(su, si));
  }
}

// Rankformer GCN weights: out_e = w_e / (max(du,1)^a * max(di,1)^b)  (two divisions, as torch evaluates
// ones / du.pow(a) / di.pow(b)); du / di are the (integer-valued) interaction counts.
__global__ void __launch_bounds__(256) k_bip_pow_norm(int64_t n_u, const int32_t* __restrict__ rowptr,
                                                      const int32_t* __restrict__ colidx,
                                                      const float* __restrict__ w, const float* __restrict__ deg_u,
                                                      const float* __restrict__ deg_i, float a, float b,
                                                      float* __restrict__ out) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_u) return;
  const float pu = powf(fmaxf(deg_u[r], 1.f), a);
  for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
    const float pi = powf(fmaxf(deg_i[colidx[j]], 1.f), b);
    out[j] = __fmul_rn(w[j], __fdiv_rn(__fdiv_rn(1.f, pu), pi));
  }
}

__global__ void k_gather_f32(int64_t n, const int32_t* __restrict__ perm, const float* __restrict__ in,
                             float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = in[perm[i]];
}

// ----------------------------------------------------------------------------
// coarsening
// ----------------------------------------------------------------------------
__global__ void k_pack_coarsen_coo(int64_t E, const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                   const float* __restrict__ w, const int32_t* __restrict__ lab_s,
                                   const int32_t* __restrict__ lab_d, int bbits, int drop_diag,
                                   uint64_t sentinel, uint64_t* __restrict__ keys,
                                   uint32_t* __restrict__ payload) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E;
       e += (int64_t)gridDim.x * blockDim.x) {
    uint32_t a = (uint32_t)lab_s[src[e]], b = (uint32_t)lab_d[dst[e]];
    keys[e] = (drop_diag && a == b) ? sentinel : (((uint64_t)a << bbits) | (uint64_t)b);
    if (payload) payload[e] = __float_as_uint(w[e]);
  }
}

__global__ void k_pack_coarsen_csr(int64_t n_rows, const int32_t* __restrict__ rowptr,
                                   const int32_t* __restrict__ colidx, const float* __restrict__ w,
                                   const int32_t* __restrict__ lab_s, const int32_t* __restrict__ lab_d,
                                   int bbits, int drop_diag, uint64_t sentinel,
                                   uint64_t* __restrict__ keys, uint32_t* __restrict__ payload) {
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = wid; r < n_rows; r += nw) {
    uint32_t a = (uint32_t)lab_s[r];
    for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
      uint32_t b = (uint32_t)lab_d[colidx[j]];
      keys[j] = (drop_diag && a == b) ? sentinel : (((uint64_t)a << bbits) | (uint64_t)b);
      if (payload) payload[j] = __float_as_uint(w[j]);
    }
  }
}

__global__ void k_emit_coarse(const int32_t* __restrict__ n_runs_dev, const uint64_t* __restrict__ ukeys,
                              const int32_t* __restrict__ run_len, const float* __restrict__ run_sum,
                              uint64_t bmask, uint64_t sentinel, int32_t* __restrict__ colidx,
                              int32_t* __restrict__ counts, float* __restrict__ wsum) {
  int64_t m = *n_runs_dev;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m;
       p += (int64_t)gridDim.x * blockDim.x) {
    if (ukeys[p] >= sentinel) continue;
    colidx[p] = (int32_t)(ukeys[p] & bmask);
    counts[p] = run_len[p];
    if (wsum) wsum[p] = run_sum[p];
  }
}

__global__ void __launch_bounds__(256) k_coarsen_scale(int64_t n_src, const int32_t* __restrict__ rowptr,
                                                       const int32_t* __restrict__ colidx,
                                                       const float* __restrict__ wsum,
                                                       const int32_t* __restrict__ size_s,
                                                       const int32_t* __restrict__ size_d,
                                                       float* __restrict__ out) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_src) return;
  float ia = __fdiv_rn(1.0f, (float)size_s[r]);
  for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
    float ib = __fdiv_rn(1.0f, (float)size_d[colidx[j]]);
    out[j] = __fmul_rn(__fmul_rn(wsum[j], ia), ib);
  }
}

// ---- multi-GPU stage 4, routing form: every edge becomes a (cell key, weight) pair tagged with the OWNER of its coarse
// row in the top byte of the key; one stable partition pass groups the pairs by owner (dropped diagonal pairs go to bucket
// 127), the owners sort + reduce what they receive.  One sort per edge instead of two (local coarsening + merge), and the
// in-cell order of the weights is the global CSR order, so the sums are bit-identical to the single-device result.
constexpr int ROUTE_SHIFT = 56;
constexpr int ROUTE_DROP = 127;
__global__ void k_pack_route_coo(int64_t E, const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                 const float* __restrict__ w, const int32_t* __restrict__ lab_s,
                                 const int32_t* __restrict__ lab_d, int bbits, int drop_diag, int cr, int world,
                                 uint64_t* __restrict__ keys, uint32_t* __restrict__ payload) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t a = (uint32_t)lab_s[src[e]], b = (uint32_t)lab_d[dst[e]];
    const uint64_t owner = (drop_diag && a == b) ? (uint64_t)ROUTE_DROP : (uint64_t)min((int)(a / (uint32_t)cr), world - 1);
    keys[e] = (owner << ROUTE_SHIFT) | ((uint64_t)a << bbits) | (uint64_t)b;
    if (payload) payload[e] = __float_as_uint(w[e]);
  }
}

__global__ void k_pack_route_csr(int64_t n_rows, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                 const float* __restrict__ w, const int32_t* __restrict__ lab_s,
                                 const int32_t* __restrict__ lab_d, int bbits, int drop_diag, int cr, int world,
                                 uint64_t* __restrict__ keys, uint32_t* __restrict__ payload) {
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = wid; r < n_rows; r += nw) {
    const uint32_t a = (uint32_t)lab_s[r];
    const uint64_t own = (uint64_t)min((int)(a / (uint32_t)cr), world - 1);
    for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
      const uint32_t b = (uint32_t)lab_d[colidx[j]];
      const uint64_t owner = (drop_diag && a == b) ? (uint64_t)ROUTE_DROP : own;
      keys[j] = (owner << ROUTE_SHIFT) | ((uint64_t)a << bbits) | (uint64_t)b;
      if (payload) payload[j] = __float_as_uint(w[j]);
    }
  }
}

__global__ void k_mask_keys(int64_t n, const uint64_t* __restrict__ in, uint64_t mask, uint64_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = in[i] & mask;
}

// vals[p] = multiplicity of the p-th unique key (duplicate COO lines summed: unit values, exact in fp32 up to 2^24)
__global__ void k_run_length_vals(const int64_t* __restrict__ nnz_dev, const int32_t* __restrict__ head_pos,
                                  float* __restrict__ vals) {
  const int64_t m = *nnz_dev;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x)
    vals[p] = (float)(head_pos[p + 1] - head_pos[p]);
}

// ---- multi-GPU stage 1, routing form: every (row, col) pair [and its mirror] becomes a key tagged with the owner rank of
// its row in the top byte; one stable partition pass groups the keys by owner.  status bit 0: index out of range,
// bit 1: the pair (0, 0) is present (the reference's `if mx[0, 0] == 0` rule needs to know).
__global__ void k_pack_edge_route(int64_t E, int64_t n_rows, int64_t n_cols, const int64_t* __restrict__ row,
                                  const int64_t* __restrict__ col, int symmetrize, int cbits, int64_t rows_per, int world,
                                  uint64_t* __restrict__ keys, int32_t* __restrict__ status) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = row[e], c = col[e];
    if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) {
      atomicOr(status, 1);
      r = 0;
      c = 0;
    } else if (r == 0 && c == 0) {
      atomicOr(status, 2);
    }
    const uint64_t o1 = (uint64_t)min((int64_t)(world - 1), r / rows_per);
    if (symmetrize) {
      const uint64_t o2 = (uint64_t)min((int64_t)(world - 1), c / rows_per);
      keys[2 * e] = (o1 << ROUTE_SHIFT) | ((uint64_t)r << cbits) | (uint64_t)c;
      keys[2 * e + 1] = (o2 << ROUTE_SHIFT) | ((uint64_t)c << cbits) | (uint64_t)r;
    } else {
      keys[e] = (o1 << ROUTE_SHIFT) | ((uint64_t)r << cbits) | (uint64_t)c;
    }
  }
}

// received keys -> keys of the local row block: owner byte cleared, row made local
__global__ void k_localise_keys(int64_t n, const uint64_t* __restrict__ in, uint64_t mask, uint64_t row_lo_shifted,
                                uint64_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (in[i] & mask) - row_lo_shifted;
}

// ---- key-range merge of per-rank coarsened graphs (multi-GPU stage 4) ----
// cell key of every entry of a coarse CSR: (a << bbits) | b
// 16-byte record per entry: [cell key | (count << 32) | weight-sum bits]
__global__ void k_coarse_records(int64_t n_src, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                 const int32_t* __restrict__ counts, const float* __restrict__ wsum, int bbits,
                                 uint64_t* __restrict__ rec) {
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = wid; r < n_src; r += nw)
    for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
      rec[2 * (int64_t)j] = ((uint64_t)r << bbits) | (uint64_t)(uint32_t)colidx[j];
      rec[2 * (int64_t)j + 1] = ((uint64_t)(uint32_t)counts[j] << 32) | (uint64_t)(wsum ? __float_as_uint(wsum[j]) : 0u);
    }
}

__global__ void k_split_records(int64_t n, const uint64_t* __restrict__ rec, uint64_t* __restrict__ keys,
                                uint32_t* __restrict__ perm) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    keys[i] = rec[2 * i];
    perm[i] = (uint32_t)i;
  }
}

// one thread per run of equal cells: integer count sum (exact) and fp32 weight sum in the stable order of the
// records (= source-rank order of the exchange: deterministic); runs are at most `world` long
__global__ void k_merge_runs(const int32_t* __restrict__ n_runs_dev, const int32_t* __restrict__ head_index,
                             const uint64_t* __restrict__ ukeys, const uint32_t* __restrict__ perm,
                             const uint64_t* __restrict__ rec, uint64_t bmask,
                             int32_t* __restrict__ colidx, int32_t* __restrict__ counts, float* __restrict__ wsum) {
  int64_t m = *n_runs_dev;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x) {
    int c = 0;
    float s = 0.f;
    for (int j = head_index[p]; j < head_index[p + 1]; ++j) {
      const uint64_t v = rec[2 * (int64_t)perm[j] + 1];
      c += (int)(uint32_t)(v >> 32);
      s = __fadd_rn(s, __uint_as_float((uint32_t)v));
    }
    colidx[p] = (int32_t)(ukeys[p] & bmask);
    counts[p] = c;
    if (wsum) wsum[p] = s;
  }
}

// rowptr of the coarse rows [a_lo, a_lo + n_rows) from the sorted unique keys
__global__ void k_rowptr_from_ukeys_range(const int32_t* __restrict__ n_runs_dev, int64_t a_lo, int64_t n_rows, int shift,
                                          const uint64_t* __restrict__ ukeys, int32_t* __restrict__ rowptr,
                                          int64_t* __restrict__ nnz_out) {
  int64_t m = *n_runs_dev;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= m; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = i == 0 ? -1 : (int64_t)(ukeys[i - 1] >> shift) - a_lo;
    int64_t hi = i == m ? n_rows : (int64_t)(ukeys[i] >> shift) - a_lo;
    if (hi > n_rows) hi = n_rows;
    if (lo < -1) lo = -1;
    for (int64_t r = lo + 1; r <= hi; ++r) rowptr[r] = (int32_t)i;
    if (i == m) *nnz_out = m;
  }
}

// sparse (rowptr, colidx, counts, wsum) -> dense n_src x n_dst (one writer per cell: no atomics)
__global__ void k_scatter_dense(int64_t n_src, int64_t n_dst, const int32_t* __restrict__ rowptr,
                                const int32_t* __restrict__ colidx, const int32_t* __restrict__ counts,
                                const float* __restrict__ wsum, int32_t* __restrict__ dc,
                                float* __restrict__ dw) {
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = wid; r < n_src; r += nw) {
    for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
      dc[r * n_dst + colidx[j]] = counts[j];
      if (dw) dw[r * n_dst + colidx[j]] = wsum[j];
    }
  }
}

// one warp per row of the dense count matrix
__global__ void __launch_bounds__(256) k_dense_row_nnz(int64_t n_src, int64_t n_dst,
                                                       const int32_t* __restrict__ dc,
                                                       int32_t* __restrict__ row_len) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_src) return;
  int c = 0;
  for (int64_t j = lane_id(); j < n_dst; j += 32) c += dc[r * n_dst + j] != 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane_id() == 0) row_len[r] = c;
}

__global__ void __launch_bounds__(256) k_dense_compact(int64_t n_src, int64_t n_dst,
                                                       const int32_t* __restrict__ dc,
                                                       const float* __restrict__ dw,
                                                       const int32_t* __restrict__ rowptr,
                                                       int32_t* __restrict__ colidx, int32_t* __restrict__ counts,
                                                       float* __restrict__ wsum, int64_t* __restrict__ nnz_out) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_src) return;
  if (r == n_src - 1 && lane_id() == 0) *nnz_out = rowptr[n_src];
  int o = rowptr[r];
  for (int64_t j0 = 0; j0 < n_dst; j0 += 32) {
    int64_t j = j0 + lane_id();
    int c = j < n_dst ? dc[r * n_dst + j] : 0;
    unsigned m = __ballot_sync(0xffffffffu, c != 0);
    if (c != 0) {
      int p = o + __popc(m & ((1u << lane_id()) - 1u));
      colidx[p] = (int32_t)j;
      counts[p] = c;
      if (wsum && dw) wsum[p] = dw[r * n_dst + j];
    }
    o += __popc(m);
  }
}

__global__ void k_csr_to_coo(int64_t n_rows, const int32_t* __restrict__ rowptr,
                             const int32_t* __restrict__ colidx, int64_t* __restrict__ row_out,
                             int64_t* __restrict__ col_out) {
  int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = wid; r < n_rows; r += nw) {
    for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
      row_out[j] = r;
      if (col_out) col_out[j] = (int64_t)colidx[j];
    }
  }
}

// ---------------- coarsening: one CTA per coarse row, cells accumulated in shared memory ----------------
// P^T A P for a CSR A (clustgdd_agent_transduct.py:234-250) without sorting the edges.  The nodes are grouped by their
// cluster (a counting sort of n_rows ids); the CTA that owns cluster a walks the adjacency rows of its nodes once and
// accumulates cell (a, b = label[col]) into a dense shared-memory row of n_dst counters:
//   count[b] += 1 (u32),  sum[b] += round(w / q_a) (i64 fixed point)
// Integer accumulation is associative, so the result does not depend on the order in which the shared-memory atomics
// land: bit-reproducible.  q_a = pow2(max |w| of the cluster) * pow2(edges of the cluster) * 2^-62 — no overflow, ~2^-48
// of the largest weight.  Each term is rounded to a multiple of q_a, so a cell of n edges is within n * q_a / 2 plus one
// fp32 rounding of its exact sum: one ulp only when the cell is at least about n * q_a * 2^24.  The row is then compacted
// in column order into a scratch slice (at the cluster's edge offset), and a second small kernel packs the slices into
// the final CSR.  HBM traffic: the edges once (8 B each), the column labels through L2, the cells twice — against four
// (key, value) radix passes over all edges before.
constexpr int CD_THREADS = 1024;
constexpr int CD_HUB = 4096;          // rows at least this long are walked by the whole CTA

__global__ void __launch_bounds__(256) k_cd_stats(int64_t n_rows, const int32_t* __restrict__ rowptr, const float* __restrict__ w,
                                                  const int32_t* __restrict__ labels, int64_t n_src,
                                                  int32_t* __restrict__ node_cnt, int32_t* __restrict__ edge_cnt,
                                                  uint32_t* __restrict__ wmax_bits, int32_t* __restrict__ status) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n_rows) return;
  const int lane = threadIdx.x & 31;
  const int32_t a = labels[i];
  if (a < 0 || a >= n_src) {
    if (lane == 0) atomicOr(status, 1);
    return;
  }
  const int32_t b = rowptr[i], e = rowptr[i + 1];
  float m = 0.f;
  if (w)
    for (int32_t k = b + lane; k < e; k += 32) m = fmaxf(m, fabsf(w[k]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) {
    atomicAdd(&node_cnt[a], 1);
    atomicAdd(&edge_cnt[a], e - b);
    if (w) atomicMax(&wmax_bits[a], __float_as_uint(m));     // non-negative floats order like their bit patterns
  }
}

__global__ void k_cd_group(int64_t n_rows, const int32_t* __restrict__ labels, const int32_t* __restrict__ starts,
                           int32_t* __restrict__ cursor, int32_t* __restrict__ nodes) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t a = labels[i];
    nodes[starts[a] + atomicAdd(&cursor[a], 1)] = (int32_t)i;
  }
}

// PAIRS: the edges of coarse row a are the (key, weight) pairs [starts[a], starts[a + 1]) of a list grouped by coarse row
// (key = column << la | local row: the owner side of the multi-GPU exchange); the fixed-point step comes from the
// GLOBAL per-cluster (edges, max |w|), so that every rank count and the single-GPU form round every term identically.
struct CdPairs {
  const uint64_t* keys;
  const float* w;
  int la;
  int64_t a_lo;
  const int32_t* g_edges;
  const uint32_t* g_wmax;
};

template <bool HAS_W, bool PAIRS>
__global__ void __launch_bounds__(CD_THREADS, 1)
k_cd_accumulate(int64_t n_src, int64_t n_dst, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                const float* __restrict__ w, const int32_t* __restrict__ labels_dst, const int32_t* __restrict__ starts,
                const int32_t* __restrict__ nodes, const int32_t* __restrict__ edge_prefix, const uint32_t* __restrict__ wmax_bits,
                int drop_diag, int32_t* __restrict__ next_cluster, int32_t* __restrict__ t_col, int32_t* __restrict__ t_cnt,
                float* __restrict__ t_sum, int32_t* __restrict__ nnz_row, int32_t* __restrict__ status, CdPairs pr) {
  extern __shared__ __align__(16) unsigned char cd_smem[];
  // 64-bit fixed-point sums as two 32-bit words with a carry (a 64-bit shared-memory add is a CAS spin loop)
  uint32_t* s_lo = reinterpret_cast<uint32_t*>(cd_smem);                                            // [HAS_W ? n_dst : 0]
  uint32_t* s_hi = s_lo + (HAS_W ? n_dst : 0);                                                      // [HAS_W ? n_dst : 0]
  uint32_t* s_cnt = s_hi + (HAS_W ? n_dst : 0);                                                     // [n_dst]
  __shared__ int s_a, s_hub_n, s_warp_tot[CD_THREADS / 32], s_hub[64];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int64_t b = tid; b < n_dst; b += CD_THREADS) {
    s_cnt[b] = 0;
    if (HAS_W) s_lo[b] = s_hi[b] = 0u;
  }
  for (;;) {
    __syncthreads();
    if (tid == 0) {
      s_a = atomicAdd(next_cluster, 1);
      s_hub_n = 0;
    }
    __syncthreads();
    const int a = s_a;
    if (a >= n_src) break;
    const int32_t nb = starts[a], ne = starts[a + 1];
    const int32_t n_edges = !HAS_W ? 0 : (PAIRS ? pr.g_edges[pr.a_lo + a] : edge_prefix[a + 1] - edge_prefix[a]);
    // fixed-point step of this cluster: |sum of any cell| <= wmax * n_edges < 2^(ew + ee)
    double inv_q = 0.0, q = 0.0;
    if (HAS_W) {
      int ew = 0, ee = 0;
      frexpf(__uint_as_float(PAIRS ? pr.g_wmax[pr.a_lo + a] : wmax_bits[a]), &ew);
      frexp((double)(n_edges > 0 ? n_edges : 1), &ee);
      q = ldexp(1.0, ew + ee - 62);
      inv_q = ldexp(1.0, 62 - ew - ee);
    }
    auto add_cell = [&](int32_t b, float wk) {
      if ((uint32_t)b >= (uint64_t)n_dst) {       // a label outside [0, n_dst) has no cell (the Python face never passes one)
        atomicOr(status, 1);
        return;
      }
      if (drop_diag && b == a) return;
      atomicAdd(&s_cnt[b], 1u);
      if (HAS_W) {
        const unsigned long long v = (unsigned long long)__double2ll_rn((double)wk * inv_q);
        const uint32_t lo = (uint32_t)v, old = atomicAdd(&s_lo[b], lo);
        atomicAdd(&s_hi[b], (uint32_t)(v >> 32) + ((uint32_t)(old + lo) < old ? 1u : 0u));
      }
    };
    // edges k, k + stride of one row together: both label gathers are in flight before the first atomic
    auto add_edges = [&](int32_t k0, int32_t re, int32_t stride) {
      for (int32_t k = k0; k < re; k += 2 * stride) {
        const bool two = k + stride < re;
        const int32_t j0 = colidx[k], j1 = two ? colidx[k + stride] : 0;
        const float w0 = HAS_W ? w[k] : 0.f, w1 = (HAS_W && two) ? w[k + stride] : 0.f;
        const int32_t c0 = __ldg(labels_dst + j0), c1 = two ? __ldg(labels_dst + j1) : 0;
        add_cell(c0, w0);
        if (two) add_cell(c1, w1);
      }
    };
    if (PAIRS) {
      for (int32_t k = nb + tid; k < ne; k += 2 * CD_THREADS) {
        const bool two = k + CD_THREADS < ne;
        const uint64_t k0 = pr.keys[k], k1 = two ? pr.keys[k + CD_THREADS] : 0ull;
        const float w0 = HAS_W ? pr.w[k] : 0.f, w1 = (HAS_W && two) ? pr.w[k + CD_THREADS] : 0.f;
        add_cell((int32_t)(k0 >> pr.la), w0);
        if (two) add_cell((int32_t)(k1 >> pr.la), w1);
      }
    }
    // one warp per adjacency row; very long rows are left to the whole CTA
    for (int32_t t = nb + warp; !PAIRS && t < ne; t += CD_THREADS / 32) {
      const int32_t i = nodes[t];
      const int32_t rb = rowptr[i], re = rowptr[i + 1];
      if (re - rb >= CD_HUB) {
        int slot = 0;
        if (lane == 0) slot = atomicAdd(&s_hub_n, 1);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot < 64) {                 // (a 65th hub row of one cluster is walked by its warp like any other row)
          if (lane == 0) s_hub[slot] = i;
          continue;
        }
      }
      add_edges(rb + lane, re, 32);
    }
    __syncthreads();
    const int hubs = PAIRS ? 0 : (s_hub_n < 64 ? s_hub_n : 64);
    for (int h = 0; h < hubs; ++h) {
      const int32_t i = s_hub[h];
      add_edges(rowptr[i] + tid, rowptr[i + 1], CD_THREADS);
    }
    __syncthreads();
    // compact the row in column order: contiguous chunk per thread, block-wide exclusive scan of the chunk counts
    const int64_t per = (n_dst + CD_THREADS - 1) / CD_THREADS;
    const int64_t b0 = (int64_t)tid * per, b1 = b0 + per < n_dst ? b0 + per : n_dst;
    int mine = 0;
    for (int64_t b = b0; b < b1; ++b) mine += s_cnt[b] != 0;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp_tot[warp] = incl;
    __syncthreads();
    int base = 0, total = 0;
#pragma unroll
    for (int ww = 0; ww < CD_THREADS / 32; ++ww) {
      if (ww < warp) base += s_warp_tot[ww];
      total += s_warp_tot[ww];
    }
    int64_t out = (int64_t)edge_prefix[a] + base + incl - mine;
    for (int64_t b = b0; b < b1; ++b) {
      const uint32_t c = s_cnt[b];
      if (c) {
        t_col[out] = (int32_t)b;
        t_cnt[out] = (int32_t)c;
        if (HAS_W) {
          t_sum[out] = (float)((double)(long long)(((unsigned long long)s_hi[b] << 32) | s_lo[b]) * q);
          s_lo[b] = s_hi[b] = 0u;
        }
        s_cnt[b] = 0;
        ++out;
      }
    }
    if (tid == 0) nnz_row[a] = total;
  }
}

// scratch slices -> final CSR arrays (one CTA per coarse row)
__global__ void __launch_bounds__(256) k_cd_pack(int64_t n_src, const int32_t* __restrict__ edge_prefix, const int32_t* __restrict__ rowptr,
                                                 const int32_t* __restrict__ t_col, const int32_t* __restrict__ t_cnt,
                                                 const float* __restrict__ t_sum, int32_t* __restrict__ colidx,
                                                 int32_t* __restrict__ counts, float* __restrict__ wsum, int64_t* __restrict__ nnz_out) {
  for (int64_t a = blockIdx.x; a < n_src; a += gridDim.x) {
    const int64_t src = edge_prefix[a], dst = rowptr[a];
    const int n = rowptr[a + 1] - rowptr[a];
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
      colidx[dst + k] = t_col[src + k];
      counts[dst + k] = t_cnt[src + k];
      if (wsum) wsum[dst + k] = t_sum[src + k];
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) nnz_out[0] = rowptr[n_src];
}

int g_coarsen_dense = 1;   // gdr_debug_set("coarsen_dense", 0): always the sort path

static int64_t cd_small_bytes(int64_t n_rows, int64_t n_src) {
  return ws_need(n_rows, 4) + 6 * ws_need(n_src + 1, 4) + scan_ws_bytes(n_src + 1) + 512;
}

// true when the dense path applies: CSR input, the coarse row fits in shared memory, the scratch fits in the workspace
static bool cd_applicable(int64_t E, int64_t n_rows, int64_t n_src, int64_t n_dst, bool has_w, int64_t ws_bytes) {
  if (!g_coarsen_dense || n_rows <= 0) return false;
  const int64_t smem = n_dst * (has_w ? 12 : 4);
  if (smem > 200 * 1024) return false;
  if (E < 4 * n_src) return false;                    // hardly any edges per coarse row: the sort is the cheaper way
  return 3 * ws_need(E, 4) + cd_small_bytes(n_rows, n_src) <= ws_bytes;
}

static int coarsen_dense(int64_t E, int64_t n_rows, const int32_t* csr_rowptr, const int32_t* csr_colidx, const float* w,
                         const int32_t* labels_src, const int32_t* labels_dst, int64_t n_src, int64_t n_dst,
                         int drop_diag, int32_t* rowptr, int32_t* colidx, int32_t* counts, float* wsum, int64_t* nnz_out_dev,
                         void* ws, int64_t ws_bytes, cudaStream_t s) {
  Workspace W(ws, ws_bytes);
  int32_t* t_col = W.take<int32_t>(E);
  int32_t* t_cnt = W.take<int32_t>(E);
  float* t_sum = W.take<float>(E);
  int32_t* nodes = W.take<int32_t>(n_rows);
  int32_t* node_cnt = W.take<int32_t>(n_src + 1);     // the next five blocks are cleared together
  int32_t* edge_cnt = W.take<int32_t>(n_src + 1);
  uint32_t* wmax = W.take<uint32_t>(n_src + 1);
  int32_t* cursor = W.take<int32_t>(n_src + 1);
  int32_t* starts = W.take<int32_t>(n_src + 1);
  int32_t* edge_prefix = W.take<int32_t>(n_src + 1);
  int32_t* misc = W.take<int32_t>(64);                 // [0] next cluster, [1] status
  const int64_t sws_b = scan_ws_bytes(n_src + 1);
  void* sws = W.take<char>(sws_b);
  if (!W.ok()) {
    set_error("coarsen: workspace too small");
    return GDR_EWORKSPACE;
  }
  GDR_CUDA(cudaMemsetAsync(node_cnt, 0, (char*)starts - (char*)node_cnt, s));
  GDR_CUDA(cudaMemsetAsync(misc, 0, 256, s));
  k_cd_stats<<<(unsigned)cdiv(n_rows * 32, 256), 256, 0, s>>>(n_rows, csr_rowptr, wsum ? w : nullptr, labels_src, n_src, node_cnt,
                                                            edge_cnt, wmax, misc + 1);
  GDR_LAUNCHED();
  int rc;
  if ((rc = exclusive_scan_i32(node_cnt, starts, n_src, sws, sws_b, s))) return rc;
  if ((rc = exclusive_scan_i32(edge_cnt, edge_prefix, n_src, sws, sws_b, s))) return rc;
  k_cd_group<<<grid_for(n_rows), 256, 0, s>>>(n_rows, labels_src, starts, cursor, nodes);
  GDR_LAUNCHED();
  int dev = 0, sms = kSMs;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const size_t smem = (size_t)n_dst * (wsum ? 12 : 4);
  const unsigned grid = (unsigned)std::min<int64_t>(n_src, sms);
  int32_t* nnz_row = node_cnt;                         // free again after the scan
  if (wsum) {
    static PerDevice<bool> attr;
    if (!attr.get()) {
      GDR_CUDA(cudaFuncSetAttribute(k_cd_accumulate<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr.get() = true;
    }
    k_cd_accumulate<true, false><<<grid, CD_THREADS, smem, s>>>(n_src, n_dst, csr_rowptr, csr_colidx, w, labels_dst, starts, nodes,
                                                               edge_prefix, wmax, drop_diag, misc, t_col, t_cnt, t_sum, nnz_row,
                                                               misc + 1, CdPairs{});
  } else {
    static PerDevice<bool> attr;
    if (!attr.get()) {
      GDR_CUDA(cudaFuncSetAttribute(k_cd_accumulate<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr.get() = true;
    }
    k_cd_accumulate<false, false><<<grid, CD_THREADS, smem, s>>>(n_src, n_dst, csr_rowptr, csr_colidx, nullptr, labels_dst, starts,
                                                                nodes, edge_prefix, wmax, drop_diag, misc, t_col, t_cnt, nullptr,
                                                                nnz_row, misc + 1, CdPairs{});
  }
  GDR_LAUNCHED();
  if ((rc = exclusive_scan_i32(nnz_row, rowptr, n_src, sws, sws_b, s))) return rc;
  k_cd_pack<<<(unsigned)std::min<int64_t>(n_src, 8 * sms), 256, 0, s>>>(n_src, edge_prefix, rowptr, t_col, t_cnt, t_sum, colidx, counts,
                                                                       wsum, nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

// key (owner tag | row << bbits | col) -> (col << la) | (row - a_lo): a stable sort on the low la bits groups by coarse row
__global__ void k_cd_swap_keys(int64_t m, const uint64_t* __restrict__ in, int bbits, int la, int64_t a_lo, uint64_t* __restrict__ out) {
  const uint64_t cell_mask = (1ull << ROUTE_SHIFT) - 1ull, bmask = (1ull << bbits) - 1ull;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t cell = in[i] & cell_mask;
    out[i] = ((cell & bmask) << la) | (uint64_t)((int64_t)(cell >> bbits) - a_lo);
  }
}
// starts[a] = first pair of local coarse row a in the grouped list (binary search), starts[n_rows] = m
__global__ void k_cd_pair_starts(int64_t m, const uint64_t* __restrict__ keys, int la, int64_t n_rows, int32_t* __restrict__ starts) {
  const int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a > n_rows) return;
  const uint64_t amask = (1ull << la) - 1ull;
  int64_t lo = 0, hi = m;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)(keys[mid] & amask) < a) lo = mid + 1;
    else hi = mid;
  }
  starts[a] = (int32_t)lo;
}

}  // namespace gdr

using namespace gdr;

extern "C" {

// ---------------- COO -> CSR ----------------
int64_t gdr_coo_to_csr_ws_bytes(int64_t n_rows, int64_t n_cols, int64_t nnz_in, int symmetrize) {
  (void)n_rows;
  (void)n_cols;
  int64_t n = nnz_in * (symmetrize ? 2 : 1);
  if (n <= 0) return 256;
  return ws_need(n, 8) + ws_need(n, 4) + sort_pairs_ws_bytes(n) + runs_ws_bytes(n, true) + 512;
}

int gdr_coo_to_csr(int64_t n_rows, int64_t n_cols, int64_t nnz_in, const int64_t* row,
                   const int64_t* col, const float* val, int symmetrize, int binarize,
                   int32_t* rowptr, int32_t* colidx, float* vals, int64_t* nnz_out_dev,
                   int32_t* status_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows >= 0 && n_cols >= 0 && nnz_in >= 0, "coo_to_csr: negative size");
  GDR_CHECK_ARG(rowptr && nnz_out_dev && status_dev, "coo_to_csr: null output");
  GDR_CHECK_ARG(!symmetrize || n_rows == n_cols, "coo_to_csr: symmetrize needs a square matrix");
  GDR_CHECK_ARG(n_rows < (1ll << 31) && n_cols < (1ll << 31), "coo_to_csr: dimension exceeds int32");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t n = nnz_in * (symmetrize ? 2 : 1);
  if (n >= (1ll << 31)) {
    set_error("coo_to_csr: %lld entries exceed the int32 CSR limit", (long long)n);
    return GDR_ERANGE;
  }
  GDR_CUDA(cudaMemsetAsync(status_dev, 0, 4, s));
  if (n == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr, 0, (n_rows + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(row && col && colidx && vals, "coo_to_csr: null pointer");
  if (ws_bytes < gdr_coo_to_csr_ws_bytes(n_rows, n_cols, nnz_in, symmetrize)) {
    set_error("coo_to_csr: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(n);
  uint32_t* payload = W.take<uint32_t>(n);
  int64_t sws_b = sort_pairs_ws_bytes(n);
  void* sws = W.take<char>(sws_b);
  RunBuffers R = carve_runs(W, n, true);
  int cbits = bits_for(n_cols), rbits = bits_for(n_rows);
  // values travel through the sort only when they are needed: binarised output is all ones and unit input values
  // sum to the run length (exact in fp32: the sequential sum of ones equals the count up to 2^24)
  const bool carry = val != nullptr && !binarize;
  k_pack_coo<<<grid_for(nnz_in), 256, 0, s>>>(nnz_in, n_rows, n_cols, row, col, val, symmetrize, cbits,
                                              keys, carry ? payload : nullptr, status_dev);
  GDR_LAUNCHED();
  uint64_t* skeys = keys;
  uint32_t* spay = carry ? payload : nullptr;
  int rc = sort_pairs_ex(n, rbits + cbits, keys, spay, sws, sws_b, &skeys, carry ? &spay : nullptr, s);
  if (rc) return rc;
  if (binarize) {
    // keys only, all values 1: count heads per tile, scan, emit CSR — two passes over the sorted keys
    const int64_t tiles = cdiv(n, UQ_TILE);
    int32_t* tile_cnt = R.pos;            // run scratch reused: [tiles + 1] ints, scan workspace behind it
    k_unique_count<<<(unsigned)tiles, UQ_THREADS, 0, s>>>(n, skeys, tile_cnt);
    GDR_LAUNCHED();
    rc = exclusive_scan_i32(tile_cnt, tile_cnt, tiles, R.scan_ws, R.scan_ws_b, s);
    if (rc) return rc;
    k_unique_emit_csr<<<(unsigned)tiles, UQ_THREADS, 0, s>>>(n, n_rows, cbits, skeys, tile_cnt, rowptr, colidx, vals,
                                                            nnz_out_dev, nullptr);
    GDR_LAUNCHED();
    return GDR_OK;
  }
  rc = reduce_runs(n, skeys, spay, R, s);
  if (rc) return rc;
  k_emit_csr_entries<<<grid_for(n), 256, 0, s>>>(R.pos + n, R.ukeys, carry ? R.run_sum : nullptr, R.run_len,
                                                 (1ull << cbits) - 1, binarize, colidx, vals);
  GDR_LAUNCHED();
  k_rowptr_from_ukeys<<<grid_for(n + 1), 256, 0, s>>>(R.pos + n, n_rows, cbits, ~0ull, R.ukeys, rowptr,
                                                      nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- transpose ----------------
int64_t gdr_csr_transpose_ws_bytes(int64_t n_rows, int64_t n_cols, int64_t nnz) {
  (void)n_rows;
  (void)n_cols;
  if (nnz <= 0) return 256;
  return ws_need(nnz, 8) + ws_need(nnz, 4) + sort_pairs_ws_bytes(nnz) + 256;
}

int gdr_csr_transpose(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* rowptr,
                      const int32_t* colidx, int32_t* t_rowptr, int32_t* t_colidx, int32_t* t_perm,
                      void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows >= 0 && n_cols >= 0 && nnz >= 0 && rowptr && t_rowptr, "csr_transpose: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  if (nnz == 0) {
    GDR_CUDA(cudaMemsetAsync(t_rowptr, 0, (n_cols + 1) * 4, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(colidx && t_colidx && t_perm, "csr_transpose: null pointer");
  if (ws_bytes < gdr_csr_transpose_ws_bytes(n_rows, n_cols, nnz)) {
    set_error("csr_transpose: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(nnz);
  uint32_t* payload = W.take<uint32_t>(nnz);
  int64_t sws_b = sort_pairs_ws_bytes(nnz);
  void* sws = W.take<char>(sws_b);
  int rbits = bits_for(n_rows), cbits = bits_for(n_cols);
  k_pack_transpose<<<grid_for(n_rows * 32), 256, 0, s>>>(n_rows, rowptr, colidx, rbits, keys, payload);
  GDR_LAUNCHED();
  // rows are already ascending inside equal columns only after a sort on the column
  // bits; the sort is stable and the input is row-major, so sorting the column bits suffices.
  int rc = sort_pairs(nnz, rbits + cbits, keys, payload, sws, sws_b, s);
  if (rc) return rc;
  k_unpack_transpose<<<grid_for(nnz + 1), 256, 0, s>>>(nnz, n_cols, rbits, keys, payload, t_rowptr,
                                                       t_colidx, t_perm);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- symmetric normalisation ----------------
int64_t gdr_sym_normalize_ws_bytes(int64_t n, int64_t nnz) {
  (void)nnz;
  return ws_need(n + 1, 4) + ws_need(n, 8) + 256 + scan_ws_bytes(n) + 256;
}

int gdr_sym_normalize(int64_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                      const float* vals, int self_loop_mode, int32_t* rowptr_out,
                      int32_t* colidx_out, float* vals_out, double* deg_out, int64_t* nnz_out_dev,
                      void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && nnz >= 0, "sym_normalize: bad sizes");
  GDR_CHECK_ARG(rowptr && rowptr_out && colidx_out && vals_out && nnz_out_dev, "sym_normalize: null pointer");
  GDR_CHECK_ARG(nnz == 0 || (colidx && vals), "sym_normalize: null input");
  GDR_CHECK_ARG(self_loop_mode >= 0 && self_loop_mode <= 2, "sym_normalize: self_loop_mode");
  if (nnz + n >= (1ll << 31)) {
    set_error("sym_normalize: nnz + n exceeds the int32 CSR limit");
    return GDR_ERANGE;
  }
  if (ws_bytes < gdr_sym_normalize_ws_bytes(n, nnz)) {
    set_error("sym_normalize: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  Workspace W(ws, ws_bytes);
  int32_t* out_len = W.take<int32_t>(n + 1);
  double* deg_ws = W.take<double>(n);
  int32_t* flag = W.take<int32_t>(1);
  int64_t sws_b = scan_ws_bytes(n);
  void* sws = W.take<char>(sws_b);
  double* deg = deg_out ? deg_out : deg_ws;
  k_selfloop_flag<<<1, 32, 0, s>>>(nnz, rowptr, colidx, vals, self_loop_mode, flag);
  GDR_LAUNCHED();
  unsigned grid = (unsigned)cdiv(n * 32, 256);
  k_row_degree<<<grid, 256, 0, s>>>(n, rowptr, colidx, vals, flag, deg, out_len, 0);
  GDR_LAUNCHED();
  int rc = exclusive_scan_i32(out_len, rowptr_out, n, sws, sws_b, s);
  if (rc) return rc;
  k_norm_fill<<<grid, 256, 0, s>>>(n, rowptr, colidx, vals, flag, deg, deg, rowptr_out, colidx_out, vals_out,
                                   nnz_out_dev, 0);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---- row-block form for the row-partitioned build (SURVEY §8e stage 1): the caller owns rows
//      [row_offset, row_offset + n_local) with GLOBAL column ids.  Phase 1 gives the block's degrees and the
//      output row pointer; the caller all-gathers the degrees; phase 2 fills the normalised block.  The values
//      are the ones gdr_sym_normalize produces for the same rows of the whole matrix (same kernels). ----
__global__ void k_set_flag(int32_t* flag, int v) { flag[0] = v; }

int64_t gdr_sym_normalize_block_ws_bytes(int64_t n_local) {
  return ws_need(n_local + 1, 4) + 256 + scan_ws_bytes(n_local) + 256;
}

int gdr_sym_normalize_block_degrees(int64_t n_local, int64_t row_offset, const int32_t* rowptr,
                                    const int32_t* colidx, const float* vals, int add_identity,
                                    double* deg_local_out, int32_t* rowptr_out, void* ws, int64_t ws_bytes,
                                    gdr_stream_t stream) {
  GDR_CHECK_ARG(n_local > 0 && row_offset >= 0 && rowptr && deg_local_out && rowptr_out && ws,
                "sym_normalize_block_degrees: bad arguments");
  if (ws_bytes < gdr_sym_normalize_block_ws_bytes(n_local)) {
    set_error("sym_normalize_block_degrees: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  Workspace W(ws, ws_bytes);
  int32_t* out_len = W.take<int32_t>(n_local + 1);
  int32_t* flag = W.take<int32_t>(1);
  int64_t sws_b = scan_ws_bytes(n_local);
  void* sws = W.take<char>(sws_b);
  k_set_flag<<<1, 1, 0, s>>>(flag, add_identity ? 1 : 0);
  GDR_LAUNCHED();
  k_row_degree<<<(unsigned)cdiv(n_local * 32, 256), 256, 0, s>>>(n_local, rowptr, colidx, vals, flag, deg_local_out,
                                                                out_len, row_offset);
  GDR_LAUNCHED();
  return exclusive_scan_i32(out_len, rowptr_out, n_local, sws, sws_b, s);
}

int gdr_sym_normalize_block_fill(int64_t n_local, int64_t row_offset, const int32_t* rowptr, const int32_t* colidx,
                                 const float* vals, int add_identity, const double* deg_global,
                                 const int32_t* rowptr_out, int32_t* colidx_out, float* vals_out,
                                 int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_local > 0 && row_offset >= 0 && rowptr && deg_global && rowptr_out && colidx_out && vals_out &&
                    nnz_out_dev && ws,
                "sym_normalize_block_fill: bad arguments");
  if (ws_bytes < 256) {
    set_error("sym_normalize_block_fill: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  int32_t* flag = (int32_t*)ws;
  k_set_flag<<<1, 1, 0, s>>>(flag, add_identity ? 1 : 0);
  GDR_LAUNCHED();
  k_norm_fill<<<(unsigned)cdiv(n_local * 32, 256), 256, 0, s>>>(n_local, rowptr, colidx, vals, flag,
                                                               deg_global + row_offset, deg_global, rowptr_out,
                                                               colidx_out, vals_out, nnz_out_dev, row_offset);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_sym_normalize_dense_ws_bytes(int64_t n) { return ws_need(n, 4) + 256; }

int gdr_sym_normalize_dense(int64_t n, const float* A, int64_t lda, float* out, int64_t ldo, void* ws,
                            int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && A && out && lda >= n && ldo >= n, "sym_normalize_dense: bad arguments");
  if (ws_bytes < gdr_sym_normalize_dense_ws_bytes(n)) {
    set_error("sym_normalize_dense: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  float* rinv = (float*)ws;
  k_dense_rowsum<<<(unsigned)cdiv(n * 32, 256), 256, 0, s>>>(n, A, lda, rinv);
  GDR_LAUNCHED();
  k_dense_scale<<<grid_for(n * n), 256, 0, s>>>(n, A, lda, rinv, out, ldo);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- bipartite normalisation ----------------
int gdr_bipartite_normalize(int64_t n_u, int64_t n_i, int64_t nnz, const int32_t* rowptr,
                            const int32_t* colidx, const float* w, const int32_t* t_rowptr,
                            const int32_t* t_perm, float eps, float* norm_out, float* t_norm_out,
                            float* deg_u, float* deg_i, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_u > 0 && n_i > 0 && nnz >= 0 && rowptr && t_rowptr && deg_u && deg_i,
                "bipartite_normalize: bad arguments");
  GDR_CHECK_ARG(nnz == 0 || (colidx && w && t_perm && norm_out), "bipartite_normalize: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  k_rowsum_seq<<<grid_for(n_u), 256, 0, s>>>(n_u, rowptr, nullptr, w, deg_u);
  GDR_LAUNCHED();
  k_rowsum_seq<<<grid_for(n_i), 256, 0, s>>>(n_i, t_rowptr, t_perm, w, deg_i);
  GDR_LAUNCHED();
  if (nnz == 0) return GDR_OK;
  k_bip_norm<<<(unsigned)cdiv(n_u * 32, 256), 256, 0, s>>>(n_u, rowptr, colidx, w, deg_u, deg_i, eps,
                                                          norm_out);
  GDR_LAUNCHED();
  if (t_norm_out) {
    k_gather_f32<<<grid_for(nnz), 256, 0, s>>>(nnz, t_perm, norm_out, t_norm_out);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

// Rankformer GCN edge weights (Rankformer/code/rec.py:118-124): degrees = row / column sums of the
// interaction counts clamped to >= 1;  out = w / du^a / di^b  and, for the transposed matrix,
// t_out = w / du^b / di^a  (written in transposed order through t_perm).
// LightGCN edge norm of a ROW BLOCK of the weight matrix (or of its transpose): norm = w / (sqrt(d_row + eps) *
// sqrt(d_col + eps)) with the block's own row degrees and the all-gathered degrees of the other side
// (distill_recsys.py:329-335 on a row partition; same arithmetic as gdr_bipartite_normalize)
int gdr_bipartite_norm_block(int64_t n_rows, int64_t nnz, const int32_t* rowptr, const int32_t* colidx, const float* w,
                             const float* deg_rows, const float* deg_cols, float eps, float* norm_out,
                             gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows >= 0 && nnz >= 0, "bipartite_norm_block: negative size");
  if (n_rows == 0 || nnz == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && colidx && w && deg_rows && deg_cols && norm_out, "bipartite_norm_block: null pointer");
  k_bip_norm<<<(unsigned)cdiv(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(n_rows, rowptr, colidx, w, deg_rows,
                                                                               deg_cols, eps, norm_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_bipartite_pow_normalize(int64_t n_u, int64_t n_i, int64_t nnz, const int32_t* rowptr,
                                const int32_t* colidx, const float* w, const int32_t* t_rowptr,
                                const int32_t* t_perm, float a, float b, float* out, float* t_out,
                                float* deg_u, float* deg_i, float* scratch /*nnz floats*/, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_u > 0 && n_i > 0 && nnz >= 0 && rowptr && t_rowptr && deg_u && deg_i,
                "bipartite_pow_normalize: bad arguments");
  GDR_CHECK_ARG(nnz == 0 || (colidx && w && t_perm && out && t_out && scratch), "bipartite_pow_normalize: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  k_rowsum_seq<<<grid_for(n_u), 256, 0, s>>>(n_u, rowptr, nullptr, w, deg_u);
  GDR_LAUNCHED();
  k_rowsum_seq<<<grid_for(n_i), 256, 0, s>>>(n_i, t_rowptr, t_perm, w, deg_i);
  GDR_LAUNCHED();
  if (nnz == 0) return GDR_OK;
  unsigned grid = (unsigned)cdiv(n_u * 32, 256);
  k_bip_pow_norm<<<grid, 256, 0, s>>>(n_u, rowptr, colidx, w, deg_u, deg_i, a, b, out);
  GDR_LAUNCHED();
  k_bip_pow_norm<<<grid, 256, 0, s>>>(n_u, rowptr, colidx, w, deg_u, deg_i, b, a, scratch);
  GDR_LAUNCHED();
  k_gather_f32<<<grid_for(nnz), 256, 0, s>>>(nnz, t_perm, scratch, t_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- coarsening ----------------
int64_t gdr_coarsen_ws_bytes(int64_t E, int64_t n_src, int64_t n_dst) {
  (void)n_src;
  (void)n_dst;
  if (E <= 0) return 256;
  return ws_need(E, 8) + ws_need(E, 4) + sort_pairs_ws_bytes(E) + runs_ws_bytes(E, true) + 512;
}

int gdr_coarsen(int64_t E, const int64_t* src, const int64_t* dst, int64_t n_rows,
                const int32_t* csr_rowptr, const int32_t* csr_colidx, const float* w,
                const int32_t* labels_src, const int32_t* labels_dst, int64_t n_src, int64_t n_dst,
                int drop_diag, int32_t* rowptr, int32_t* colidx, int32_t* counts, float* wsum,
                int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(E >= 0 && n_src > 0 && n_dst > 0 && rowptr && nnz_out_dev, "coarsen: bad arguments");
  GDR_CHECK_ARG(n_src < (1ll << 31) && n_dst < (1ll << 31) && E < (1ll << 31), "coarsen: size exceeds int32");
  cudaStream_t s = (cudaStream_t)stream;
  if (E == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr, 0, (n_src + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(labels_src && labels_dst && colidx && counts, "coarsen: null pointer");
  GDR_CHECK_ARG((src && dst) || (csr_rowptr && csr_colidx && n_rows > 0), "coarsen: need COO or CSR edges");
  GDR_CHECK_ARG(!wsum || w, "coarsen: wsum requested without weights");
  if (ws_bytes < gdr_coarsen_ws_bytes(E, n_src, n_dst)) {
    set_error("coarsen: workspace too small");
    return GDR_EWORKSPACE;
  }
  if (!src && cd_applicable(E, n_rows, n_src, n_dst, wsum != nullptr, ws_bytes))
    return coarsen_dense(E, n_rows, csr_rowptr, csr_colidx, w, labels_src, labels_dst, n_src, n_dst, drop_diag,
                         rowptr, colidx, counts, wsum, nnz_out_dev, ws, ws_bytes, s);
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(E);
  uint32_t* payload = W.take<uint32_t>(E);
  int64_t sws_b = sort_pairs_ws_bytes(E);
  void* sws = W.take<char>(sws_b);
  RunBuffers R = carve_runs(W, E, true);
  int abits = bits_for(n_src), bbits = bits_for(n_dst);
  uint64_t sentinel = 1ull << (abits + bbits);
  uint32_t* pl = wsum ? payload : nullptr;
  if (src) {
    k_pack_coarsen_coo<<<grid_for(E), 256, 0, s>>>(E, src, dst, w, labels_src, labels_dst, bbits,
                                                   drop_diag, sentinel, keys, pl);
  } else {
    k_pack_coarsen_csr<<<grid_for(n_rows * 32), 256, 0, s>>>(n_rows, csr_rowptr, csr_colidx, w,
                                                             labels_src, labels_dst, bbits, drop_diag,
                                                             sentinel, keys, pl);
  }
  GDR_LAUNCHED();
  int rc = sort_pairs(E, abits + bbits + (drop_diag ? 1 : 0), keys, pl, sws, sws_b, s);
  if (rc) return rc;
  rc = reduce_runs(E, keys, pl, R, s);
  if (rc) return rc;
  k_emit_coarse<<<grid_for(E), 256, 0, s>>>(R.pos + E, R.ukeys, R.run_len, R.run_sum,
                                            (1ull << bbits) - 1, sentinel, colidx, counts, wsum);
  GDR_LAUNCHED();
  k_rowptr_from_ukeys<<<grid_for(E + 1), 256, 0, s>>>(R.pos + E, n_src, bbits, sentinel, R.ukeys, rowptr,
                                                      nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_coarsen_scale(int64_t n_src, const int32_t* rowptr, const int32_t* colidx, const float* wsum,
                      const int32_t* size_src, const int32_t* size_dst, float* vals_out,
                      gdr_stream_t stream) {
  GDR_CHECK_ARG(n_src > 0 && rowptr && colidx && wsum && size_src && size_dst && vals_out,
                "coarsen_scale: bad arguments");
  k_coarsen_scale<<<(unsigned)cdiv(n_src * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      n_src, rowptr, colidx, wsum, size_src, size_dst, vals_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_csr_to_coo(int64_t n_rows, const int32_t* rowptr, const int32_t* colidx, int64_t* row_out,
                   int64_t* col_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows >= 0, "csr_to_coo: negative size");
  if (n_rows == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && colidx && row_out, "csr_to_coo: null pointer");
  k_csr_to_coo<<<grid_for(n_rows * 32), 256, 0, (cudaStream_t)stream>>>(n_rows, rowptr, colidx, row_out,
                                                                       col_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- routing form of the multi-GPU stage 1 ----------------
int64_t gdr_edges_route_ws_bytes(int64_t E, int symmetrize) {
  const int64_t n = E * (symmetrize ? 2 : 1);
  if (n <= 0) return 256;
  return ws_need(n, 8) + sort_pairs_ws_bytes(n) + 512;
}

int gdr_edges_route(int64_t E, const int64_t* row, const int64_t* col, int64_t n_rows, int64_t n_cols, int symmetrize,
                    int64_t rows_per, int world, uint64_t* keys_out, int64_t* owner_starts_dev, int32_t* status_dev, void* ws,
                    int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(E >= 0 && n_rows > 0 && n_cols > 0 && rows_per > 0 && world >= 1 && world < ROUTE_DROP && owner_starts_dev &&
                    status_dev,
                "edges_route: bad arguments");
  GDR_CHECK_ARG(!symmetrize || n_rows == n_cols, "edges_route: symmetrize needs a square matrix");
  const int64_t n = E * (symmetrize ? 2 : 1);
  GDR_CHECK_ARG(n < (1ll << 31) && bits_for(n_rows) + bits_for(n_cols) <= ROUTE_SHIFT, "edges_route: size out of range");
  cudaStream_t s = (cudaStream_t)stream;
  GDR_CUDA(cudaMemsetAsync(status_dev, 0, 4, s));
  if (n == 0) {
    GDR_CUDA(cudaMemsetAsync(owner_starts_dev, 0, 129 * 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(row && col && keys_out, "edges_route: null pointer");
  if (ws_bytes < gdr_edges_route_ws_bytes(E, symmetrize)) {
    set_error("edges_route: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(n);
  const int64_t sws_b = sort_pairs_ws_bytes(n);
  void* sws = W.take<char>(sws_b);
  k_pack_edge_route<<<grid_for(E), 256, 0, s>>>(E, n_rows, n_cols, row, col, symmetrize, bits_for(n_cols), rows_per, world, keys,
                                                status_dev);
  GDR_LAUNCHED();
  uint64_t* ks = nullptr;
  return sort_pairs_digit(n, ROUTE_SHIFT, 7, keys, nullptr, sws, sws_b, &ks, nullptr, owner_starts_dev, s, keys_out, nullptr);
}

int64_t gdr_csr_from_keys_ws_bytes(int64_t m) {
  m = m > 0 ? m : 1;
  return ws_need(m, 8) + sort_pairs_ws_bytes(m) + runs_ws_bytes(m, false) + 512;
}

// keys received from every rank -> CSR of the local rows [row_lo, row_lo + n_rows_local), columns global.
// binarize = 1: all values 1 (utils_graphsaint.py:20-22); 0: value = number of equal pairs (distill_recsys.py:110-117).
int gdr_csr_from_keys(int64_t m, const uint64_t* keys_in, int64_t row_lo, int64_t n_rows_local, int64_t n_cols, int binarize,
                      int32_t* rowptr, int32_t* colidx, float* vals, int64_t* nnz_out_dev, void* ws, int64_t ws_bytes,
                      gdr_stream_t stream) {
  GDR_CHECK_ARG(m >= 0 && row_lo >= 0 && n_rows_local >= 0 && n_cols > 0 && rowptr && nnz_out_dev, "csr_from_keys: bad arguments");
  GDR_CHECK_ARG(m < (1ll << 31), "csr_from_keys: size exceeds int32");
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0 || n_rows_local == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr, 0, (n_rows_local + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(keys_in && colidx && vals, "csr_from_keys: null pointer");
  if (ws_bytes < gdr_csr_from_keys_ws_bytes(m)) {
    set_error("csr_from_keys: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(m);
  const int64_t sws_b = sort_pairs_ws_bytes(m);
  void* sws = W.take<char>(sws_b);
  RunBuffers R = carve_runs(W, m, false);
  const int cbits = bits_for(n_cols), rbits = bits_for(n_rows_local);
  k_localise_keys<<<grid_for(m), 256, 0, s>>>(m, keys_in, (1ull << ROUTE_SHIFT) - 1ull, (uint64_t)row_lo << cbits, keys);
  GDR_LAUNCHED();
  uint64_t* skeys = keys;
  int rc = sort_pairs_ex(m, rbits + cbits, keys, nullptr, sws, sws_b, &skeys, nullptr, s);
  if (rc) return rc;
  const int64_t tiles = cdiv(m, UQ_TILE);
  int32_t* tile_cnt = R.pos;
  k_unique_count<<<(unsigned)tiles, UQ_THREADS, 0, s>>>(m, skeys, tile_cnt);
  GDR_LAUNCHED();
  rc = exclusive_scan_i32(tile_cnt, tile_cnt, tiles, R.scan_ws, R.scan_ws_b, s);
  if (rc) return rc;
  k_unique_emit_csr<<<(unsigned)tiles, UQ_THREADS, 0, s>>>(m, n_rows_local, cbits, skeys, tile_cnt, rowptr, colidx, vals,
                                                          nnz_out_dev, binarize ? nullptr : R.head_index);
  GDR_LAUNCHED();
  if (!binarize) {
    k_run_length_vals<<<grid_for(m), 256, 0, s>>>(nnz_out_dev, R.head_index, vals);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

// ---------------- routing form of the multi-GPU stage 4 ----------------
int64_t gdr_coarsen_route_ws_bytes(int64_t E) {
  if (E <= 0) return 256;
  return ws_need(E, 8) + ws_need(E, 4) + sort_pairs_ws_bytes(E) + 512;
}

int gdr_coarsen_route(int64_t E, const int64_t* src, const int64_t* dst, int64_t n_rows, const int32_t* csr_rowptr,
                      const int32_t* csr_colidx, const float* w, const int32_t* labels_src, const int32_t* labels_dst,
                      int64_t n_src, int64_t n_dst, int drop_diag, int world, uint64_t* keys_out, float* w_out,
                      int64_t* owner_starts_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(E >= 0 && n_src > 0 && n_dst > 0 && world >= 1 && world < ROUTE_DROP && owner_starts_dev,
                "coarsen_route: bad arguments");
  GDR_CHECK_ARG(E < (1ll << 31) && bits_for(n_src) + bits_for(n_dst) <= ROUTE_SHIFT, "coarsen_route: size out of range");
  cudaStream_t s = (cudaStream_t)stream;
  if (E == 0) {
    GDR_CUDA(cudaMemsetAsync(owner_starts_dev, 0, 129 * 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(labels_src && labels_dst && keys_out && (!w || w_out), "coarsen_route: null pointer");
  GDR_CHECK_ARG((src && dst) || (csr_rowptr && csr_colidx && n_rows > 0), "coarsen_route: need COO or CSR edges");
  if (ws_bytes < gdr_coarsen_route_ws_bytes(E)) {
    set_error("coarsen_route: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(E);
  uint32_t* payload = W.take<uint32_t>(E);
  const int64_t sws_b = sort_pairs_ws_bytes(E);
  void* sws = W.take<char>(sws_b);
  const int bbits = bits_for(n_dst);
  const int cr = (int)cdiv(n_src, world);
  uint32_t* pl = w ? payload : nullptr;
  if (src)
    k_pack_route_coo<<<grid_for(E), 256, 0, s>>>(E, src, dst, w, labels_src, labels_dst, bbits, drop_diag, cr, world, keys, pl);
  else
    k_pack_route_csr<<<grid_for(n_rows * 32), 256, 0, s>>>(n_rows, csr_rowptr, csr_colidx, w, labels_src, labels_dst, bbits,
                                                           drop_diag, cr, world, keys, pl);
  GDR_LAUNCHED();
  uint64_t* ks = nullptr;
  uint32_t* vs = nullptr;
  return sort_pairs_digit(E, ROUTE_SHIFT, 7, keys, pl, sws, sws_b, &ks, pl ? &vs : nullptr, owner_starts_dev, s, keys_out,
                          (uint32_t*)w_out);
}

int64_t gdr_coarse_merge_edges_ws_bytes(int64_t m) {
  m = m > 0 ? m : 1;
  return ws_need(m, 8) + ws_need(m, 4) + sort_pairs_ws_bytes(m) + runs_ws_bytes(m, true) + 512;
}

int gdr_coarse_merge_edges(int64_t m, const uint64_t* keys_in, const float* w_in, int64_t a_lo, int64_t n_rows, int64_t n_src,
                           int64_t n_dst, int32_t* rowptr, int32_t* colidx, int32_t* counts, float* wsum,
                           int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(m >= 0 && n_rows >= 0 && n_src > 0 && n_dst > 0 && a_lo >= 0 && rowptr && nnz_out_dev,
                "coarse_merge_edges: bad arguments");
  GDR_CHECK_ARG(m < (1ll << 31), "coarse_merge_edges: size exceeds int32");
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr, 0, (n_rows + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(keys_in && colidx && counts && (!wsum || w_in), "coarse_merge_edges: null pointer");
  if (ws_bytes < gdr_coarse_merge_edges_ws_bytes(m)) {
    set_error("coarse_merge_edges: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(m);
  uint32_t* payload = W.take<uint32_t>(m);
  const int64_t sws_b = sort_pairs_ws_bytes(m);
  void* sws = W.take<char>(sws_b);
  RunBuffers R = carve_runs(W, m, true);
  const int abits = bits_for(n_src), bbits = bits_for(n_dst);
  k_mask_keys<<<grid_for(m), 256, 0, s>>>(m, keys_in, (1ull << ROUTE_SHIFT) - 1ull, keys);
  GDR_LAUNCHED();
  uint32_t* pl = wsum ? payload : nullptr;
  if (pl) GDR_CUDA(cudaMemcpyAsync(payload, w_in, m * 4, cudaMemcpyDeviceToDevice, s));
  uint64_t* skeys = keys;
  uint32_t* spay = pl;
  int rc = sort_pairs_ex(m, abits + bbits, keys, pl, sws, sws_b, &skeys, pl ? &spay : nullptr, s);
  if (rc) return rc;
  rc = reduce_runs(m, skeys, spay, R, s);
  if (rc) return rc;
  k_emit_coarse<<<grid_for(m), 256, 0, s>>>(R.pos + m, R.ukeys, R.run_len, pl ? R.run_sum : nullptr, (1ull << bbits) - 1, ~0ull,
                                            colidx, counts, wsum);
  GDR_LAUNCHED();
  k_rowptr_from_ukeys_range<<<grid_for(m + 1), 256, 0, s>>>(R.pos + m, a_lo, n_rows, bbits, R.ukeys, rowptr, nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- owner-side merge of routed edges in shared memory (multi-GPU stage 4) ----------------
// per-cluster (edges, max |w|, nodes) of this rank's rows: summed / maxed over the ranks they fix the fixed-point step
int gdr_cluster_stats(int64_t n_rows, const int32_t* rowptr, const float* w, const int32_t* labels, int64_t n_src,
                      int32_t* nodes_out, int32_t* edges_out, uint32_t* wmax_bits_out, int32_t* status_dev, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows >= 0 && n_src > 0 && nodes_out && edges_out && wmax_bits_out && status_dev, "cluster_stats: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  GDR_CUDA(cudaMemsetAsync(nodes_out, 0, n_src * 4, s));
  GDR_CUDA(cudaMemsetAsync(edges_out, 0, n_src * 4, s));
  GDR_CUDA(cudaMemsetAsync(wmax_bits_out, 0, n_src * 4, s));
  GDR_CUDA(cudaMemsetAsync(status_dev, 0, 4, s));
  if (n_rows == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && labels, "cluster_stats: null pointer");
  k_cd_stats<<<(unsigned)cdiv(n_rows * 32, 256), 256, 0, s>>>(n_rows, rowptr, w, labels, n_src, nodes_out, edges_out, wmax_bits_out,
                                                            status_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_coarse_merge_edges_dense_ws_bytes(int64_t m, int64_t n_rows) {
  m = m > 0 ? m : 1;
  return ws_need(m, 8) + ws_need(m, 4) + sort_pairs_ws_bytes(m) + 3 * ws_need(m, 4) + 3 * ws_need(n_rows + 1, 4) +
         scan_ws_bytes(n_rows + 1) + 1024;
}

// 1 when gdr_coarse_merge_edges_dense applies to this shape (the coarse row fits in shared memory), else 0
int gdr_coarse_merge_edges_dense_ok(int64_t n_rows, int64_t n_dst, int has_weights) {
  return (g_coarsen_dense && n_rows > 0 && n_rows < (1ll << 24) && n_dst * (has_weights ? 12 : 4) <= 200 * 1024) ? 1 : 0;
}

int gdr_coarse_merge_edges_dense(int64_t m, const uint64_t* keys_in, const float* w_in, int64_t a_lo, int64_t n_rows, int64_t n_src,
                                 int64_t n_dst, const int32_t* cluster_edges, const uint32_t* cluster_wmax_bits, int32_t* rowptr,
                                 int32_t* colidx, int32_t* counts, float* wsum, int64_t* nnz_out_dev, void* ws, int64_t ws_bytes,
                                 gdr_stream_t stream) {
  GDR_CHECK_ARG(m >= 0 && n_rows >= 0 && n_src > 0 && n_dst > 0 && a_lo >= 0 && a_lo + n_rows <= n_src && rowptr && nnz_out_dev,
                "coarse_merge_edges_dense: bad arguments");
  GDR_CHECK_ARG(m < (1ll << 31), "coarse_merge_edges_dense: size exceeds int32");
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0 || n_rows == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr, 0, (n_rows + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(keys_in && colidx && counts && (!wsum || (w_in && cluster_edges && cluster_wmax_bits)),
                "coarse_merge_edges_dense: null pointer");
  if (!gdr_coarse_merge_edges_dense_ok(n_rows, n_dst, wsum != nullptr)) {
    set_error("coarse_merge_edges_dense: a coarse row of %lld cells does not fit in shared memory", (long long)n_dst);
    return GDR_EUNSUPPORTED;
  }
  if (ws_bytes < gdr_coarse_merge_edges_dense_ws_bytes(m, n_rows)) {
    set_error("coarse_merge_edges_dense: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(m);
  uint32_t* payload = W.take<uint32_t>(m);
  const int64_t sws_b = sort_pairs_ws_bytes(m);
  void* sws = W.take<char>(sws_b);
  int32_t* t_col = W.take<int32_t>(m);
  int32_t* t_cnt = W.take<int32_t>(m);
  float* t_sum = W.take<float>(m);
  int32_t* starts = W.take<int32_t>(n_rows + 1);
  int32_t* nnz_row = W.take<int32_t>(n_rows + 1);
  int32_t* misc = W.take<int32_t>(64);
  const int64_t scan_b = scan_ws_bytes(n_rows + 1);
  void* scan_ws = W.take<char>(scan_b);
  const int bbits = bits_for(n_dst), la = std::max(7, bits_for(n_rows));      // >= 7: the sort leaves the bits above alone
  k_cd_swap_keys<<<grid_for(m), 256, 0, s>>>(m, keys_in, bbits, la, a_lo, keys);
  GDR_LAUNCHED();
  uint32_t* pl = wsum ? payload : nullptr;
  if (pl) GDR_CUDA(cudaMemcpyAsync(payload, w_in, m * 4, cudaMemcpyDeviceToDevice, s));
  uint64_t* skeys = keys;
  uint32_t* spay = pl;
  int rc = sort_pairs_ex(m, la, keys, pl, sws, sws_b, &skeys, pl ? &spay : nullptr, s);      // stable: groups by coarse row
  if (rc) return rc;
  k_cd_pair_starts<<<(unsigned)cdiv(n_rows + 1, 256), 256, 0, s>>>(m, skeys, la, n_rows, starts);
  GDR_LAUNCHED();
  GDR_CUDA(cudaMemsetAsync(misc, 0, 256, s));
  int dev = 0, sms = kSMs;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const size_t smem = (size_t)n_dst * (wsum ? 12 : 4);
  const unsigned grid = (unsigned)std::min<int64_t>(n_rows, sms);
  CdPairs pr{skeys, reinterpret_cast<const float*>(spay), la, a_lo, cluster_edges, cluster_wmax_bits};
  if (wsum) {
    static PerDevice<bool> attr;
    if (!attr.get()) {
      GDR_CUDA(cudaFuncSetAttribute(k_cd_accumulate<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr.get() = true;
    }
    k_cd_accumulate<true, true><<<grid, CD_THREADS, smem, s>>>(n_rows, n_dst, nullptr, nullptr, nullptr, nullptr, starts, nullptr, starts,
                                                              nullptr, 0, misc, t_col, t_cnt, t_sum, nnz_row, misc + 1, pr);
  } else {
    static PerDevice<bool> attr;
    if (!attr.get()) {
      GDR_CUDA(cudaFuncSetAttribute(k_cd_accumulate<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr.get() = true;
    }
    k_cd_accumulate<false, true><<<grid, CD_THREADS, smem, s>>>(n_rows, n_dst, nullptr, nullptr, nullptr, nullptr, starts, nullptr,
                                                               starts, nullptr, 0, misc, t_col, t_cnt, nullptr, nnz_row, misc + 1, pr);
  }
  GDR_LAUNCHED();
  if ((rc = exclusive_scan_i32(nnz_row, rowptr, n_rows, scan_ws, scan_b, s))) return rc;
  k_cd_pack<<<(unsigned)std::min<int64_t>(n_rows, 8 * sms), 256, 0, s>>>(n_rows, starts, rowptr, t_col, t_cnt, t_sum, colidx, counts, wsum,
                                                                        nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- key-range merge of per-rank coarsened graphs (multi-GPU stage 4) ----------------
int gdr_coarse_records(int64_t n_src, int64_t n_dst, const int32_t* rowptr, const int32_t* colidx, const int32_t* counts,
                       const float* wsum, uint64_t* records_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_src > 0 && n_dst > 0 && rowptr && colidx && counts && records_out, "coarse_records: bad arguments");
  k_coarse_records<<<grid_for(n_src * 32), 256, 0, (cudaStream_t)stream>>>(n_src, rowptr, colidx, counts, wsum,
                                                                          bits_for(n_dst), records_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_coarse_merge_ws_bytes(int64_t m) {
  m = m > 0 ? m : 1;
  return ws_need(m, 8) + ws_need(m, 4) + sort_pairs_ws_bytes(m) + runs_ws_bytes(m, false) + 512;
}

int gdr_coarse_merge(int64_t m, const uint64_t* records, int64_t a_lo, int64_t n_rows, int64_t n_src, int64_t n_dst,
                     int32_t* rowptr, int32_t* colidx, int32_t* counts, float* wsum, int64_t* nnz_out_dev, void* ws,
                     int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(m >= 0 && n_rows >= 0 && n_src > 0 && n_dst > 0 && a_lo >= 0 && rowptr && nnz_out_dev,
                "coarse_merge: bad arguments");
  GDR_CHECK_ARG(m < (1ll << 31), "coarse_merge: size exceeds int32");
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr, 0, (n_rows + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(records && colidx && counts, "coarse_merge: null pointer");
  if (ws_bytes < gdr_coarse_merge_ws_bytes(m)) {
    set_error("coarse_merge: workspace too small");
    return GDR_EWORKSPACE;
  }
  Workspace W(ws, ws_bytes);
  uint64_t* keys = W.take<uint64_t>(m);
  uint32_t* perm = W.take<uint32_t>(m);
  const int64_t sws_b = sort_pairs_ws_bytes(m);
  void* sws = W.take<char>(sws_b);
  RunBuffers R = carve_runs(W, m, false);
  k_split_records<<<grid_for(m), 256, 0, s>>>(m, records, keys, perm);
  GDR_LAUNCHED();
  const int abits = bits_for(n_src), bbits = bits_for(n_dst);
  int rc = sort_pairs(m, abits + bbits, keys, perm, sws, sws_b, s);   // stable: equal cells keep the exchange order
  if (rc) return rc;
  rc = reduce_runs(m, keys, nullptr, R, s);
  if (rc) return rc;
  k_merge_runs<<<grid_for(m), 256, 0, s>>>(R.pos + m, R.head_index, R.ukeys, perm, records, (1ull << bbits) - 1, colidx,
                                           counts, wsum);
  GDR_LAUNCHED();
  k_rowptr_from_ukeys_range<<<grid_for(m + 1), 256, 0, s>>>(R.pos + m, a_lo, n_rows, bbits, R.ukeys, rowptr, nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

// ---------------- dense merge of per-rank coarsened graphs (multi-GPU stage 4) ----------------
int gdr_coarse_scatter_dense(int64_t n_src, int64_t n_dst, const int32_t* rowptr, const int32_t* colidx,
                             const int32_t* counts, const float* wsum, int32_t* dense_counts,
                             float* dense_wsum, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_src > 0 && n_dst > 0 && rowptr && dense_counts, "coarse_scatter_dense: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  GDR_CUDA(cudaMemsetAsync(dense_counts, 0, n_src * n_dst * 4, s));
  if (dense_wsum) GDR_CUDA(cudaMemsetAsync(dense_wsum, 0, n_src * n_dst * 4, s));
  k_scatter_dense<<<grid_for(n_src * 32), 256, 0, s>>>(n_src, n_dst, rowptr, colidx, counts, wsum, dense_counts,
                                                       dense_wsum);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_dense_to_coarse_ws_bytes(int64_t n_src) { return ws_need(n_src + 1, 4) + scan_ws_bytes(n_src) + 256; }

int gdr_dense_to_coarse(int64_t n_src, int64_t n_dst, const int32_t* dense_counts, const float* dense_wsum,
                        int32_t* rowptr, int32_t* colidx, int32_t* counts, float* wsum, int64_t* nnz_out_dev,
                        void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_src > 0 && n_dst > 0 && dense_counts && rowptr && colidx && counts && nnz_out_dev,
                "dense_to_coarse: bad arguments");
  if (ws_bytes < gdr_dense_to_coarse_ws_bytes(n_src)) {
    set_error("dense_to_coarse: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  Workspace W(ws, ws_bytes);
  int32_t* row_len = W.take<int32_t>(n_src + 1);
  void* sws = W.take<char>(scan_ws_bytes(n_src));
  unsigned grid = (unsigned)cdiv(n_src * 32, 256);
  k_dense_row_nnz<<<grid, 256, 0, s>>>(n_src, n_dst, dense_counts, row_len);
  GDR_LAUNCHED();
  int rc = exclusive_scan_i32(row_len, rowptr, n_src, sws, scan_ws_bytes(n_src), s);
  if (rc) return rc;
  k_dense_compact<<<grid, 256, 0, s>>>(n_src, n_dst, dense_counts, dense_wsum, rowptr, colidx, counts, wsum,
                                       nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

}  // extern "C"
