// lightgcn_grad.cu — backward of the bipartite LightGCN propagation with respect to the edge weights
// (LightGCNCondensed.propagate, distill_recsys.py:319-353, whose condensed edge weights are trained in the
// refinement loop :684-733).
//
// Forward (recsys.py):  norm_e = w_e / (sqrt(du[a]+eps) sqrt(di[b]+eps)) for the CSR entry e = (a, b),
// M = [[0, A], [A^T, 0]] with A_ab = norm_e, X_l = M^l [u0; i0], out = c sum_{l<=L} X_l, c = 1/(L+1).
// With g = dL/dout and Y_m = M^m g (the adjoint is the same propagation: M is symmetric):
//   G_e = dL/dA_ab = c sum_{j<L} ( Xi_j[b] . PY_{L-1-j}[a]  +  Yi_j[b] . PX_{L-1-j}[a] ),
//   PY_k = sum_{m<=k} Yu_m,  PX_k = sum_{m<=k} Xu_m              (row-side prefix sums, built once per row)
//   S_u[a] = sum_{e in row a} G_e norm_e,  S_i[b] = sum_{e in col b} G_e norm_e                       (fp64)
//   dL/dw_e = G_e / (sqrt(du+eps) sqrt(di+eps)) - S_u[a] / (2 (du+eps)) - S_i[b] / (2 (di+eps)).
//
// k_edge_grad follows the anatomy of k_spmm: a CTA owns up to 64 consecutive rows and hands them to lane groups of LPR
// lanes through a shared counter; (colidx, norm) are read coalesced, LPR at a time, and broadcast with shuffles; a
// lane holds float4 column chunks of the row-side prefix sums in registers and gathers the 2L column-side rows of
// each edge with 128-bit loads; the per-edge dot product is reduced by a butterfly inside the group.  Rows longer
// than EG_HEAVY_NNZ are split over every group of the CTA afterwards.  Wide rows (d > 256) and deep models (L > 4)
// run as several passes over column windows / layer chunks; each pass adds its part to G in pass order.  Every sum
// has one fixed order and no float atomics are used, so results are bit-identical run to run.
#include "common.cuh"

namespace gdr {

constexpr int EG_THREADS = 256;
constexpr int EG_ROWS_PER_CTA = 64;   // at most; fewer when the matrix has few rows, so that every SM gets blocks
constexpr int EG_HEAVY_NNZ = 1024;   // rows longer than this are processed by the whole CTA
constexpr int EG_MAX_JC = 4;         // layers per pass (row-side registers: 2 * JC * NCH float4 per lane)
constexpr int EG_WIN4 = 64;          // column window of one pass, in float4 (256 columns)

struct EgArgs {
  int64_t n_u;
  const int32_t* rowptr;
  const int32_t* colidx;
  const float* norm;
  const float *Xu, *Xi, *Yu, *Yi;   // [L][n][ld]
  int64_t ld, lsu, lsi;             // leading dimension, layer strides of the user / item stacks
  int L, j0;                        // this pass covers the layer terms j0 .. j0 + JC - 1
  int d;
  float c;
  int first, last;                  // first pass writes G, later passes add to it; the last one scales and sums S_u
  float* G;
  double* S_u;
};

template <int LPR, int NCH, int JC>
struct EgRow {
  float4 py[JC][NCH];   // PY_{L-1-j}[a], j = j0 + jj
  float4 px[JC][NCH];   // PX_{L-1-j}[a]
};

__device__ __forceinline__ void add4(float4& s, const float4& v) {
  s.x = __fadd_rn(s.x, v.x);
  s.y = __fadd_rn(s.y, v.y);
  s.z = __fadd_rn(s.z, v.z);
  s.w = __fadd_rn(s.w, v.w);
}

// row-side prefix sums of row a for this pass's layer terms and column window; columns >= d are zeroed
template <int LPR, int NCH, int JC>
__device__ __forceinline__ void eg_load_row(const EgArgs& a, int64_t row, int col4_base, int c4_end, int gl,
                                            EgRow<LPR, NCH, JC>& R) {
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const int c4 = col4_base + c * LPR + gl;
    const bool in = c4 < c4_end;
    float4 sy = make_float4(0.f, 0.f, 0.f, 0.f), sx = sy;
    int m = 0;
#pragma unroll
    for (int jj = JC - 1; jj >= 0; --jj) {
      const int upto = a.L - 1 - (a.j0 + jj);   // PY / PX index of this layer term (ascending in m as jj falls)
      for (; m <= upto; ++m) {
        if (in) {
          add4(sy, ldg_f4(a.Yu + m * a.lsu + row * a.ld + 4 * c4));
          add4(sx, ldg_f4(a.Xu + m * a.lsu + row * a.ld + 4 * c4));
        }
      }
      float4 y = sy, x = sx;
      const int e0 = 4 * c4;
      if (!in || e0 + 0 >= a.d) y.x = x.x = 0.f;
      if (!in || e0 + 1 >= a.d) y.y = x.y = 0.f;
      if (!in || e0 + 2 >= a.d) y.z = x.z = 0.f;
      if (!in || e0 + 3 >= a.d) y.w = x.w = 0.f;
      R.py[jj][c] = y;
      R.px[jj][c] = x;
    }
  }
}

// G for the entries [start, end) of row `row` (this pass's part); returns the lane's fp64 share of
// sum G_e norm_e over the entries it owns (last pass only)
template <int LPR, int NCH, int JC>
__device__ __forceinline__ double eg_edges(const EgArgs& a, const EgRow<LPR, NCH, JC>& R, int start, int end,
                                           int col4_base, int c4_end, int gl, unsigned gmask) {
  double su = 0.0;
  for (int k = start; k < end; k += LPR) {
    const int my = k + gl;
    int c_l = 0;
    float n_l = 0.f;
    if (my < end) {
      c_l = __ldg(a.colidx + my);
      if (a.last) n_l = __ldg(a.norm + my);
    }
    const int cnt = min(LPR, end - k);
    float g_mine = 0.f;
#pragma unroll 1
    for (int j = 0; j < cnt; ++j) {
      const int64_t b = __shfl_sync(gmask, c_l, j, LPR);
      float4 xi[JC][NCH], yi[JC][NCH];
#pragma unroll
      for (int jj = 0; jj < JC; ++jj) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const int c4 = col4_base + c * LPR + gl;
          if (c4 < c4_end) {
            const int64_t off = (int64_t)(a.j0 + jj) * a.lsi + b * a.ld + 4 * c4;
            xi[jj][c] = ldg_f4(a.Xi + off);
            yi[jj][c] = ldg_f4(a.Yi + off);
          } else {
            xi[jj][c] = yi[jj][c] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      }
      float p = 0.f;
#pragma unroll
      for (int jj = 0; jj < JC; ++jj) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          p = fmaf(xi[jj][c].x, R.py[jj][c].x, p);
          p = fmaf(xi[jj][c].y, R.py[jj][c].y, p);
          p = fmaf(xi[jj][c].z, R.py[jj][c].z, p);
          p = fmaf(xi[jj][c].w, R.py[jj][c].w, p);
          p = fmaf(yi[jj][c].x, R.px[jj][c].x, p);
          p = fmaf(yi[jj][c].y, R.px[jj][c].y, p);
          p = fmaf(yi[jj][c].z, R.px[jj][c].z, p);
          p = fmaf(yi[jj][c].w, R.px[jj][c].w, p);
        }
      }
#pragma unroll
      for (int o = LPR / 2; o > 0; o >>= 1) p = __fadd_rn(p, __shfl_xor_sync(gmask, p, o, LPR));
      if (gl == j) g_mine = p;
    }
    if (my < end) {
      float g = a.first ? g_mine : __fadd_rn(a.G[my], g_mine);
      if (a.last) {
        g = __fmul_rn(a.c, g);
        su = fma((double)g, (double)n_l, su);
      }
      a.G[my] = g;
    }
  }
  return su;
}

template <int LPR>
__device__ __forceinline__ double group_sum_f64(double v, unsigned gmask) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o, LPR);
  return v;
}

template <int LPR, int NCH, int JC>
__global__ void __launch_bounds__(EG_THREADS) k_edge_grad(const EgArgs a, int rows_per_cta, int col4_base, int c4_end) {
  __shared__ int s_rowptr[EG_ROWS_PER_CTA + 1];
  __shared__ int s_heavy[EG_ROWS_PER_CTA];
  __shared__ int s_next, s_nheavy;
  constexpr int GROUPS = 32 / LPR;
  constexpr int NPART = (EG_THREADS / 32) * GROUPS;
  __shared__ double s_part[NPART];
  const int64_t row0 = (int64_t)blockIdx.x * rows_per_cta;
  const int nrows = (int)min((int64_t)rows_per_cta, a.n_u - row0);
  for (int i = threadIdx.x; i <= nrows; i += EG_THREADS) s_rowptr[i] = a.rowptr[row0 + i];
  if (threadIdx.x == 0) {
    s_next = 0;
    s_nheavy = 0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int g = lane / LPR, gl = lane % LPR;
  const unsigned gmask = LPR == 32 ? 0xffffffffu : (((1u << LPR) - 1u) << (g * LPR));

  // ---- phase 1: light rows, one lane group per row; heavy rows are deferred ----
  while (true) {
    int r_base = 0;
    if (lane == 0) r_base = atomicAdd(&s_next, GROUPS);
    r_base = __shfl_sync(0xffffffffu, r_base, 0);
    if (r_base >= nrows) break;
    // every lane reaches the warp-wide shuffle above on every trip: a dead or deferred row runs an empty range
    // (groups of one warp may diverge in between; their shuffles name only the group's own lanes)
    const int r = r_base + g;
    int start = 0, end = 0;
    bool live = r < nrows;
    if (live) {
      start = s_rowptr[r];
      end = s_rowptr[r + 1];
      if (end - start > EG_HEAVY_NNZ) {
        if (gl == 0) s_heavy[atomicAdd(&s_nheavy, 1)] = r;
        live = false;
        start = end = 0;
      }
    }
    EgRow<LPR, NCH, JC> R;
    if (live) eg_load_row<LPR, NCH, JC>(a, row0 + r, col4_base, c4_end, gl, R);
    double su = eg_edges<LPR, NCH, JC>(a, R, start, end, col4_base, c4_end, gl, gmask);
    su = group_sum_f64<LPR>(su, gmask);
    if (live && a.last && gl == 0) a.S_u[row0 + r] = su;
  }
  __syncthreads();

  // ---- phase 2: each heavy row is split over all lane groups of the CTA in fixed chunks; the fp64 partial sums
  //      are combined in chunk order ----
  const int nheavy = s_nheavy;
  const int part = (threadIdx.x >> 5) * GROUPS + g;
  for (int h = 0; h < nheavy; ++h) {
    const int r = s_heavy[h];
    const int hs = s_rowptr[r], he = s_rowptr[r + 1];
    int chunk = (he - hs + NPART - 1) / NPART;
    chunk = (chunk + LPR - 1) / LPR * LPR;
    const int cs = min(he, hs + part * chunk), ce = min(he, cs + chunk);
    EgRow<LPR, NCH, JC> R;
    eg_load_row<LPR, NCH, JC>(a, row0 + r, col4_base, c4_end, gl, R);
    double su = eg_edges<LPR, NCH, JC>(a, R, cs, ce, col4_base, c4_end, gl, gmask);
    su = group_sum_f64<LPR>(su, gmask);
    if (gl == 0) s_part[part] = su;
    __syncthreads();
    if (threadIdx.x == 0 && a.last) {
      double s = 0.0;
      for (int p = 0; p < NPART; ++p) s += s_part[p];
      a.S_u[row0 + r] = s;
    }
    __syncthreads();
  }
}

template <int LPR, int NCH>
static int launch_eg(const EgArgs& a, int jc, int col4_base, int c4_end, cudaStream_t s) {
  // >= 4 blocks per SM where the rows allow it (a condensed graph has a few thousand rows)
  const int rpc = (int)std::min<int64_t>(EG_ROWS_PER_CTA, std::max<int64_t>(4, cdiv(a.n_u, kSMs * 4)));
  const unsigned grid = (unsigned)cdiv(a.n_u, rpc);
  switch (jc) {
    case 1: k_edge_grad<LPR, NCH, 1><<<grid, EG_THREADS, 0, s>>>(a, rpc, col4_base, c4_end); break;
    case 2: k_edge_grad<LPR, NCH, 2><<<grid, EG_THREADS, 0, s>>>(a, rpc, col4_base, c4_end); break;
    case 3: k_edge_grad<LPR, NCH, 3><<<grid, EG_THREADS, 0, s>>>(a, rpc, col4_base, c4_end); break;
    default: k_edge_grad<LPR, NCH, 4><<<grid, EG_THREADS, 0, s>>>(a, rpc, col4_base, c4_end); break;
  }
  GDR_LAUNCHED();
  return GDR_OK;
}

static int eg_window(const EgArgs& a, int jc, int base, int width, cudaStream_t s) {
  const int c4_end = base + width;
  if (width <= 8) return launch_eg<8, 1>(a, jc, base, c4_end, s);
  if (width <= 16) return launch_eg<16, 1>(a, jc, base, c4_end, s);
  if (width <= 32) return launch_eg<32, 1>(a, jc, base, c4_end, s);
  return launch_eg<32, 2>(a, jc, base, c4_end, s);
}

// ---------------------------------------------------------------------------------------------------------------
// edge location: position of every input (row, col) pair in the CSR (binary search inside the row)
__global__ void k_csr_locate(int64_t n_rows, int64_t n_cols, const int32_t* __restrict__ rowptr,
                             const int32_t* __restrict__ colidx, int64_t E, const int64_t* __restrict__ row,
                             const int64_t* __restrict__ col, int32_t* __restrict__ pos, int32_t* __restrict__ status) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < E; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = row[k], c = col[k];
    int p = -1;
    if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) {
      atomicOr(status, 1);
    } else {
      int lo = rowptr[r], hi = rowptr[r + 1];   // first entry >= c in [lo, hi)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (colidx[mid] < c) lo = mid + 1;
        else hi = mid;
      }
      if (lo < rowptr[r + 1] && colidx[lo] == c) p = lo;
      else atomicOr(status, 2);
    }
    pos[k] = p;
  }
}

// S_i[b] = sum over the transposed row b (ascending transposed position) of G_e norm_e, e = t_perm[t]; one warp per
// column, lane-strided partial sums combined by a fixed butterfly
__global__ void __launch_bounds__(256) k_col_gnorm(int64_t n_i, const int32_t* __restrict__ t_rowptr,
                                                   const int32_t* __restrict__ t_perm, const float* __restrict__ G,
                                                   const float* __restrict__ norm, double* __restrict__ S_i) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= n_i) return;
  double s = 0.0;
  for (int t = t_rowptr[b] + lane_id(); t < t_rowptr[b + 1]; t += 32) {
    const int e = t_perm[t];
    s = fma((double)G[e], (double)norm[e], s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane_id() == 0) S_i[b] = s;
}

// dL/dw in CSR order (one warp per row), fp64 arithmetic and one rounding
__global__ void __launch_bounds__(256) k_dw_csr(int64_t n_u, const int32_t* __restrict__ rowptr,
                                                const int32_t* __restrict__ colidx, const float* __restrict__ deg_u,
                                                const float* __restrict__ deg_i, float eps, const float* __restrict__ G,
                                                const double* __restrict__ S_u, const double* __restrict__ S_i,
                                                float* __restrict__ dw_csr) {
  const int64_t a = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (a >= n_u) return;
  const float du = __fadd_rn(deg_u[a], eps);
  const double su = (double)__fsqrt_rn(du);
  const double tu = 0.5 * S_u[a] / (double)du;
  for (int e = rowptr[a] + lane_id(); e < rowptr[a + 1]; e += 32) {
    const int b = colidx[e];
    const float di = __fadd_rn(deg_i[b], eps);
    const double si = (double)__fsqrt_rn(di);
    const double v = (double)G[e] / (su * si) - tu - 0.5 * S_i[b] / (double)di;
    dw_csr[e] = (float)v;
  }
}

__global__ void k_dw_gather(int64_t E, int64_t nnz, const int32_t* __restrict__ pos, const float* __restrict__ dw_csr,
                            float* __restrict__ dw) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < E; k += (int64_t)gridDim.x * blockDim.x) {
    const int p = pos[k];
    dw[k] = (p >= 0 && p < nnz) ? dw_csr[p] : __int_as_float(0x7fc00000);
  }
}

static unsigned grid_1d(int64_t n) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(n, 256), kSMs * 16)); }

}  // namespace gdr

extern "C" {

int gdr_csr_locate(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* rowptr, const int32_t* colidx, int64_t E,
                   const int64_t* row, const int64_t* col, int32_t* edge_pos_out, int32_t* status_dev,
                   gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows >= 0 && n_cols >= 0 && nnz >= 0 && E >= 0, "csr_locate: negative size");
  GDR_CHECK_ARG(n_rows < INT32_MAX && n_cols < INT32_MAX && nnz < INT32_MAX, "csr_locate: sizes must fit int32");
  GDR_CHECK_ARG(rowptr && status_dev, "csr_locate: null pointer");
  if (E == 0) return GDR_OK;
  GDR_CHECK_ARG(row && col && edge_pos_out && (nnz == 0 || colidx), "csr_locate: null pointer");
  gdr::k_csr_locate<<<gdr::grid_1d(E), 256, 0, (cudaStream_t)stream>>>(n_rows, n_cols, rowptr, colidx, E, row, col,
                                                                      edge_pos_out, status_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_lightgcn_edge_grad(int64_t n_u, int64_t n_i, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                           const float* norm, int num_layers, int64_t d, const float* Xu, const float* Xi,
                           const float* Yu, const float* Yi, int64_t ld, float c, float* G_out, double* S_u_out,
                           gdr_stream_t stream) {
  GDR_CHECK_ARG(n_u >= 0 && n_i >= 0 && nnz >= 0 && d >= 0, "lightgcn_edge_grad: negative size");
  GDR_CHECK_ARG(num_layers >= 0, "lightgcn_edge_grad: num_layers must be >= 0");
  GDR_CHECK_ARG(n_u < INT32_MAX && n_i < INT32_MAX && nnz < INT32_MAX, "lightgcn_edge_grad: sizes must fit int32");
  if (n_u == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && S_u_out, "lightgcn_edge_grad: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  if (nnz == 0 || num_layers == 0 || d == 0) {   // no entries, or out does not depend on A: G = 0, S_u = 0
    if (nnz > 0) {
      GDR_CHECK_ARG(G_out, "lightgcn_edge_grad: null pointer");
      GDR_CUDA(cudaMemsetAsync(G_out, 0, nnz * sizeof(float), s));
    }
    GDR_CUDA(cudaMemsetAsync(S_u_out, 0, n_u * sizeof(double), s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(colidx && norm && Xu && Xi && Yu && Yi && G_out, "lightgcn_edge_grad: null pointer");
  GDR_CHECK_ARG(ld % 4 == 0 && ld >= gdr::align_up(d, 4), "lightgcn_edge_grad: ld must be a multiple of 4 and >= d");
  GDR_CHECK_ARG(((uintptr_t)Xu & 15) == 0 && ((uintptr_t)Xi & 15) == 0 && ((uintptr_t)Yu & 15) == 0 &&
                    ((uintptr_t)Yi & 15) == 0,
                "lightgcn_edge_grad: layer stacks must be 16-byte aligned");
  gdr::EgArgs a;
  a.n_u = n_u;
  a.rowptr = rowptr;
  a.colidx = colidx;
  a.norm = norm;
  a.Xu = Xu;
  a.Xi = Xi;
  a.Yu = Yu;
  a.Yi = Yi;
  a.ld = ld;
  a.lsu = n_u * ld;
  a.lsi = n_i * ld;
  a.L = num_layers;
  a.d = (int)d;
  a.c = c;
  a.G = G_out;
  a.S_u = S_u_out;
  const int F4 = (int)gdr::cdiv(d, 4);
  const int n_win = (int)gdr::cdiv(F4, gdr::EG_WIN4);
  const int n_jc = (int)gdr::cdiv(num_layers, gdr::EG_MAX_JC);
  for (int w = 0; w < n_win; ++w) {
    const int base = w * gdr::EG_WIN4, width = std::min(gdr::EG_WIN4, F4 - base);
    for (int q = 0; q < n_jc; ++q) {
      a.j0 = q * gdr::EG_MAX_JC;
      a.first = w == 0 && q == 0;
      a.last = w == n_win - 1 && q == n_jc - 1;
      int rc = gdr::eg_window(a, std::min(gdr::EG_MAX_JC, num_layers - a.j0), base, width, s);
      if (rc) return rc;
    }
  }
  return GDR_OK;
}

int64_t gdr_bipartite_normalize_backward_ws_bytes(int64_t n_i, int64_t nnz) {
  if (n_i < 0 || nnz < 0) return 256;
  return gdr::ws_need(n_i, 8) + gdr::ws_need(nnz, 4) + 256;
}

int gdr_bipartite_normalize_backward(int64_t n_u, int64_t n_i, int64_t nnz, const int32_t* rowptr,
                                     const int32_t* colidx, const int32_t* t_rowptr, const int32_t* t_perm,
                                     const float* norm, const float* deg_u, const float* deg_i, float eps,
                                     const float* G, const double* S_u, int64_t E, const int32_t* edge_pos,
                                     float* dw_out, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_u >= 0 && n_i >= 0 && nnz >= 0 && E >= 0, "bipartite_normalize_backward: negative size");
  GDR_CHECK_ARG(n_u < INT32_MAX && n_i < INT32_MAX && nnz < INT32_MAX,
                "bipartite_normalize_backward: sizes must fit int32");
  if (E == 0) return GDR_OK;
  GDR_CHECK_ARG(nnz > 0 && n_u > 0 && n_i > 0, "bipartite_normalize_backward: E > 0 edges on an empty matrix");
  GDR_CHECK_ARG(rowptr && colidx && t_rowptr && t_perm && norm && deg_u && deg_i && G && S_u && edge_pos && dw_out && ws,
                "bipartite_normalize_backward: null pointer");
  if (ws_bytes < gdr_bipartite_normalize_backward_ws_bytes(n_i, nnz)) {
    gdr::set_error("bipartite_normalize_backward: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  gdr::Workspace W(ws, ws_bytes);
  double* S_i = W.take<double>(n_i);
  float* dw_csr = W.take<float>(nnz);
  gdr::k_col_gnorm<<<(unsigned)gdr::cdiv(n_i * 32, 256), 256, 0, s>>>(n_i, t_rowptr, t_perm, G, norm, S_i);
  GDR_LAUNCHED();
  gdr::k_dw_csr<<<(unsigned)gdr::cdiv(n_u * 32, 256), 256, 0, s>>>(n_u, rowptr, colidx, deg_u, deg_i, eps, G, S_u, S_i,
                                                                   dw_csr);
  GDR_LAUNCHED();
  gdr::k_dw_gather<<<gdr::grid_1d(E), 256, 0, s>>>(E, nnz, edge_pos, dw_csr, dw_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

}  // extern "C"
