// spmm.cu — stage 2: one propagation hop  Y = (alpha*A) @ X ; T += beta*Y  as a
// CSR SpMM for sm_100a.
//
// Replaces the reference expression `alpha*adj_norm @ prop_feat` + the axpy on
// the next line (clustgdd_agent_transduct.py:64-65, clustgdd_agent_induct.py
// :77-94) which the reference runs as ATen mul(sparse,scalar) + coalesce +
// cuSPARSE/MKL SpMM, and the index_add_ message passing of
// distill_recsys.py:340-345.
//
// Mapping (HBM / L2-gather bound, no tensor cores):
//   * a CTA owns a block of SPMM_ROWS_PER_CTA consecutive rows; their rowptr
//     slice is staged in shared memory once, and the CTA's warps pull rows from
//     it through a shared counter (dynamic balance inside the block);
//   * a row is processed by a group of LPR lanes (8/16/32, chosen from the
//     column window) so a gathered X row is one fully coalesced run of 128-bit
//     loads;
//   * the row's (colidx, val) pairs are read coalesced, LPR at a time, and
//     broadcast with warp shuffles; UNROLL gathers are in flight per lane
//     before the first FMA consumes one (MLP); accumulation order stays CSR
//     order, one fp32 chain per output element => deterministic;
//   * streamed operands (colidx, vals, T, Y) use no-allocate / streaming cache
//     hints so that they do not evict the gathered X rows from L1/L2;
//   * wide feature matrices can be processed in column windows (col_split) so
//     that the window of X stays L2-resident across the whole pass.
#include "common.cuh"
#include "comm.cuh"
#include <stdlib.h>
#include <string.h>

namespace gdr {

constexpr int SPMM_THREADS = 256;
constexpr int SPMM_ROWS_PER_CTA = 64;     // row blocks without a plan
constexpr int SPMM_MAX_ROWS = 128;        // rows per block with an nnz-balanced plan
constexpr int SPMM_BLOCK_WEIGHT = 2048;   // plan: weight(row) = nnz(row) + SPMM_ROW_COST, blocks of equal weight
constexpr int SPMM_ROW_COST = 16;         // => at most SPMM_BLOCK_WEIGHT / SPMM_ROW_COST = 128 rows per block
constexpr int SPMM_HEAVY_NNZ = 1024;   // rows longer than this are processed by the whole CTA

// run-time tuning (gdr_debug_set): 0 = automatic choice
static int g_spmm_unroll = 0;     // 4 or 8
static int g_spmm_hints = -1;     // 0 off, 1 streaming hints on colidx/vals/T/Y
static int g_spmm_split = 0;      // number of column windows (1, 2, 4)
extern int g_lloyd_graph;         // lloyd.cu
extern int g_kpp_skip_score;      // kmeans_init.cu
extern int g_tc_screen;           // kmeans_tc.cu
extern int g_tc_gate;             // kmeans_tc.cu
extern int g_tc_cand;             // kmeans_tc.cu
extern int g_tc_cand_cap;         // kmeans_tc.cu
extern int g_coarsen_dense;       // graph.cu
extern int g_rs_match;            // primitives.cu
extern int g_rs_max_bits;         // primitives.cu
extern int g_tc_ablate;
extern int g_topk_path;           // topk.cu
extern int g_topk_condensed_path; // topk_condensed.cu
}  // namespace gdr
extern "C" int g_sparsify_batch_cap;   // sparsify.cu
namespace gdr {

__device__ __forceinline__ int ld_stream_i32(const int32_t* p) {
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f32(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_cs_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.cs.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_cs_f4(float* p, const float4& v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Multicast epilogue (multi-GPU hop fused with its all-gather): besides Y, every output row is stored into the gathered
// operand of the NEXT hop on every rank — dst[p] are peer-mapped (NVLink) pointers to rank p's copy of that matrix, row
// `row_off + r`, leading dimension `ld`.  n == 0: plain single-device epilogue.
struct SpmmPeers {
  float* dst[GDR_MAX_RANKS];
  int n;
  int64_t row_off;
  int64_t ld;
};

template <int LPR, int NCH, int UNROLL, bool HINTS>
__device__ __forceinline__ void spmm_row(const int32_t* __restrict__ colidx,
                                         const float* __restrict__ vals, float alpha,
                                         const float* __restrict__ X, int64_t ldx, int start, int end,
                                         int c4_end, int gl /*lane in group*/, unsigned gmask,
                                         int col4_base, float4 (&acc)[NCH]) {
#pragma unroll
  for (int c = 0; c < NCH; ++c) acc[c] = make_float4(0.f, 0.f, 0.f, 0.f);
  // start/end are uniform inside a lane group; groups of one warp may diverge (the
  // shuffles below name only the group's own lanes in gmask).
  for (int k = start; k < end; k += LPR) {
    int my = k + gl;
    int c_l = 0;
    float v_l = 0.f;
    if (my < end) {
      c_l = HINTS ? ld_stream_i32(colidx + my) : __ldg(colidx + my);
      v_l = vals ? __fmul_rn(HINTS ? ld_stream_f32(vals + my) : __ldg(vals + my), alpha) : alpha;
    }
    int cnt = min(LPR, end - k);
#pragma unroll 1
    for (int j = 0; j < cnt; j += UNROLL) {
      int cj[UNROLL];
      float vj[UNROLL];
      float4 xv[UNROLL][NCH];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        cj[u] = __shfl_sync(gmask, c_l, (j + u) & (LPR - 1), LPR);
        vj[u] = __shfl_sync(gmask, v_l, (j + u) & (LPR - 1), LPR);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        if (j + u < cnt) {
          const float* xr = X + (int64_t)cj[u] * ldx;
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            int c4 = col4_base + c * LPR + gl;
            if (c4 < c4_end) xv[u][c] = ldg_f4(xr + 4 * c4);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        if (j + u < cnt) {
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            int c4 = col4_base + c * LPR + gl;
            if (c4 < c4_end) {
              acc[c].x = fmaf(vj[u], xv[u][c].x, acc[c].x);
              acc[c].y = fmaf(vj[u], xv[u][c].y, acc[c].y);
              acc[c].z = fmaf(vj[u], xv[u][c].z, acc[c].z);
              acc[c].w = fmaf(vj[u], xv[u][c].w, acc[c].w);
            }
          }
        }
      }
    }
  }
}

template <int LPR, int NCH, int UNROLL, bool HINTS, bool MC>
__global__ void __launch_bounds__(SPMM_THREADS, MC ? (NCH == 1 ? 4 : 1) : ((NCH == 1 && UNROLL <= 2) ? 8 : ((NCH == 1 && UNROLL <= 4) ? 6 : 1)))
k_spmm(int64_t rows, int c4_end, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
       const float* __restrict__ vals, float alpha, const float* __restrict__ X, int64_t ldx,
       float* __restrict__ Y, int64_t ldy, float* __restrict__ T, int64_t ldt, float beta,
       int col4_base, const int32_t* __restrict__ bounds, const SpmmPeers mc) {
  __shared__ int s_rowptr[SPMM_MAX_ROWS + 1];
  __shared__ int s_heavy[SPMM_MAX_ROWS];
  __shared__ int s_next, s_nheavy;
  constexpr int GROUPS = 32 / LPR;  // rows processed concurrently by one warp
  // row block of this CTA: from the nnz-balanced plan when there is one, else 64 consecutive rows
  const int64_t row0 = bounds ? (int64_t)bounds[blockIdx.x] : (int64_t)blockIdx.x * SPMM_ROWS_PER_CTA;
  const int nrows = bounds ? (bounds[blockIdx.x + 1] - (int)row0)
                           : (int)min((int64_t)SPMM_ROWS_PER_CTA, rows - row0);
  if (nrows <= 0) return;
  for (int i = threadIdx.x; i <= nrows; i += SPMM_THREADS) s_rowptr[i] = rowptr[row0 + i];
  if (threadIdx.x == 0) {
    s_next = 0;
    s_nheavy = 0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int g = lane / LPR, gl = lane % LPR;
  const unsigned gmask = LPR == 32 ? 0xffffffffu : (((1u << LPR) - 1u) << (g * LPR));

  // epilogue of one float4 column chunk: Y = acc ; T += beta * acc (two roundings, as the reference)
  auto store = [&](int64_t row, int c4, const float4& a) {
    if (Y) {
      float* yp = Y + row * ldy + 4 * c4;
      if (HINTS) st_cs_f4(yp, a);
      else *reinterpret_cast<float4*>(yp) = a;
    }
    if (MC) {
      for (int p = 0; p < mc.n; ++p)   // posted NVLink stores: the row lands in every rank's gathered operand
        *reinterpret_cast<float4*>(mc.dst[p] + (mc.row_off + row) * mc.ld + 4 * c4) = a;
    }
    if (T) {
      float* tp = T + row * ldt + 4 * c4;
      float4 t = HINTS ? ld_cs_f4(tp) : *reinterpret_cast<float4*>(tp);
      t.x = __fadd_rn(t.x, __fmul_rn(beta, a.x));
      t.y = __fadd_rn(t.y, __fmul_rn(beta, a.y));
      t.z = __fadd_rn(t.z, __fmul_rn(beta, a.z));
      t.w = __fadd_rn(t.w, __fmul_rn(beta, a.w));
      if (HINTS) st_cs_f4(tp, t);
      else *reinterpret_cast<float4*>(tp) = t;
    }
  };

  // ---- phase 1: light rows, one lane group per row; heavy rows are deferred ----
  while (true) {
    int r_base = 0;
    if (lane == 0) r_base = atomicAdd(&s_next, GROUPS);
    r_base = __shfl_sync(0xffffffffu, r_base, 0);
    if (r_base >= nrows) break;
    int r = r_base + g;
    int start = 0, end = 0;
    bool live = r < nrows;
    if (live) {
      start = s_rowptr[r];
      end = s_rowptr[r + 1];
      if (end - start > SPMM_HEAVY_NNZ) {
        if (gl == 0) s_heavy[atomicAdd(&s_nheavy, 1)] = r;
        live = false;
        start = end = 0;
      }
    }
    float4 acc[NCH];
    spmm_row<LPR, NCH, UNROLL, HINTS>(colidx, vals, alpha, X, ldx, start, end, c4_end, gl, gmask, col4_base, acc);
    if (live) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        int c4 = col4_base + c * LPR + gl;
        if (c4 < c4_end) store(row0 + r, c4, acc[c]);
      }
    }
  }
  __syncthreads();

  // ---- phase 2: each heavy (hub) row is split over all lane groups of the CTA; the
  //      partial sums are combined in fixed chunk order (deterministic) ----
  const int nheavy = s_nheavy;
  if (nheavy == 0) return;
  constexpr int NPART = (SPMM_THREADS / 32) * GROUPS;
  __shared__ float4 s_part[NPART][NCH * LPR];
  const int part = (threadIdx.x >> 5) * GROUPS + g;
  for (int h = 0; h < nheavy; ++h) {
    const int r = s_heavy[h];
    const int hs = s_rowptr[r], he = s_rowptr[r + 1];
    int chunk = (he - hs + NPART - 1) / NPART;
    chunk = (chunk + LPR - 1) / LPR * LPR;
    const int cs = min(he, hs + part * chunk), ce = min(he, cs + chunk);
    float4 acc[NCH];
    spmm_row<LPR, NCH, UNROLL, HINTS>(colidx, vals, alpha, X, ldx, cs, ce, c4_end, gl, gmask, col4_base, acc);
#pragma unroll
    for (int c = 0; c < NCH; ++c) s_part[part][c * LPR + gl] = acc[c];
    __syncthreads();
    for (int t = threadIdx.x; t < NCH * LPR; t += SPMM_THREADS) {
      const int c4 = col4_base + t;
      if (c4 < c4_end) {
        float4 s = s_part[0][t];
#pragma unroll 4
        for (int p = 1; p < NPART; ++p) {
          const float4 q = s_part[p][t];
          s.x = __fadd_rn(s.x, q.x);
          s.y = __fadd_rn(s.y, q.y);
          s.z = __fadd_rn(s.z, q.z);
          s.w = __fadd_rn(s.w, q.w);
        }
        store(row0 + r, c4, s);
      }
    }
    __syncthreads();
  }
}

struct SpmmArgs {
  int64_t rows;
  const int32_t *rowptr, *colidx;
  const float* vals;
  float alpha;
  const float* X;
  int64_t ldx;
  float* Y;
  int64_t ldy;
  float* T;
  int64_t ldt;
  float beta;
  cudaStream_t s;
  const int32_t* bounds;   // nnz-balanced row-block plan (nullable)
  int64_t n_blocks;
  SpmmPeers mc;
};

template <int LPR, int NCH, int UNROLL, bool HINTS>
static int launch_spmm(const SpmmArgs& a, int col4_base, int c4_end) {
  unsigned grid = a.bounds ? (unsigned)a.n_blocks : (unsigned)cdiv(a.rows, SPMM_ROWS_PER_CTA);
  {
    ProfileScope prof(PROF_SPMM, a.s);
    if constexpr (!HINTS && UNROLL == (NCH >= 8 ? 1 : (NCH >= 4 ? 2 : 4))) {
      if (a.mc.n > 0) {   // multi-GPU hop fused with its all-gather (built for the default tuning of every width)
        k_spmm<LPR, NCH, UNROLL, HINTS, true><<<grid, SPMM_THREADS, 0, a.s>>>(a.rows, c4_end, a.rowptr, a.colidx, a.vals,
                                                                              a.alpha, a.X, a.ldx, a.Y, a.ldy, a.T, a.ldt,
                                                                              a.beta, col4_base, a.bounds, a.mc);
        GDR_LAUNCHED();
        return GDR_OK;
      }
    }
    if (a.mc.n > 0) {
      set_error("spmm: the fused all-gather epilogue is built for the default tuning only (spmm_unroll / spmm_hints unset)");
      return GDR_EUNSUPPORTED;
    }
    k_spmm<LPR, NCH, UNROLL, HINTS, false><<<grid, SPMM_THREADS, 0, a.s>>>(a.rows, c4_end, a.rowptr, a.colidx, a.vals, a.alpha,
                                                                           a.X, a.ldx, a.Y, a.ldy, a.T, a.ldt, a.beta,
                                                                           col4_base, a.bounds, a.mc);
  }
  GDR_LAUNCHED();
  return GDR_OK;
}

template <int LPR, int NCH>
static int dispatch_tuning(const SpmmArgs& a, int base, int c4_end, int unroll, bool hints) {
  if constexpr (NCH == 1) {
    if (unroll == 2)
      return hints ? launch_spmm<LPR, NCH, 2, true>(a, base, c4_end) : launch_spmm<LPR, NCH, 2, false>(a, base, c4_end);
  }
  if constexpr (NCH <= 2) {
    if (unroll >= 8)
      return hints ? launch_spmm<LPR, NCH, 8, true>(a, base, c4_end) : launch_spmm<LPR, NCH, 8, false>(a, base, c4_end);
  }
  constexpr int U = NCH >= 8 ? 1 : (NCH >= 4 ? 2 : 4);
  return hints ? launch_spmm<LPR, NCH, U, true>(a, base, c4_end) : launch_spmm<LPR, NCH, U, false>(a, base, c4_end);
}

// one column window [base, base + width) in float4 units
static int spmm_window(const SpmmArgs& a, int base, int width, int unroll, bool hints) {
  const int c4_end = base + width;
  if (width <= 8) return dispatch_tuning<8, 1>(a, base, c4_end, unroll, hints);
  if (width <= 16) return dispatch_tuning<16, 1>(a, base, c4_end, unroll, hints);
  if (width <= 32) return dispatch_tuning<32, 1>(a, base, c4_end, unroll, hints);
  if (width <= 64) return dispatch_tuning<32, 2>(a, base, c4_end, unroll, hints);
  if (width <= 128) return dispatch_tuning<32, 4>(a, base, c4_end, unroll, hints);
  for (int b = base; b < c4_end; b += 256) {
    int rc = dispatch_tuning<32, 8>(a, b, std::min(c4_end, b + 256), unroll, hints);
    if (rc) return rc;
  }
  return GDR_OK;
}

// bounds[c] = first row r with rowptr[r] + SPMM_ROW_COST * r >= c * SPMM_BLOCK_WEIGHT
__global__ void k_spmm_plan(int64_t n_rows, const int32_t* __restrict__ rowptr, int64_t n_blocks,
                            int32_t* __restrict__ bounds) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c > n_blocks) return;
  if (c == n_blocks) {
    bounds[c] = (int32_t)n_rows;
    return;
  }
  const int64_t target = c * SPMM_BLOCK_WEIGHT;
  int64_t lo = 0, hi = n_rows;   // answer in [0, n_rows]
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if ((int64_t)rowptr[mid] + SPMM_ROW_COST * mid >= target) hi = mid;
    else lo = mid + 1;
  }
  bounds[c] = (int32_t)lo;
}

int spmm_launch_planned(int64_t rows, int64_t F, const int32_t* rowptr, const int32_t* colidx,
                        const float* vals, float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy,
                        float* T, int64_t ldt, float beta, const int32_t* bounds, int64_t n_blocks, cudaStream_t s);
int spmm_launch_mc(int64_t rows, int64_t F, const int32_t* rowptr, const int32_t* colidx, const float* vals, float alpha,
                   const float* X, int64_t ldx, float* Y, int64_t ldy, float* T, int64_t ldt, float beta,
                   const int32_t* bounds, int64_t n_blocks, const SpmmPeers& mc, cudaStream_t s);

int spmm_launch(int64_t rows, int64_t F, const int32_t* rowptr, const int32_t* colidx,
                const float* vals, float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy,
                float* T, int64_t ldt, float beta, cudaStream_t s) {
  return spmm_launch_planned(rows, F, rowptr, colidx, vals, alpha, X, ldx, Y, ldy, T, ldt, beta, nullptr, 0, s);
}

int spmm_launch_planned(int64_t rows, int64_t F, const int32_t* rowptr, const int32_t* colidx,
                        const float* vals, float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy,
                        float* T, int64_t ldt, float beta, const int32_t* bounds, int64_t n_blocks, cudaStream_t s) {
  SpmmPeers none;
  none.n = 0;
  none.row_off = 0;
  none.ld = 0;
  return spmm_launch_mc(rows, F, rowptr, colidx, vals, alpha, X, ldx, Y, ldy, T, ldt, beta, bounds, n_blocks, none, s);
}

int spmm_launch_mc(int64_t rows, int64_t F, const int32_t* rowptr, const int32_t* colidx, const float* vals, float alpha,
                   const float* X, int64_t ldx, float* Y, int64_t ldy, float* T, int64_t ldt, float beta,
                   const int32_t* bounds, int64_t n_blocks, const SpmmPeers& mc, cudaStream_t s) {
  if (rows == 0 || F == 0) return GDR_OK;
  const int F4 = (int)cdiv(F, 4);
  SpmmArgs a{rows, rowptr, colidx, vals, alpha, X, ldx, Y, ldy, T, ldt, beta, s, bounds, n_blocks, mc};
  const int unroll = g_spmm_unroll > 0 ? g_spmm_unroll : 4;
  const bool hints = g_spmm_hints >= 0 ? g_spmm_hints != 0 : false;
  int split = g_spmm_split > 0 ? g_spmm_split : 1;
  if (split > 1 && F4 >= 8 * split) {
    const int w = (int)cdiv(F4, split);
    for (int b = 0; b < F4; b += w) {
      int rc = spmm_window(a, b, std::min(w, F4 - b), unroll, hints);
      if (rc) return rc;
    }
    return GDR_OK;
  }
  return spmm_window(a, 0, F4, unroll, hints);
}

__global__ void k_scale_rows(int64_t rows, int F4, float a, const float* __restrict__ X, int64_t ldx,
                             float* __restrict__ out, int64_t ldo) {
  int64_t total = rows * (int64_t)F4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / F4;
    int c4 = (int)(i - r * F4);
    float4 x = ldg_nc_f4(X + r * ldx + 4 * c4);
    x.x = __fmul_rn(a, x.x);
    x.y = __fmul_rn(a, x.y);
    x.z = __fmul_rn(a, x.z);
    x.w = __fmul_rn(a, x.w);
    *reinterpret_cast<float4*>(out + r * ldo + 4 * c4) = x;
  }
}

// column ids of a row-partitioned matrix -> rows of the chunk-major gathered operand (parallel.py, row-chunk
// pipelined hop): node (rank r, local row i = c*cr + o)  ->  c*world*cr + r*cr + o
__global__ void k_remap_chunk_major(int64_t nnz, const int32_t* __restrict__ in, int rows_per, int cr, int world,
                                    int32_t* __restrict__ out) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nnz; j += (int64_t)gridDim.x * blockDim.x) {
    const int g = in[j];
    const int r = g / rows_per, i = g - r * rows_per;
    const int c = i / cr, o = i - c * cr;
    out[j] = c * (world * cr) + r * cr + o;
  }
}

}  // namespace gdr

extern "C" {

int gdr_remap_chunk_major(int64_t nnz, const int32_t* colidx_in, int64_t rows_per, int64_t chunk_rows, int64_t world,
                          int32_t* colidx_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(nnz >= 0 && rows_per > 0 && chunk_rows > 0 && world > 0, "remap_chunk_major: bad sizes");
  if (nnz == 0) return GDR_OK;
  GDR_CHECK_ARG(colidx_in && colidx_out, "remap_chunk_major: null pointer");
  GDR_CHECK_ARG(((rows_per + chunk_rows - 1) / chunk_rows) * chunk_rows * world < (1ll << 31), "remap_chunk_major: range");
  unsigned grid = (unsigned)std::min<int64_t>(gdr::cdiv(nnz, 256), gdr::kSMs * 32);
  gdr::k_remap_chunk_major<<<grid, 256, 0, (cudaStream_t)stream>>>(nnz, colidx_in, (int)rows_per, (int)chunk_rows,
                                                                  (int)world, colidx_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

// Tuning / experiment knobs (not part of the stable surface; see tools/spmm_sweep.py).
int gdr_debug_set(const char* key, int value) {
  GDR_CHECK_ARG(key, "debug_set: null key");
  if (!strcmp(key, "spmm_unroll")) gdr::g_spmm_unroll = value;
  else if (!strcmp(key, "spmm_hints")) gdr::g_spmm_hints = value;
  else if (!strcmp(key, "spmm_split")) gdr::g_spmm_split = value;
  else if (!strcmp(key, "lloyd_graph")) gdr::g_lloyd_graph = value;
  else if (!strcmp(key, "kpp_dist_skip_score")) gdr::g_kpp_skip_score = value;
  else if (!strcmp(key, "tc_screen")) gdr::g_tc_screen = value;
  else if (!strcmp(key, "topk_path")) gdr::g_topk_path = value;
  else if (!strcmp(key, "topk_condensed_path")) gdr::g_topk_condensed_path = value;
  else if (!strcmp(key, "coarsen_dense")) gdr::g_coarsen_dense = value;
  else if (!strcmp(key, "tc_ablate")) gdr::g_tc_ablate = value;
  else if (!strcmp(key, "tc_gate")) gdr::g_tc_gate = value;
  else if (!strcmp(key, "tc_cand")) gdr::g_tc_cand = value;
  else if (!strcmp(key, "tc_cand_cap")) gdr::g_tc_cand_cap = value;
  else if (!strcmp(key, "rs_match")) gdr::g_rs_match = value;
  else if (!strcmp(key, "rs_max_bits")) gdr::g_rs_max_bits = value;
  else if (!strcmp(key, "sparsify_batch")) g_sparsify_batch_cap = value;
  else {
    gdr::set_error("debug_set: unknown key %s", key);
    return GDR_EINVAL;
  }
  return GDR_OK;
}

int gdr_spmm_prop(int64_t rows_local, int64_t F, const int32_t* rowptr, const int32_t* colidx,
                  const float* vals, float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy,
                  float* T, int64_t ldt, float beta, gdr_stream_t stream) {
  GDR_CHECK_ARG(rows_local >= 0 && F >= 0, "spmm_prop: negative size");
  if (rows_local == 0 || F == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && colidx && X && Y, "spmm_prop: null pointer");
  GDR_CHECK_ARG(ldx % 4 == 0 && ldy % 4 == 0 && ldx >= gdr::align_up(F, 4) &&
                    ldy >= gdr::align_up(F, 4),
                "spmm_prop: ldx/ldy must be multiples of 4 and >= F rounded up to 4");
  GDR_CHECK_ARG(((uintptr_t)X & 15) == 0 && ((uintptr_t)Y & 15) == 0, "spmm_prop: X/Y not 16B aligned");
  if (T) {
    GDR_CHECK_ARG(ldt % 4 == 0 && ldt >= gdr::align_up(F, 4) && ((uintptr_t)T & 15) == 0,
                  "spmm_prop: T misaligned");
  }
  GDR_CHECK_ARG(X != Y, "spmm_prop: in-place propagation is not supported");
  return gdr::spmm_launch(rows_local, F, rowptr, colidx, vals, alpha, X, ldx, Y, ldy, T, ldt, beta,
                          (cudaStream_t)stream);
}

int64_t gdr_spmm_plan_blocks(int64_t n_rows, int64_t nnz) {
  if (n_rows <= 0) return 0;
  return gdr::cdiv(nnz + (int64_t)gdr::SPMM_ROW_COST * n_rows, gdr::SPMM_BLOCK_WEIGHT) + 1;
}

int gdr_spmm_plan(int64_t n_rows, int64_t nnz, const int32_t* rowptr, int32_t* bounds_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows >= 0 && nnz >= 0, "spmm_plan: negative size");
  if (n_rows == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && bounds_out, "spmm_plan: null pointer");
  const int64_t nb = gdr_spmm_plan_blocks(n_rows, nnz);
  gdr::k_spmm_plan<<<(unsigned)gdr::cdiv(nb + 1, 256), 256, 0, (cudaStream_t)stream>>>(n_rows, rowptr, nb, bounds_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_spmm_prop_planned(int64_t rows_local, int64_t F, const int32_t* rowptr, const int32_t* colidx,
                          const float* vals, float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy,
                          float* T, int64_t ldt, float beta, const int32_t* bounds, int64_t n_blocks,
                          gdr_stream_t stream) {
  GDR_CHECK_ARG(rows_local >= 0 && F >= 0, "spmm_prop: negative size");
  if (rows_local == 0 || F == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && colidx && X && Y && bounds && n_blocks > 0, "spmm_prop_planned: null pointer");
  GDR_CHECK_ARG(ldx % 4 == 0 && ldy % 4 == 0 && ldx >= gdr::align_up(F, 4) && ldy >= gdr::align_up(F, 4),
                "spmm_prop: ldx/ldy must be multiples of 4 and >= F rounded up to 4");
  GDR_CHECK_ARG(((uintptr_t)X & 15) == 0 && ((uintptr_t)Y & 15) == 0, "spmm_prop: X/Y not 16B aligned");
  if (T) {
    GDR_CHECK_ARG(ldt % 4 == 0 && ldt >= gdr::align_up(F, 4) && ((uintptr_t)T & 15) == 0, "spmm_prop: T misaligned");
  }
  GDR_CHECK_ARG(X != Y, "spmm_prop: in-place propagation is not supported");
  return gdr::spmm_launch_planned(rows_local, F, rowptr, colidx, vals, alpha, X, ldx, Y, ldy, T, ldt, beta, bounds,
                                  n_blocks, (cudaStream_t)stream);
}

// One hop of a row-partitioned propagation FUSED with the all-gather of its result: every output row is stored (posted
// NVLink stores from the SpMM epilogue) into row dst_row_offset + r of the matrix at dst_offset_bytes of EVERY rank's
// copy of the symmetric buffer, i.e. straight into the gathered operand of the next hop; no separate collective, no
// staging copy.  Y (this rank's plain copy of the block) is optional.  Follow with gdr_symm_barrier before any rank
// reads the gathered matrix.
int gdr_spmm_prop_mc(gdr_symm_t* symm, int64_t dst_offset_bytes, int64_t dst_ld, int64_t dst_row_offset,
                     int64_t rows_local, int64_t F, const int32_t* rowptr, const int32_t* colidx, const float* vals,
                     float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy, float* T, int64_t ldt, float beta,
                     const int32_t* bounds, int64_t n_blocks, gdr_stream_t stream) {
  GDR_CHECK_ARG(symm && rows_local >= 0 && F >= 0 && dst_offset_bytes >= 0 && dst_offset_bytes % 16 == 0 && dst_row_offset >= 0,
                "spmm_prop_mc: bad arguments");
  if (rows_local == 0 || F == 0) return GDR_OK;
  GDR_CHECK_ARG(rowptr && colidx && X && bounds && n_blocks > 0, "spmm_prop_mc: null pointer");
  GDR_CHECK_ARG(ldx % 4 == 0 && ldx >= gdr::align_up(F, 4) && dst_ld % 4 == 0 && dst_ld >= gdr::align_up(F, 4) &&
                    ((uintptr_t)X & 15) == 0,
                "spmm_prop_mc: leading dimensions must be multiples of 4 and >= F rounded up to 4");
  if (Y) GDR_CHECK_ARG(ldy % 4 == 0 && ldy >= gdr::align_up(F, 4) && ((uintptr_t)Y & 15) == 0, "spmm_prop_mc: Y misaligned");
  if (T) GDR_CHECK_ARG(ldt % 4 == 0 && ldt >= gdr::align_up(F, 4) && ((uintptr_t)T & 15) == 0, "spmm_prop_mc: T misaligned");
  GDR_CHECK_ARG(dst_offset_bytes + (dst_row_offset + rows_local) * dst_ld * 4 <= symm->bytes,
                "spmm_prop_mc: destination rows exceed the symmetric buffer");
  gdr::SpmmPeers mc;
  mc.n = symm->comm->world;
  mc.row_off = dst_row_offset;
  mc.ld = dst_ld;
  for (int p = 0; p < mc.n; ++p) mc.dst[p] = (float*)(symm->peer[p] + dst_offset_bytes);
  {   // the source operand must not overlap the rows this call writes into the local copy
    const char* d0 = symm->local + dst_offset_bytes + dst_row_offset * dst_ld * 4;
    const char* d1 = d0 + rows_local * dst_ld * 4;
    const char* x0 = (const char*)X;
    GDR_CHECK_ARG(!(x0 < d1 && x0 + 1 > d0), "spmm_prop_mc: in-place propagation is not supported");
  }
  return gdr::spmm_launch_mc(rows_local, F, rowptr, colidx, vals, alpha, X, ldx, Y, ldy, T, ldt, beta, bounds, n_blocks, mc,
                             (cudaStream_t)stream);
}

int gdr_scale_rows(int64_t rows, int64_t F, float a, const float* X, int64_t ldx, float* out,
                   int64_t ldo, gdr_stream_t stream) {
  GDR_CHECK_ARG(rows >= 0 && F >= 0, "scale_rows: negative size");
  if (rows == 0 || F == 0) return GDR_OK;
  GDR_CHECK_ARG(X && out && ldx % 4 == 0 && ldo % 4 == 0 && ((uintptr_t)X & 15) == 0 &&
                    ((uintptr_t)out & 15) == 0,
                "scale_rows: null or misaligned");
  int F4 = (int)gdr::cdiv(F, 4);
  int64_t total = rows * F4;
  unsigned grid = (unsigned)std::min<int64_t>(gdr::cdiv(total, 256), gdr::kSMs * 16);
  gdr::k_scale_rows<<<grid, 256, 0, (cudaStream_t)stream>>>(rows, F4, a, X, ldx, out, ldo);
  GDR_LAUNCHED();
  return GDR_OK;
}

}  // extern "C"
