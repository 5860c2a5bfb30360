// sparsify.cu — SURVEY §8(f) item 1: edge scoring and top-k sparsification, the step between
// k-means (stage 3) and the coarsened graph (stage 4).
//
// Replaces, on a device CSR (rows = src, colidx = dst, both in the coalesced order the reference's
// `adj.coalesce()._indices()` has):
//   ER_estimator            utils_clustgdd.py:151-162   degree = adj @ 1 ; v/deg[src] + v/deg[dst]
//   attaw_ER_estimator      utils_clustgdd.py:165-184   v * cosine_similarity(ebd[src], ebd[dst]) then ER
//   ClustGDD.graph_sparse   clustgdd_agent_transduct.py:131-232   softmax class probabilities,
//                           src_prob * dst_prob * ER_low, torch.topk(int(nedges * ratio)), COO rebuild
// The reference does D2H copies and a scipy COO rebuild per class; here everything stays on the
// device: the k-th largest weight comes from a 4-pass radix select on the order-preserving integer
// image of the fp32 weights, the selection is compacted with two scans (CSR order is kept, so the
// output is a sorted CSR without any sort).  All of it is HBM-bound integer / elementwise work.
#include <vector>

#include "common.cuh"
#include "comm.cuh"

namespace gdr {

static unsigned grid_for(int64_t n, int threads = 256) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(n, threads), kSMs * 32));
}

// fp32 row sums in stored order (one thread per row: the CPU reference's sequential order)
__global__ void k_row_sums(int64_t n, const int32_t* __restrict__ rowptr, const float* __restrict__ vals,
                           float* __restrict__ deg) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j) s = __fadd_rn(s, vals[j]);
    deg[r] = s;
  }
}

// one warp per row: er[j] = v/deg[row_lo + r] + v/deg[c]  (rows of a block starting at global row row_lo; deg global)
__global__ void __launch_bounds__(256) k_er_lower(int64_t n, int64_t row_lo, const int32_t* __restrict__ rowptr,
                                                  const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                                                  const float* __restrict__ deg, float* __restrict__ er) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const float dr = deg[row_lo + r];
  for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32) {
    const float v = vals[j];
    er[j] = __fadd_rn(__fdiv_rn(v, dr), __fdiv_rn(v, deg[colidx[j]]));
  }
}

// inv[i] = 1 / max(|e_i|, eps)
__global__ void k_inv_norm(int64_t n, int C, const float* __restrict__ E, int64_t ld, float eps,
                           float* __restrict__ inv) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < C; ++k) s = fmaf(E[i * ld + k], E[i * ld + k], s);
    inv[i] = 1.f / fmaxf(sqrtf(s), eps);
  }
}

// 8 lanes per edge: out[j] = vals[j] * cos(e_{row_lo + r}, e_c)  (E and inv indexed by global row)
__global__ void __launch_bounds__(256) k_edge_cosine_scale(int64_t n, int64_t row_lo, int C, const int32_t* __restrict__ rowptr,
                                                           const int32_t* __restrict__ colidx,
                                                           const float* __restrict__ vals,
                                                           const float* __restrict__ E, int64_t ld,
                                                           const float* __restrict__ inv, float* __restrict__ out) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const int lane = lane_id(), g = lane >> 3, gl = lane & 7;
  const float* er = E + (row_lo + r) * ld;
  const float ir = inv[row_lo + r];
  const int b = rowptr[r], e = rowptr[r + 1];
  for (int j0 = b; j0 < e; j0 += 4) {
    const int j = j0 + g;
    float dot = 0.f;
    int c = 0;
    if (j < e) {
      c = colidx[j];
      const float* ec = E + (int64_t)c * ld;
      for (int k = gl; k < C; k += 8) dot = fmaf(er[k], ec[k], dot);
    }
    dot += __shfl_xor_sync(0xffffffffu, dot, 4);
    dot += __shfl_xor_sync(0xffffffffu, dot, 2);
    dot += __shfl_xor_sync(0xffffffffu, dot, 1);
    if (j < e && gl == 0) out[j] = __fmul_rn(vals[j], __fmul_rn(__fmul_rn(dot, ir), inv[c]));
  }
}

// fp32 softmax of every row (one warp per row): exp(x - max) / sum
__global__ void __launch_bounds__(256) k_softmax_rows(int64_t n, int C, const float* __restrict__ X, int64_t ld,
                                                      float* __restrict__ out, int64_t ldo) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  float m = -INFINITY;
  for (int k = lane_id(); k < C; k += 32) m = fmaxf(m, X[r * ld + k]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float s = 0.f;
  for (int k = lane_id(); k < C; k += 32) s += expf(X[r * ld + k] - m);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  for (int k = lane_id(); k < C; k += 32) out[r * ldo + k] = __fdiv_rn(expf(X[r * ld + k] - m), s);
}

// w[j] = (p[r] * p[c]) * er[j]   with p = column `cls` of the probability matrix
__global__ void __launch_bounds__(256) k_class_weight(int64_t n, const int32_t* __restrict__ rowptr,
                                                      const int32_t* __restrict__ colidx, const float* __restrict__ er,
                                                      const float* __restrict__ P, int64_t ldp, int cls,
                                                      float* __restrict__ w) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const float pr = P[r * ldp + cls];
  for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32)
    w[j] = __fmul_rn(__fmul_rn(pr, P[(int64_t)colidx[j] * ldp + cls]), er[j]);
}

// ---------------------------------------------------------------------------------
// top-k by radix select
// ---------------------------------------------------------------------------------
// order-preserving image of an fp32 value (ascending); NaN sorts above +inf like torch.topk treats it
__device__ __forceinline__ uint32_t f32_key(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

struct SelState {
  uint32_t prefix;    // bytes of the k-th largest key fixed so far (high to low)
  uint32_t mask;      // which bits of prefix are fixed
  int64_t k_rem;      // how many entries >= the final key are still to be taken among the candidates
};

__global__ void k_sel_init(SelState* st, int32_t* hist, int32_t k) {
  if (threadIdx.x == 0) {
    st->prefix = 0;
    st->mask = 0;
    st->k_rem = k;
  }
  hist[threadIdx.x] = 0;
}

__global__ void __launch_bounds__(256) k_sel_hist(int64_t n, const float* __restrict__ w, const SelState* __restrict__ st,
                                                  int shift, int32_t* __restrict__ hist) {
  __shared__ int sh[256];
  sh[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t prefix = st->prefix, mask = st->mask;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t u = f32_key(w[i]);
    if ((u & mask) == prefix) atomicAdd(&sh[(u >> shift) & 0xff], 1);
  }
  __syncthreads();
  if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

// walk the bins from the largest digit down until k_rem entries are covered; fixes one more byte
__global__ void k_sel_pick(SelState* st, int32_t* hist, int shift) {
  __shared__ int sh[256];
  sh[threadIdx.x] = hist[threadIdx.x];
  hist[threadIdx.x] = 0;   // ready for the next pass
  __syncthreads();
  if (threadIdx.x == 0) {
    int k = st->k_rem, d = 255;
    for (; d > 0; --d) {
      if (sh[d] >= k) break;
      k -= sh[d];
    }
    st->prefix |= (uint32_t)d << shift;
    st->mask |= 0xffu << shift;
    st->k_rem = k;
  }
}

__global__ void k_sel_eqflag(int64_t n, const float* __restrict__ w, const SelState* __restrict__ st,
                             int32_t* __restrict__ eq) {
  const uint32_t T = st->prefix;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    eq[i] = f32_key(w[i]) == T;
}

// sel = above the threshold, or one of the first k_rem entries equal to it (index order)
__global__ void k_sel_flag(int64_t n, const float* __restrict__ w, const SelState* __restrict__ st,
                           const int32_t* __restrict__ eqrank, int32_t* __restrict__ sel) {
  const uint32_t T = st->prefix;
  const int k_rem = st->k_rem;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t u = f32_key(w[i]);
    sel[i] = (u > T) || (u == T && eqrank[i] < k_rem);
  }
}

__global__ void k_sel_compact(int64_t n_rows, int64_t nnz, const int32_t* __restrict__ rowptr,
                              const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                              const int32_t* __restrict__ pos /*nnz + 1*/, int32_t* __restrict__ rowptr_out,
                              int32_t* __restrict__ colidx_out, float* __restrict__ vals_out,
                              int64_t* __restrict__ nnz_out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t i = t0; i < nnz; i += stride) {
    const int p = pos[i];
    if (pos[i + 1] != p) {
      colidx_out[p] = colidx[i];
      vals_out[p] = vals[i];
    }
  }
  for (int64_t r = t0; r <= n_rows; r += stride) rowptr_out[r] = pos[rowptr[r]];
  if (t0 == 0) *nnz_out = pos[nnz];
}

// ---------------------------------------------------------------------------------
// class-batched variants (blockIdx.y = class inside the batch): at arxiv size one class is ~10 MB of
// traffic per pass — a launch, not a bandwidth problem — so the per-class loop of ~20 short launches
// is replaced by ~20 launches per BATCH of classes.
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_class_weight_b(int64_t n, int64_t nnz, int64_t row_lo, const int32_t* __restrict__ rowptr,
                                                        const int32_t* __restrict__ colidx, const float* __restrict__ er,
                                                        const float* __restrict__ P, int64_t ldp, int cls0,
                                                        float* __restrict__ w /*[classes][nnz]*/) {
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const int cls = cls0 + blockIdx.y;
  float* wc = w + (int64_t)blockIdx.y * nnz;
  const float pr = P[(row_lo + r) * ldp + cls];
  for (int j = rowptr[r] + lane_id(); j < rowptr[r + 1]; j += 32)
    wc[j] = __fmul_rn(__fmul_rn(pr, P[(int64_t)colidx[j] * ldp + cls]), er[j]);
}

__global__ void k_sel_init_b(SelState* st, int32_t* hist, int64_t k) {
  if (threadIdx.x == 0) {
    st[blockIdx.x].prefix = 0;
    st[blockIdx.x].mask = 0;
    st[blockIdx.x].k_rem = k;
  }
  hist[blockIdx.x * 256 + threadIdx.x] = 0;
}

__global__ void __launch_bounds__(256) k_sel_hist_b(int64_t n, const float* __restrict__ w, const SelState* __restrict__ st,
                                                    int shift, int32_t* __restrict__ hist) {
  __shared__ int sh[256];
  sh[threadIdx.x] = 0;
  __syncthreads();
  const float* wc = w + (int64_t)blockIdx.y * n;
  const uint32_t prefix = st[blockIdx.y].prefix, mask = st[blockIdx.y].mask;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t u = f32_key(wc[i]);
    if ((u & mask) == prefix) atomicAdd(&sh[(u >> shift) & 0xff], 1);
  }
  __syncthreads();
  if (sh[threadIdx.x]) atomicAdd(&hist[blockIdx.y * 256 + threadIdx.x], sh[threadIdx.x]);
}

__global__ void k_sel_pick_b(SelState* st, int32_t* hist, int shift) {
  __shared__ int sh[256];
  sh[threadIdx.x] = hist[blockIdx.x * 256 + threadIdx.x];
  hist[blockIdx.x * 256 + threadIdx.x] = 0;
  __syncthreads();
  if (threadIdx.x == 0) {
    SelState* s = st + blockIdx.x;
    int k = s->k_rem, d = 255;
    for (; d > 0; --d) {
      if (sh[d] >= k) break;
      k -= sh[d];
    }
    s->prefix |= (uint32_t)d << shift;
    s->mask |= 0xffu << shift;
    s->k_rem = k;
  }
}

// flags of all classes into ONE array of classes * (n + 1) ints (the slot n of every class stays 0), so that a single
// exclusive scan serves every class: position inside class c = scan[c (n+1) + i] - scan[c (n+1)]
__global__ void k_sel_eqflag_b(int64_t n, const float* __restrict__ w, const SelState* __restrict__ st,
                               int32_t* __restrict__ eq) {
  const float* wc = w + (int64_t)blockIdx.y * n;
  int32_t* e = eq + (int64_t)blockIdx.y * (n + 1);
  const uint32_t T = st[blockIdx.y].prefix;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x)
    e[i] = i < n ? (int32_t)(f32_key(wc[i]) == T) : 0;
}

__global__ void k_sel_flag_b(int64_t n, const float* __restrict__ w, const SelState* __restrict__ st,
                             const int32_t* __restrict__ eqrank, int32_t* __restrict__ sel) {
  const float* wc = w + (int64_t)blockIdx.y * n;
  const int32_t* er = eqrank + (int64_t)blockIdx.y * (n + 1);
  int32_t* sl = sel + (int64_t)blockIdx.y * (n + 1);
  const uint32_t T = st[blockIdx.y].prefix;
  const int k_rem = st[blockIdx.y].k_rem;
  const int base = er[0];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x) {
    int v = 0;
    if (i < n) {
      const uint32_t u = f32_key(wc[i]);
      v = (u > T) || (u == T && er[i] - base < k_rem);
    }
    sl[i] = v;
  }
}

__global__ void k_sel_compact_b(int64_t n_rows, int64_t nnz, int64_t k, const int32_t* __restrict__ rowptr,
                                const int32_t* __restrict__ colidx, const float* __restrict__ vals,
                                const int32_t* __restrict__ pos /*[classes][nnz + 1]*/, int32_t* __restrict__ rowptr_out,
                                int32_t* __restrict__ colidx_out, float* __restrict__ vals_out,
                                int64_t* __restrict__ nnz_out) {
  const int32_t* pc = pos + (int64_t)blockIdx.y * (nnz + 1);
  const int base = pc[0];
  int32_t* rp = rowptr_out + (int64_t)blockIdx.y * (n_rows + 1);
  int32_t* co = colidx_out + (int64_t)blockIdx.y * k;
  float* vo = vals_out + (int64_t)blockIdx.y * k;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t i = t0; i < nnz; i += stride) {
    const int p = pc[i];
    if (pc[i + 1] != p) {
      co[p - base] = colidx[i];
      vo[p - base] = vals[i];
    }
  }
  for (int64_t r = t0; r <= n_rows; r += stride) rp[r] = pc[rowptr[r]] - base;
  if (t0 == 0) nnz_out[blockIdx.y] = pc[nnz] - base;
}

__global__ void k_copy_i32_to_i64(const int32_t* src, int64_t* dst) { dst[0] = src[0]; }

// ---------------------------------------------------------------------------------
// the class-batched select on a row partition (gdr_sparsify_classes_dist).  The local passes are the kernels above;
// these three carry what is global: 64-bit histogram counts, k_rem, and each rank's share of the threshold ties.
// ---------------------------------------------------------------------------------
// local int32 histograms -> int64 (the all-reduce operand); the int32 ones are cleared for the next pass
__global__ void k_seld_widen(int32_t* __restrict__ hist, int64_t* __restrict__ hl) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  hl[i] = hist[i];
  hist[i] = 0;
}

// k_sel_pick_b on the global histograms hg; after the last byte (shift 0) the local histogram's count of the threshold
// key is this rank's number of ties
__global__ void k_seld_pick(SelState* st, const int64_t* __restrict__ hg, const int64_t* __restrict__ hl, int shift,
                            int64_t* __restrict__ ties_mine) {
  __shared__ int64_t sh[256];
  sh[threadIdx.x] = hg[blockIdx.x * 256 + threadIdx.x];
  __syncthreads();
  if (threadIdx.x == 0) {
    SelState* s = st + blockIdx.x;
    int64_t k = s->k_rem;
    int d = 255;
    for (; d > 0; --d) {
      if (sh[d] >= k) break;
      k -= sh[d];
    }
    s->prefix |= (uint32_t)d << shift;
    s->mask |= 0xffu << shift;
    s->k_rem = k;
    if (shift == 0) ties_mine[blockIdx.x] = hl[blockIdx.x * 256 + d];
  }
}

// the blocks in rank order are the global stored order, so the first k_rem ties overall are rank p's first
// clamp(k_rem - sum_{q<p} ties_q, 0, ties_p); k_rem becomes that local quota, which k_sel_flag_b then applies
__global__ void k_seld_quota(SelState* st, const int64_t* __restrict__ ties /*[world][nb]*/, int nb, int rank) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nb) return;
  int64_t before = 0;
  for (int q = 0; q < rank; ++q) before += ties[(int64_t)q * nb + c];
  const int64_t left = st[c].k_rem - before;
  st[c].k_rem = left < 0 ? 0 : (left < ties[(int64_t)rank * nb + c] ? left : ties[(int64_t)rank * nb + c]);
}

// ---------------------------------------------------------------------------------
// induced subgraph  adj[np.ix_(idx, idx)]  (utils_graphsaint.py:34-36, utils.py:127-129)
// ---------------------------------------------------------------------------------
__global__ void k_sub_map(int64_t m, const int64_t* __restrict__ idx, int32_t* __restrict__ map) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
    map[idx[i]] = (int32_t)i;   // position of node idx[i] in the selection (a repeated node keeps one of its positions)
}

// one warp per selected row: how many of its entries stay (pass 0) / write them as relabelled COO (pass 1)
__global__ void __launch_bounds__(256) k_sub_rows(int64_t m, const int64_t* __restrict__ idx,
                                                  const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                                  const float* __restrict__ vals, const int32_t* __restrict__ map,
                                                  int32_t* __restrict__ cnt_or_pos, int fill, int64_t* __restrict__ out_row,
                                                  int64_t* __restrict__ out_col, float* __restrict__ out_val) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= m) return;
  const int64_t r = idx[i];
  const int b = rowptr[r], e = rowptr[r + 1];
  int base = fill ? cnt_or_pos[i] : 0, total = 0;
  for (int j0 = b; j0 < e; j0 += 32) {
    const int j = j0 + lane_id();
    const int c = j < e ? map[colidx[j]] : -1;
    const unsigned keep = __ballot_sync(0xffffffffu, c >= 0);
    if (fill && c >= 0) {
      const int o = base + total + __popc(keep & ((1u << lane_id()) - 1u));
      out_row[o] = i;
      out_col[o] = c;
      out_val[o] = vals[j];
    }
    total += __popc(keep);
  }
  if (!fill && lane_id() == 0) cnt_or_pos[i] = total;
}

}  // namespace gdr

using namespace gdr;

namespace {

struct SpdBuffers {
  float* w;          // [bmax][nnz]        class weights of the batch
  int32_t* a;        // [bmax][nnz + 1]    tie flags -> their local ranks
  int32_t* b;        // [bmax][nnz + 1]    selection flags -> output positions
  int32_t* hist;     // [bmax][256]        local pass histograms
  int64_t* hl;       // [bmax][256]        the same widened (all-reduce send buffer)
  int64_t* hg;       // [bmax][256]        global histograms
  int64_t* ties;     // [world][bmax]      ties per rank and class (all-gathered in place)
  SelState* st;      // [bmax]
  void* sws;
  int64_t sws_b, off;
};

SpdBuffers spd_carve(void* ws, int64_t nnz, int64_t bmax, int world) {
  Workspace W(ws, INT64_MAX);
  SpdBuffers B;
  B.w = W.take<float>(bmax * nnz);
  B.a = W.take<int32_t>(bmax * (nnz + 1) + 1);
  B.b = W.take<int32_t>(bmax * (nnz + 1) + 1);
  B.hist = W.take<int32_t>(bmax * 256);
  B.hl = W.take<int64_t>(bmax * 256);
  B.hg = W.take<int64_t>(bmax * 256);
  B.ties = W.take<int64_t>((int64_t)world * bmax);
  B.st = W.take<SelState>(bmax);
  B.sws_b = scan_ws_bytes(bmax * (nnz + 1));
  B.sws = W.take<char>(B.sws_b);
  B.off = W.off + 256;
  return B;
}

}  // namespace

extern "C" {

int gdr_row_sums_f32(int64_t n, const int32_t* rowptr, const float* vals, float* deg_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && rowptr && deg_out, "row_sums_f32: bad arguments");
  k_row_sums<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(n, rowptr, vals, deg_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_er_lower(int64_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx, const float* vals,
                 float* deg_scratch, float* er_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && nnz >= 0 && rowptr && deg_scratch, "er_lower: bad arguments");
  GDR_CHECK_ARG(nnz == 0 || (colidx && vals && er_out), "er_lower: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  k_row_sums<<<grid_for(n), 256, 0, s>>>(n, rowptr, vals, deg_scratch);
  GDR_LAUNCHED();
  if (nnz == 0) return GDR_OK;
  k_er_lower<<<(unsigned)cdiv(n * 32, 256), 256, 0, s>>>(n, 0, rowptr, colidx, vals, deg_scratch, er_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_er_lower_rows(int64_t n_local, int64_t nnz, int64_t row_lo, const int32_t* rowptr, const int32_t* colidx,
                      const float* vals, const float* deg, float* er_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_local > 0 && nnz >= 0 && row_lo >= 0 && rowptr && deg, "er_lower_rows: bad arguments");
  GDR_CHECK_ARG(nnz == 0 || (colidx && vals && er_out), "er_lower_rows: null pointer");
  if (nnz == 0) return GDR_OK;
  k_er_lower<<<(unsigned)cdiv(n_local * 32, 256), 256, 0, (cudaStream_t)stream>>>(n_local, row_lo, rowptr, colidx, vals,
                                                                                  deg, er_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_edge_cosine_scale_rows(int64_t n_local, int64_t nnz, int64_t C, int64_t row_lo, int64_t n_global,
                               const int32_t* rowptr, const int32_t* colidx, const float* vals, const float* ebd,
                               int64_t ld, float eps, float* inv_norm_scratch, float* vals_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_local > 0 && nnz >= 0 && C > 0 && row_lo >= 0 && row_lo + n_local <= n_global && rowptr && ebd &&
                    ld >= C && inv_norm_scratch,
                "edge_cosine_scale: bad arguments");
  GDR_CHECK_ARG(nnz == 0 || (colidx && vals && vals_out), "edge_cosine_scale: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  k_inv_norm<<<grid_for(n_global), 256, 0, s>>>(n_global, (int)C, ebd, ld, eps, inv_norm_scratch);
  GDR_LAUNCHED();
  if (nnz == 0) return GDR_OK;
  k_edge_cosine_scale<<<(unsigned)cdiv(n_local * 32, 256), 256, 0, s>>>(n_local, row_lo, (int)C, rowptr, colidx, vals,
                                                                        ebd, ld, inv_norm_scratch, vals_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_edge_cosine_scale(int64_t n, int64_t nnz, int64_t C, const int32_t* rowptr, const int32_t* colidx,
                          const float* vals, const float* ebd, int64_t ld, float eps, float* inv_norm_scratch,
                          float* vals_out, gdr_stream_t stream) {
  return gdr_edge_cosine_scale_rows(n, nnz, C, 0, n, rowptr, colidx, vals, ebd, ld, eps, inv_norm_scratch, vals_out,
                                    stream);
}

int gdr_softmax_rows(int64_t n, int64_t C, const float* X, int64_t ld, float* out, int64_t ldo, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && C > 0 && X && out && ld >= C && ldo >= C, "softmax_rows: bad arguments");
  k_softmax_rows<<<(unsigned)cdiv(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(n, (int)C, X, ld, out, ldo);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_class_edge_weight(int64_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx, const float* er,
                          const float* prob, int64_t ldp, int64_t cls, float* w_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && nnz >= 0 && rowptr && prob && cls >= 0 && cls < ldp, "class_edge_weight: bad arguments");
  if (nnz == 0) return GDR_OK;
  GDR_CHECK_ARG(colidx && er && w_out, "class_edge_weight: null pointer");
  k_class_weight<<<(unsigned)cdiv(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(n, rowptr, colidx, er, prob, ldp,
                                                                               (int)cls, w_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_topk_filter_ws_bytes(int64_t n, int64_t nnz) {
  (void)n;
  return 2 * ws_need(nnz + 1, 4) + ws_need(256, 4) + 256 + scan_ws_bytes(nnz) + 256;
}

int gdr_topk_filter_csr(int64_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx, const float* vals,
                        const float* weight, int64_t k, int32_t* rowptr_out, int32_t* colidx_out, float* vals_out,
                        int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && nnz >= 0 && k >= 0 && k <= nnz && rowptr && rowptr_out && nnz_out_dev && ws,
                "topk_filter_csr: bad arguments (0 <= k <= nnz)");
  GDR_CHECK_ARG(nnz == 0 || (colidx && vals && weight && colidx_out && vals_out), "topk_filter_csr: null pointer");
  if (nnz >= (1ll << 31) - 1) {
    set_error("topk_filter_csr: nnz exceeds the int32 CSR limit");
    return GDR_ERANGE;
  }
  if (ws_bytes < gdr_topk_filter_ws_bytes(n, nnz)) {
    set_error("topk_filter_csr: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  Workspace W(ws, ws_bytes);
  int32_t* a = W.take<int32_t>(nnz + 1);   // equal-to-threshold flags -> their ranks
  int32_t* b = W.take<int32_t>(nnz + 1);   // selection flags -> output positions
  int32_t* hist = W.take<int32_t>(256);
  SelState* st = (SelState*)W.take<char>(256);
  const int64_t sws_b = scan_ws_bytes(nnz);
  void* sws = W.take<char>(sws_b);
  if (k == 0 || nnz == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr_out, 0, (n + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  k_sel_init<<<1, 256, 0, s>>>(st, hist, (int32_t)k);
  GDR_LAUNCHED();
  for (int shift = 24; shift >= 0; shift -= 8) {
    k_sel_hist<<<grid_for(nnz), 256, 0, s>>>(nnz, weight, st, shift, hist);
    GDR_LAUNCHED();
    k_sel_pick<<<1, 256, 0, s>>>(st, hist, shift);
    GDR_LAUNCHED();
  }
  k_sel_eqflag<<<grid_for(nnz), 256, 0, s>>>(nnz, weight, st, a);
  GDR_LAUNCHED();
  int rc = exclusive_scan_i32(a, a, nnz, sws, sws_b, s);
  if (rc) return rc;
  k_sel_flag<<<grid_for(nnz), 256, 0, s>>>(nnz, weight, st, a, b);
  GDR_LAUNCHED();
  if ((rc = exclusive_scan_i32(b, b, nnz, sws, sws_b, s))) return rc;
  k_sel_compact<<<grid_for(std::max(nnz, n + 1)), 256, 0, s>>>(n, nnz, rowptr, colidx, vals, b, rowptr_out, colidx_out,
                                                              vals_out, nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

/* adj[np.ix_(idx, idx)] as relabelled COO triplets (row i of the result = node idx[i]); the caller sorts them
 * into a CSR with gdr_coo_to_csr.  map_scratch: n int32, pos_scratch: m + 1 int32.  *nnz_out_dev = entries kept;
 * capacity of the outputs: nnz of the source matrix. */
int64_t gdr_induced_subgraph_ws_bytes(int64_t n, int64_t m) {
  return ws_need(n, 4) + ws_need(m + 1, 4) + scan_ws_bytes(m) + 256;
}

int gdr_induced_subgraph_coo(int64_t n, const int32_t* rowptr, const int32_t* colidx, const float* vals, int64_t m,
                             const int64_t* idx, int64_t* out_row, int64_t* out_col, float* out_val,
                             int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && m >= 0 && rowptr && nnz_out_dev && ws, "induced_subgraph: bad arguments");
  if (ws_bytes < gdr_induced_subgraph_ws_bytes(n, m)) {
    set_error("induced_subgraph: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (m == 0) {
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(idx && colidx && vals && out_row && out_col && out_val, "induced_subgraph: null pointer");
  Workspace W(ws, ws_bytes);
  int32_t* map = W.take<int32_t>(n);
  int32_t* pos = W.take<int32_t>(m + 1);
  const int64_t sws_b = scan_ws_bytes(m);
  void* sws = W.take<char>(sws_b);
  GDR_CUDA(cudaMemsetAsync(map, 0xff, n * 4, s));   // -1
  k_sub_map<<<grid_for(m), 256, 0, s>>>(m, idx, map);
  GDR_LAUNCHED();
  const unsigned grid = (unsigned)cdiv(m * 32, 256);
  k_sub_rows<<<grid, 256, 0, s>>>(m, idx, rowptr, colidx, vals, map, pos, 0, nullptr, nullptr, nullptr);
  GDR_LAUNCHED();
  int rc = exclusive_scan_i32(pos, pos, m, sws, sws_b, s);
  if (rc) return rc;
  k_sub_rows<<<grid, 256, 0, s>>>(m, idx, rowptr, colidx, vals, map, pos, 1, out_row, out_col, out_val);
  GDR_LAUNCHED();
  k_copy_i32_to_i64<<<1, 1, 0, s>>>(pos + m, nnz_out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

/* All classes of the 'attaw' sparsifier in ONE call (clustgdd_agent_transduct.py:160-181): for class c the edge
 * weights (prob[src,c] * prob[dst,c]) * er, their top-k and the rebuilt CSR, written to slice c of the outputs
 * (rowptr_out [C][n+1], colidx_out / vals_out [C][k]).  ~20 launches per class issued back to back from here. */
// classes per batch: bounded by ~1.5 GB of scratch (3 arrays of nnz + 1 words per class) and by int32 scan totals
int g_sparsify_batch_cap = 0;   // gdr_debug_set("sparsify_batch", v): cap the classes per batch (tests)
static int64_t sparsify_batch(int64_t nnz, int64_t C) {
  if (g_sparsify_batch_cap > 0) C = std::min<int64_t>(C, g_sparsify_batch_cap);
  int64_t by_mem = std::max<int64_t>(1, (int64_t)(1500ll << 20) / (12 * (nnz + 1)));
  int64_t by_int = std::max<int64_t>(1, ((1ll << 31) - 1) / (nnz + 1));
  return std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(by_mem, by_int), std::min<int64_t>(C, 65535)));
}

int64_t gdr_sparsify_classes_ws_bytes(int64_t n, int64_t nnz, int64_t C) {
  (void)n;
  const int64_t b = sparsify_batch(nnz, C);
  return ws_need(b * nnz, 4) + 2 * ws_need(b * (nnz + 1) + 1, 4) + ws_need(b * 256, 4) + ws_need(b * 16, 1) +
         scan_ws_bytes(b * (nnz + 1)) + 256;
}

int gdr_sparsify_classes(int64_t n, int64_t nnz, int64_t C, const int32_t* rowptr, const int32_t* colidx,
                         const float* vals, const float* er, const float* prob, int64_t ldp, int64_t k,
                         int32_t* rowptr_out, int32_t* colidx_out, float* vals_out, int64_t* nnz_out_dev /*[C]*/,
                         void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && nnz >= 0 && C > 0 && C <= ldp && k >= 0 && k <= nnz && rowptr && prob && rowptr_out &&
                    nnz_out_dev && ws,
                "sparsify_classes: bad arguments");
  if (ws_bytes < gdr_sparsify_classes_ws_bytes(n, nnz, C)) {
    set_error("sparsify_classes: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (k == 0 || nnz == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr_out, 0, C * (n + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, C * 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(colidx && vals && er && colidx_out && vals_out, "sparsify_classes: null pointer");
  const int64_t bmax = sparsify_batch(nnz, C);
  Workspace W(ws, ws_bytes);
  float* w = W.take<float>(bmax * nnz);
  int32_t* a = W.take<int32_t>(bmax * (nnz + 1) + 1);
  int32_t* b = W.take<int32_t>(bmax * (nnz + 1) + 1);
  int32_t* hist = W.take<int32_t>(bmax * 256);
  SelState* st = (SelState*)W.take<char>(bmax * 16);
  const int64_t sws_b = scan_ws_bytes(bmax * (nnz + 1));
  void* sws = W.take<char>(sws_b);
  const unsigned gx = grid_for(nnz);
  for (int64_t c0 = 0; c0 < C; c0 += bmax) {
    const unsigned nb = (unsigned)std::min<int64_t>(bmax, C - c0);
    const int64_t tot = (int64_t)nb * (nnz + 1);
    k_class_weight_b<<<dim3((unsigned)cdiv(n * 32, 256), nb), 256, 0, s>>>(n, nnz, 0, rowptr, colidx, er, prob, ldp, (int)c0,
                                                                         w);
    GDR_LAUNCHED();
    k_sel_init_b<<<nb, 256, 0, s>>>(st, hist, k);
    GDR_LAUNCHED();
    for (int shift = 24; shift >= 0; shift -= 8) {
      k_sel_hist_b<<<dim3(gx, nb), 256, 0, s>>>(nnz, w, st, shift, hist);
      GDR_LAUNCHED();
      k_sel_pick_b<<<nb, 256, 0, s>>>(st, hist, shift);
      GDR_LAUNCHED();
    }
    k_sel_eqflag_b<<<dim3(gx, nb), 256, 0, s>>>(nnz, w, st, a);
    GDR_LAUNCHED();
    int rc = exclusive_scan_i32(a, a, tot, sws, sws_b, s);
    if (rc) return rc;
    k_sel_flag_b<<<dim3(gx, nb), 256, 0, s>>>(nnz, w, st, a, b);
    GDR_LAUNCHED();
    if ((rc = exclusive_scan_i32(b, b, tot, sws, sws_b, s))) return rc;
    k_sel_compact_b<<<dim3(grid_for(std::max(nnz, n + 1)), nb), 256, 0, s>>>(
        n, nnz, k, rowptr, colidx, vals, b, rowptr_out + c0 * (n + 1), colidx_out + c0 * k, vals_out + c0 * k,
        nnz_out_dev + c0);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

/* gdr_sparsify_classes on a row partition (see gdr.h).  One class batch:
 *   weights   k_class_weight_b on the local rows (global row ids for prob), or er itself without prob
 *   4 passes  k_sel_hist_b (local, int32) -> widen to int64 -> all-reduce -> k_seld_pick on every rank
 *   quota     each rank's ties of the threshold (local histogram bin) all-gathered; rank p keeps its first
 *             clamp(k_rem - sum_{q<p} ties_q, 0, ties_p)
 *   compact   k_sel_eqflag_b, scan, k_sel_flag_b, scan, k_sel_compact_b as on one GPU
 * The batch size comes from the LARGEST local nnz so that every rank issues the same collectives; the workspace of
 * gdr_sparsify_classes_dist_ws_bytes (sized with the local nnz's batch, which is never smaller) holds it. */
int64_t gdr_sparsify_classes_dist_ws_bytes(int64_t n_local, int64_t nnz_local, int64_t C, int world) {
  (void)n_local;
  return spd_carve(nullptr, nnz_local, sparsify_batch(nnz_local, C), world).off;
}

int gdr_sparsify_classes_dist(gdr_comm_t* comm, int64_t n_local, int64_t nnz, int64_t row_lo, int64_t n_global, int64_t C,
                              const int32_t* rowptr, const int32_t* colidx, const float* vals, const float* er,
                              const float* prob, int64_t ldp, int64_t k, int32_t* rowptr_out, int32_t* colidx_out,
                              float* vals_out, int64_t* nnz_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(comm, "sparsify_classes_dist: null communicator");
  const int world = comm->world, rank = comm->rank;
  cudaStream_t s = (cudaStream_t)stream;
  // local checks are decided collectively in comm_entry_check: an early return would leave the others in a collective
  int local_rc = GDR_OK;
  if (!(n_local >= 0 && nnz >= 0 && row_lo >= 0 && C > 0 && k >= 0 && (prob ? C <= ldp : C == 1) &&
        rowptr_out && nnz_out_dev && ws && (n_local == 0 || rowptr) &&
        (nnz == 0 || (n_local > 0 && colidx && vals && er && colidx_out && vals_out)))) {
    set_error("sparsify_classes_dist: bad arguments");
    local_rc = GDR_EINVAL;
  } else if (nnz >= (1ll << 31) - 1) {
    set_error("sparsify_classes_dist: local nnz exceeds the int32 CSR limit");
    local_rc = GDR_ERANGE;
  } else if (ws_bytes < gdr_sparsify_classes_dist_ws_bytes(n_local, nnz, C, world)) {
    set_error("sparsify_classes_dist: workspace too small");
    local_rc = GDR_EWORKSPACE;
  }
  std::vector<int64_t> nnz_of((size_t)world);
  int rc = comm_entry_check(comm, s, "sparsify_classes_dist", local_rc, row_lo, n_local, n_global,
                            {C, k, n_global, prob != nullptr, g_sparsify_batch_cap}, "C, k, n_global, prob or batch cap",
                            nnz, nullptr, nnz_of.data());
  if (rc != GDR_OK) return rc;
  int64_t nnz_global = 0, nnz_max = 0;
  for (int64_t m : nnz_of) {
    nnz_global += m;
    nnz_max = std::max(nnz_max, m);
  }
  GDR_CHECK_ARG(k <= nnz_global, "sparsify_classes_dist: k = %lld exceeds the %lld stored entries", (long long)k,
                (long long)nnz_global);

  if (k == 0 || nnz == 0) {
    GDR_CUDA(cudaMemsetAsync(rowptr_out, 0, C * (n_local + 1) * 4, s));
    GDR_CUDA(cudaMemsetAsync(nnz_out_dev, 0, C * 8, s));
  }
  if (k == 0) return GDR_OK;   // the same k on every rank: no rank enters a collective
  const int64_t cap = std::min(k, nnz);   // output slice per class
  const int64_t bmax = sparsify_batch(nnz_max, C);
  SpdBuffers B = spd_carve(ws, nnz, bmax, world);
  const unsigned gx = grid_for(nnz);
  for (int64_t c0 = 0; c0 < C; c0 += bmax) {
    const unsigned nb = (unsigned)std::min<int64_t>(bmax, C - c0);
    const int64_t tot = (int64_t)nb * (nnz + 1);
    int64_t* ties_mine = B.ties + (int64_t)rank * nb;
    const float* w = er;
    if (prob) {
      if (nnz > 0) {
        k_class_weight_b<<<dim3((unsigned)cdiv(n_local * 32, 256), nb), 256, 0, s>>>(n_local, nnz, row_lo, rowptr, colidx,
                                                                                   er, prob, ldp, (int)c0, B.w);
        GDR_LAUNCHED();
      }
      w = B.w;
    }
    k_sel_init_b<<<nb, 256, 0, s>>>(B.st, B.hist, k);
    GDR_LAUNCHED();
    for (int shift = 24; shift >= 0; shift -= 8) {
      if (nnz > 0) {
        k_sel_hist_b<<<dim3(gx, nb), 256, 0, s>>>(nnz, w, B.st, shift, B.hist);
        GDR_LAUNCHED();
      }
      k_seld_widen<<<nb, 256, 0, s>>>(B.hist, B.hl);
      GDR_LAUNCHED();
      if ((rc = comm_allreduce_i64(comm, B.hl, B.hg, (int64_t)nb * 256, s))) return rc;
      k_seld_pick<<<nb, 256, 0, s>>>(B.st, B.hg, B.hl, shift, ties_mine);
      GDR_LAUNCHED();
    }
    if ((rc = comm_allgather(comm, ties_mine, B.ties, (int64_t)nb * 8, s))) return rc;
    k_seld_quota<<<(unsigned)cdiv(nb, 256), 256, 0, s>>>(B.st, B.ties, (int)nb, rank);
    GDR_LAUNCHED();
    if (nnz == 0) continue;
    k_sel_eqflag_b<<<dim3(gx, nb), 256, 0, s>>>(nnz, w, B.st, B.a);
    GDR_LAUNCHED();
    if ((rc = exclusive_scan_i32(B.a, B.a, tot, B.sws, B.sws_b, s))) return rc;
    k_sel_flag_b<<<dim3(gx, nb), 256, 0, s>>>(nnz, w, B.st, B.a, B.b);
    GDR_LAUNCHED();
    if ((rc = exclusive_scan_i32(B.b, B.b, tot, B.sws, B.sws_b, s))) return rc;
    k_sel_compact_b<<<dim3(grid_for(std::max(nnz, n_local + 1)), nb), 256, 0, s>>>(
        n_local, nnz, cap, rowptr, colidx, vals, B.b, rowptr_out + c0 * (n_local + 1), colidx_out + c0 * cap,
        vals_out + c0 * cap, nnz_out_dev + c0);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

}  // extern "C"
