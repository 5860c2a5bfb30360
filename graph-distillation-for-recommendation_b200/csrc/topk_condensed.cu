// topk_condensed.cu — full-ranking top-K of a condensed model from its cluster tables.
//
// A condensed model has n_cu super-user rows U and n_ci super-item rows I; user u is U[user_map[u]] and item j is
// I[item_map[j]].  The output is byte-identical to gdr_topk_scores on the expanded tables U[user_map], I[item_map]:
//   s(u, j) = the fmaf chain of U[g] and I[c], g = user_map[u], c = item_map[j]: one value per (g, c) pair,
// so every item of cluster c has the same score for every user of group g, and a user's ranking is its group's order
// of the clusters with each cluster expanded to its members in id order (clusters with bit-equal scores merged by id).
//   k_tkc_maps     map ranges (status bit 2), member counts m[c]
//   k_tkc_check    user ids of the rows (bit 1), non-finite super-user rows of evaluated rows and super-item rows with a
//                  member (bit 0); marks the used groups and need_g = k + max |exclusion row| over their rows
//   sort_pairs     members CSR: items grouped by cluster, ascending inside each (stable radix sort)
//   per slab of used groups:
//     k_topk_score   S[g][c] for the slab (topk.cu's kernel: the same fmaf chain, the same bits)
//     k_tkc_prefix   one CTA per group: radix select of the score level at which the member count of the clusters at or
//                    above it reaches min(n_items, need_g) (whole tie runs), compaction, sort by (score desc, cluster)
//     k_tkc_walk     one warp per row: tie run by tie run, members in id order, exclusions by binary search, stop at k
// A row that meets a tie run of more than 32 clusters before it has k items (a zero super-user ties every cluster) is
// finished by the exact path of topk.cu on the expanded rows, as the tensor-core screen's overflow rows are.
#include "topk_common.cuh"

namespace gdr {

constexpr int64_t TKC_SLAB_BYTES = 384ll << 20;   // score rows + sorted prefixes of one slab of groups
constexpr int TKC_PREFIX_THREADS = 256;
constexpr int TKC_MAX_RUN = 32;                    // a warp merges tie runs of up to 32 clusters
int g_topk_condensed_path = 0;             // gdr_debug_set("topk_condensed_path"): 1 = every row on the fallback
int64_t g_topk_condensed_last_fallback = -1;   // rows the last gdr_topk_condensed finished on the exact path

// status bit 2 for a map value outside its range; m[c] = members of cluster c
__global__ void __launch_bounds__(256) k_tkc_maps(int64_t n_users, int64_t n_items, int64_t n_cu, int64_t n_ci,
                                                  const int64_t* __restrict__ user_map,
                                                  const int64_t* __restrict__ item_map, int32_t* __restrict__ cnt,
                                                  int32_t* __restrict__ status) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool bad = false;
  if (i < n_users) {
    const int64_t g = user_map[i];
    bad |= g < 0 || g >= n_cu;
  }
  if (i < n_items) {
    const int64_t c = item_map[i];
    if (c < 0 || c >= n_ci) bad = true;
    else atomicAdd(&cnt[c], 1);
  }
  if (bad) atomicOr(status, 4);
}

// one warp per evaluated row (used[g], need via maxdeg[g], non-finite U[g]), then one per super-item with members
__global__ void __launch_bounds__(256) k_tkc_check(int64_t n_rows, int64_t n_users, int64_t n_cu, int64_t n_ci,
                                                   int64_t d, const float* __restrict__ U, int64_t ldu,
                                                   const float* __restrict__ I, int64_t ldi,
                                                   const int64_t* __restrict__ rows,
                                                   const int64_t* __restrict__ user_map,
                                                   const int32_t* __restrict__ ex_rowptr,
                                                   const int32_t* __restrict__ cnt, int32_t* __restrict__ used,
                                                   int32_t* __restrict__ maxdeg, int32_t* __restrict__ status) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= n_rows + n_ci) return;
  const float* p;
  if (w < n_rows) {
    const int64_t u = rows ? rows[w] : w;
    if (u < 0 || u >= n_users) {
      if (lane_id() == 0) atomicOr(status, 2);
      return;
    }
    const int64_t g = user_map[u];
    if (g < 0 || g >= n_cu) return;   // reported by k_tkc_maps
    if (lane_id() == 0) {
      used[g] = 1;
      atomicMax(&maxdeg[g], ex_rowptr ? ex_rowptr[u + 1] - ex_rowptr[u] : 0);
    }
    p = U + g * ldu;
  } else {
    const int64_t c = w - n_rows;
    if (cnt[c] == 0) return;   // a cluster without members is never read
    p = I + c * ldi;
  }
  bool bad = false;
  for (int64_t t = lane_id(); t < d; t += 32) bad |= !isfinite(p[t]);
  if (__any_sync(0xffffffffu, bad) && lane_id() == 0) atomicOr(status, 1);
}

__global__ void __launch_bounds__(256) k_tkc_glist(int64_t n_cu, const int32_t* __restrict__ used,
                                                   const int32_t* __restrict__ gpos, int64_t* __restrict__ glist) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n_cu && used[g]) glist[gpos[g]] = g;
}

__global__ void __launch_bounds__(256) k_tkc_keys(int64_t n_items, const int64_t* __restrict__ item_map,
                                                  uint64_t* __restrict__ keys, uint32_t* __restrict__ members) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n_items) {
    keys[j] = (uint64_t)item_map[j];
    members[j] = (uint32_t)j;
  }
}

// dst[r] = src[map[r]] (the expanded rows the fallback scores)
__global__ void __launch_bounds__(256) k_tkc_gather(int64_t n, int64_t d, const float* __restrict__ src, int64_t lds,
                                                    const int64_t* __restrict__ map, float* __restrict__ dst) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const float* p = src + map[r] * lds;
  for (int64_t t = lane_id(); t < d; t += 32) dst[r * d + t] = p[t];
}

// Group slot s0 + blockIdx.x: the clusters with members whose score level is >= v, v = the largest level at which the
// member count at or above it reaches need = min(n_items, k + maxdeg[g]) (the prefix every row of the group can need,
// whole tie runs included), as keys (ordered score << 32 | ~c) sorted descending into P[0..plen).
__global__ void __launch_bounds__(TKC_PREFIX_THREADS) k_tkc_prefix(int64_t s0, int64_t n_ci, int64_t n_items, int64_t k,
                                                                   const int64_t* __restrict__ glist,
                                                                   const int32_t* __restrict__ maxdeg,
                                                                   const float* __restrict__ S, int64_t lds,
                                                                   const int32_t* __restrict__ cstart,
                                                                   uint64_t* __restrict__ pkeys, int64_t ldp,
                                                                   int32_t* __restrict__ plen) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t s_prefix;
  __shared__ int64_t s_need;
  __shared__ unsigned int s_pos;
  const int64_t b = blockIdx.x;
  const int64_t g = glist[s0 + b];
  const uint32_t* Sb = reinterpret_cast<const uint32_t*>(S + b * lds);
  uint64_t* P = pkeys + b * ldp;
  if (threadIdx.x == 0) {
    const int64_t need = k + (int64_t)maxdeg[g];
    s_need = need < n_items ? need : n_items;
    s_prefix = 0;
    s_pos = 0;
  }
  // radix select on the 32-bit score level, weighted by the member counts, 8 bits per pass from the top
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const uint32_t prefix = s_prefix;
    const uint32_t hmask = shift == 24 ? 0u : (~0u << (shift + 8));
    for (int64_t c = threadIdx.x; c < n_ci; c += blockDim.x) {
      const int32_t m = cstart[c + 1] - cstart[c];
      if (m == 0) continue;
      const uint32_t lvl = (uint32_t)(tk_key(Sb[c], c) >> 32);
      if ((lvl & hmask) == prefix) atomicAdd(&hist[(lvl >> shift) & 255], (uint32_t)m);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int64_t above = 0;
      int bin = 255;
      for (; bin > 0; --bin) {
        if (above + (int64_t)hist[bin] >= s_need) break;
        above += hist[bin];
      }
      s_prefix = prefix | ((uint32_t)bin << shift);
      s_need -= above;
    }
    __syncthreads();
  }
  const uint32_t v = s_prefix;
  for (int64_t c = threadIdx.x; c < n_ci; c += blockDim.x) {
    if (cstart[c + 1] == cstart[c]) continue;
    const uint64_t key = tk_key(Sb[c], c);
    if ((uint32_t)(key >> 32) >= v) P[atomicAdd(&s_pos, 1u)] = key;
  }
  __syncthreads();
  const int64_t n = s_pos, np = next_pow2_dev(n);
  for (int64_t i = n + threadIdx.x; i < np; i += blockDim.x) P[i] = 0ull;
  __syncthreads();
  tk_bitonic_desc(P, np);
  if (threadIdx.x == 0) plen[b] = (int32_t)n;
}

__device__ __forceinline__ bool tkc_excluded(const int32_t* __restrict__ ex, int32_t lo, int32_t hi, int32_t j) {
  const int32_t end = hi;
  while (lo < hi) {
    const int32_t mid = lo + ((hi - lo) >> 1);
    if (ex[mid] < j) lo = mid + 1;
    else hi = mid;
  }
  return lo < end && ex[lo] == j;
}

// one warp per output row whose group slot lies in [s0, s0 + ns): the group's sorted prefix, one tie run at a time
__global__ void __launch_bounds__(256) k_tkc_walk(int64_t n_rows, int64_t s0, int64_t ns, int64_t k, int force_fallback,
                                                  const int64_t* __restrict__ rows,
                                                  const int64_t* __restrict__ user_map,
                                                  const int32_t* __restrict__ gpos, const uint64_t* __restrict__ pkeys,
                                                  int64_t ldp, const int32_t* __restrict__ plen,
                                                  const int32_t* __restrict__ cstart,
                                                  const uint32_t* __restrict__ members,
                                                  const int32_t* __restrict__ ex_rowptr,
                                                  const int32_t* __restrict__ ex_colidx, float* __restrict__ scores_out,
                                                  int64_t lds, int32_t* __restrict__ items_out, int64_t ldit,
                                                  int32_t* __restrict__ fb_list, int32_t* __restrict__ fb_count) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_rows) return;
  const int lane = lane_id();
  const int64_t u = rows ? rows[r] : r;
  const int64_t b = (int64_t)gpos[user_map[u]] - s0;
  if (b < 0 || b >= ns) return;
  if (force_fallback) {
    if (lane == 0) fb_list[atomicAdd(fb_count, 1)] = (int32_t)r;
    return;
  }
  const uint64_t* P = pkeys + b * ldp;
  const int64_t n = plen[b];
  const int32_t e0 = ex_rowptr ? ex_rowptr[u] : 0, e1 = ex_rowptr ? ex_rowptr[u + 1] : 0;
  float* so = scores_out + r * lds;
  int32_t* io = items_out + r * ldit;
  int64_t o = 0, p = 0;
  while (o < k && p < n) {
    const uint32_t lvl = (uint32_t)(P[p] >> 32);
    const uint64_t mykey = p + lane < n ? P[p + lane] : 0ull;
    const uint32_t run = __ballot_sync(0xffffffffu, p + lane < n && (uint32_t)(mykey >> 32) == lvl);
    const int L = run == 0xffffffffu ? 32 : __ffs(~run) - 1;
    if (L == TKC_MAX_RUN && p + TKC_MAX_RUN < n && (uint32_t)(P[p + TKC_MAX_RUN] >> 32) == lvl) {
      if (lane == 0) fb_list[atomicAdd(fb_count, 1)] = (int32_t)r;   // the exact path writes this row
      return;
    }
    const float score = tk_key_score(P[p]);
    if (L == 1) {   // one cluster: its members in id order, 32 at a time
      const uint32_t c = ~(uint32_t)P[p];
      const int32_t mb = cstart[c], me = cstart[c + 1];
      for (int32_t q = mb; q < me && o < k; q += 32) {
        const bool in = q + lane < me;
        const int32_t j = in ? (int32_t)members[q + lane] : -1;
        const bool ok = in && !tkc_excluded(ex_colidx, e0, e1, j);
        const uint32_t bal = __ballot_sync(0xffffffffu, ok);
        const int64_t at = o + __popc(bal & ((1u << lane) - 1u));
        if (ok && at < k) {
          io[at] = j;
          so[at] = score;
        }
        o += __popc(bal);
      }
      if (o > k) o = k;
    } else {        // 2..32 clusters of one score: k-way merge of their members by id, lane l holding cluster l
      int32_t h = 0, he = 0;
      if (lane < L) {
        const uint32_t c = ~(uint32_t)mykey;
        h = cstart[c];
        he = cstart[c + 1];
      }
      uint32_t cur = h < he ? members[h] : 0xFFFFFFFFu;
      while (o < k) {
        const uint32_t mn = __reduce_min_sync(0xffffffffu, cur);
        if (mn == 0xFFFFFFFFu) break;   // the run is exhausted
        const bool mine = cur == mn;    // item ids are unique: exactly one lane
        const bool ex = mine && tkc_excluded(ex_colidx, e0, e1, (int32_t)mn);
        if (mine) cur = ++h < he ? members[h] : 0xFFFFFFFFu;
        if (!__any_sync(0xffffffffu, ex)) {
          if (lane == 0) {
            io[o] = (int32_t)mn;
            so[o] = score;
          }
          ++o;
        }
      }
    }
    p += L;
  }
  for (int64_t i = o + lane; i < k; i += 32) {
    io[i] = -1;
    so[i] = -INFINITY;
  }
}

// workspace: persistent arrays, then one region shared in turn by the scan / sort scratch, the slabs of groups and
// the fallback's exact path
struct TkcShape {
  int64_t n_rows, n_users, n_items, n_cu, n_ci, d, k;
};
static int64_t tkc_lds(const TkcShape& z) { return align_up(z.n_ci, 4); }
static int64_t tkc_ldp(const TkcShape& z) { return next_pow2(z.n_ci); }
static int64_t tkc_slab_groups(const TkcShape& z) {
  const int64_t per = tkc_lds(z) * 4 + tkc_ldp(z) * 8 + 4;
  int64_t sg = TKC_SLAB_BYTES / per;
  if (sg >= 128) sg = sg / 128 * 128;
  if (sg < 1) sg = 1;
  const int64_t most = z.n_rows < z.n_cu ? z.n_rows : z.n_cu;
  return sg < most ? sg : most;
}
static int64_t tkc_region_bytes(const TkcShape& z) {
  const int64_t sg = tkc_slab_groups(z);
  const int64_t slab = ws_need(sg * tkc_lds(z), 4) + ws_need(sg * tkc_ldp(z), 8) + ws_need(sg, 4);
  const int64_t scan = scan_ws_bytes(z.n_cu > z.n_ci ? z.n_cu : z.n_ci);
  const int64_t sort = ws_need(z.n_items, 8) + sort_pairs_ws_bytes(z.n_items);
  const int64_t exact = topk_exact_ws_bytes(z.n_rows, z.n_items, z.k);
  int64_t b = slab > scan ? slab : scan;
  b = b > sort ? b : sort;
  return (b > exact ? b : exact) + 256;
}

struct TkcWs {
  int32_t *cnt, *cstart, *used, *gpos, *maxdeg, *fb_list, *fb_count;
  int64_t* glist;
  uint32_t* members;
  float *u_exp, *i_exp;
  char* region;
  int64_t region_bytes;
};
static int64_t tkc_carve(const TkcShape& z, void* base, TkcWs* w) {
  Workspace W(base, 0);
  w->cnt = W.take<int32_t>(z.n_ci + 1);
  w->cstart = W.take<int32_t>(z.n_ci + 1);
  w->used = W.take<int32_t>(z.n_cu + 1);
  w->gpos = W.take<int32_t>(z.n_cu + 1);
  w->maxdeg = W.take<int32_t>(z.n_cu);
  w->glist = W.take<int64_t>(z.n_cu);
  w->members = W.take<uint32_t>(z.n_items);
  w->fb_list = W.take<int32_t>(z.n_rows);
  w->fb_count = W.take<int32_t>(1);
  w->u_exp = W.take<float>(z.n_users * z.d);
  w->i_exp = W.take<float>(z.n_items * z.d);
  w->region_bytes = tkc_region_bytes(z);
  w->region = W.take<char>(w->region_bytes);
  return W.off;
}

int64_t topk_condensed_ws_bytes(const TkcShape& z) {
  TkcWs w;
  return tkc_carve(z, nullptr, &w);
}

static int topk_condensed(const TkcShape& z, const float* U, int64_t ldu, const float* I, int64_t ldi,
                          const int64_t* user_map, const int64_t* item_map, const int64_t* rows,
                          const int32_t* ex_rowptr, const int32_t* ex_colidx, float* scores_out, int64_t lds,
                          int32_t* items_out, int64_t ldit, int32_t* status, void* ws, cudaStream_t s) {
  TkcWs w;
  tkc_carve(z, ws, &w);
  // the map / row checks, member counts and used groups
  GDR_CUDA(cudaMemsetAsync(w.cnt, 0, (z.n_ci + 1) * 4, s));
  GDR_CUDA(cudaMemsetAsync(w.used, 0, (z.n_cu + 1) * 4, s));
  GDR_CUDA(cudaMemsetAsync(w.maxdeg, 0, z.n_cu * 4, s));
  GDR_CUDA(cudaMemsetAsync(w.fb_count, 0, 4, s));
  const int64_t nm = z.n_users > z.n_items ? z.n_users : z.n_items;
  k_tkc_maps<<<(unsigned)cdiv(nm, 256), 256, 0, s>>>(z.n_users, z.n_items, z.n_cu, z.n_ci, user_map, item_map, w.cnt,
                                                     status);
  GDR_LAUNCHED();
  k_tkc_check<<<(unsigned)cdiv((z.n_rows + z.n_ci) * 32, 256), 256, 0, s>>>(
      z.n_rows, z.n_users, z.n_cu, z.n_ci, z.d, U, ldu, I, ldi, rows, user_map, ex_rowptr, w.cnt, w.used, w.maxdeg,
      status);
  GDR_LAUNCHED();
  int rc = exclusive_scan_i32(w.cnt, w.cstart, z.n_ci, w.region, w.region_bytes, s);
  if (rc) return rc;
  if ((rc = exclusive_scan_i32(w.used, w.gpos, z.n_cu, w.region, w.region_bytes, s))) return rc;
  k_tkc_glist<<<(unsigned)cdiv(z.n_cu, 256), 256, 0, s>>>(z.n_cu, w.used, w.gpos, w.glist);
  GDR_LAUNCHED();
  // the status and the number of used groups size everything that follows
  int32_t st = 0, n_g = 0;
  GDR_CUDA(cudaMemcpyAsync(&st, status, 4, cudaMemcpyDeviceToHost, s));
  GDR_CUDA(cudaMemcpyAsync(&n_g, w.gpos + z.n_cu, 4, cudaMemcpyDeviceToHost, s));
  GDR_CUDA(cudaStreamSynchronize(s));
  g_topk_condensed_last_fallback = -1;
  if (st) return GDR_OK;   // the caller reports the status; no output is written
  // members CSR: items by cluster, ascending inside each
  {
    uint64_t* keys = reinterpret_cast<uint64_t*>(w.region);
    void* sws = w.region + ws_need(z.n_items, 8);
    k_tkc_keys<<<(unsigned)cdiv(z.n_items, 256), 256, 0, s>>>(z.n_items, item_map, keys, w.members);
    GDR_LAUNCHED();
    int bits = 0;
    while ((1ll << bits) < z.n_ci) ++bits;
    if ((rc = sort_pairs(z.n_items, bits, keys, w.members, sws, sort_pairs_ws_bytes(z.n_items), s))) return rc;
  }
  const int64_t sg = tkc_slab_groups(z), ld_s = tkc_lds(z), ldp = tkc_ldp(z);
  Workspace R(w.region, w.region_bytes);
  float* S = R.take<float>(sg * ld_s);
  uint64_t* pkeys = R.take<uint64_t>(sg * ldp);
  int32_t* plen = R.take<int32_t>(sg);
  for (int64_t s0 = 0; s0 < n_g; s0 += sg) {
    const int64_t ns = n_g - s0 < sg ? n_g - s0 : sg;
    if ((rc = topk_score_rows(ns, s0, z.n_cu, z.n_ci, z.d, U, ldu, w.glist, I, ldi, S, ld_s, s))) return rc;
    k_tkc_prefix<<<(unsigned)ns, TKC_PREFIX_THREADS, 0, s>>>(s0, z.n_ci, z.n_items, z.k, w.glist, w.maxdeg, S, ld_s,
                                                             w.cstart, pkeys, ldp, plen);
    GDR_LAUNCHED();
    k_tkc_walk<<<(unsigned)cdiv(z.n_rows * 32, 256), 256, 0, s>>>(
        z.n_rows, s0, ns, z.k, g_topk_condensed_path == 1, rows, user_map, w.gpos, pkeys, ldp, plen, w.cstart,
        w.members, ex_rowptr, ex_colidx, scores_out, lds, items_out, ldit, w.fb_list, w.fb_count);
    GDR_LAUNCHED();
  }
  // rows stopped by a long tie run: the exact path on their expanded user rows and the expanded items
  int32_t n_fb = 0;
  GDR_CUDA(cudaMemcpyAsync(&n_fb, w.fb_count, 4, cudaMemcpyDeviceToHost, s));
  GDR_CUDA(cudaStreamSynchronize(s));
  g_topk_condensed_last_fallback = n_fb;
  if (n_fb == 0) return GDR_OK;
  k_tkc_gather<<<(unsigned)cdiv(z.n_users * 32, 256), 256, 0, s>>>(z.n_users, z.d, U, ldu, user_map, w.u_exp);
  GDR_LAUNCHED();
  k_tkc_gather<<<(unsigned)cdiv(z.n_items * 32, 256), 256, 0, s>>>(z.n_items, z.d, I, ldi, item_map, w.i_exp);
  GDR_LAUNCHED();
  return topk_exact(n_fb, z.n_users, z.n_items, z.d, z.k, w.u_exp, z.d, rows, w.fb_list, w.i_exp, z.d, ex_rowptr,
                    ex_colidx, scores_out, lds, items_out, ldit, nullptr, w.region, w.region_bytes, s);
}

}  // namespace gdr

extern "C" {

int64_t gdr_topk_condensed_ws_bytes(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t n_cu, int64_t n_ci,
                                    int64_t d, int64_t k) {
  if (n_rows <= 0 || n_users <= 0 || n_items <= 0 || n_cu <= 0 || n_ci <= 0 || d <= 0 || k <= 0) return 256;
  return gdr::topk_condensed_ws_bytes({n_rows, n_users, n_items, n_cu, n_ci, d, k});
}

int gdr_topk_condensed(int64_t n_rows, int64_t n_users, int64_t n_items, int64_t n_cu, int64_t n_ci, int64_t d,
                       int64_t k, const float* U, int64_t ldu, const float* I, int64_t ldi, const int64_t* user_map,
                       const int64_t* item_map, const int64_t* rows, const int32_t* ex_rowptr,
                       const int32_t* ex_colidx, float* scores_out, int64_t lds, int32_t* items_out, int64_t ldit,
                       int32_t* status_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_rows > 0 && n_users > 0 && n_items > 0 && n_cu > 0 && n_ci > 0 && d > 0,
                "topk_condensed: sizes must be positive");
  GDR_CHECK_ARG(k >= 1 && k <= n_items, "topk_condensed: k=%lld outside [1, n_items=%lld]", (long long)k,
                (long long)n_items);
  GDR_CHECK_ARG(n_items < INT32_MAX && n_users < INT32_MAX && n_rows < INT32_MAX && n_cu < INT32_MAX &&
                    n_ci < INT32_MAX,
                "topk_condensed: ids must fit int32");
  GDR_CHECK_ARG(U && I && user_map && item_map && scores_out && items_out && status_dev && ws,
                "topk_condensed: null pointer");
  GDR_CHECK_ARG((ex_rowptr == nullptr) == (ex_colidx == nullptr), "topk_condensed: exclusion CSR needs both arrays");
  GDR_CHECK_ARG(ldu >= d && ldi >= d && lds >= k && ldit >= k, "topk_condensed: leading dimension too small");
  GDR_CHECK_ARG(rows || n_rows <= n_users, "topk_condensed: n_rows > n_users without a rows list");
  const gdr::TkcShape z{n_rows, n_users, n_items, n_cu, n_ci, d, k};
  if (ws_bytes < gdr::topk_condensed_ws_bytes(z)) {
    gdr::set_error("topk_condensed: workspace too small");
    return GDR_EWORKSPACE;
  }
  return gdr::topk_condensed(z, U, ldu, I, ldi, user_map, item_map, rows, ex_rowptr, ex_colidx, scores_out, lds,
                             items_out, ldit, status_dev, ws, (cudaStream_t)stream);
}

}  // extern "C"
