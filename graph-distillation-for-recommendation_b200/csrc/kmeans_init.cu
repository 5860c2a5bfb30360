// kmeans_init.cu — greedy k-means++ seeding on the device.
//
// Algorithm of sklearn's _kmeans_plusplus (sklearn/cluster/_kmeans.py:180-278), the default
// initialisation behind the reference's `KMeans(n_clusters=n).fit(...)`
// (clustgdd_agent_transduct.py:105, distill_recsys.py:178):
//   first centre = a uniformly drawn sample; then for every further centre draw
//   n_local_trials = 2 + int(log K) candidates with probability proportional to the squared
//   distance to the closest centre so far (searchsorted on the cumulative sum), keep the
//   candidate that lowers the total potential most.
// The random numbers are drawn by the HOST from numpy's RandomState exactly as sklearn
// consumes them (one choice(), then uniform(size=n_local_trials) per round) and handed in;
// every arithmetic step runs here, and the K rounds need no host synchronisation.
// Potentials / cumulative sums are accumulated in fp64 in a fixed order (deterministic); sklearn
// uses an fp32 cumsum, so a draw that lands within rounding of a boundary may pick a neighbour.
#include "common.cuh"
#include "comm.cuh"
#include <vector>

namespace gdr {

constexpr int PP_THREADS = 256;
constexpr int PP_ROWS_PER_BLOCK = 1024;   // rows summarised by one block-sum entry
constexpr int PP_MAX_TRIALS = 16;   // 2 + int(log K) <= 16 up to K ~ 1.2e6

struct PpState {
  int64_t cur_id;      // centre chosen in the previous round
  double pot;          // current potential
  int64_t cand[PP_MAX_TRIALS];
};

// |x - c|^2 of one row by one warp: lane-strided __fsub_rn + fmaf chains, then the xor butterfly 16..1.  Every
// k-means++ pass (one-GPU and row-partitioned) computes a row's distance with exactly these bits.
__device__ __forceinline__ float pp_row_dist(const float* __restrict__ x, const float* c, int D, int lane) {
  float d = 0.f;
  for (int k = lane; k < D; k += 32) {
    float t = __fsub_rn(x[k], c[k]);
    d = fmaf(t, t, d);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
  return d;
}

// k_pp_pick's fixed-order prefix over the block sums (1024 threads): per-thread runs of ceil(nblocks / 1024) sums, a
// Hillis-Steele scan of the 1024 partials; bprefix[b] = exclusive prefix, bprefix[nblocks] = total (visible to the
// whole block on return)
__device__ __forceinline__ void pp_block_prefix(int nblocks, const double* __restrict__ bsum, double* __restrict__ bprefix,
                                                double* s_part) {
  const int t = threadIdx.x;
  const int per = (nblocks + 1023) / 1024;
  const int b0 = t * per, b1 = min(nblocks, b0 + per);
  double s = 0.0;
  for (int b = b0; b < b1; ++b) s += bsum[b];
  s_part[t] = s;
  __syncthreads();
  // exclusive scan of the 1024 partials (Hillis-Steele on shared memory, fixed order)
  for (int o = 1; o < 1024; o <<= 1) {
    double v = t >= o ? s_part[t - o] : 0.0;
    __syncthreads();
    s_part[t] += v;
    __syncthreads();
  }
  double run = t == 0 ? 0.0 : s_part[t - 1];
  for (int b = b0; b < b1; ++b) {
    bprefix[b] = run;
    run += bsum[b];
  }
  if (t == 1023) bprefix[nblocks] = s_part[1023];
  __syncthreads();
}

// np.searchsorted(cumsum, thr, side='left') inside one block of rows [r0, r1) by one warp: the first row whose
// inclusive fp64 running sum base + closest[r0..i] reaches thr (warp scan of 32 rows at a time); `none` when no row does
__device__ __forceinline__ int64_t pp_block_search(const float* __restrict__ closest, int64_t r0, int64_t r1, double base,
                                                   double thr, int lane, int64_t none) {
  int64_t found = none;
  bool done = false;
  for (int64_t r = r0; r < r1 && !done; r += 32) {
    int64_t i = r + lane;
    double v = i < r1 ? (double)closest[i] : 0.0;
    double incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      double u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
    }
    unsigned hit = __ballot_sync(0xffffffffu, i < r1 && base + incl >= thr);
    if (hit) {
      found = r + (__ffs(hit) - 1);
      done = true;
    }
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
  return found;
}

// k_pp_choose's fixed order of one candidate's total: lane-strided over the block sums bpot[b * stride + l], then the
// xor butterfly (one warp; every lane returns the total)
__device__ __forceinline__ double pp_cand_total(const double* bpot, int stride, int l, int nblocks, int lane) {
  double s = 0.0;
  for (int b = lane; b < nblocks; b += 32) s += bpot[(int64_t)b * stride + l];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}

// closest[i] = min(closest[i], |x_i - x_cur|^2)  (first round: plain assignment);
// bsum[b] = sum of closest over the block's rows (fp64, fixed order)
__global__ void __launch_bounds__(PP_THREADS) k_pp_update(int64_t N, int D, const float* __restrict__ X, int64_t ldx,
                                                          const PpState* __restrict__ st, int first,
                                                          float* __restrict__ closest, double* __restrict__ bsum) {
  extern __shared__ float s_c[];   // D floats: the current centre
  __shared__ double s_w[PP_THREADS / 32];
  const int64_t cur = st->cur_id;
  for (int k = threadIdx.x; k < D; k += PP_THREADS) s_c[k] = X[cur * ldx + k];
  __syncthreads();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t r0 = (int64_t)blockIdx.x * PP_ROWS_PER_BLOCK;
  const int64_t r1 = min(N, r0 + PP_ROWS_PER_BLOCK);
  double acc = 0.0;
  for (int64_t r = r0 + w; r < r1; r += PP_THREADS / 32) {
    const float d = pp_row_dist(X + r * ldx, s_c, D, lane);
    float c = first ? d : fminf(closest[r], d);
    if (lane == 0) closest[r] = c;
    acc += (double)c;
  }
  if (lane == 0) s_w[w] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < PP_THREADS / 32; ++i) s += s_w[i];
    bsum[blockIdx.x] = s;
  }
}

// single CTA: prefix over the block sums, potential, and the searchsorted of the L draws
__global__ void __launch_bounds__(1024) k_pp_pick(int64_t N, int nblocks, const double* __restrict__ bsum,
                                                  double* __restrict__ bprefix /*[nblocks + 1]*/,
                                                  const float* __restrict__ closest,
                                                  const double* __restrict__ rand_vals, int L,
                                                  PpState* __restrict__ st) {
  __shared__ double s_part[1024];
  const int t = threadIdx.x;
  pp_block_prefix(nblocks, bsum, bprefix, s_part);
  const double pot = bprefix[nblocks];
  if (t == 0) st->pot = pot;
  // warp l resolves draw l: first index i with cumsum[i] >= rand * pot  (np.searchsorted, side='left')
  const int w = t >> 5, lane = t & 31;
  if (w < L) {
    const double thr = rand_vals[w] * pot;
    // first block whose inclusive prefix reaches thr
    int lo = 0, hi = nblocks;  // search in [0, nblocks)
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      if (bprefix[mid + 1] >= thr) hi = mid;
      else lo = mid + 1;
    }
    int64_t found = N - 1;  // np.clip(candidate_ids, None, n - 1)
    if (lo < nblocks) {
      const int64_t r0 = (int64_t)lo * PP_ROWS_PER_BLOCK, r1 = min(N, r0 + PP_ROWS_PER_BLOCK);
      found = pp_block_search(closest, r0, r1, bprefix[lo], thr, lane, N - 1);
    }
    if (lane == 0) st->cand[w] = found;
  }
}

// per block: for every candidate l the sum over the block's rows of min(closest_i, |x_i - x_cand_l|^2)
__global__ void __launch_bounds__(PP_THREADS) k_pp_score(int64_t N, int D, const float* __restrict__ X, int64_t ldx,
                                                         const PpState* __restrict__ st, int L,
                                                         const float* __restrict__ closest,
                                                         double* __restrict__ bpot /*[nblocks][L]*/) {
  extern __shared__ float s_cand[];   // L * D floats
  __shared__ double s_w[PP_THREADS / 32][PP_MAX_TRIALS];
  for (int i = threadIdx.x; i < L * D; i += PP_THREADS) {
    int l = i / D, k = i - l * D;
    s_cand[i] = X[st->cand[l] * ldx + k];
  }
  __syncthreads();
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t r0 = (int64_t)blockIdx.x * PP_ROWS_PER_BLOCK;
  const int64_t r1 = min(N, r0 + PP_ROWS_PER_BLOCK);
  double acc[PP_MAX_TRIALS];
#pragma unroll
  for (int l = 0; l < PP_MAX_TRIALS; ++l) acc[l] = 0.0;
  for (int64_t r = r0 + w; r < r1; r += PP_THREADS / 32) {
    const float cl = closest[r];
#pragma unroll
    for (int l = 0; l < PP_MAX_TRIALS; ++l) {
      if (l >= L) break;
      const float d = pp_row_dist(X + r * ldx, s_cand + l * D, D, lane);
      acc[l] += (double)fminf(cl, d);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int l = 0; l < PP_MAX_TRIALS; ++l)
      if (l < L) s_w[w][l] = acc[l];
  }
  __syncthreads();
  if (threadIdx.x < L) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < PP_THREADS / 32; ++i) s += s_w[i][threadIdx.x];
    bpot[(int64_t)blockIdx.x * L + threadIdx.x] = s;
  }
}

// single CTA: total potential per candidate (fixed order), first argmin, commit the winner
__global__ void __launch_bounds__(1024) k_pp_choose(int nblocks, int L, int D, const double* __restrict__ bpot,
                                                    const float* __restrict__ X, int64_t ldx,
                                                    PpState* __restrict__ st, float* __restrict__ centers, int64_t ldc,
                                                    int64_t* __restrict__ indices, int c) {
  __shared__ double s_pot[PP_MAX_TRIALS];
  __shared__ int s_best;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (w < L) {
    double s = 0.0;
    for (int b = lane; b < nblocks; b += 32) s += bpot[(int64_t)b * L + w];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) s_pot[w] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int best = 0;
    for (int l = 1; l < L; ++l)
      if (s_pot[l] < s_pot[best]) best = l;   // np.argmin: first minimum
    s_best = best;
    st->pot = s_pot[best];
    st->cur_id = st->cand[best];
    if (indices) indices[c] = st->cand[best];
  }
  __syncthreads();
  const int64_t id = st->cand[s_best];
  for (int k = threadIdx.x; k < D; k += 1024) centers[(int64_t)c * ldc + k] = X[id * ldx + k];
}

__global__ void k_pp_first(int64_t first, int D, const float* __restrict__ X, int64_t ldx, PpState* __restrict__ st,
                           float* __restrict__ centers, int64_t* __restrict__ indices) {
  if (threadIdx.x == 0) {
    st->cur_id = first;
    st->pot = 0.0;
    if (indices) indices[0] = first;
  }
  for (int k = threadIdx.x; k < D; k += blockDim.x) centers[k] = X[first * ldx + k];
}


// ---- k-means++ on a row partition (gdr_kmeans_plusplus_dist) -------------------------------------------------------
// Every rank holds a contiguous block of rows; the blocks in rank order are the global row order.  One round (centre c):
//   pick     every rank derives pot = sum_r T_r and the rank prefixes P_r (rank order) from the totals of exchange B;
//            the owner of draw l (first rank with rows and P_r + T_r >= u_l * pot) searches its rows as k_pp_pick does
//   exch. A  the owners' candidate rows and global ids are all-gathered; every rank copies (never sums) candidate l
//            from its owner's slot
//   score    ONE pass over the local rows: dcol[l][i] = min(closest_i, |x_i - cand_l|^2) for every candidate, and the
//            per-block fp64 sums bpot[l][b] in k_pp_score's order.  The winner's column is the next round's `closest`
//            and its block sums are the next round's bsum (double-buffered by round parity), so X is read once a round
//   reduce   per candidate the rank total in k_pp_choose's order (S) and in k_pp_pick's order (T)
//   exch. B  [S | T] all-gathered; every rank adds pot_l = sum_r S_r[l] in rank order, takes the first argmin and
//            commits the centre from the exchange-A rows
// The per-row fp32 distances have the one-GPU bits; only the fp64 totals are grouped by rank.
int g_kpp_skip_score = 0;   // gdr_debug_set("kpp_dist_skip_score", 1): rounds without the score pass (exchange timing only)

struct PpdState {
  int64_t round;                     // index of the centre the next choose commits
  int64_t n_total;
  int64_t off[GDR_MAX_RANKS + 1];    // global row offset of every rank's block
  double T[GDR_MAX_RANKS];           // per-rank total of the current `closest` in k_pp_pick's order
  int world, rank, last;             // last: the last rank with rows (it owns row n_total - 1)
  int best;                          // winning column of the last pass
  int src[PP_MAX_TRIALS];            // owner rank of draw l (-1: none; the draw is clipped to row n_total - 1)
};

// exchange-A slot of one rank: int64 ids[Lmax] | float rows[Lmax + 1][D]; row Lmax is the rank's last row (published
// by the last rank: the row every clipped draw resolves to)
__device__ __forceinline__ const float* ppd_cand(const PpdState* st, const char* exa, int64_t slot, int Lmax, int D, int l,
                                                 int64_t* id) {
  const int o = st->src[l];
  if (o >= 0) {
    const char* p = exa + o * slot;
    const int64_t g = ((const int64_t*)p)[l];
    if (g >= st->off[o] && g < st->off[o + 1]) {
      *id = g;
      return (const float*)(p + Lmax * 8) + (int64_t)l * D;
    }
  }
  *id = st->n_total - 1;
  return (const float*)(exa + st->last * slot + Lmax * 8) + (int64_t)Lmax * D;
}

// start-up: state, and the owner of the first centre publishes it as candidate 0
__global__ void k_ppd_first(PpdState init, int64_t first, int64_t N, int D, const float* __restrict__ X, int64_t ldx, int Lmax,
                            PpdState* __restrict__ st, char* __restrict__ my_slot) {
  int owner = 0;
  while (owner + 1 < init.world && first >= init.off[owner + 1]) ++owner;
  if (threadIdx.x == 0) {
    *st = init;
    st->round = 0;
    st->best = 0;
    st->src[0] = owner;
    if (owner == init.rank) ((int64_t*)my_slot)[0] = first;
  }
  float* rows = (float*)(my_slot + Lmax * 8);
  if (owner == init.rank)
    for (int k = threadIdx.x; k < D; k += blockDim.x) rows[k] = X[(first - init.off[init.rank]) * ldx + k];
  if (init.rank == init.last)
    for (int k = threadIdx.x; k < D; k += blockDim.x) rows[(int64_t)Lmax * D + k] = X[(N - 1) * ldx + k];
}

// single CTA: prefix over the last winner's block sums, owners of the L draws, the owned draws' rows into this rank's slot
__global__ void __launch_bounds__(1024) k_ppd_pick(int64_t N, int nb, int D, const float* __restrict__ X, int64_t ldx,
                                                   const double* __restrict__ bpot, const float* __restrict__ dcol, int Lmax,
                                                   const double* __restrict__ rand_vals, double* __restrict__ bprefix,
                                                   PpdState* __restrict__ st, char* __restrict__ my_slot) {
  __shared__ double s_part[1024];
  const int64_t c = st->round;
  const int p_in = (int)((c - 1) & 1), best = st->best;
  const double* bsum = bpot + (int64_t)(p_in * Lmax + best) * nb;
  const float* closest = dcol + (int64_t)(p_in * Lmax + best) * N;
  pp_block_prefix(nb, bsum, bprefix, s_part);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (w >= Lmax) return;
  const int world = st->world, rank = st->rank;
  double pot = 0.0;
  for (int r = 0; r < world; ++r) pot += st->T[r];
  const double thr = rand_vals[(c - 1) * Lmax + w] * pot;
  int owner = -1;
  double P = 0.0;
  for (int r = 0; r < world; ++r) {
    if (st->off[r + 1] > st->off[r] && P + st->T[r] >= thr) {
      owner = r;
      break;
    }
    P += st->T[r];
  }
  if (lane == 0) st->src[w] = owner;
  if (owner != rank) return;
  int lo = 0, hi = nb;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (P + bprefix[mid + 1] >= thr) hi = mid;
    else lo = mid + 1;
  }
  int64_t found = -1;
  if (lo < nb) {
    const int64_t r0 = (int64_t)lo * PP_ROWS_PER_BLOCK, r1 = min(N, r0 + PP_ROWS_PER_BLOCK);
    found = pp_block_search(closest, r0, r1, P + bprefix[lo], thr, lane, -1);
  }
  // a draw no row reaches is np.clip'ed to the last global row: id -1 lies in no rank's range, so every rank takes the
  // row the last rank published once (slot row Lmax), never this slot's row w (the previous round's candidate)
  if (lane == 0) ((int64_t*)my_slot)[w] = found >= 0 ? st->off[rank] + found : -1;
  if (found >= 0) {
    float* row = (float*)(my_slot + Lmax * 8) + (int64_t)w * D;
    for (int k = lane; k < D; k += 32) row[k] = X[found * ldx + k];
  }
}

// the one pass over the local rows for L candidates (start-up: L = 1 and `first`, closest = d as in k_pp_update)
__global__ void __launch_bounds__(PP_THREADS, 4) k_ppd_score(int64_t N, int nb, int D, const float* __restrict__ X, int64_t ldx,
                                                          const PpdState* __restrict__ st, const char* __restrict__ exa,
                                                          int64_t slot, int Lmax, int L, int first,
                                                          float* __restrict__ dcol, double* __restrict__ bpot) {
  extern __shared__ float s_cand[];   // L * D floats
  __shared__ double s_w[PP_THREADS / 32][PP_MAX_TRIALS];
  for (int l = 0; l < L; ++l) {
    int64_t id;
    const float* src = ppd_cand(st, exa, slot, Lmax, D, l, &id);
    for (int k = threadIdx.x; k < D; k += PP_THREADS) s_cand[l * D + k] = src[k];
  }
  __syncthreads();
  const int p_out = (int)(st->round & 1), p_in = p_out ^ 1;
  const float* closest = dcol + (int64_t)(p_in * Lmax + st->best) * N;
  float* out = dcol + (int64_t)p_out * Lmax * N;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t r0 = (int64_t)blockIdx.x * PP_ROWS_PER_BLOCK;
  const int64_t r1 = min(N, r0 + PP_ROWS_PER_BLOCK);
  double acc[PP_MAX_TRIALS];
#pragma unroll
  for (int l = 0; l < PP_MAX_TRIALS; ++l) acc[l] = 0.0;
  for (int64_t r = r0 + w; r < r1; r += PP_THREADS / 32) {
    const float cl = first ? 0.f : closest[r];
#pragma unroll
    for (int l = 0; l < PP_MAX_TRIALS; ++l) {
      if (l >= L) break;
      const float d = pp_row_dist(X + r * ldx, s_cand + l * D, D, lane);
      const float v = first ? d : fminf(cl, d);
      if (lane == 0) out[(int64_t)l * N + r] = v;
      acc[l] += (double)v;
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int l = 0; l < PP_MAX_TRIALS; ++l)
      if (l < L) s_w[w][l] = acc[l];
  }
  __syncthreads();
  if (threadIdx.x < L) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < PP_THREADS / 32; ++i) s += s_w[i][threadIdx.x];
    bpot[(int64_t)(p_out * Lmax + threadIdx.x) * nb + blockIdx.x] = s;
  }
}

// single CTA: this rank's [S[Lmax] | T[Lmax]] for exchange B
__global__ void __launch_bounds__(1024) k_ppd_reduce(int nb, int Lmax, int L, const double* __restrict__ bpot,
                                                     const PpdState* __restrict__ st, double* __restrict__ scratch,
                                                     double* __restrict__ my_slot) {
  __shared__ double s_part[1024];
  const int p_out = (int)(st->round & 1);
  const double* cols = bpot + (int64_t)p_out * Lmax * nb;
  for (int l = 0; l < L; ++l) {
    pp_block_prefix(nb, cols + (int64_t)l * nb, scratch, s_part);
    if (threadIdx.x == 0) my_slot[Lmax + l] = scratch[nb];
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (w < L) {
    const double s = pp_cand_total(cols + (int64_t)w * nb, 1, 0, nb, lane);
    if (lane == 0) my_slot[w] = s;
  }
}

// single CTA: pot_l = sum_r S_r[l] in rank order, first argmin, commit centre `round`, T_r := T_r[best]
__global__ void k_ppd_choose(int Lmax, int L, int D, const double* __restrict__ exb, const char* __restrict__ exa, int64_t slot,
                             PpdState* __restrict__ st, float* __restrict__ centers, int64_t ldc, int64_t* __restrict__ indices) {
  __shared__ int s_best;
  const int world = st->world;
  const int64_t c = st->round;
  if (threadIdx.x == 0) {
    int best = 0;
    double bp = 0.0;
    for (int l = 0; l < L; ++l) {
      double s = exb[l];
      for (int r = 1; r < world; ++r) s += exb[(int64_t)r * 2 * Lmax + l];
      if (l == 0 || s < bp) {   // np.argmin: first minimum
        bp = s;
        best = l;
      }
    }
    s_best = best;
  }
  __syncthreads();
  const int best = s_best;
  int64_t id;
  const float* row = ppd_cand(st, exa, slot, Lmax, D, best, &id);
  for (int k = threadIdx.x; k < D; k += blockDim.x) centers[c * ldc + k] = row[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    if (indices) indices[c] = id;
    for (int r = 0; r < world; ++r) st->T[r] = exb[(int64_t)r * 2 * Lmax + Lmax + best];
    st->best = best;
    st->round = c + 1;
  }
}

bool profiling_enabled();

}  // namespace gdr

using namespace gdr;

namespace {

struct PpdBuffers {
  int64_t* meta;     // [world][8]     entry check (first in the workspace: see gdr_kmeans_plusplus_dist)
  float* dcol;       // [2][Lmax][N]   candidate columns of the last two passes
  double* bpot;      // [2][Lmax][nb]  their block sums
  double* bprefix;   // [nb + 1]
  double* rand_dev;  // [K - 1][Lmax]
  char* exa;         // [world][slot]  exchange A (in place: this rank's slot is its send buffer)
  double* exb;       // [world][2 Lmax] exchange B
  PpdState* st;
  int64_t slot, off;
};

PpdBuffers ppd_carve(void* ws, int64_t N, int64_t K, int64_t D, int Lmax, int world) {
  const int64_t n = N > 0 ? N : 1, nb = cdiv(n, PP_ROWS_PER_BLOCK);
  Workspace W(ws, INT64_MAX);
  PpdBuffers b;
  b.slot = align_up(Lmax * 8 + (Lmax + 1) * D * 4, 16);
  b.meta = W.take<int64_t>(world * 8);
  b.dcol = W.take<float>(2 * Lmax * n);
  b.bpot = W.take<double>(2 * Lmax * nb);
  b.bprefix = W.take<double>(nb + 1);
  b.rand_dev = W.take<double>((K > 1 ? K - 1 : 1) * Lmax);
  b.exa = W.take<char>(world * b.slot);
  b.exb = W.take<double>(world * 2 * Lmax);
  b.st = W.take<PpdState>(1);
  b.off = W.off + 256;
  return b;
}

uint64_t fnv1a(const void* p, size_t n) {
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; ++i) h = (h ^ ((const unsigned char*)p)[i]) * 1099511628211ull;
  return h;
}

struct PpdGraph {
  cudaStream_t gs = nullptr;
  cudaEvent_t ev = nullptr;
  cudaGraphExec_t exec = nullptr;
  ~PpdGraph() {
    if (exec) cudaGraphExecDestroy(exec);
    if (ev) cudaEventDestroy(ev);
    if (gs) cudaStreamDestroy(gs);
  }
};

}  // namespace


extern "C" {

int64_t gdr_kmeans_plusplus_ws_bytes(int64_t N, int64_t K, int64_t D, int n_trials) {
  (void)D;
  int64_t nb = cdiv(N > 0 ? N : 1, PP_ROWS_PER_BLOCK);
  return ws_need(N, 4) + 2 * ws_need(nb + 1, 8) + ws_need(nb * n_trials, 8) + ws_need((K > 1 ? K - 1 : 1) * n_trials, 8) +
         ws_need(1, sizeof(PpState)) + 256;
}

int gdr_kmeans_plusplus(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx, int64_t first_center,
                        const double* rand_vals_host, int n_trials, float* centers_out, int64_t ldc,
                        int64_t* indices_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && K > 0 && D > 0 && X && centers_out && ws, "kmeans_plusplus: bad arguments");
  GDR_CHECK_ARG(K <= N, "kmeans_plusplus: n_samples=%lld should be >= n_clusters=%lld", (long long)N, (long long)K);
  GDR_CHECK_ARG(first_center >= 0 && first_center < N, "kmeans_plusplus: first centre out of range");
  GDR_CHECK_ARG(n_trials >= 1 && n_trials <= PP_MAX_TRIALS, "kmeans_plusplus: n_trials must be in [1, 16]");
  GDR_CHECK_ARG(K == 1 || rand_vals_host, "kmeans_plusplus: null random numbers");
  GDR_CHECK_ARG(ldx >= D && ldc >= D, "kmeans_plusplus: leading dimension");
  if (ws_bytes < gdr_kmeans_plusplus_ws_bytes(N, K, D, n_trials)) {
    set_error("kmeans_plusplus: workspace too small");
    return GDR_EWORKSPACE;
  }
  const size_t smem_score = (size_t)n_trials * D * 4, smem_upd = (size_t)D * 4;
  if (smem_score > 200 * 1024 || smem_upd > 48 * 1024) {
    set_error("kmeans_plusplus: n_trials * D = %lld floats exceeds the shared-memory plan", (long long)n_trials * D);
    return GDR_EUNSUPPORTED;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int nb = (int)cdiv(N, PP_ROWS_PER_BLOCK);
  Workspace W(ws, ws_bytes);
  float* closest = W.take<float>(N);
  double* bsum = W.take<double>(nb + 1);
  double* bprefix = W.take<double>(nb + 1);
  double* bpot = W.take<double>((int64_t)nb * n_trials);
  double* rand_dev = W.take<double>((K > 1 ? K - 1 : 1) * n_trials);
  PpState* st = W.take<PpState>(1);
  if (K > 1)
    GDR_CUDA(cudaMemcpyAsync(rand_dev, rand_vals_host, (K - 1) * n_trials * 8, cudaMemcpyHostToDevice, s));
  if (smem_score > 48 * 1024)
    GDR_CUDA(cudaFuncSetAttribute(k_pp_score, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_score));
  k_pp_first<<<1, 256, 0, s>>>(first_center, (int)D, X, ldx, st, centers_out, indices_out_dev);
  GDR_LAUNCHED();
  for (int64_t c = 1; c < K; ++c) {
    k_pp_update<<<nb, PP_THREADS, smem_upd, s>>>(N, (int)D, X, ldx, st, c == 1, closest, bsum);
    GDR_LAUNCHED();
    k_pp_pick<<<1, 1024, 0, s>>>(N, nb, bsum, bprefix, closest, rand_dev + (c - 1) * n_trials, n_trials, st);
    GDR_LAUNCHED();
    k_pp_score<<<nb, PP_THREADS, smem_score, s>>>(N, (int)D, X, ldx, st, n_trials, closest, bpot);
    GDR_LAUNCHED();
    k_pp_choose<<<1, 1024, 0, s>>>(nb, n_trials, (int)D, bpot, X, ldx, st, centers_out, ldc, indices_out_dev, (int)c);
    GDR_LAUNCHED();
  }
  // the pageable host buffer must stay valid until the copy above has executed
  if (K > 1) GDR_CUDA(cudaStreamSynchronize(s));
  return GDR_OK;
}

int64_t gdr_kmeans_plusplus_dist_ws_bytes(int64_t N_local, int64_t K, int64_t D, int n_trials, int world) {
  return ppd_carve(nullptr, N_local, K, D, n_trials, world).off;
}

int gdr_kmeans_plusplus_dist(gdr_comm_t* comm, int64_t N_local, int64_t K, int64_t D, const float* X_local, int64_t ldx,
                             int64_t first_center, const double* rand_vals_host, int n_trials, float* centers_out,
                             int64_t ldc, int64_t* indices_out_dev, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(comm, "kmeans_plusplus_dist: null communicator");
  const int world = comm->world, rank = comm->rank;
  cudaStream_t caller = (cudaStream_t)stream;
  // local checks are decided collectively below: a rank that returned early would leave the others in a collective
  int local_rc = GDR_OK;
  const size_t smem_score = (size_t)n_trials * D * 4;
  if (!(N_local >= 0 && K > 0 && D > 0 && centers_out && ws && (N_local == 0 || X_local) && ldx >= D && ldc >= D &&
        (K == 1 || rand_vals_host))) {
    set_error("kmeans_plusplus_dist: bad arguments");
    local_rc = GDR_EINVAL;
  } else if (n_trials < 1 || n_trials > PP_MAX_TRIALS) {
    set_error("kmeans_plusplus_dist: n_trials must be in [1, 16]");
    local_rc = GDR_EINVAL;
  } else if (world > GDR_MAX_RANKS) {
    set_error("kmeans_plusplus_dist: more than %d ranks", GDR_MAX_RANKS);
    local_rc = GDR_EUNSUPPORTED;
  } else if (smem_score > 200 * 1024 || (size_t)D * 4 > 48 * 1024) {
    set_error("kmeans_plusplus_dist: n_trials * D = %lld floats exceeds the shared-memory plan", (long long)n_trials * D);
    local_rc = GDR_EUNSUPPORTED;
  } else if (ws_bytes < gdr_kmeans_plusplus_dist_ws_bytes(N_local, K, D, n_trials, world)) {
    set_error("kmeans_plusplus_dist: workspace too small");
    local_rc = GDR_EWORKSPACE;
  }
  // entry check: every rank must pass the same first centre, n_trials, K, D and random numbers
  const uint64_t sum = (local_rc == GDR_OK && K > 1) ? fnv1a(rand_vals_host, (size_t)(K - 1) * n_trials * 8) : 0;
  int64_t mine[8] = {N_local, first_center, n_trials, (int64_t)sum, K, D, local_rc, 0};
  std::vector<int64_t> all((size_t)world * 8);
  // the gather buffer is the head of the workspace; a rank whose workspace cannot hold it still takes part in the
  // check (through a temporary buffer: a rejected call only) so that every rank learns the verdict
  const int64_t meta_bytes = (int64_t)all.size() * 8;
  int64_t* meta = ws && ws_bytes >= meta_bytes ? (int64_t*)ws : nullptr;   // ppd_carve's first block
  int64_t* meta_tmp = nullptr;
  if (!meta) {
    GDR_CUDA(cudaMalloc(&meta_tmp, meta_bytes));
    meta = meta_tmp;
  }
  int rc = GDR_OK;
  if (cudaMemcpyAsync(meta + rank * 8, mine, 64, cudaMemcpyHostToDevice, caller) != cudaSuccess) {
    set_error("kmeans_plusplus_dist: copy of the argument check failed");
    rc = GDR_ECUDA;
  }
  if (rc == GDR_OK) rc = comm_allgather(comm, meta + rank * 8, meta, 64, caller);
  if (rc == GDR_OK && (cudaMemcpyAsync(all.data(), meta, meta_bytes, cudaMemcpyDeviceToHost, caller) != cudaSuccess ||
                       cudaStreamSynchronize(caller) != cudaSuccess)) {
    set_error("kmeans_plusplus_dist: read-back of the argument check failed");
    rc = GDR_ECUDA;
  }
  if (meta_tmp) cudaFree(meta_tmp);
  if (rc != GDR_OK) return rc;
  if (local_rc != GDR_OK) return local_rc;
  PpdState init = {};
  init.world = world;
  init.rank = rank;
  init.last = 0;
  for (int r = 0; r < world; ++r) {
    const int64_t* m = &all[(size_t)r * 8];
    if (m[6] != GDR_OK) {
      set_error("kmeans_plusplus_dist: rank %d rejected its arguments", r);
      return GDR_EINVAL;
    }
    if (m[1] != mine[1] || m[2] != mine[2] || m[3] != mine[3] || m[4] != mine[4] || m[5] != mine[5]) {
      set_error("kmeans_plusplus_dist: rank %d passed a different first centre, n_trials, K, D or random numbers", r);
      return GDR_EINVAL;
    }
    init.off[r + 1] = init.off[r] + m[0];
    if (m[0] > 0) init.last = r;
  }
  const int64_t N_total = init.off[world];
  init.n_total = N_total;
  GDR_CHECK_ARG(K <= N_total, "kmeans_plusplus_dist: n_samples=%lld should be >= n_clusters=%lld", (long long)N_total,
                (long long)K);
  GDR_CHECK_ARG(first_center >= 0 && first_center < N_total, "kmeans_plusplus_dist: first centre out of range");

  // graph replay needs a capturable stream: the rounds run on an internal stream ordered after the caller's
  PpdGraph G;
  bool use_graph = K >= 3 && !profiling_enabled();
  cudaStream_t s = caller;
  if (use_graph) {
    if (cudaStreamCreateWithFlags(&G.gs, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&G.ev, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      use_graph = false;
    } else {
      GDR_CUDA(cudaEventRecord(G.ev, caller));
      GDR_CUDA(cudaStreamWaitEvent(G.gs, G.ev, 0));
      s = G.gs;
    }
  }
  const int L = n_trials, nb = (int)cdiv(N_local, PP_ROWS_PER_BLOCK);
  PpdBuffers B = ppd_carve(ws, N_local, K, D, L, world);
  char* my_a = B.exa + rank * B.slot;
  double* my_b = B.exb + (int64_t)rank * 2 * L;
  if (K > 1) GDR_CUDA(cudaMemcpyAsync(B.rand_dev, rand_vals_host, (K - 1) * L * 8, cudaMemcpyHostToDevice, s));
  if (smem_score > 48 * 1024)
    GDR_CUDA(cudaFuncSetAttribute(k_ppd_score, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_score));
  auto pass_and_choose = [&](int n_cand, int first) -> int {
    if (nb > 0 && (first || !g_kpp_skip_score)) {
      k_ppd_score<<<nb, PP_THREADS, (size_t)n_cand * D * 4, s>>>(N_local, nb, (int)D, X_local, ldx, B.st, B.exa, B.slot, L,
                                                                 n_cand, first, B.dcol, B.bpot);
      GDR_LAUNCHED();
    }
    k_ppd_reduce<<<1, 1024, 0, s>>>(nb, L, n_cand, B.bpot, B.st, B.bprefix, my_b);
    GDR_LAUNCHED();
    int r = comm_allgather(comm, my_b, B.exb, 2 * L * 8, s);
    if (r) return r;
    k_ppd_choose<<<1, 256, 0, s>>>(L, n_cand, (int)D, B.exb, B.exa, B.slot, B.st, centers_out, ldc, indices_out_dev);
    GDR_LAUNCHED();
    return GDR_OK;
  };
  auto enqueue_round = [&]() -> int {
    k_ppd_pick<<<1, 1024, 0, s>>>(N_local, nb, (int)D, X_local, ldx, B.bpot, B.dcol, L, B.rand_dev, B.bprefix, B.st, my_a);
    GDR_LAUNCHED();
    int r = comm_allgather(comm, my_a, B.exa, B.slot, s);
    if (r) return r;
    return pass_and_choose(L, 0);
  };
  // start-up: centre 0 is the drawn row; closest = d(x, first)
  k_ppd_first<<<1, 256, 0, s>>>(init, first_center, N_local, (int)D, X_local, ldx, L, B.st, my_a);
  GDR_LAUNCHED();
  if ((rc = comm_allgather(comm, my_a, B.exa, B.slot, s))) return rc;
  if ((rc = pass_and_choose(1, 1))) return rc;
  // rounds 1 .. K-1; NCCL sets up its channels on the first collectives (not capturable): round 1 runs eagerly, round
  // 2 is captured and the graph replayed K - 2 times (each replay reads its round index from the device state)
  for (int64_t c = 1; c < K; ++c) {
    if (use_graph && c >= 2) {
      if (!G.exec) {
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
          int r = enqueue_round();
          cudaError_t e = cudaStreamEndCapture(s, &graph);
          if (r == GDR_OK && e == cudaSuccess && graph && cudaGraphInstantiate(&G.exec, graph, 0) == cudaSuccess) {
            cudaGraphDestroy(graph);
          } else {
            if (graph) cudaGraphDestroy(graph);
            G.exec = nullptr;
            cudaGetLastError();
            use_graph = false;   // capture not possible here: issue the launches directly
            if (r != GDR_OK) return r;
          }
        } else {
          cudaGetLastError();
          use_graph = false;
        }
      }
      if (use_graph && G.exec) {
        GDR_CUDA(cudaGraphLaunch(G.exec, s));
        count_launch(1);
        continue;
      }
    }
    if ((rc = enqueue_round())) return rc;
  }
  // the pageable host buffer must stay valid until the copy above has executed
  GDR_CUDA(cudaStreamSynchronize(s));
  if (s != caller) {
    GDR_CUDA(cudaEventRecord(G.ev, s));
    GDR_CUDA(cudaStreamWaitEvent(caller, G.ev, 0));
  }
  return GDR_OK;
}

}  // extern "C"
