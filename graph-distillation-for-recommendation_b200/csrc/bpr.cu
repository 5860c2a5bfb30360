// bpr.cu — BPR triplet sampling and the fused BPR loss + gradient of the refinement loop (distill_recsys.py:684-733:
// sample (user, positive, negative) triplets, propagate, BPR, backward, Adam).  With these two entry points and
// LightGCNPropagate a refinement step runs on the device without a host round trip.
//
// Sampler (k_bpr_sample, one thread per triplet).  Philox4x32-10 (Salmon et al., SC'11; the Random123 constants),
// key = (seed lo, seed hi), counter = (b, step, j, 0).  Call j = 0: user draw from (w1:w0), positive draw from (w3:w2);
// call j = 1: negative draw from (w1:w0).  A 64-bit word x becomes an integer in [0, n) as umulhi64(x, n).  The
// negative is the r-th item of the complement of the user's row: with sorted columns c_0 < ... < c_{k-1},
// neg = r + #{t : c_t - t <= r}, a binary search because c_t - t does not decrease.  That is the distribution of a
// rejection sampler with no loop that can fail to end.  Any (seed, step) can be regenerated on its own.
//
// Loss (k_bpr_score, one thread per triplet): x_b = dot(U[u], I[p]) - dot(U[u], I[n]), each dot a fp32 fmaf chain in
// column order over 128-bit row loads (a chain is sequential, so a thread owns a triplet: 32 independent chains per
// warp); l_b = softplus(-x_b) in the stable fp32 form, c_b = -sigmoid(-x_b) / B.  The loss is a fp64 sum of l_b with
// per-CTA partials in a fixed tree and a fixed-order combine (k_bpr_loss_combine).
//
// Gradients: gU[u] = sum c_b (I[p_b] - I[n_b]),  gI[j] = sum_{p_b = j} c_b U[u_b] - sum_{n_b = j} c_b U[u_b].
// k_bpr_score also writes the 3B slots (row key, slot = 3b + role), item keys offset by n_u; the stable radix sort
// (sort_pairs) groups them by row with slots ascending; k_bpr_heads lists the distinct rows; k_bpr_accumulate gives
// each row to a lane group that walks its slots in (b, role) order, float4 column chunks gathered with 128-bit loads
// and accumulated in fp64 registers (a row can take 2^21 terms of nearly one value, where a fp32 chain would drift by
// a few 1e-3), rounded once.  Rows with more than ACC_HEAVY slots are split over every group of the CTA in fixed
// chunks whose fp64 partials are added in chunk order.  No float atomics: the gradients are bit-identical from run
// to run.
#include "common.cuh"

namespace gdr {

constexpr int64_t BPR_MAX_BATCH = (1ll << 31) / 3;   // 3B slots must fit the sort's int32 positions
constexpr int BPR_THREADS = 256;
constexpr int ACC_THREADS = 256;
constexpr int ACC_SEGS_PER_CTA = 64;
constexpr int ACC_HEAVY = 2048;   // rows with more slots are split over the whole CTA
constexpr int ACC_WIN4 = 64;      // column window of one accumulate pass, in float4 (256 columns)

// ---------------------------------------------------------------------------------------------------------------
// Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// integer in [0, n) from a 64-bit word (bias <= n / 2^64)
__device__ __forceinline__ int64_t draw_below(uint32_t lo, uint32_t hi, int64_t n) {
  return (int64_t)__umul64hi(((uint64_t)hi << 32) | lo, (uint64_t)n);
}

__global__ void __launch_bounds__(BPR_THREADS) k_bpr_sample(int64_t B, uint32_t step, uint32_t k0, uint32_t k1,
                                                            const int32_t* __restrict__ rowptr,
                                                            const int32_t* __restrict__ colidx, int64_t n_items,
                                                            int64_t n_elig, const int32_t* __restrict__ elig,
                                                            int64_t* __restrict__ users, int64_t* __restrict__ pos,
                                                            int64_t* __restrict__ neg) {
  const int64_t b = (int64_t)blockIdx.x * BPR_THREADS + threadIdx.x;
  if (b >= B) return;
  const uint4 w = philox4x32_10(make_uint4((uint32_t)b, step, 0u, 0u), k0, k1);
  const uint4 v = philox4x32_10(make_uint4((uint32_t)b, step, 1u, 0u), k0, k1);
  const int32_t u = elig[draw_below(w.x, w.y, n_elig)];
  const int32_t s = rowptr[u], deg = rowptr[u + 1] - s;
  const int32_t p = colidx[s + draw_below(w.z, w.w, deg)];
  const int64_t r = draw_below(v.x, v.y, n_items - deg);
  int lo = 0, hi = deg;   // m = #{t : c_t - t <= r}
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (colidx[s + mid] - mid <= r) lo = mid + 1;
    else hi = mid;
  }
  users[b] = u;
  pos[b] = p;
  neg[b] = r + lo;
}

// ---------------------------------------------------------------------------------------------------------------
// loss terms, coefficients and slots
__device__ __forceinline__ float4 ld_row4(const float* row, int c4, int d) {
  float4 v = ldg_f4(row + 4 * c4);
  const int e = 4 * c4;
  if (e + 1 >= d) v.y = 0.f;
  if (e + 2 >= d) v.z = 0.f;
  if (e + 3 >= d) v.w = 0.f;
  return v;
}

__global__ void __launch_bounds__(BPR_THREADS) k_bpr_score(int64_t B, int64_t n_u, int64_t n_i, int d,
                                                           const float* __restrict__ U, int64_t ldu,
                                                           const float* __restrict__ I, int64_t ldi,
                                                           const int64_t* __restrict__ users,
                                                           const int64_t* __restrict__ pos,
                                                           const int64_t* __restrict__ neg, float* __restrict__ coef,
                                                           uint64_t* __restrict__ keys, uint32_t* __restrict__ slots,
                                                           double* __restrict__ part, int32_t* __restrict__ status) {
  __shared__ double s_w[BPR_THREADS / 32];
  const int64_t b = (int64_t)blockIdx.x * BPR_THREADS + threadIdx.x;
  double l = 0.0;
  if (b < B) {
    const int64_t u = users[b], p = pos[b], n = neg[b];
    const uint64_t bad = (uint64_t)(n_u + n_i);   // sorts after every row and is skipped by the accumulation
    uint64_t ku = bad, kp = bad, kn = bad;
    float c = 0.f;
    if (u < 0 || u >= n_u || p < 0 || p >= n_i || n < 0 || n >= n_i) {
      atomicOr(status, 1);
    } else {
      const float *ru = U + u * ldu, *rp = I + p * ldi, *rn = I + n * ldi;
      float sp = 0.f, sn = 0.f;
      const int F4 = (d + 3) >> 2;
      for (int c4 = 0; c4 < F4; ++c4) {
        const float4 a = ld_row4(ru, c4, d), x = ld_row4(rp, c4, d), y = ld_row4(rn, c4, d);
        sp = fmaf(a.x, x.x, sp);
        sn = fmaf(a.x, y.x, sn);
        sp = fmaf(a.y, x.y, sp);
        sn = fmaf(a.y, y.y, sn);
        sp = fmaf(a.z, x.z, sp);
        sn = fmaf(a.z, y.z, sn);
        sp = fmaf(a.w, x.w, sp);
        sn = fmaf(a.w, y.w, sn);
      }
      const float z = -__fsub_rn(sp, sn);
      if (!isfinite(z)) {
        atomicOr(status, 2);
      } else {
        const float e = expf(-fabsf(z));
        l = (double)__fadd_rn(fmaxf(z, 0.f), log1pf(e));                      // softplus(z)
        const float sig = z >= 0.f ? __fdiv_rn(1.f, __fadd_rn(1.f, e)) : __fdiv_rn(e, __fadd_rn(1.f, e));
        c = (float)(-(double)sig / (double)B);
        ku = (uint64_t)u;
        kp = (uint64_t)(n_u + p);
        kn = (uint64_t)(n_u + n);
      }
    }
    if (keys) {
      coef[b] = c;
      keys[3 * b] = ku;
      keys[3 * b + 1] = kp;
      keys[3 * b + 2] = kn;
      slots[3 * b] = (uint32_t)(3 * b);
      slots[3 * b + 1] = (uint32_t)(3 * b + 1);
      slots[3 * b + 2] = (uint32_t)(3 * b + 2);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
  if (lane_id() == 0) s_w[threadIdx.x >> 5] = l;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < BPR_THREADS / 32; ++w) s += s_w[w];
    part[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(256) k_bpr_loss_combine(int64_t nparts, const double* __restrict__ part, int64_t B,
                                                          float* __restrict__ loss) {
  __shared__ double s_w[8];
  double s = 0.0;
  for (int64_t k = threadIdx.x; k < nparts; k += 256) s += part[k];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane_id() == 0) s_w[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += s_w[w];
    loss[0] = (float)(t / (double)B);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// gradient accumulation over the sorted slots
__global__ void k_bpr_heads(int64_t M, const uint64_t* __restrict__ skeys, uint64_t n_rows, int32_t* __restrict__ seg,
                            int32_t* __restrict__ n_seg) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < M; k += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t key = skeys[k];
    if (key < n_rows && (k == 0 || skeys[k - 1] != key)) seg[atomicAdd(n_seg, 1)] = (int32_t)k;   // list order is free
  }
}

struct AccArgs {
  int64_t M, n_u;
  const uint64_t* skeys;
  const uint32_t* sslots;
  const float* coef;
  const int64_t *users, *pos, *neg;
  const float *U, *I;
  int64_t ldu, ldi;
  float *gU, *gI;
  int64_t ldgu, ldgi;
  int d;
  const int32_t* seg;
  const int32_t* n_seg;
};

struct Acc4 {
  double x, y, z, w;
};

// the group's fp64 fma chain over the slots [s, e) of row `key`, for its float4 chunks of the window
template <int LPR, int NCH>
__device__ __forceinline__ void acc_walk(const AccArgs& a, bool user_row, int s, int e, int col4_base, int c4_end,
                                         int gl, unsigned gmask, Acc4 (&acc)[NCH]) {
#pragma unroll
  for (int c = 0; c < NCH; ++c) acc[c] = Acc4{0.0, 0.0, 0.0, 0.0};
  for (int k = s; k < e; k += LPR) {
    const int my = k + gl;
    float cf = 0.f;
    int64_t ra = 0, rb = 0;
    if (my < e) {
      const uint32_t slot = a.sslots[my];
      const uint32_t b = slot / 3u, role = slot - 3u * b;
      cf = a.coef[b];
      if (role == 0) {
        ra = a.pos[b];
        rb = a.neg[b];
      } else {
        ra = a.users[b];
        if (role == 2) cf = -cf;
      }
    }
    const int cnt = min(LPR, e - k);
#pragma unroll 1
    for (int j = 0; j < cnt; ++j) {
      const double cj = (double)__shfl_sync(gmask, cf, j, LPR);
      const int64_t aj = __shfl_sync(gmask, ra, j, LPR);
      const int64_t bj = __shfl_sync(gmask, rb, j, LPR);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int c4 = col4_base + c * LPR + gl;
        if (c4 < c4_end) {
          Acc4 v;
          if (user_row) {   // I[p] - I[n] in fp64: exact
            const float4 x = ldg_f4(a.I + aj * a.ldi + 4 * c4), y = ldg_f4(a.I + bj * a.ldi + 4 * c4);
            v = Acc4{(double)x.x - y.x, (double)x.y - y.y, (double)x.z - y.z, (double)x.w - y.w};
          } else {
            const float4 x = ldg_f4(a.U + aj * a.ldu + 4 * c4);
            v = Acc4{x.x, x.y, x.z, x.w};
          }
          acc[c].x = fma(cj, v.x, acc[c].x);
          acc[c].y = fma(cj, v.y, acc[c].y);
          acc[c].z = fma(cj, v.z, acc[c].z);
          acc[c].w = fma(cj, v.w, acc[c].w);
        }
      }
    }
  }
}

__device__ __forceinline__ void acc_store(const AccArgs& a, uint64_t key, int c4, const Acc4& r) {
  const float4 v = make_float4((float)r.x, (float)r.y, (float)r.z, (float)r.w);
  float* out = key < (uint64_t)a.n_u ? (a.gU ? a.gU + (int64_t)key * a.ldgu : nullptr)
                                     : (a.gI ? a.gI + ((int64_t)key - a.n_u) * a.ldgi : nullptr);
  if (!out) return;
  const int e = 4 * c4;
  if (e + 3 < a.d) {
    *reinterpret_cast<float4*>(out + e) = v;
  } else {
    out[e] = v.x;
    if (e + 1 < a.d) out[e + 1] = v.y;
    if (e + 2 < a.d) out[e + 2] = v.z;
  }
}

__device__ __forceinline__ int seg_end(const AccArgs& a, int s, uint64_t key) {
  int lo = s + 1, hi = (int)a.M;   // first position past the run of `key`
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a.skeys[mid] == key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

template <int LPR, int NCH>
__global__ void __launch_bounds__(ACC_THREADS) k_bpr_accumulate(const AccArgs a, int col4_base, int c4_end) {
  constexpr int GROUPS = 32 / LPR;
  constexpr int NPART = (ACC_THREADS / 32) * GROUPS;
  __shared__ Acc4 s_part[NPART][LPR * NCH];
  __shared__ int s_heavy[ACC_SEGS_PER_CTA];
  __shared__ int s_next, s_nheavy;
  const int total = *a.n_seg;
  const int seg0 = blockIdx.x * ACC_SEGS_PER_CTA;
  if (seg0 >= total) return;
  const int nsegs = min(ACC_SEGS_PER_CTA, total - seg0);
  if (threadIdx.x == 0) {
    s_next = 0;
    s_nheavy = 0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int g = lane / LPR, gl = lane % LPR;
  const unsigned gmask = LPR == 32 ? 0xffffffffu : (((1u << LPR) - 1u) << (g * LPR));

  // ---- phase 1: a lane group per row; heavy rows are deferred ----
  while (true) {
    int r_base = 0;
    if (lane == 0) r_base = atomicAdd(&s_next, GROUPS);
    r_base = __shfl_sync(0xffffffffu, r_base, 0);
    if (r_base >= nsegs) break;
    const int r = r_base + g;
    int s = 0, e = 0;
    uint64_t key = 0;
    if (r < nsegs) {
      s = a.seg[seg0 + r];
      key = a.skeys[s];
      e = seg_end(a, s, key);
      if (e - s > ACC_HEAVY) {
        if (gl == 0) s_heavy[atomicAdd(&s_nheavy, 1)] = s;
        s = e = 0;
      }
    }
    Acc4 acc[NCH];
    acc_walk<LPR, NCH>(a, key < (uint64_t)a.n_u, s, e, col4_base, c4_end, gl, gmask, acc);
    if (e > s) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int c4 = col4_base + c * LPR + gl;
        if (c4 < c4_end) acc_store(a, key, c4, acc[c]);
      }
    }
  }
  __syncthreads();

  // ---- phase 2: each heavy row split over all lane groups in fixed chunks, partials added in chunk order ----
  const int nheavy = s_nheavy;
  const int part = (threadIdx.x >> 5) * GROUPS + g;
  for (int h = 0; h < nheavy; ++h) {
    const int hs = s_heavy[h];
    const uint64_t key = a.skeys[hs];
    const int he = seg_end(a, hs, key);
    int chunk = (he - hs + NPART - 1) / NPART;
    chunk = (chunk + LPR - 1) / LPR * LPR;
    const int cs = min(he, hs + part * chunk), ce = min(he, cs + chunk);
    Acc4 acc[NCH];
    acc_walk<LPR, NCH>(a, key < (uint64_t)a.n_u, cs, ce, col4_base, c4_end, gl, gmask, acc);
#pragma unroll
    for (int c = 0; c < NCH; ++c) s_part[part][c * LPR + gl] = acc[c];
    __syncthreads();
    for (int q = threadIdx.x; q < LPR * NCH; q += ACC_THREADS) {
      const int c4 = col4_base + q;   // q = c * LPR + gl
      if (c4 < c4_end) {
        Acc4 t = s_part[0][q];
        for (int p = 1; p < NPART; ++p) {
          const Acc4 v = s_part[p][q];
          t = Acc4{t.x + v.x, t.y + v.y, t.z + v.z, t.w + v.w};
        }
        acc_store(a, key, c4, t);
      }
    }
    __syncthreads();
  }
}

template <int LPR, int NCH>
static int launch_acc(const AccArgs& a, int64_t max_segs, int col4_base, int c4_end, cudaStream_t s) {
  const unsigned grid = (unsigned)std::max<int64_t>(1, cdiv(max_segs, ACC_SEGS_PER_CTA));
  k_bpr_accumulate<LPR, NCH><<<grid, ACC_THREADS, 0, s>>>(a, col4_base, c4_end);
  GDR_LAUNCHED();
  return GDR_OK;
}

static int acc_window(const AccArgs& a, int64_t max_segs, int base, int width, cudaStream_t s) {
  const int c4_end = base + width;
  if (width <= 4) return launch_acc<4, 1>(a, max_segs, base, c4_end, s);
  if (width <= 8) return launch_acc<8, 1>(a, max_segs, base, c4_end, s);
  if (width <= 16) return launch_acc<16, 1>(a, max_segs, base, c4_end, s);
  if (width <= 32) return launch_acc<32, 1>(a, max_segs, base, c4_end, s);
  return launch_acc<32, 2>(a, max_segs, base, c4_end, s);
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace gdr

extern "C" {

int gdr_bpr_sample(int64_t n_users, int64_t n_items, const int32_t* rowptr, const int32_t* colidx, int64_t n_eligible,
                   const int32_t* eligible, uint64_t seed, int64_t step, int64_t batch, int64_t* users_out,
                   int64_t* pos_out, int64_t* neg_out, gdr_stream_t stream) {
  GDR_CHECK_ARG(n_users >= 0 && n_items >= 0 && n_eligible >= 0 && batch >= 0, "bpr_sample: negative size");
  GDR_CHECK_ARG(n_users < INT32_MAX && n_items < INT32_MAX, "bpr_sample: sizes must fit int32");
  GDR_CHECK_ARG(n_eligible >= 1 && n_eligible <= n_users, "bpr_sample: n_eligible must lie in [1, n_users]");
  GDR_CHECK_ARG(n_items >= 2, "bpr_sample: a user with a positive and a negative needs n_items >= 2");
  GDR_CHECK_ARG(batch >= 1 && batch <= gdr::BPR_MAX_BATCH, "bpr_sample: batch must lie in [1, 2^31 / 3]");
  GDR_CHECK_ARG(step >= 0 && step <= (int64_t)UINT32_MAX, "bpr_sample: step must lie in [0, 2^32)");
  GDR_CHECK_ARG(rowptr && colidx && eligible && users_out && pos_out && neg_out, "bpr_sample: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  gdr::k_bpr_sample<<<(unsigned)gdr::cdiv(batch, gdr::BPR_THREADS), gdr::BPR_THREADS, 0, s>>>(
      batch, (uint32_t)step, (uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32), rowptr, colidx, n_items, n_eligible,
      eligible, users_out, pos_out, neg_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_bpr_loss_ws_bytes(int64_t batch, int64_t n_u, int64_t n_i) {
  if (batch < 1 || batch > gdr::BPR_MAX_BATCH || n_u < 0 || n_i < 0) return 256;
  const int64_t M = 3 * batch;
  return gdr::ws_need(batch, 4) + gdr::ws_need(M, 8) + gdr::ws_need(M, 4) +
         gdr::ws_need(gdr::cdiv(batch, gdr::BPR_THREADS), 8) + gdr::ws_need(std::min(M, n_u + n_i), 4) +
         gdr::ws_need(1, 4) + gdr::sort_pairs_ws_bytes(M) + 256;
}

int gdr_bpr_loss(int64_t batch, int64_t n_u, int64_t n_i, int64_t d, const float* U, int64_t ldu, const float* I,
                 int64_t ldi, const int64_t* users, const int64_t* pos, const int64_t* neg, float* loss_out,
                 float* gU, int64_t ldgu, float* gI, int64_t ldgi, int32_t* status_dev, void* ws, int64_t ws_bytes,
                 gdr_stream_t stream) {
  GDR_CHECK_ARG(batch >= 0 && n_u >= 0 && n_i >= 0 && d >= 0, "bpr_loss: negative size");
  GDR_CHECK_ARG(batch >= 1 && batch <= gdr::BPR_MAX_BATCH, "bpr_loss: batch must lie in [1, 2^31 / 3]");
  GDR_CHECK_ARG(n_u >= 1 && n_i >= 1 && d >= 1, "bpr_loss: n_u, n_i and d must be >= 1");
  GDR_CHECK_ARG(n_u + n_i < INT32_MAX && d < INT32_MAX, "bpr_loss: sizes must fit int32");
  GDR_CHECK_ARG(U && I && users && pos && neg && loss_out && status_dev && ws, "bpr_loss: null pointer");
  GDR_CHECK_ARG(ldu % 4 == 0 && ldu >= d && ldi % 4 == 0 && ldi >= d,
                "bpr_loss: ldu / ldi must be multiples of 4 and >= d");
  GDR_CHECK_ARG(gdr::aligned16(U) && gdr::aligned16(I), "bpr_loss: U and I must be 16-byte aligned");
  GDR_CHECK_ARG(!gU || (ldgu % 4 == 0 && ldgu >= d && gdr::aligned16(gU)),
                "bpr_loss: gU needs a 16-byte aligned base and ldgu a multiple of 4, >= d");
  GDR_CHECK_ARG(!gI || (ldgi % 4 == 0 && ldgi >= d && gdr::aligned16(gI)),
                "bpr_loss: gI needs a 16-byte aligned base and ldgi a multiple of 4, >= d");
  if (ws_bytes < gdr_bpr_loss_ws_bytes(batch, n_u, n_i)) {
    gdr::set_error("bpr_loss: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const bool grads = gU || gI;
  const int64_t M = 3 * batch;
  const int64_t nparts = gdr::cdiv(batch, gdr::BPR_THREADS);
  const int64_t max_segs = std::min(M, n_u + n_i);
  gdr::Workspace W(ws, ws_bytes);
  float* coef = W.take<float>(batch);
  uint64_t* keys = W.take<uint64_t>(M);
  uint32_t* slots = W.take<uint32_t>(M);
  double* part = W.take<double>(nparts);
  int32_t* seg = W.take<int32_t>(max_segs);
  int32_t* n_seg = W.take<int32_t>(1);
  void* sort_ws = W.take<char>(gdr::sort_pairs_ws_bytes(M));
  gdr::k_bpr_score<<<(unsigned)nparts, gdr::BPR_THREADS, 0, s>>>(batch, n_u, n_i, (int)d, U, ldu, I, ldi, users, pos,
                                                                 neg, grads ? coef : nullptr, grads ? keys : nullptr,
                                                                 grads ? slots : nullptr, part, status_dev);
  GDR_LAUNCHED();
  gdr::k_bpr_loss_combine<<<1, 256, 0, s>>>(nparts, part, batch, loss_out);
  GDR_LAUNCHED();
  if (!grads) return GDR_OK;

  if (gU) GDR_CUDA(cudaMemset2DAsync(gU, ldgu * sizeof(float), 0, d * sizeof(float), n_u, s));
  if (gI) GDR_CUDA(cudaMemset2DAsync(gI, ldgi * sizeof(float), 0, d * sizeof(float), n_i, s));
  int key_bits = 1;
  while ((1ll << key_bits) <= n_u + n_i) ++key_bits;   // the key n_u + n_i marks a skipped triplet
  uint64_t* skeys = keys;
  uint32_t* sslots = slots;
  int rc = gdr::sort_pairs_ex(M, key_bits, keys, slots, sort_ws, gdr::sort_pairs_ws_bytes(M), &skeys, &sslots, s);
  if (rc) return rc;
  GDR_CUDA(cudaMemsetAsync(n_seg, 0, sizeof(int32_t), s));
  gdr::k_bpr_heads<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>(gdr::cdiv(M, 256), gdr::kSMs * 16)), 256, 0, s>>>(
      M, skeys, (uint64_t)(n_u + n_i), seg, n_seg);
  GDR_LAUNCHED();
  gdr::AccArgs a;
  a.M = M;
  a.n_u = n_u;
  a.skeys = skeys;
  a.sslots = sslots;
  a.coef = coef;
  a.users = users;
  a.pos = pos;
  a.neg = neg;
  a.U = U;
  a.I = I;
  a.ldu = ldu;
  a.ldi = ldi;
  a.gU = gU;
  a.gI = gI;
  a.ldgu = ldgu;
  a.ldgi = ldgi;
  a.d = (int)d;
  a.seg = seg;
  a.n_seg = n_seg;
  const int F4 = (int)gdr::cdiv(d, 4);
  for (int base = 0; base < F4; base += gdr::ACC_WIN4) {
    rc = gdr::acc_window(a, max_segs, base, std::min(gdr::ACC_WIN4, F4 - base), s);
    if (rc) return rc;
  }
  return GDR_OK;
}

}  // extern "C"
