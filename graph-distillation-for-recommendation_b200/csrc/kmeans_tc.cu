// kmeans_tc.cu — stage 3 E-step on the 5th-gen tensor cores (precision_mode 1).
//
//   d(i,j) = |c_j|^2 - 2 x_i . c_j          (sklearn/_k_means_lloyd.pyx:196-213)
//
// X.C^T is the only dense contraction of the distillation core.  Inputs are fp32 and
// the contract is "labels bit-exact wherever the distance margin exceeds 1e-6", so the
// GEMM runs as 3xTF32:  x = x_hi + x_lo, c = c_hi + c_lo (each a TF32 value),
//   x.c ~= x_lo.c_hi + x_hi.c_lo + x_hi.c_hi        (fp32 accumulation in TMEM)
// and every row whose best/second-best margin falls inside a proven error band is
// re-scored by the exact fp32 SIMT kernel of kmeans.cu (screen-then-refine).
//
// Kernel anatomy (persistent, one CTA per SM, 192 threads):
//   warp 0   TMA producer   cp.async.bulk.tensor.2d, 128B-swizzled K-blocks of 32 floats
//   warp 1   MMA issuer     tcgen05.mma.cta_group::1.kind::tf32, M=128 N=128 K=8, one lane
//   warps 2-5 epilogue      tcgen05.ld 32x32b.x32 -> +|c|^2 -> running (best, second, argmin)
//   * the 128-row X tile (hi and lo) stays resident in shared memory while all centre
//     tiles stream past it through a 3-stage mbarrier ring;
//   * two 128-column fp32 accumulators in TMEM, so the argmin epilogue of centre tile t
//     overlaps the MMAs of tile t+1.
#include "tc_common.cuh"
#include <cuda.h>
#include <string.h>

namespace gdr {

int launch_row_sqnorm(int64_t K, int D, const float* C, int64_t ldc, float* out, cudaStream_t s);
int launch_assign_simt_rows(int64_t max_rows, int64_t K, int64_t D, const float* X, int64_t ldx,
                            const float* CT, int64_t ldct, const float* cnorm, const int32_t* rows,
                            const int32_t* n_rows_dev, unsigned long long* packed, int32_t* labels,
                            const int32_t* labels_prev, int32_t* n_changed, float* best_out, cudaStream_t s);

constexpr int TC_BN = 128;        // centres per tile (UMMA N)
constexpr int TC_MAX_KB = 4;      // D padded <= 128
constexpr int TC_BAR_KB = 5;      // K-blocks of the augmented first-level operand (D + 4 padded <= 160)
constexpr int TC_STAGES = 3;      // centre-tile ring
constexpr int TC_THREADS = 320;      // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quarter)
constexpr int TC_EPI_THREADS = 256;
constexpr int TC_TMEM_COLS = 256;                 // two 128-column accumulators
// error band of the 3xTF32 screen, relative to |x_i| * max_j |c_j| (see DESIGN.md)
constexpr float TC_BAND = 3.0517578125e-05f;      // 2^-15
// first-level screen: one TF32 product over the augmented operands of k_split_tf32; its error radius is built
// from the measured rounding residuals |x - tf32(x)|, |c - tf32(c)| (see k_split_tf32 / k_tc_select1).
static const int32_t* g_last_count1 = nullptr;   // device counter of the last two-level run (debug read-back)
int g_tc_gate = 1;      // gdr_debug_set("tc_gate", v): first-level epilogue gate — 0 off (exact running top-2 over all columns), otherwise (default) gate on the running best
extern int64_t g_topk_last_overflow;   // topk.cu
extern int64_t g_topk_condensed_last_fallback;   // topk_condensed.cu
int g_tc_cand = 1;      // gdr_debug_set("tc_cand", v): second level of the default two-level screen — 1 (default) seeded candidate pass + exact re-score of the candidates, 0 3xTF32 + exact re-score over all centres
int g_tc_cand_cap = 0;  // gdr_debug_set("tc_cand_cap", v): candidate list capacity per row and column half, 1..TC_CAND_CAP (0: TC_CAND_CAP)
static const int32_t* g_last_cand = nullptr;     // candidate counters of the last run that used the candidate level (debug read-back)
int g_tc_screen = 0;    // gdr_debug_set("tc_screen", v): 0 auto, 1 direct 3xTF32, >= 2 two-level

// smallest TF32 value >= v (v finite); used where a bound must not shrink under the operand rounding
__device__ __forceinline__ float tf32_up(float v) {
  uint32_t u = __float_as_uint(v);
  if (v >= 0.f) u = (u + 0x1FFFu) & ~0x1FFFu;   // magnitude up
  else u &= ~0x1FFFu;                           // magnitude down
  return __uint_as_float(u);
}

// aug_mode 1 (rows of X) / 2 (centres): additionally write the first-level operand row
//   aug[r] = [ tf32(x_0..x_{D-1}), e1, e2, p, q, 0... ]   (Dp1 = D + 4 rounded up to 32 floats)
//   X rows : e1 = up(|dx|),  e2 = up(|x|),             p = q = 1           (dx = x - tf32(x), exact in fp32)
//   centres: e1 = up(|c|),   e2 = up(|dc| + 2^-15|c|), p + q >= w = -|c|^2/2 (1 - 2^-15) in two TF32 values
//            (padding centres: p = -1e30)                       (the e's carry a 1.001 factor for the fp32 norms)
// so that ONE TF32 GEMM over the augmented rows yields the SCORE
//   s_ij = x^.c^ + E_ij - |c|^2/2 + slack,   E_ij = |dx_i||c_j| + |x_i||dc_j| + 2^-15|x_i||c_j|
// E_ij bounds the error of the rounded dot product (|x^.c^ - x.c| <= |dx||c| + |x^||dc|) plus the TMEM
// accumulation error, with the MEASURED rounding residuals of this row and this centre instead of the worst
// case 2^-11 — about 2.4x tighter.  s_ij >= t_ij = x.c - |c|^2/2 (= -d_ij / 2) and s_ij - t_ij <= 2 rad_ij.
__global__ void __launch_bounds__(256) k_split_tf32(int64_t rows, int64_t rows_pad, int D, int Dp,
                                                    const float* __restrict__ X, int64_t ldx,
                                                    float* __restrict__ hi, float* __restrict__ lo,
                                                    float* __restrict__ norm_out /*|x| per row, nullable*/,
                                                    float* __restrict__ xt /*[Dp][rows_pad] transposed copy, nullable*/,
                                                    float* __restrict__ sqnorm_out /*|x|^2, +inf on padding rows, nullable*/,
                                                    float* __restrict__ aug /*nullable*/, int Dp1, int aug_mode,
                                                    float* __restrict__ dnorm_out /*|x - tf32(x)|, with aug*/) {
  // one warp per row
  int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= rows_pad) return;
  float s = 0.f, sd = 0.f;
  for (int c = lane_id(); c < Dp; c += 32) {
    float x = (r < rows && c < D) ? X[r * ldx + c] : 0.f;
    float h = to_tf32(x);
    float dx = __fsub_rn(x, h);
    float l = to_tf32(dx);
    hi[r * Dp + c] = h;
    lo[r * Dp + c] = l;
    if (xt) xt[(int64_t)c * rows_pad + r] = x;
    if (aug && c < D) aug[r * Dp1 + c] = h;
    s = fmaf(x, x, s);
    sd = fmaf(dx, dx, sd);
  }
  // same per-lane fmaf order and xor-shuffle tree as k_row_sqnorm: bit-identical |row|^2
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    sd += __shfl_xor_sync(0xffffffffu, sd, o);
  }
  if (lane_id() == 0) {
    if (norm_out && r < rows) norm_out[r] = sqrtf(s);
    if (sqnorm_out) sqnorm_out[r] = r < rows ? s : INFINITY;   // padding rows can never win the argmin
  }
  if (aug) {
    const float nrm = sqrtf(s), dn = sqrtf(sd);
    float e1, e2, p, q;
    if (aug_mode == 1) {
      e1 = tf32_up(1.001f * dn);
      e2 = tf32_up(1.001f * nrm);
      p = q = 1.f;
    } else if (r < rows) {
      e1 = tf32_up(1.001f * nrm);
      e2 = tf32_up(1.001f * (dn + 3.0517578125e-05f * nrm));
      const float w = -0.5f * s * (1.f - 3.0517578125e-05f);
      p = to_tf32(w);
      q = tf32_up(__fsub_rn(w, p));
    } else {
      e1 = e2 = q = 0.f;
      p = to_tf32(-1e30f);
    }
    if (lane_id() == 0 && dnorm_out) dnorm_out[r] = r < rows ? dn : 0.f;
    for (int c = D + lane_id(); c < Dp1; c += 32)
      aug[r * Dp1 + c] = c == D ? e1 : (c == D + 1 ? e2 : (c == D + 2 ? p : (c == D + 3 ? q : 0.f)));
  }
}

// cmax = max_j |c_j| over the real centres, |c_j| per centre (0 on padding); also resets the list lengths and counters
__global__ void __launch_bounds__(1024) k_cnorm_finish(int64_t K, int64_t Kp, const float* __restrict__ cnorm,
                                                       const float* __restrict__ cdnorm /*nullable*/,
                                                       float* __restrict__ cnorm_sqrt, float* __restrict__ cmax /*[2]*/,
                                                       int32_t* __restrict__ amb_count, int32_t* __restrict__ count1,
                                                       int32_t* __restrict__ zero /*nullable*/, int n_zero) {
  __shared__ float s_m[1024];
  __shared__ float s_d[1024];
  float m = 0.f, md = 0.f;
  if (threadIdx.x == 0) {
    if (amb_count) amb_count[0] = 0;
    if (count1) count1[0] = 0;
  }
  if (zero && (int)threadIdx.x < n_zero) zero[threadIdx.x] = 0;
  for (int64_t j = threadIdx.x; j < Kp; j += 1024) {
    const float c2 = j < K ? cnorm[j] : 0.f;
    m = fmaxf(m, c2);
    if (cdnorm && j < K) md = fmaxf(md, cdnorm[j]);
    cnorm_sqrt[j] = sqrtf(c2);
  }
  s_m[threadIdx.x] = m;
  s_d[threadIdx.x] = md;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_m[threadIdx.x] = fmaxf(s_m[threadIdx.x], s_m[threadIdx.x + o]);
      s_d[threadIdx.x] = fmaxf(s_d[threadIdx.x], s_d[threadIdx.x + o]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    cmax[0] = sqrtf(s_m[0]);
    cmax[1] = s_d[0];
  }
}

// ---------------------------------------------------------------------------------
// the tensor-core kernel
// ---------------------------------------------------------------------------------
// NPASS = 3: 3xTF32 (x_lo.c_hi + x_hi.c_lo + x_hi.c_hi), outputs (best, second, argmin) of the distances.
// NPASS = 1: the first-level screen — ONE TF32 product per K-step over the augmented operands of
//            k_split_tf32 (aug_mode 1 / 2), whose accumulator is directly the score s_ij >= x_i.c_j - |c_j|^2/2;
//            the epilogue is a bare running (max, second max, argmax) — no norm add, no per-centre loads —
//            and k_tc_select1 accepts the row when s_best - s_second exceeds twice the error radius.
// BN      = centres per accumulator tile (UMMA N): 128 (NPASS 3) or 256 (NPASS 1); a CTA tile holds TC_BM = 128 rows.
constexpr int TC_MAX_STAGES = 8;
constexpr int TC_SMEM_LIMIT = 227 * 1024;

// First-level epilogue gate.  k_tc_select1 only needs to know (a) the best score of a row and (b) whether ANY other
// centre comes within tol(i, best) of it, and tol(i, j) <= tolmax_i = the same expression with max_j |c_j|, max_j |dc_j|.
// So the running top-2 has to look only at chunks that hold a score within tolmax_i of a lower bound of the row's
// final best: the running best (k_tc_cand starts from the row's level-1 best instead).  A warp (32 rows) then takes
// the per-element path for a few percent of the 8-column chunks instead of ~a third.
struct TcGate {
  const float* xnorm;    // |x_i|           (nullptr: gate off, exact running top-2 over all columns)
  const float* xdnorm;   // |x_i - tf32(x_i)|
  const float* cscal;    // [0] = max_j |c_j|, [1] = max_j (|c_j - tf32(c_j)|)
  const float* seed;     // k_tc_cand only: the row's level-1 best (negated score)
  float band;
};

// First-level epilogue step: running (max, second max, argmax) over one 32-column chunk of scores (kept negated).  A row's
// running top-2 changes only ~2 ln(K) times, so most chunks hold nothing below any lane's bound: the four 8-column maxima
// are formed as independent trees, ONE warp vote on their maximum dismisses the whole chunk, and only otherwise do the
// 8-column votes and the per-element path run (in column order with the running bounds: the result does not depend on
// the filtering).  The per-warp dependency chain of a dismissed chunk is one tree + one vote instead of four.
__device__ __forceinline__ void epi_chunk32(const uint32_t (&v)[32], int jbase, bool chunk_skip, bool gated, float tolmax,
                                            float& limt, float& best, float& second, int& bidx) {
  float m8[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int u0 = 8 * q;
    const float m = fmaxf(fmaxf(__uint_as_float(v[u0]), __uint_as_float(v[u0 + 1])),
                          fmaxf(__uint_as_float(v[u0 + 2]), __uint_as_float(v[u0 + 3])));
    m8[q] = fmaxf(m, fmaxf(fmaxf(__uint_as_float(v[u0 + 4]), __uint_as_float(v[u0 + 5])),
                           fmaxf(__uint_as_float(v[u0 + 6]), __uint_as_float(v[u0 + 7]))));
  }
  const float m32 = fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3]));
  if (chunk_skip && !__any_sync(0xffffffffu, -m32 < (gated ? limt : second))) return;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (!chunk_skip || __any_sync(0xffffffffu, -m8[q] < (gated ? limt : second))) {
#pragma unroll
      for (int u = 8 * q; u < 8 * q + 8; ++u) {
        const float d = -__uint_as_float(v[u]);
        second = fminf(second, fmaxf(d, best));
        bidx = d < best ? jbase + u : bidx;
        best = fminf(best, d);
      }
      if (gated) limt = fminf(limt, best + tolmax);
    }
  }
}

// slack of the candidate pass's starting limit over the level-1 best it is seeded with: the two passes multiply the
// same operands but may accumulate differently
__device__ __forceinline__ float tc_cand_slack(float xn, float cm) { return 3.814697265625e-06f * (xn * cm + cm * cm); }

// Candidate-pass epilogue step (k_tc_cand): as epi_chunk32 with the gate always on, plus every per-element score below
// the limit in force is appended to this (row, column half)'s list.  The limit only falls, from seed + slack + tolmax
// to best-so-far + tolmax, so every centre with d < min(seed + slack, final best) + tolmax is recorded.
__device__ __forceinline__ void epi_chunk32_rec(const uint32_t (&v)[32], int jbase, float tolmax, float& limt,
                                                float& best, int& n, int2* rec, int cap) {
  float m8[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int u0 = 8 * q;
    const float m = fmaxf(fmaxf(__uint_as_float(v[u0]), __uint_as_float(v[u0 + 1])),
                          fmaxf(__uint_as_float(v[u0 + 2]), __uint_as_float(v[u0 + 3])));
    m8[q] = fmaxf(m, fmaxf(fmaxf(__uint_as_float(v[u0 + 4]), __uint_as_float(v[u0 + 5])),
                           fmaxf(__uint_as_float(v[u0 + 6]), __uint_as_float(v[u0 + 7]))));
  }
  const float m32 = fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3]));
  if (!__any_sync(0xffffffffu, -m32 < limt)) return;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (__any_sync(0xffffffffu, -m8[q] < limt)) {
#pragma unroll
      for (int u = 8 * q; u < 8 * q + 8; ++u) {
        const float d = -__uint_as_float(v[u]);
        if (d < limt) {
          if (n < cap) rec[n] = make_int2(jbase + u, __float_as_int(d));
          ++n;
        }
        best = fminf(best, d);
      }
      limt = fminf(limt, best + tolmax);
    }
  }
}

template <int NPASS, int BN>
struct TcCfg {
  static constexpr int kXCopies = NPASS == 3 ? 2 : 1;                        // hi (+ lo) copy of the row tile
  static constexpr int kStageBytes = kXCopies * BN * TC_BK * 4;              // one centre K-block (hi [+ lo])
  static constexpr int kTmemCols = 2 * BN;                                   // two accumulators
  static constexpr int kTail = 512 /*barriers*/ + 1536 /*epilogue merge buffer*/;
  __host__ __device__ static constexpr int x_hi(int kb) { return kb * TC_KBLK_BYTES; }
  __host__ __device__ static constexpr int x_lo(int nkb, int kb) { return (nkb + kb) * TC_KBLK_BYTES; }   // NPASS 3
  __host__ __device__ static constexpr int x_bytes(int nkb) { return kXCopies * nkb * TC_KBLK_BYTES; }
  __host__ __device__ static constexpr int c_stage(int nkb, int s) { return x_bytes(nkb) + s * kStageBytes; }
  // as many centre stages as fit beside the resident rows (<= TC_MAX_STAGES)
  __host__ __device__ static constexpr int stages(int nkb) {
    int n = (TC_SMEM_LIMIT - 1024 /*alignment slack*/ - kTail - x_bytes(nkb)) / kStageBytes;
    return n > TC_MAX_STAGES ? TC_MAX_STAGES : n;
  }
  __host__ __device__ static constexpr int bars(int nkb) { return c_stage(nkb, stages(nkb)); }
  __host__ __device__ static constexpr int total(int nkb) { return bars(nkb) + kTail + 1024; }
};

// Candidate recording of the seeded first-level pass (k_tc_cand): per (compacted row, column half) the centres whose
// negated score is below the row's limit, in column order; count[] may exceed cap (overflow: the row takes the fallback).
struct TcCand {
  int2* list;       // [rows][2][cap] (centre, negated score bits)
  int32_t* count;   // [rows][2] centres met below the limit per column half
  int cap;
};

// The kernel body, shared by the first level / 3xTF32 level (k_assign_tc) and the seeded candidate pass (k_tc_cand,
// REC = true).  REC: the gate is always on, the limit starts at the row's seed and every per-element score below it
// is recorded; best / second / argmin are not written.
template <int NPASS, int BN, bool REC>
__device__ __forceinline__ void assign_tc_body(const CUtensorMap& map_xhi, const CUtensorMap& map_xlo,
                                               const CUtensorMap& map_chi, const CUtensorMap& map_clo, int64_t N_host,
                                               const int32_t* __restrict__ n_rows_dev, int D, int n_col_tiles, int nkb,
                                               const float* __restrict__ cnorm, float* __restrict__ best_out,
                                               float* __restrict__ second_out, int32_t* __restrict__ idx_out,
                                               TcGate gate, TcCand cand) {
  using Cfg = TcCfg<NPASS, BN>;
  static_assert(Cfg::kTmemCols <= 512, "tile plan");
  static_assert(!REC || NPASS == 1, "candidate recording: first-level shape only");
  const int S = Cfg::stages(nkb);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::bars(nkb));
  uint64_t* x_full = bars;                              // [TC_BAR_KB]
  uint64_t* x_empty = bars + TC_BAR_KB;                 // [TC_BAR_KB]
  uint64_t* c_full = bars + 2 * TC_BAR_KB;              // [TC_MAX_STAGES]
  uint64_t* c_empty = c_full + TC_MAX_STAGES;           // [TC_MAX_STAGES]
  uint64_t* t_full = c_empty + TC_MAX_STAGES;           // [2]
  uint64_t* t_empty = t_full + 2;                       // [2]
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(t_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t N = n_rows_dev ? (int64_t)n_rows_dev[0] : N_host;
  const int n_row_tiles = (int)((N + TC_BM - 1) / TC_BM);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < TC_BAR_KB; ++i) {
      mbar_init(&x_full[i], 1);
      mbar_init(&x_empty[i], 1);
    }
    for (int i = 0; i < TC_MAX_STAGES; ++i) {
      mbar_init(&c_full[i], 1);
      mbar_init(&c_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&t_full[i], 1);
      mbar_init(&t_empty[i], TC_EPI_THREADS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_base_smem)),
                 "r"(Cfg::kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;

  // Producer and MMA warps keep WARP-UNIFORM control flow and let one elected lane issue the asynchronous
  // instructions.  (Running the loops inside `if (lane == 0)` makes every descriptor a per-thread value: the
  // compiler then wraps each UTCHMMA in an ELECT / R2UR.BROADCAST waterfall and the issue path — ~350 cycles per
  // MMA, measured with clock64 inside the kernel — becomes the bottleneck instead of the tensor pipe, which runs a
  // 128 x 256 x 8 TF32 MMA in 171 cycles.)
  if (warp == 0) {
    // ================= TMA producer =================
    uint32_t tile_it = 0;
    int s = 0;
    uint32_t ph = 0;   // ring position and its phase, advanced incrementally (no division on the issue path)
    for (int rt = blockIdx.x; rt < n_row_tiles; rt += gridDim.x, ++tile_it) {
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&x_empty[kb], (tile_it & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&x_full[kb], Cfg::kXCopies * TC_KBLK_BYTES);
          tma_load_2d(smem + Cfg::x_hi(kb), &map_xhi, kb * TC_BK, rt * TC_BM, &x_full[kb]);
          if (NPASS == 3) tma_load_2d(smem + Cfg::x_lo(nkb, kb), &map_xlo, kb * TC_BK, rt * TC_BM, &x_full[kb]);
        }
        __syncwarp();
      }
      for (int ct = 0; ct < n_col_tiles; ++ct) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&c_empty[s], ph ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&c_full[s], Cfg::kStageBytes);
            uint8_t* dst = smem + Cfg::c_stage(nkb, s);
            tma_load_2d(dst, &map_chi, kb * TC_BK, ct * BN, &c_full[s]);
            if (NPASS == 3) tma_load_2d(dst + BN * TC_BK * 4, &map_clo, kb * TC_BK, ct * BN, &c_full[s]);
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
    // ================= MMA issuer =================
    // The per-K-block issue path is kept to a handful of uniform instructions (descriptor = base + offset, ring
    // position advanced incrementally, K steps unrolled): at ~128 cycles per 128 x 256 x 8 MMA the tensor pipe
    // drains a K-block in ~500 cycles, and a path with integer divisions and descriptor rebuilds took longer
    // than that (measured: 250 cycles per MMA with every wait removed, 128 on a bare stream of MMAs).
    constexpr uint32_t idesc = umma_idesc_tf32(TC_BM, BN);
    uint32_t tile_it = 0, g = 0;
    int s = 0;
    uint32_t ph = 0;
    const uint64_t dx0 = umma_desc_sw128(smem_u32(smem));                                  // row tile, K-block 0
    const uint64_t dc0 = umma_desc_sw128(smem_u32(smem + Cfg::c_stage(nkb, 0)));             // centre stage 0
    constexpr uint64_t kKb = TC_KBLK_BYTES >> 4, kStage = Cfg::kStageBytes >> 4, kLo = (uint64_t)(BN * TC_BK * 4) >> 4;
    for (int rt = blockIdx.x; rt < n_row_tiles; rt += gridDim.x, ++tile_it) {
      for (int ct = 0; ct < n_col_tiles; ++ct, ++g) {
        const uint32_t a = g & 1, aph = (g >> 1) & 1;
        mbar_wait(&t_empty[a], aph ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + a * BN;
        const bool last_ct = ct == n_col_tiles - 1;
        for (int kb = 0; kb < nkb; ++kb) {
          if (ct == 0) mbar_wait(&x_full[kb], tile_it & 1);
          mbar_wait(&c_full[s], ph);
          tc_fence_after();
          const uint64_t d_chi = dc0 + (uint64_t)s * kStage;
          // K = 8 steps that still hold real columns (the rest of the 32-float block is zero padding)
          const int ksteps = min(TC_BK / 8, (D - kb * TC_BK + 7) >> 3);
          if (elect_one()) {
            if (NPASS == 3) {
              const uint64_t d_xhi = dx0 + (uint64_t)kb * kKb;
              const uint64_t d_xlo = dx0 + (uint64_t)(nkb + kb) * kKb;
              const uint64_t d_clo = d_chi + kLo;
              if (ksteps == 4) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);  // 32 bytes per K = 8 step
                  // small terms first, the dominant hi*hi product last
                  tc_mma_tf32(tmem_d, d_xlo + adv, d_chi + adv, idesc, (kb | k) != 0);
                  tc_mma_tf32(tmem_d, d_xhi + adv, d_clo + adv, idesc, 1);
                  tc_mma_tf32(tmem_d, d_xhi + adv, d_chi + adv, idesc, 1);
                }
              } else {
                for (int k = 0; k < ksteps; ++k) {
                  const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);
                  tc_mma_tf32(tmem_d, d_xlo + adv, d_chi + adv, idesc, (kb | k) != 0);
                  tc_mma_tf32(tmem_d, d_xhi + adv, d_clo + adv, idesc, 1);
                  tc_mma_tf32(tmem_d, d_xhi + adv, d_chi + adv, idesc, 1);
                }
              }
            } else {
              const uint64_t d_x = dx0 + (uint64_t)kb * kKb;
              if (ksteps == 4) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);
                  tc_mma_tf32(tmem_d, d_x + adv, d_chi + adv, idesc, (kb | k) != 0);
                }
              } else {
                for (int k = 0; k < ksteps; ++k) {
                  const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);
                  tc_mma_tf32(tmem_d, d_x + adv, d_chi + adv, idesc, (kb | k) != 0);
                }
              }
            }
            tc_commit(&c_empty[s]);                          // frees the centre stage
            if (last_ct) tc_commit(&x_empty[kb]);            // X K-block no longer needed
            if (kb == nkb - 1) tc_commit(&t_full[a]);        // accumulator ready
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
    // ================= epilogue: 8 warps; warp w reads TMEM lanes [32*(w%4), +32).  The two warps of a lane
    //                    quarter take one column half of the accumulator each (merged at the end of the row
    //                    tile); two warps per SM sub-partition hide each other's tcgen05.ld and min-chain
    //                    latencies =================
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;
    constexpr int COLS = BN / 2;                                      // columns per warp and accumulator
    float* s_merge = reinterpret_cast<float*>(tmem_base_smem + 4);   // [3][128] exchange buffer after the barriers
    const int rl = quarter * 32 + lane;
    const bool chunk_skip = REC || n_col_tiles * BN >= 4096;   // the vote only pays once most chunks can be skipped
    uint32_t g = 0;
    for (int rt = blockIdx.x; rt < n_row_tiles; rt += gridDim.x) {
      const int64_t row = (int64_t)rt * TC_BM + rl;
      // NPASS 3: (best, second) = two smallest distances; NPASS 1: two largest scores, stored negated so that
      // both variants share the min-tracking code and the merge below
      float best = INFINITY, second = INFINITY;
      int bidx = 0;
      // gate (NPASS 1): limt = (lower bound of the final best, as a negated score) + tolmax_i; a chunk whose smallest
      // negated score is not below limt for any lane cannot hold the row's best nor anything within tol of it
      float tolmax = 0.f, limt = INFINITY;
      const bool gated = REC || (NPASS == 1 && chunk_skip && gate.xnorm != nullptr);
      if (gated) {
        const float xn = row < N ? gate.xnorm[row] : 0.f, xd = row < N ? gate.xdnorm[row] : 0.f;
        const float cm = gate.cscal[0], cdm = gate.cscal[1];
        tolmax = 1.001f * (2.02f * (xd * cm + xn * (cdm + 3.0517578125e-05f * cm) + 1.52587890625e-05f * cm * cm) +
                           gate.band * xn * cm + 9.5367431640625e-07f * (xn * cm + cm * cm));
        if constexpr (REC) limt = row < N ? gate.seed[row] + tc_cand_slack(xn, cm) + tolmax : -INFINITY;   // padding rows record nothing
      }
      int n_rec = 0;   // REC: this (row, column half)'s list
      int2* rec = nullptr;
      if constexpr (REC) rec = cand.list + ((int64_t)row * 2 + half) * cand.cap;
      for (int ct = 0; ct < n_col_tiles; ++ct, ++g) {
        const uint32_t a = g & 1, aph = (g >> 1) & 1;
        mbar_wait(&t_full[a], aph);
        tc_fence_after();
#pragma unroll 1
        for (int h2 = 0; h2 < COLS / 64; ++h2) {
          const int col0 = half * COLS + h2 * 64;   // column inside the centre tile
          const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + a * BN + col0;
          uint32_t v[2][32];
          tc_ld_32x32(taddr, v[0]);
          tc_ld_32x32(taddr + 32, v[1]);          // both chunks in flight before the first is consumed
          tc_wait_ld();
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const int jbase = ct * BN + col0 + c * 32;
            if constexpr (REC) {
              epi_chunk32_rec(v[c], jbase, tolmax, limt, best, n_rec, rec, cand.cap);
            } else if (NPASS == 1) {
              epi_chunk32(v[c], jbase, chunk_skip, gated, tolmax, limt, best, second, bidx);
            } else {
              const float4* cn4 = reinterpret_cast<const float4*>(cnorm + jbase);
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 cn = __ldg(cn4 + q);
                const float cc[4] = {cn.x, cn.y, cn.z, cn.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const float d = fmaf(-2.f, __uint_as_float(v[c][q * 4 + u]), cc[u]);
                  second = fminf(second, fmaxf(d, best));
                  bidx = d < best ? jbase + q * 4 + u : bidx;   // strict '<': first minimum wins
                  best = fminf(best, d);
                }
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(&t_empty[a]);
      }
      if constexpr (REC) {
        if (row < N) cand.count[row * 2 + half] = n_rec;
      } else {
        // merge the two column halves of each row: lower columns win ties
        if (half == 1) {
          s_merge[rl] = best;
          s_merge[128 + rl] = second;
          reinterpret_cast<int*>(s_merge)[256 + rl] = bidx;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_THREADS) : "memory");
        if (half == 0) {
          const float b1 = s_merge[rl], s1 = s_merge[128 + rl];
          const int i1 = reinterpret_cast<int*>(s_merge)[256 + rl];
          const float nb = fminf(best, b1);
          const float ns = fminf(fminf(second, s1), fmaxf(best, b1));
          const int ni = b1 < best ? i1 : bidx;
          if (row < N) {
            best_out[row] = nb;
            second_out[row] = ns;
            idx_out[row] = ni;
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_THREADS) : "memory");
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::kTmemCols) : "memory");
  }
}

template <int NPASS, int BN>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_assign_tc(const __grid_constant__ CUtensorMap map_xhi, const __grid_constant__ CUtensorMap map_xlo,
            const __grid_constant__ CUtensorMap map_chi, const __grid_constant__ CUtensorMap map_clo,
            int64_t N_host, const int32_t* __restrict__ n_rows_dev /*nullable: row count on the device*/,
            int D /*contraction width incl. the 3 augmented columns for NPASS 1*/, int n_col_tiles, int nkb,
            const float* __restrict__ cnorm /*NPASS 3: |c_j|^2*/,
            float* __restrict__ best_out, float* __restrict__ second_out, int32_t* __restrict__ idx_out, TcGate gate) {
  assign_tc_body<NPASS, BN, false>(map_xhi, map_xlo, map_chi, map_clo, N_host, n_rows_dev, D, n_col_tiles, nkb, cnorm,
                                   best_out, second_out, idx_out, gate, TcCand{nullptr, nullptr, 0});
}

// Seeded candidate pass over the compacted undecided rows: k_assign_tc<1, 256>'s schedule and arithmetic on the
// compacted augmented rows (row count on the device), with gate.seed / xnorm / xdnorm indexed by compacted slot.
__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc_cand(const __grid_constant__ CUtensorMap map_x1, const __grid_constant__ CUtensorMap map_c1, int64_t N_host,
          const int32_t* __restrict__ n_rows_dev, int D, int n_col_tiles, int nkb, TcGate gate, TcCand cand) {
  assign_tc_body<1, 256, true>(map_x1, map_x1, map_c1, map_c1, N_host, n_rows_dev, D, n_col_tiles, nkb, nullptr,
                               nullptr, nullptr, nullptr, gate, cand);
}

// first-level decision.  best = -s_idx, second = -s_second (negated scores of the first-level kernel).  With
//   E_ij   = |dx_i||c_j| + |x_i|(|dc_j| + 2^-15|c_j|)   (operand rounding incl. the dx.dc cross term; TMEM
//            accumulation <= (D + 4) 2^-23 |x||c| <= 2^-15.9 |x||c| for D <= 128)
//   rad_ij = 1.01 (E_ij + 2^-16 |c_j|^2)   and   t_ij <= s_ij <= t_ij + 2 rad_ij
// (t = true score x.c - |c|^2/2; the factor 1.01 covers the 1.001 factors and the round-ups inside the operands),
// s_idx - s_second > 2 rad_idx implies t_idx > t_j for every other centre: idx is the unique exact argmin.
// eta = 2^-15 |x| cmax keeps the margin above the rounding noise of the exact fp32 kernel (same term as the
// second-level band), 2^-21 |s| covers the last accumulator rounding.  Everything else goes to the
// second-level list (3xTF32 on the compacted rows).
__global__ void __launch_bounds__(256) k_tc_select1(int64_t N, const float* __restrict__ best,
                                                    const float* __restrict__ second,
                                                    const int32_t* __restrict__ idx,
                                                    const float* __restrict__ xnorm, const float* __restrict__ xdnorm,
                                                    const float* __restrict__ cnorm,
                                                    const float* __restrict__ cnorm_sqrt,
                                                    const float* __restrict__ cdnorm,
                                                    const float* __restrict__ cmax, float band,
                                                    int32_t* __restrict__ labels,
                                                    const int32_t* __restrict__ labels_prev,
                                                    int32_t* __restrict__ n_changed,
                                                    int32_t* __restrict__ list1, int32_t* __restrict__ count1) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int changed = 0;
  if (i < N) {
    const int l = idx[i];
    const float b = best[i], s2 = second[i], xn = xnorm[i], cr = cnorm_sqrt[l];
    const float E = xdnorm[i] * cr + xn * (cdnorm[l] + 3.0517578125e-05f * cr);
    // s2 = +inf: the gated epilogue met no other centre within tolmax_i >= tol of the best -> decided
    const float tol = 2.02f * (E + 1.52587890625e-05f * cnorm[l]) + band * xn * cmax[0] +
                      4.76837158e-07f * fmaxf(fabsf(b), s2 == INFINITY ? 0.f : fabsf(s2));
    const bool ambiguous = !(s2 - b > tol);   // also catches NaN / inf - inf
    if (ambiguous) {
      list1[atomicAdd(count1, 1)] = (int32_t)i;
    } else {
      labels[i] = l;
      if (labels_prev && labels_prev[i] != l) changed = 1;
    }
  }
  if (n_changed) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
    if (lane_id() == 0 && changed) atomicAdd(n_changed, changed);
  }
}

// compact the hi/lo operand rows (and |x|) of the second-level list; one warp per listed row
__global__ void __launch_bounds__(256) k_tc_gather(const int32_t* __restrict__ list1, const int32_t* __restrict__ count1,
                                                   int Dp, const float* __restrict__ hi, const float* __restrict__ lo,
                                                   const float* __restrict__ xnorm, float* __restrict__ ghi,
                                                   float* __restrict__ glo, float* __restrict__ gnorm) {
  const int n = count1[0];
  const int wpg = (gridDim.x * blockDim.x) >> 5;
  const int Dp4 = Dp >> 2;
  for (int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; slot < n; slot += wpg) {
    const int64_t r = list1[slot];
    const float4* h = reinterpret_cast<const float4*>(hi + r * Dp);
    const float4* l = reinterpret_cast<const float4*>(lo + r * Dp);
    float4* gh = reinterpret_cast<float4*>(ghi + (int64_t)slot * Dp);
    float4* gl = reinterpret_cast<float4*>(glo + (int64_t)slot * Dp);
    for (int c = lane_id(); c < Dp4; c += 32) {
      gh[c] = __ldg(h + c);
      gl[c] = __ldg(l + c);
    }
    if (lane_id() == 0) gnorm[slot] = xnorm[r];
  }
}

// ---------------------------------------------------------------------------------
// second level on candidate centres (the default two-level screen)
// ---------------------------------------------------------------------------------
// For every row level 1 left undecided, k_tc_cand re-runs the first-level product over the compacted rows with the
// limit fixed from the start at seed + slack + tolmax_i (seed = the row's level-1 best, as a negated score) and records
// each centre j met below the limit in force; k_tc_cand_resolve then decides the row on those centres alone.
//
// Why that is exact.  Let b = the smallest recorded negated score, l its centre (lowest index on ties), and tol(i, l)
// the expression of k_tc_select1 (with 2^-21 max(|b|, |d_j|) as its last term).  For a centre j with
// d_j - b > tol(i, l), i.e. s_l - s_j > tol(i, l), the inequality k_tc_select1 relies on gives, for this pair,
//   t_j <= s_j < s_l - 2 rad_l - eta <= t_l - eta,
// so j loses to l in the exact fp32 chain, ties included: such a j is excluded.  Every other centre is recorded:
// the limit in force is min(seed + slack, running best) + tolmax_i >= b + tolmax_i whenever b <= seed + slack (then b
// is also the row's true minimum, which the limit always admits), and tol(i, .) < tolmax_i.  k_tc_cand_resolve checks
// b <= seed + slack itself — it does not assume that the two TF32 passes produce the same bits — and sends a row that
// fails it, a row with an empty list and a row whose list overflowed in either column half to the fallback list,
// which takes the 3xTF32 level and the exact re-score over all centres as before.  The kept centres are re-scored with
// the exact fp32 chain of k_assign_simt / k_refine_partial (ed_chain) and the (distance, index) minimum of rf_pack.

// compact the first-level operand rows, |x|, |x - tf32(x)| and the level-1 best (the seed) of the listed rows
__global__ void __launch_bounds__(256) k_tc_gather_cand(const int32_t* __restrict__ list1, const int32_t* __restrict__ count1,
                                                        int Dp1, const float* __restrict__ x1, const float* __restrict__ xnorm,
                                                        const float* __restrict__ xdnorm, const float* __restrict__ best,
                                                        float* __restrict__ gx1, float* __restrict__ gnorm,
                                                        float* __restrict__ gdnorm, float* __restrict__ gseed) {
  const int n = count1[0];
  const int wpg = (gridDim.x * blockDim.x) >> 5;
  for (int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; slot < n; slot += wpg) {
    const int64_t r = list1[slot];
    const float4* a = reinterpret_cast<const float4*>(x1 + r * Dp1);
    float4* g = reinterpret_cast<float4*>(gx1 + (int64_t)slot * Dp1);
    for (int c = lane_id(); c < (Dp1 >> 2); c += 32) g[c] = __ldg(a + c);
    if (lane_id() == 0) {
      gnorm[slot] = xnorm[r];
      gdnorm[slot] = xdnorm[r];
      gseed[slot] = best[r];
    }
  }
}

// cand_ctr: [0] fallback rows, [1] candidate rows whose exact margin lies inside the band, [2] rows decided on their
// candidates, [3] rows whose list overflowed, [4..5] recorded entries (uint64)
constexpr int TC_CAND_CTRS = 6;

// one warp per compacted row: merge the two half lists, filter, exact re-score of the kept centres, label.  The row and
// up to RS_BATCH kept centre rows are staged in shared memory by the whole warp (coalesced, all loads in flight), then
// one lane per kept centre runs the exact chain from there.
constexpr int RS_BATCH = 8;
constexpr int RS_LD = 132;   // floats per staged row (D <= 128; rows 4 banks apart)
__global__ void __launch_bounds__(256) k_tc_cand_resolve(
    const int32_t* __restrict__ list1, const int32_t* __restrict__ count1, const int2* __restrict__ cand,
    const int32_t* __restrict__ cand_n, int cap, const float* __restrict__ gseed, const float* __restrict__ gnorm,
    const float* __restrict__ gdnorm, int D, const float* __restrict__ X, int64_t ldx, const float* __restrict__ C,
    int64_t ldc, const float* __restrict__ cnorm, const float* __restrict__ cnorm_sqrt, const float* __restrict__ cdnorm,
    const float* __restrict__ cmax, float band, int32_t* __restrict__ labels, const int32_t* __restrict__ labels_prev,
    int32_t* __restrict__ n_changed, int32_t* __restrict__ list2, int32_t* __restrict__ ctr) {
  __shared__ __align__(16) float s_rows[8][(1 + RS_BATCH) * RS_LD];   // per warp: [0] x row, [1 + b] kept centre b
  __shared__ int s_j[8][32];                                          // per warp: kept centres
  const int n = count1[0];
  const int lane = lane_id();
  const int wpg = (gridDim.x * blockDim.x) >> 5;
  float* sx = s_rows[threadIdx.x >> 5];
  float* sc = sx + RS_LD;
  int* sj = s_j[threadIdx.x >> 5];
  const int D4 = (D + 3) >> 2;   // rows of X and C are 16-byte aligned with ld % 4 == 0
  int changed = 0;
  for (int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; slot < n; slot += wpg) {
    const int32_t row = list1[slot];
    const int n0 = cand_n[2 * slot], n1 = cand_n[2 * slot + 1];
    bool fallback = n0 > cap || n1 > cap || n0 + n1 == 0;
    // lane holds merged entries lane and lane + 32 (half 0 first; 2 cap <= 64)
    unsigned long long key[2] = {~0ull, ~0ull};
    if (!fallback) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int e = lane + 32 * h;
        if (e < n0 + n1) {
          const int2 p = e < n0 ? cand[(int64_t)(2 * slot) * cap + e] : cand[(int64_t)(2 * slot + 1) * cap + (e - n0)];
          key[h] = rf_pack(__int_as_float(p.y), p.x);
        }
      }
    }
    if (lane == 0 && !fallback) atomicAdd(reinterpret_cast<unsigned long long*>(ctr + 4), (unsigned long long)(n0 + n1));
    unsigned long long kmin = key[0] < key[1] ? key[0] : key[1];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, kmin, o);
      kmin = other < kmin ? other : kmin;
    }
    const int l = (int)(unsigned)(kmin & 0xffffffffull);
    const float b = rf_unpack(kmin);
    const float xn = gnorm[slot], cm = cmax[0];
    if (!fallback && !(b <= gseed[slot] + tc_cand_slack(xn, cm))) fallback = true;   // also catches NaN
    if (fallback) {
      if (lane == 0) {
        list2[atomicAdd(ctr, 1)] = row;
        if (n0 > cap || n1 > cap) atomicAdd(ctr + 3, 1);
      }
      continue;
    }
    // tol(i, l) of k_tc_select1 without its last term, which is taken per candidate below
    const float cr = cnorm_sqrt[l];
    const float E = gdnorm[slot] * cr + xn * (cdnorm[l] + 3.0517578125e-05f * cr);
    const float tol0 = 2.02f * (E + 1.52587890625e-05f * cnorm[l]) + band * xn * cm;
    bool keep[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float d = rf_unpack(key[h]);
      const float tol = tol0 + 4.76837158e-07f * fmaxf(fabsf(b), fabsf(d));
      keep[h] = key[h] != ~0ull && !(d - b > tol);   // an excluded centre loses to l in the exact chain
    }
    const unsigned m0 = __ballot_sync(0xffffffffu, keep[0]), m1 = __ballot_sync(0xffffffffu, keep[1]);
    const unsigned lt = (1u << lane) - 1u;
    __syncwarp();   // the previous row's chains have read sx / sc / sj
    if (keep[0]) sj[__popc(m0 & lt)] = (int)(unsigned)(key[0] & 0xffffffffull);
    if (keep[1]) sj[__popc(m0) + __popc(m1 & lt)] = (int)(unsigned)(key[1] & 0xffffffffull);
    for (int q = lane; q < D4; q += 32)
      reinterpret_cast<float4*>(sx)[q] = __ldg(reinterpret_cast<const float4*>(X + (int64_t)row * ldx) + q);
    const int nk = __popc(m0) + __popc(m1);
    unsigned long long k1 = ~0ull, k2 = ~0ull;   // two smallest exact keys of this lane
    for (int t0 = 0; t0 < nk; t0 += RS_BATCH) {
      const int nb = min(RS_BATCH, nk - t0);
      __syncwarp();
      for (int bb = 0; bb < nb; ++bb) {
        const float4* c4 = reinterpret_cast<const float4*>(C + (int64_t)sj[t0 + bb] * ldc);
        for (int q = lane; q < D4; q += 32) reinterpret_cast<float4*>(sc + bb * RS_LD)[q] = __ldg(c4 + q);
      }
      __syncwarp();
      if (lane < nb) {
        const int j = sj[t0 + lane];
        const float* c = sc + lane * RS_LD;
        float acc = 0.f;
#pragma unroll 4
        for (int k = 0; k < D; ++k) acc = ed_chain(acc, sx[k], c[k]);
        const float dist = ed_finish(acc, cnorm[j]);
        const unsigned long long kk = dist == dist ? rf_pack(dist, j) : ~0ull;
        if (kk < k1) {
          k2 = k1;
          k1 = kk;
        } else if (kk < k2) {
          k2 = kk;
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long o1 = __shfl_xor_sync(0xffffffffu, k1, o), o2 = __shfl_xor_sync(0xffffffffu, k2, o);
      const unsigned long long lo = k1 < o1 ? k1 : o1, hi = k1 < o1 ? o1 : k1;
      const unsigned long long s2 = k2 < o2 ? k2 : o2;
      k1 = lo;
      k2 = hi < s2 ? hi : s2;
    }
    if (k1 == ~0ull) {   // no finite exact distance: leave the row to the full exact path
      if (lane == 0) list2[atomicAdd(ctr, 1)] = row;
      continue;
    }
    if (lane == 0) {
      const int lab = (int)(unsigned)(k1 & 0xffffffffull);
      labels[row] = lab;
      if (labels_prev && labels_prev[row] != lab) ++changed;
      const float d1 = rf_unpack(k1), d2 = k2 == ~0ull ? INFINITY : rf_unpack(k2);
      if (!(d2 - d1 > band * xn * cm)) atomicAdd(ctr + 1, 1);
      atomicAdd(ctr + 2, 1);
    }
  }
  if (n_changed) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
    if (lane == 0 && changed) atomicAdd(n_changed, changed);
  }
}

// *dst += *src (the candidate rows' band count joins the re-scored rows' count in *n_refined)
__global__ void k_add_i32(int32_t* __restrict__ dst, const int32_t* __restrict__ src) { *dst += *src; }

// second-level decision on the compacted rows (slot -> row through list1): same band as k_tc_select
__global__ void __launch_bounds__(256) k_tc_select2(const int32_t* __restrict__ list1, const int32_t* __restrict__ count1,
                                                    const float* __restrict__ best, const float* __restrict__ second,
                                                    const int32_t* __restrict__ idx, const float* __restrict__ gnorm,
                                                    const float* __restrict__ cmax, float band,
                                                    int32_t* __restrict__ labels, const int32_t* __restrict__ labels_prev,
                                                    int32_t* __restrict__ n_changed, int32_t* __restrict__ amb_list,
                                                    int32_t* __restrict__ amb_count,
                                                    unsigned long long* __restrict__ amb_packed) {
  const int n = count1[0];
  const int stride = gridDim.x * blockDim.x;
  int changed = 0;
  for (int slot = blockIdx.x * blockDim.x + threadIdx.x; slot < n; slot += stride) {
    const int32_t i = list1[slot];
    const float tol = band * gnorm[slot] * cmax[0];
    const float b = best[slot], s2 = second[slot];
    if (!(s2 - b > tol)) {
      const int a = atomicAdd(amb_count, 1);
      amb_list[a] = i;
      amb_packed[a] = ~0ull;
    } else {
      const int l = idx[slot];
      labels[i] = l;
      if (labels_prev && labels_prev[i] != l) ++changed;
    }
  }
  if (n_changed) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
    if (lane_id() == 0 && changed) atomicAdd(n_changed, changed);
  }
}

// rows whose margin is inside the error band go to the exact re-score list
__global__ void __launch_bounds__(256) k_tc_select(int64_t N, const float* __restrict__ best,
                                                   const float* __restrict__ second,
                                                   const int32_t* __restrict__ idx,
                                                   const float* __restrict__ xnorm,
                                                   const float* __restrict__ cmax, float band,
                                                   int32_t* __restrict__ labels,
                                                   const int32_t* __restrict__ labels_prev,
                                                   int32_t* __restrict__ n_changed, float* __restrict__ best_out,
                                                   int32_t* __restrict__ amb_list, int32_t* __restrict__ amb_count,
                                                   unsigned long long* __restrict__ amb_packed) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int changed = 0;
  if (i < N) {
    float tol = band * xnorm[i] * cmax[0];
    float b = best[i], s2 = second[i];
    bool ambiguous = !(s2 - b > tol);  // also catches NaN / inf - inf
    if (ambiguous) {
      int slot = atomicAdd(amb_count, 1);
      amb_list[slot] = (int32_t)i;
      amb_packed[slot] = ~0ull;   // identity of the re-score kernel's atomicMin
    } else {
      int l = idx[i];
      labels[i] = l;
      if (best_out) best_out[i] = b;
      if (labels_prev && labels_prev[i] != l) changed = 1;
    }
  }
  if (n_changed) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
    if (lane_id() == 0 && changed) atomicAdd(n_changed, changed);
  }
}

// ---------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------
static inline int dpad(int64_t D) { return (int)align_up(D, TC_BK); }
constexpr int TC_AUG = 4;   // augmented columns of the first-level operands
static inline int dpad1(int64_t D) { return (int)align_up(D + TC_AUG, TC_BK); }
constexpr int TC_KPAD = 256;   // centres padded to the widest accumulator tile
// candidates recorded per row and column half.  tools/cand_estimate.py, config-E-shaped data after one Lloyd update,
// 20 000-row sample: 3.7 % (D = 100) / 3.0 % (D = 47) of the rows undecided, 2.2 recorded per row on average, at most 4
// in one column half (profiles/r3_cand_estimate_configE.txt): 16 leaves ample room at 256 bytes of list per row
constexpr int TC_CAND_CAP = 16;
static_assert(TC_CAND_CAP <= 32, "k_tc_cand_resolve holds the two half lists in two entries per lane");

int64_t kmeans_tc_xsplit_bytes(int64_t N, int64_t D) {
  return 2 * ws_need(N * dpad(D), 4) + 2 * ws_need(N, 4) + ws_need(N * dpad1(D), 4) + 256;
}

struct XSplit {
  float *hi, *lo, *norm, *x1, *dnorm;
};
static XSplit carve_xsplit(void* buf, int64_t N, int64_t D) {
  Workspace W(buf, kmeans_tc_xsplit_bytes(N, D));
  XSplit x;
  int Dp = dpad(D);
  x.hi = W.take<float>(N * Dp);
  x.lo = W.take<float>(N * Dp);
  x.norm = W.take<float>(N);
  x.x1 = W.take<float>(N * dpad1(D));
  x.dnorm = W.take<float>(N);
  return x;
}

int kmeans_tc_prepare(int64_t N, int64_t D, const float* X, int64_t ldx, void* xsplit, cudaStream_t s) {
  XSplit x = carve_xsplit(xsplit, N, D);
  k_split_tf32<<<(unsigned)cdiv(N * 32, 256), 256, 0, s>>>(N, N, (int)D, dpad(D), X, ldx, x.hi, x.lo, x.norm, nullptr,
                                                          nullptr, x.x1, dpad1(D), 1, x.dnorm);
  GDR_LAUNCHED();
  return GDR_OK;
}

// two-level screen (1xTF32 over all rows, 3xTF32 over the compacted undecided rows) pays off once the
// row tiles fill the machine a few times over; below that the direct 3xTF32 kernel is one launch instead of five
static bool tc_two_level(int64_t N, bool want_best) {
  if (want_best) return false;              // best_out is defined by the 3xTF32 / exact distances
  if (g_tc_screen == 1) return false;
  if (g_tc_screen >= 2) return true;
  return cdiv(N, TC_BM) >= 4 * kSMs;
}

int64_t kmeans_assign_tc_ws_bytes(int64_t N, int64_t K, int64_t D) {
  int Dp = dpad(D);
  int64_t Kp = align_up(K, TC_KPAD);
  return 3 * ws_need(Kp * Dp, 4) /*c_hi, c_lo, c^T*/ + ws_need(Kp * dpad1(D), 4) /*augmented centres*/ +
         3 * ws_need(Kp, 4) /*|c|^2, |c|, |c - tf32(c)|*/ + 256 /*cmax*/ +
         3 * ws_need(N, 4) /*best, second, idx*/ + ws_need(N, 4) /*amb list*/ + ws_need(N, 8) /*amb packed*/ +
         256 /*amb count*/ + ws_need(N, 4) /*second-level list*/ + 256 /*its count*/ +
         2 * ws_need(N * Dp, 4) + ws_need(N, 4) /*compacted hi, lo, |x|*/ + 2 * ws_need(N, 4) /*compacted |dx|, seed*/ +
         ws_need(2 * N, 4) + ws_need(2 * N * TC_CAND_CAP, 8) /*candidate counts, lists*/ + ws_need(N, 4) /*fallback list*/ +
         256 /*candidate counters*/ + 256;
}

// D_eff = contraction width (D, or D + 4 for the augmented first level); nkb = its 32-float K-blocks
template <int NPASS, int BN>
static int launch_assign_tc(const CUtensorMap& m_xhi, const CUtensorMap& m_xlo, const CUtensorMap& m_chi,
                            const CUtensorMap& m_clo, int64_t N_max, const int32_t* n_rows_dev, int D_eff, int64_t Kp,
                            int nkb, const float* cnorm, float* best, float* second, int32_t* idx, cudaStream_t s,
                            TcGate gate = TcGate{nullptr, nullptr, nullptr, nullptr, 0.f}) {
  using Cfg = TcCfg<NPASS, BN>;
  static PerDevice<bool> attr_set_dev;
  bool& attr_set = attr_set_dev.get();
  if (!attr_set) {
    GDR_CUDA(cudaFuncSetAttribute(k_assign_tc<NPASS, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_LIMIT));
    attr_set = true;
  }
  int sms = kSMs;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  const int64_t tiles = cdiv(N_max, TC_BM);
  const int grid = (int)(tiles < sms ? tiles : sms);
  k_assign_tc<NPASS, BN><<<grid, TC_THREADS, Cfg::total(nkb), s>>>(m_xhi, m_xlo, m_chi, m_clo, N_max, n_rows_dev, D_eff,
                                                                   (int)(Kp / BN), nkb, cnorm, best, second, idx, gate);
  GDR_LAUNCHED();
  return GDR_OK;
}

static int launch_tc_cand(const CUtensorMap& m_x1, const CUtensorMap& m_c1, int64_t N_max, const int32_t* n_rows_dev,
                          int D_eff, int64_t Kp, int nkb, TcGate gate, TcCand cand, cudaStream_t s) {
  using Cfg = TcCfg<1, 256>;
  static PerDevice<bool> attr_set_dev;
  bool& attr_set = attr_set_dev.get();
  if (!attr_set) {
    GDR_CUDA(cudaFuncSetAttribute(k_tc_cand, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_LIMIT));
    attr_set = true;
  }
  int sms = kSMs;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  const int64_t tiles = cdiv(N_max, TC_BM);
  const int grid = (int)(tiles < sms ? tiles : sms);
  k_tc_cand<<<grid, TC_THREADS, Cfg::total(nkb), s>>>(m_x1, m_c1, N_max, n_rows_dev, D_eff, (int)(Kp / 256), nkb, gate, cand);
  GDR_LAUNCHED();
  return GDR_OK;
}

static int kmeans_assign_tc_run(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx, const void* xsplit,
                                const float* C, int64_t ldc, int32_t* labels, const int32_t* labels_prev,
                                int32_t* n_changed_dev, float* best_out, int32_t* n_refined_dev, void* ws,
                                int64_t ws_bytes, cudaStream_t s) {
  if (D > TC_MAX_KB * TC_BK) {
    set_error("kmeans_assign(tc): D=%lld > %d is not supported by the tensor-core path", (long long)D,
              TC_MAX_KB * TC_BK);
    return GDR_EUNSUPPORTED;
  }
  if (N >= (1ll << 31) - TC_BM || K >= (1ll << 31) - TC_KPAD) {
    set_error("kmeans_assign(tc): N or K exceeds int32 tile coordinates");
    return GDR_ERANGE;
  }
  const int Dp = dpad(D), Dp1 = dpad1(D);
  const int nkb = Dp / TC_BK, nkb1 = Dp1 / TC_BK;
  const int64_t Kp = align_up(K, TC_KPAD);
  XSplit xs = carve_xsplit(const_cast<void*>(xsplit), N, D);
  Workspace W(ws, ws_bytes);
  float* c_hi = W.take<float>(Kp * Dp);
  float* c_lo = W.take<float>(Kp * Dp);
  float* c_t = W.take<float>(Kp * Dp);   // fp32 centres transposed [Dp][Kp] for the re-score kernel
  float* c1 = W.take<float>(Kp * Dp1);   // augmented first-level centres
  float* cnorm = W.take<float>(Kp);
  float* cnorm_sqrt = W.take<float>(Kp);
  float* cdnorm = W.take<float>(Kp);
  float* cmax = W.take<float>(2);   // [max |c|, max |c - tf32(c)|]
  float* best = W.take<float>(N);
  float* second = W.take<float>(N);
  int32_t* idx = W.take<int32_t>(N);
  int32_t* amb_list = W.take<int32_t>(N);
  unsigned long long* amb_packed = W.take<unsigned long long>(N);
  int32_t* amb_count_ws = W.take<int32_t>(1);
  int32_t* list1 = W.take<int32_t>(N);
  int32_t* count1 = W.take<int32_t>(1);
  float* g_hi = W.take<float>(N * Dp);
  float* g_lo = W.take<float>(N * Dp);
  float* g_norm = W.take<float>(N);
  float* g_dnorm = W.take<float>(N);
  float* g_seed = W.take<float>(N);
  int32_t* cand_n = W.take<int32_t>(2 * N);
  int2* cand_list = W.take<int2>(2 * N * TC_CAND_CAP);
  int32_t* list2 = W.take<int32_t>(N);
  int32_t* cand_ctr = W.take<int32_t>(TC_CAND_CTRS);
  int32_t* amb_count = n_refined_dev ? n_refined_dev : amb_count_ws;
  if (!W.ok()) {
    set_error("kmeans_assign(tc): workspace too small");
    return GDR_EWORKSPACE;
  }
  const bool two_level = tc_two_level(N, best_out != nullptr);
  // per-iteration centre preparation: split, norms, padding (+ the augmented rows of the first level)
  k_split_tf32<<<(unsigned)cdiv(Kp * 32, 256), 256, 0, s>>>(K, Kp, (int)D, Dp, C, ldc, c_hi, c_lo, nullptr, c_t, cnorm,
                                                           two_level ? c1 : nullptr, Dp1, 2, cdnorm);
  GDR_LAUNCHED();
  int rc;
  k_cnorm_finish<<<1, 1024, 0, s>>>(K, Kp, cnorm, two_level ? cdnorm : nullptr, cnorm_sqrt, cmax, amb_count, count1,
                                    two_level ? cand_ctr : nullptr, TC_CAND_CTRS);
  GDR_LAUNCHED();

  CUtensorMap m_xhi, m_xlo, m_chi, m_clo;
  if ((rc = make_map(&m_chi, c_hi, Kp, Dp, 128))) return rc;
  if ((rc = make_map(&m_clo, c_lo, Kp, Dp, 128))) return rc;

  if (!two_level) {
    if ((rc = make_map(&m_xhi, xs.hi, N, Dp, TC_BM))) return rc;
    if ((rc = make_map(&m_xlo, xs.lo, N, Dp, TC_BM))) return rc;
    {
      ProfileScope prof(PROF_ASSIGN, s);
      if ((rc = launch_assign_tc<3, 128>(m_xhi, m_xlo, m_chi, m_clo, N, nullptr, (int)D, Kp, nkb, cnorm, best, second,
                                         idx, s)))
        return rc;
    }
    k_tc_select<<<(unsigned)cdiv(N, 256), 256, 0, s>>>(N, best, second, idx, xs.norm, cmax, TC_BAND, labels,
                                                      labels_prev, n_changed_dev, best_out, amb_list, amb_count,
                                                      amb_packed);
    GDR_LAUNCHED();
  } else {
    // the profile scope spans the whole tensor-core screen: level 1, decision, compaction, level 2
    ProfileScope prof(PROF_ASSIGN, s);
    CUtensorMap m_x1, m_c1;
    if ((rc = make_map(&m_x1, xs.x1, N, Dp1, TC_BM))) return rc;
    if ((rc = make_map(&m_c1, c1, Kp, Dp1, 256))) return rc;
    TcGate gate{nullptr, nullptr, nullptr, nullptr, TC_BAND};
    if (g_tc_gate) {
      gate.xnorm = xs.norm;
      gate.xdnorm = xs.dnorm;
      gate.cscal = cmax;
    }
    if ((rc = launch_assign_tc<1, 256>(m_x1, m_x1, m_c1, m_c1, N, nullptr, (int)D + TC_AUG, Kp, nkb1, cnorm, best, second, idx,
                                       s, gate)))
      return rc;
    const bool cand_level = g_tc_cand != 0;   // second level on candidate centres
    g_last_count1 = count1;
    k_tc_select1<<<(unsigned)cdiv(N, 256), 256, 0, s>>>(N, best, second, idx, xs.norm, xs.dnorm, cnorm, cnorm_sqrt,
                                                       cdnorm, cmax, TC_BAND, labels, labels_prev, n_changed_dev,
                                                       list1, count1);
    GDR_LAUNCHED();
    // rows (and their count, on the device) that take the 3xTF32 level over all centres
    const int32_t* list_f = list1;
    const int32_t* count_f = count1;
    g_last_cand = cand_level ? cand_ctr : nullptr;
    if (cand_level) {
      float* g_x1 = g_hi;   // N Dp1 <= 2 N Dp floats: g_hi and g_lo are free until the fallback gathers into them
      k_tc_gather_cand<<<4 * kSMs, 256, 0, s>>>(list1, count1, Dp1, xs.x1, xs.norm, xs.dnorm, best, g_x1, g_norm, g_dnorm,
                                                g_seed);
      GDR_LAUNCHED();
      CUtensorMap m_gx1;
      if ((rc = make_map(&m_gx1, g_x1, N, Dp1, TC_BM))) return rc;
      const int cap = g_tc_cand_cap > 0 ? std::min(g_tc_cand_cap, TC_CAND_CAP) : TC_CAND_CAP;
      if ((rc = launch_tc_cand(m_gx1, m_c1, N, count1, (int)D + TC_AUG, Kp, nkb1, TcGate{g_norm, g_dnorm, cmax, g_seed, TC_BAND},
                               TcCand{cand_list, cand_n, cap}, s)))
        return rc;
      k_tc_cand_resolve<<<4 * kSMs, 256, 0, s>>>(list1, count1, cand_list, cand_n, cap, g_seed, g_norm, g_dnorm, (int)D, X, ldx,
                                                 C, ldc, cnorm, cnorm_sqrt, cdnorm, cmax, TC_BAND, labels, labels_prev,
                                                 n_changed_dev, list2, cand_ctr);
      GDR_LAUNCHED();
      list_f = list2;
      count_f = cand_ctr;   // [0]: fallback rows
    }
    k_tc_gather<<<4 * kSMs, 256, 0, s>>>(list_f, count_f, Dp, xs.hi, xs.lo, xs.norm, g_hi, g_lo, g_norm);
    GDR_LAUNCHED();
    CUtensorMap m_ghi, m_glo;
    if ((rc = make_map(&m_ghi, g_hi, N, Dp, TC_BM))) return rc;
    if ((rc = make_map(&m_glo, g_lo, N, Dp, TC_BM))) return rc;
    if ((rc = launch_assign_tc<3, 128>(m_ghi, m_glo, m_chi, m_clo, N, count_f, (int)D, Kp, nkb, cnorm, best, second, idx,
                                       s)))
      return rc;
    k_tc_select2<<<2 * kSMs, 256, 0, s>>>(list_f, count_f, best, second, idx, g_norm, cmax, TC_BAND, labels,
                                         labels_prev, n_changed_dev, amb_list, amb_count, amb_packed);
    GDR_LAUNCHED();
  }
  // exact fp32 re-score of the ambiguous rows (list length stays on the device)
  rc = launch_assign_simt_rows(N, K, D, X, ldx, c_t, Kp, cnorm, amb_list, amb_count, amb_packed, labels, labels_prev,
                               n_changed_dev, best_out, s);
  if (rc || !two_level || !g_last_cand || !n_refined_dev) return rc;
  k_add_i32<<<1, 1, 0, s>>>(n_refined_dev, cand_ctr + 1);   // + candidate rows whose exact margin lies in the band
  GDR_LAUNCHED();
  return GDR_OK;
}

// gdr_kmeans_assign(precision_mode = 1): split X into the tail of the workspace, then run
int64_t kmeans_assign_tc_total_ws_bytes(int64_t N, int64_t K, int64_t D) {
  return kmeans_assign_tc_ws_bytes(N, K, D) + kmeans_tc_xsplit_bytes(N, D);
}

int kmeans_assign_tc(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx, const float* C, int64_t ldc,
                     int32_t* labels, const int32_t* labels_prev, int32_t* n_changed_dev, float* best_out,
                     void* ws, int64_t ws_bytes, cudaStream_t s) {
  if (ws_bytes < kmeans_assign_tc_total_ws_bytes(N, K, D)) {
    set_error("kmeans_assign(tc): workspace too small");
    return GDR_EWORKSPACE;
  }
  char* xsplit = (char*)ws + kmeans_assign_tc_ws_bytes(N, K, D);
  int rc = kmeans_tc_prepare(N, D, X, ldx, xsplit, s);
  if (rc) return rc;
  return kmeans_assign_tc_run(N, K, D, X, ldx, xsplit, C, ldc, labels, labels_prev, n_changed_dev, best_out,
                              nullptr, ws, kmeans_assign_tc_ws_bytes(N, K, D), s);
}

}  // namespace gdr

extern "C" {

// debug read-back (synchronises the device): "tc_level2_rows" = rows the last two-level screen sent to level 2
int gdr_debug_get(const char* key, int64_t* value_host) {
  GDR_CHECK_ARG(key && value_host, "debug_get: bad arguments");
  if (!strcmp(key, "tc_level2_rows")) {
    int32_t v = -1;
    if (gdr::g_last_count1) GDR_CUDA(cudaMemcpy(&v, gdr::g_last_count1, 4, cudaMemcpyDeviceToHost));
    *value_host = v;
    return GDR_OK;
  }
  if (!strcmp(key, "tc_cand_rows") || !strcmp(key, "tc_cand_overflow_rows") || !strcmp(key, "tc_cand_entries")) {
    int32_t h[gdr::TC_CAND_CTRS];
    for (int i = 0; i < gdr::TC_CAND_CTRS; ++i) h[i] = -1;
    if (gdr::g_last_cand) GDR_CUDA(cudaMemcpy(h, gdr::g_last_cand, sizeof(h), cudaMemcpyDeviceToHost));
    long long e = -1;
    if (gdr::g_last_cand) memcpy(&e, h + 4, 8);
    *value_host = !strcmp(key, "tc_cand_rows") ? h[2] : (!strcmp(key, "tc_cand_overflow_rows") ? h[3] : e);
    return GDR_OK;
  }
  if (!strcmp(key, "topk_overflow_rows")) {
    *value_host = gdr::g_topk_last_overflow;
    return GDR_OK;
  }
  if (!strcmp(key, "topk_condensed_fallback_rows")) {
    *value_host = gdr::g_topk_condensed_last_fallback;
    return GDR_OK;
  }
  gdr::set_error("debug_get: unknown key %s", key);
  return GDR_EINVAL;
}

int64_t gdr_kmeans_tc_xsplit_bytes(int64_t N, int64_t D) { return gdr::kmeans_tc_xsplit_bytes(N, D); }

int gdr_kmeans_tc_prepare(int64_t N, int64_t D, const float* X, int64_t ldx, void* xsplit, int64_t xsplit_bytes,
                          gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && D > 0 && X && xsplit && ldx >= D, "kmeans_tc_prepare: bad arguments");
  GDR_CHECK_ARG(D <= gdr::TC_MAX_KB * gdr::TC_BK, "kmeans_tc_prepare: D > 128 is not supported by the tensor-core path");
  if (xsplit_bytes < gdr::kmeans_tc_xsplit_bytes(N, D)) {
    gdr::set_error("kmeans_tc_prepare: buffer too small");
    return GDR_EWORKSPACE;
  }
  return gdr::kmeans_tc_prepare(N, D, X, ldx, xsplit, (cudaStream_t)stream);
}

int64_t gdr_kmeans_assign_tc_ws_bytes(int64_t N, int64_t K, int64_t D) {
  return gdr::kmeans_assign_tc_ws_bytes(N, K, D);
}

int gdr_kmeans_assign_tc(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx, const void* xsplit,
                         const float* C, int64_t ldc, int32_t* labels, const int32_t* labels_prev,
                         int32_t* n_changed_dev, float* best_out, int32_t* n_refined_dev, void* ws,
                         int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && K > 0 && D > 0 && X && xsplit && C && labels && ws, "kmeans_assign_tc: bad arguments");
  GDR_CHECK_ARG(ldx % 4 == 0 && ldc % 4 == 0 && ldx >= D && ldc >= D && ((uintptr_t)X & 15) == 0 &&
                    ((uintptr_t)C & 15) == 0,
                "kmeans_assign_tc: X/C need 16B alignment and ld %% 4 == 0");
  if (ws_bytes < gdr::kmeans_assign_tc_ws_bytes(N, K, D)) {
    gdr::set_error("kmeans_assign_tc: workspace too small");
    return GDR_EWORKSPACE;
  }
  return gdr::kmeans_assign_tc_run(N, K, D, X, ldx, xsplit, C, ldc, labels, labels_prev, n_changed_dev, best_out,
                                   n_refined_dev, ws, ws_bytes, (cudaStream_t)stream);
}

}  // extern "C"
