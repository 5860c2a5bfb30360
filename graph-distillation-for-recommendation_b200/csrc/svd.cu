// svd.cu — the small dense steps of the truncated SVD embeddings (compute_svd_embeddings,
// distill_recsys.py:124-155; the reference calls scipy's ARPACK svds on the host).
//
// The factorisation is a block Krylov Rayleigh-Ritz (svd.py): its sparse products R.Q / R^T.Q run on the stage-2
// CSR SpMM kernel; this file holds everything else, in fp64, hand-written (no cuSOLVER / cuBLAS):
//   gdr_dense_gram         C = A^T B for tall-skinny A [N x p], B [N x r]   (Gram matrices, projections Q^T Z)
//   gdr_dense_chol         lower Cholesky factor of a small SPD matrix       (CholeskyQR)
//   gdr_dense_trsm_rows    Y <- Y L^-T, one thread per row                   (CholeskyQR)
//   gdr_dense_gemm_small   Z <- beta Z + alpha A P, A tall, P small           (block Gram-Schmidt, Ritz vectors)
//   gdr_sym_eig_jacobi     eigen-decomposition of a small symmetric matrix    (the (q b)^2 Ritz problem)
//   gdr_dense_gram_dist    gdr_dense_gram of row blocks split over the ranks, the same bits on every rank
// All reductions have a fixed order (two-stage partial sums): results are run-to-run deterministic.
#include "common.cuh"
#include "comm.cuh"
#include <algorithm>

namespace gdr {

constexpr int GT = 32;          // output tile of the Gram kernel
constexpr int GR = 32;          // rows staged per step
constexpr int GRAM_MAX_SLABS = 16;

// partial[slab][i][j] = sum over the slab's rows of A[r][i] * B[r][j]
__global__ void __launch_bounds__(256) k_gram_partial(int64_t N, int p, int r, const double* __restrict__ A, int64_t lda,
                                                      const double* __restrict__ B, int64_t ldb, int slabs,
                                                      double* __restrict__ part) {
  __shared__ double sA[GR][GT + 1];
  __shared__ double sB[GR][GT + 1];
  const int ti = blockIdx.x * GT, tj = blockIdx.y * GT, slab = blockIdx.z;
  const int64_t rows_per = (N + slabs - 1) / slabs;
  const int64_t r0 = slab * rows_per, r1 = min(N, r0 + rows_per);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;        // 16 x 16 threads, 2 x 2 outputs each
  double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
  for (int64_t rr = r0; rr < r1; rr += GR) {
    for (int t = threadIdx.x; t < GR * GT; t += 256) {
      const int row = t / GT, col = t % GT;
      const int64_t g = rr + row;
      sA[row][col] = (g < r1 && ti + col < p) ? A[g * lda + ti + col] : 0.0;
      sB[row][col] = (g < r1 && tj + col < r) ? B[g * ldb + tj + col] : 0.0;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < GR; ++k) {
      const double a0 = sA[k][ty * 2], a1 = sA[k][ty * 2 + 1];
      const double b0 = sB[k][tx * 2], b1 = sB[k][tx * 2 + 1];
      acc[0][0] = fma(a0, b0, acc[0][0]);
      acc[0][1] = fma(a0, b1, acc[0][1]);
      acc[1][0] = fma(a1, b0, acc[1][0]);
      acc[1][1] = fma(a1, b1, acc[1][1]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const int i = ti + ty * 2 + a, j = tj + tx * 2 + b;
      if (i < p && j < r) part[((int64_t)slab * p + i) * r + j] = acc[a][b];
    }
}

__global__ void k_gram_reduce(int p, int r, int slabs, const double* __restrict__ part, double* __restrict__ C, int64_t ldc) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)p * r) return;
  double s = 0.0;
  for (int z = 0; z < slabs; ++z) s += part[(int64_t)z * p * r + t];
  C[(t / r) * ldc + (t % r)] = s;
}

// ---- the Gram on a row partition (gdr_dense_gram_dist) ----
// A rank's rows cut at the global slab boundaries: segment z (blockIdx.z) runs k_gram_partial's chain over local rows
// [r0, r1), from 0.0 when it starts its slab or from init (the accumulators the previous rank's part of the slab ended
// with), and stores the chain's end in out [p][r]: the slab's partial, or the carry for the next rank.  The steps of GR
// rows start at the segment, not at the slab, so zero rows pad a step at a rank boundary too; they leave a chain as it
// is (fma(0, 0, c) = c for every c but -0.0, which only an fp64 underflow can produce).
struct GramSegs {
  int64_t r0[GRAM_MAX_SLABS], r1[GRAM_MAX_SLABS];
  const double* init[GRAM_MAX_SLABS];
  double* out[GRAM_MAX_SLABS];
};

__global__ void __launch_bounds__(256) k_gram_segments(int p, int r, const double* __restrict__ A, int64_t lda,
                                                       const double* __restrict__ B, int64_t ldb, GramSegs sg) {
  __shared__ double sA[GR][GT + 1];
  __shared__ double sB[GR][GT + 1];
  const int ti = blockIdx.x * GT, tj = blockIdx.y * GT, z = blockIdx.z;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const double* init = sg.init[z];
  double acc[2][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const int i = ti + ty * 2 + a, j = tj + tx * 2 + b;
      acc[a][b] = (init && i < p && j < r) ? init[(int64_t)i * r + j] : 0.0;
    }
  const int64_t r0 = sg.r0[z], r1 = sg.r1[z];
  for (int64_t rr = r0; rr < r1; rr += GR) {
    for (int t = threadIdx.x; t < GR * GT; t += 256) {
      const int row = t / GT, col = t % GT;
      const int64_t g = rr + row;
      sA[row][col] = (g < r1 && ti + col < p) ? A[g * lda + ti + col] : 0.0;
      sB[row][col] = (g < r1 && tj + col < r) ? B[g * ldb + tj + col] : 0.0;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < GR; ++k) {
      const double a0 = sA[k][ty * 2], a1 = sA[k][ty * 2 + 1];
      const double b0 = sB[k][tx * 2], b1 = sB[k][tx * 2 + 1];
      acc[0][0] = fma(a0, b0, acc[0][0]);
      acc[0][1] = fma(a0, b1, acc[0][1]);
      acc[1][0] = fma(a1, b0, acc[1][0]);
      acc[1][1] = fma(a1, b1, acc[1][1]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const int i = ti + ty * 2 + a, j = tj + tx * 2 + b;
      if (i < p && j < r) sg.out[z][(int64_t)i * r + j] = acc[a][b];
    }
}

// sum_out = sum_in + part[0] + ... + part[n - 1]: k_gram_reduce's slab-order chain, continued from the running sum of the
// slabs that ended on earlier ranks (0.0 on the first rank)
__global__ void k_gram_reduce_dist(int64_t pr, int n, const double* __restrict__ part, const double* __restrict__ sum_in,
                                   double* __restrict__ sum_out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= pr) return;
  double s = sum_in[t];
  for (int z = 0; z < n; ++z) s += part[(int64_t)z * pr + t];
  sum_out[t] = s;
}

// lower Cholesky of an n x n SPD matrix (n <= 128) in shared memory; info[0] = 0 ok, j + 1 = pivot j not positive
__global__ void __launch_bounds__(256) k_chol(int n, const double* __restrict__ S, int64_t lds, double* __restrict__ L,
                                              int64_t ldl, int32_t* __restrict__ info, double rel_tol) {
  extern __shared__ double sm[];     // [n][n + 1]
  const int ld = n + 1;
  double dmax = 0.0;
  for (int t = threadIdx.x; t < n * n; t += blockDim.x) sm[(t / n) * ld + (t % n)] = S[(int64_t)(t / n) * lds + (t % n)];
  __syncthreads();
  for (int i = 0; i < n; ++i) dmax = fmax(dmax, sm[i * ld + i]);
  __shared__ int s_fail;
  if (threadIdx.x == 0) s_fail = 0;
  __syncthreads();
  for (int j = 0; j < n; ++j) {
    if (threadIdx.x == 0) {
      const double d = sm[j * ld + j];
      if (!(d > rel_tol * dmax)) s_fail = j + 1;
      else sm[j * ld + j] = sqrt(d);
    }
    __syncthreads();
    if (s_fail) break;
    const double dj = sm[j * ld + j];
    for (int i = j + 1 + threadIdx.x; i < n; i += blockDim.x) sm[i * ld + j] /= dj;
    __syncthreads();
    // trailing update: A[i][k] -= L[i][j] L[k][j] for j < k <= i
    const int m = n - j - 1;
    for (int t = threadIdx.x; t < m * m; t += blockDim.x) {
      const int i = j + 1 + t / m, k = j + 1 + t % m;
      if (k <= i) sm[i * ld + k] = fma(-sm[i * ld + j], sm[k * ld + j], sm[i * ld + k]);
    }
    __syncthreads();
  }
  for (int t = threadIdx.x; t < n * n; t += blockDim.x) {
    const int i = t / n, k = t % n;
    L[(int64_t)i * ldl + k] = k <= i ? sm[i * ld + k] : 0.0;
  }
  if (threadIdx.x == 0) info[0] = s_fail;
}

// Y <- Y L^-T : row y solves x L^T = y, i.e. x_j = (y_j - sum_{i<j} x_i L[j][i]) / L[j][j]
__global__ void __launch_bounds__(128) k_trsm_rows(int64_t N, int n, double* __restrict__ Y, int64_t ldy,
                                                   const double* __restrict__ L, int64_t ldl) {
  extern __shared__ double sL[];     // [n][n]
  for (int t = threadIdx.x; t < n * n; t += blockDim.x) sL[t] = L[(int64_t)(t / n) * ldl + (t % n)];
  __syncthreads();
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= N) return;
  double* y = Y + row * ldy;
  for (int j = 0; j < n; ++j) {
    double s = y[j];
    for (int i = 0; i < j; ++i) s = fma(-y[i], sL[j * n + i], s);
    y[j] = s / sL[j * n + j];
  }
}

// Z[N x r] = beta * Z + alpha * A[N x m] P[m x r]  (optionally each output column j scaled by colscale[j]),
// output to fp64 Z and/or fp32 Zf
__global__ void __launch_bounds__(256) k_gemm_small(int64_t N, int m, int r, double alpha, const double* __restrict__ A,
                                                    int64_t lda, const double* __restrict__ P, int64_t ldp, double beta,
                                                    double* __restrict__ Z, int64_t ldz, float* __restrict__ Zf,
                                                    int64_t ldzf, const double* __restrict__ colscale) {
  __shared__ double sA[64][33];
  __shared__ double sP[32][33];
  const int64_t row0 = (int64_t)blockIdx.x * 64;
  const int col0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // thread: column tx, rows ty, ty + 8, ... (8 rows)
  double acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = 0.0;
  for (int k0 = 0; k0 < m; k0 += 32) {
    for (int t = threadIdx.x; t < 64 * 32; t += 256) {
      const int rr = t >> 5, kk = t & 31;
      sA[rr][kk] = (row0 + rr < N && k0 + kk < m) ? A[(row0 + rr) * lda + k0 + kk] : 0.0;
    }
    for (int t = threadIdx.x; t < 32 * 32; t += 256) {
      const int kk = t >> 5, cc = t & 31;
      sP[kk][cc] = (k0 + kk < m && col0 + cc < r) ? P[(int64_t)(k0 + kk) * ldp + col0 + cc] : 0.0;
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < 32; ++kk) {
      const double pv = sP[kk][tx];
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q] = fma(sA[ty + 8 * q][kk], pv, acc[q]);
    }
    __syncthreads();
  }
  const int col = col0 + tx;
  if (col >= r) return;
  const double cs = colscale ? colscale[col] : 1.0;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int64_t row = row0 + ty + 8 * q;
    if (row < N) {
      double v = alpha * acc[q];
      if (beta != 0.0) v += beta * Z[row * ldz + col];
      v *= cs;
      if (Z) Z[row * ldz + col] = v;
      if (Zf) Zf[row * ldzf + col] = (float)v;
    }
  }
}

// ---- symmetric eigen-decomposition: parallel cyclic Jacobi (round-robin pairing) ----------------------------
// round `rd` of an n-player tournament (n even): pair k = (a, b)
__device__ __forceinline__ void rr_pair(int n, int rd, int k, int& a, int& b) {
  const int m = n - 1;
  if (k == 0) {
    a = m;
    b = rd % m;
  } else {
    a = (rd + k) % m;
    b = (rd - k + m) % m;
  }
  if (a > b) {
    const int t = a;
    a = b;
    b = t;
  }
}

// One round = all n/2 disjoint rotations at once: A <- J^T A J, W <- W J with J the product of the round's rotations.
// k_jacobi_angles: (c, s) of every pair from a_pp, a_qq, a_pq of the matrix at the START of the round.
// k_jacobi_apply: the 2 x 2 block A[{p,q}][{p',q'}] depends only on itself and the two pairs' angles — columns first, rows
// second, the same arithmetic per element as rotating whole columns and then whole rows — so every block is updated in
// place by one thread, and CTA k walks the row pair (p, q): all its accesses lie in two contiguous rows (the column-wise
// formulation read and wrote with a stride of n doubles: 29 us per round at n = 600 against 6 us for the row phase).
// The same CTA rotates rows 2k, 2k + 1 of W.
__global__ void __launch_bounds__(256) k_jacobi_angles(int n, int npad, int rd, const double* __restrict__ A, double* __restrict__ cs) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= npad / 2) return;
  int p, q;
  rr_pair(npad, rd, k, p, q);
  double c = 1.0, s = 0.0;
  if (q < n) {
    const double apq = A[(int64_t)p * n + q];
    if (apq != 0.0) {
      const double tau = (A[(int64_t)q * n + q] - A[(int64_t)p * n + p]) / (2.0 * apq);
      const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
      c = 1.0 / sqrt(1.0 + t * t);
      s = t * c;
    }
  }
  cs[2 * k] = c;
  cs[2 * k + 1] = s;
}

__global__ void __launch_bounds__(128) k_jacobi_apply(int n, int npad, int rd, double* __restrict__ A, double* __restrict__ W,
                                                      const double* __restrict__ cs) {
  const int k1 = blockIdx.x, half = npad / 2;
  int p, q;
  rr_pair(npad, rd, k1, p, q);
  const double c1 = cs[2 * k1], s1 = cs[2 * k1 + 1];
  const bool q_ok = q < n;                    // the padding index of an odd n has no row / column
  double* Ap = A + (int64_t)p * n;
  double* Aq = A + (int64_t)(q_ok ? q : p) * n;
  const int w0 = 2 * k1, w1 = 2 * k1 + 1;     // the rows of W this CTA rotates
  for (int k2 = threadIdx.x; k2 < half; k2 += blockDim.x) {
    int pc, qc;
    rr_pair(npad, rd, k2, pc, qc);
    const double c2 = cs[2 * k2], s2 = cs[2 * k2 + 1];
    const bool qc_ok = qc < n;
    if (s1 != 0.0 || s2 != 0.0) {
      // columns (pc, qc) of rows p and q, then rows (p, q)
      double tpp = Ap[pc], tpq = qc_ok ? Ap[qc] : 0.0;
      double tqp = q_ok ? Aq[pc] : 0.0, tqq = (q_ok && qc_ok) ? Aq[qc] : 0.0;
      if (s2 != 0.0) {
        const double a = tpp, b = tpq, d = tqp, e = tqq;
        tpp = c2 * a - s2 * b;
        tpq = s2 * a + c2 * b;
        tqp = c2 * d - s2 * e;
        tqq = s2 * d + c2 * e;
      }
      if (s1 != 0.0) {
        const double a = tpp, b = tpq, d = tqp, e = tqq;
        tpp = c1 * a - s1 * d;
        tqp = s1 * a + c1 * d;
        tpq = c1 * b - s1 * e;
        tqq = s1 * b + c1 * e;
      }
      Ap[pc] = tpp;
      if (qc_ok) Ap[qc] = tpq;
      if (q_ok) {
        Aq[pc] = tqp;
        if (qc_ok) Aq[qc] = tqq;
      }
    }
    if (s2 != 0.0) {                         // (s2 != 0 implies qc < n)
      if (w0 < n) {
        const double wp = W[(int64_t)w0 * n + pc], wq = W[(int64_t)w0 * n + qc];
        W[(int64_t)w0 * n + pc] = c2 * wp - s2 * wq;
        W[(int64_t)w0 * n + qc] = s2 * wp + c2 * wq;
      }
      if (w1 < n) {
        const double wp = W[(int64_t)w1 * n + pc], wq = W[(int64_t)w1 * n + qc];
        W[(int64_t)w1 * n + pc] = c2 * wp - s2 * wq;
        W[(int64_t)w1 * n + qc] = s2 * wp + c2 * wq;
      }
    }
  }
}

// out[0] = sum of squared off-diagonal entries, out[1] = sum of squared diagonal entries (single CTA, fixed order)
__global__ void __launch_bounds__(1024) k_offdiag_norm(int n, const double* __restrict__ A, double* __restrict__ out) {
  __shared__ double so[1024], sd[1024];
  double o = 0.0, d = 0.0;
  for (int64_t t = threadIdx.x; t < (int64_t)n * n; t += 1024) {
    const double v = A[t];
    if (t / n == t % n) d += v * v;
    else o += v * v;
  }
  so[threadIdx.x] = o;
  sd[threadIdx.x] = d;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      so[threadIdx.x] += so[threadIdx.x + s];
      sd[threadIdx.x] += sd[threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[0] = so[0];
    out[1] = sd[0];
  }
}

__global__ void k_set_identity(int n, double* __restrict__ W) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < (int64_t)n * n) W[t] = (t / n == t % n) ? 1.0 : 0.0;
}

// eigenvalues (diagonal) sorted descending: order[k] = index of the k-th largest; single CTA rank sort (n <= 2048)
__global__ void __launch_bounds__(1024) k_eig_order(int n, const double* __restrict__ A, double* __restrict__ evals,
                                                    int32_t* __restrict__ order) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = A[(int64_t)i * n + i];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const double u = A[(int64_t)j * n + j];
      rank += (u > v || (u == v && j < i)) ? 1 : 0;
    }
    evals[rank] = v;
    order[rank] = i;
  }
}

// Wk[i][k] = W[i][order[k]] for k < kcols
__global__ void k_gather_cols(int n, int kcols, const double* __restrict__ W, const int32_t* __restrict__ order,
                              double* __restrict__ Wk) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)n * kcols) return;
  const int i = (int)(t / kcols), k = (int)(t % kcols);
  Wk[t] = W[(int64_t)i * n + order[k]];
}

// the slabs of an N-row Gram: contiguous blocks of cdiv(N, slabs) rows, summed in slab order
static int gram_slabs(int64_t N) { return (int)std::max<int64_t>(1, std::min<int64_t>(GRAM_MAX_SLABS, cdiv(N, 2048))); }

}  // namespace gdr

using namespace gdr;

namespace {

struct GramDistBuffers {
  double* part;    // [slabs][p][r] partials of the slabs that end on this rank, in slab order
  double* x;       // [4][p][r]  carry in, running sum in | carry out, running sum out
  int64_t off;
};

GramDistBuffers gram_dist_carve(void* ws, int64_t N, int64_t p, int64_t r) {
  Workspace W(ws, INT64_MAX);
  GramDistBuffers b;
  b.part = W.take<double>(gram_slabs(N) * p * r);
  b.x = W.take<double>(4 * p * r);
  b.off = W.off + 256;
  return b;
}

}  // namespace

extern "C" {

int64_t gdr_dense_gram_ws_bytes(int64_t N, int64_t p, int64_t r) {
  (void)N;
  return ws_need((int64_t)GRAM_MAX_SLABS * p * r, 8) + 256;
}

int gdr_dense_gram(int64_t N, int64_t p, int64_t r, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                   int64_t ldc, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && p > 0 && r > 0 && A && B && C && lda >= p && ldb >= r && ldc >= r, "dense_gram: bad arguments");
  if (ws_bytes < gdr_dense_gram_ws_bytes(N, p, r)) {
    set_error("dense_gram: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int slabs = gram_slabs(N);
  double* part = (double*)ws;
  dim3 grid((unsigned)cdiv(p, GT), (unsigned)cdiv(r, GT), (unsigned)slabs);
  k_gram_partial<<<grid, 256, 0, s>>>(N, (int)p, (int)r, A, lda, B, ldb, slabs, part);
  GDR_LAUNCHED();
  k_gram_reduce<<<(unsigned)cdiv(p * r, 256), 256, 0, s>>>((int)p, (int)r, slabs, part, C, ldc);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_dense_gram_dist_ws_bytes(int64_t N_global, int64_t p, int64_t r, int world) {
  (void)world;
  return gram_dist_carve(nullptr, N_global, p, r).off;
}

int gdr_dense_gram_dist(gdr_comm_t* comm, int64_t N_global, int64_t row_lo, int64_t n_local, int64_t p, int64_t r,
                        const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, void* ws,
                        int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(comm, "dense_gram_dist: null communicator");
  const int world = comm->world, rank = comm->rank;
  cudaStream_t s = (cudaStream_t)stream;
  // local checks are decided collectively in comm_entry_check: an early return would leave the others in a collective
  int local_rc = GDR_OK;
  if (!(N_global >= 0 && row_lo >= 0 && n_local >= 0 && row_lo + n_local <= N_global && p > 0 && r > 0 && C && ldc >= r &&
        ws && (n_local == 0 || (A && B && lda >= p && ldb >= r)))) {
    set_error("dense_gram_dist: bad arguments");
    local_rc = GDR_EINVAL;
  } else if (ws_bytes < gdr_dense_gram_dist_ws_bytes(N_global, p, r, world)) {
    set_error("dense_gram_dist: workspace too small");
    local_rc = GDR_EWORKSPACE;
  }
  int rc = comm_entry_check(comm, s, "dense_gram_dist", local_rc, row_lo, n_local, N_global, {N_global, p, r},
                            "N_global, p or r");
  if (rc != GDR_OK) return rc;

  // this rank's rows cut at the global slab boundaries (gdr_dense_gram's geometry): the segments that start their slab
  // need nothing from the previous rank; at most one, the first, continues the carry of a slab begun on an earlier rank
  const int64_t pr = p * r, rows_per = cdiv(N_global, gram_slabs(N_global));
  GramDistBuffers G = gram_dist_carve(ws, N_global, p, r);
  double *carry_in = G.x, *sum_in = G.x + pr, *carry_out = G.x + 2 * pr, *sum_out = G.x + 3 * pr;
  GramSegs starts = {}, cont = {};
  int n_starts = 0, n_cont = 0, n_done = 0;
  for (int64_t a = row_lo, hi = row_lo + n_local; a < hi;) {
    const int64_t z0 = a / rows_per * rows_per, z1 = std::min(N_global, z0 + rows_per), b = std::min(hi, z1);
    GramSegs& g = a == z0 ? starts : cont;
    int& n = a == z0 ? n_starts : n_cont;
    g.r0[n] = a - row_lo;
    g.r1[n] = b - row_lo;
    g.init[n] = a == z0 ? nullptr : carry_in;
    g.out[n] = b == z1 ? G.part + (int64_t)(n_done++) * pr : carry_out;
    ++n;
    a = b;
  }
  const unsigned tx = (unsigned)cdiv(p, GT), ty = (unsigned)cdiv(r, GT);
  if (n_starts) {
    k_gram_segments<<<dim3(tx, ty, (unsigned)n_starts), 256, 0, s>>>((int)p, (int)r, A, lda, B, ldb, starts);
    GDR_LAUNCHED();
  }
  // (carry, running sum) from the previous rank; the first rank starts the running sum from 0.0
  if (rank > 0) {
    if ((rc = comm_recv(comm, G.x, 2 * pr * 8, rank - 1, s))) return rc;
  } else {
    GDR_CUDA(cudaMemsetAsync(G.x, 0, 2 * pr * 8, s));
  }
  if (n_cont) {
    k_gram_segments<<<dim3(tx, ty, 1), 256, 0, s>>>((int)p, (int)r, A, lda, B, ldb, cont);
    GDR_LAUNCHED();
  }
  // an empty rank hands on what it received
  double* handed = G.x;
  if (n_local > 0) {
    k_gram_reduce_dist<<<(unsigned)cdiv(pr, 256), 256, 0, s>>>(pr, n_done, G.part, sum_in, sum_out);
    GDR_LAUNCHED();
    handed = carry_out;
  }
  if (rank + 1 < world && (rc = comm_send(comm, handed, 2 * pr * 8, rank + 1, s))) return rc;
  // the last rank's running sum is C: every other rank receives it into its (already sent) running-sum slot
  double* total = handed + pr;
  if ((rc = comm_broadcast(comm, total, pr * 8, world - 1, s))) return rc;
  GDR_CUDA(cudaMemcpy2DAsync(C, (size_t)ldc * 8, total, (size_t)r * 8, (size_t)r * 8, (size_t)p, cudaMemcpyDeviceToDevice, s));
  return GDR_OK;
}

int gdr_dense_chol(int64_t n, const double* S, int64_t lds, double* L, int64_t ldl, int32_t* info_dev, double rel_tol,
                   gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && n <= 128 && S && L && info_dev && lds >= n && ldl >= n, "dense_chol: bad arguments (n <= 128)");
  const size_t smem = (size_t)n * (n + 1) * 8;
  static PerDevice<bool> attr_set_dev;
  bool& attr_set = attr_set_dev.get();
  if (!attr_set) {
    GDR_CUDA(cudaFuncSetAttribute(k_chol, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 129 * 8));
    attr_set = true;
  }
  k_chol<<<1, 256, smem, (cudaStream_t)stream>>>((int)n, S, lds, L, ldl, info_dev, rel_tol);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_dense_trsm_rows(int64_t N, int64_t n, double* Y, int64_t ldy, const double* L, int64_t ldl, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && n > 0 && n <= 128 && L && ldl >= n && ldy >= n, "dense_trsm_rows: bad arguments (n <= 128)");
  if (N == 0) return GDR_OK;
  GDR_CHECK_ARG(Y, "dense_trsm_rows: null Y");
  static PerDevice<bool> attr_set_dev;
  bool& attr_set = attr_set_dev.get();
  if (!attr_set) {
    GDR_CUDA(cudaFuncSetAttribute(k_trsm_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 128 * 8));
    attr_set = true;
  }
  k_trsm_rows<<<(unsigned)cdiv(N, 128), 128, (size_t)n * n * 8, (cudaStream_t)stream>>>(N, (int)n, Y, ldy, L, ldl);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_dense_gemm_small(int64_t N, int64_t m, int64_t r, double alpha, const double* A, int64_t lda, const double* P,
                         int64_t ldp, double beta, double* Z, int64_t ldz, float* Zf, int64_t ldzf, const double* colscale,
                         gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && m > 0 && r > 0 && A && P && (Z || Zf) && lda >= m && ldp >= r, "dense_gemm_small: bad arguments");
  GDR_CHECK_ARG(beta == 0.0 || Z, "dense_gemm_small: beta needs the fp64 output");
  if (N == 0) return GDR_OK;
  dim3 grid((unsigned)cdiv(N, 64), (unsigned)cdiv(r, 32));
  k_gemm_small<<<grid, 256, 0, (cudaStream_t)stream>>>(N, (int)m, (int)r, alpha, A, lda, P, ldp, beta, Z, ldz, Zf, ldzf,
                                                       colscale);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_sym_eig_jacobi_ws_bytes(int64_t n) { return ws_need(n + 2, 8) + ws_need(4, 8) + 512; }

// A (n x n symmetric, contiguous, DESTROYED) -> evals[n] descending, W (n x n, contiguous): column order[k] of W is the
// eigenvector of evals[k].  Sweeps until the off-diagonal mass is below tol^2 of the diagonal mass (host read per sweep).
int gdr_sym_eig_jacobi(int64_t n, double* A, double* W, double* evals, int32_t* order, int max_sweeps, double tol,
                       int32_t* sweeps_out_host, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && n <= 2048 && A && W && evals && order && max_sweeps > 0, "sym_eig_jacobi: bad arguments (n <= 2048)");
  if (ws_bytes < gdr_sym_eig_jacobi_ws_bytes(n)) {
    set_error("sym_eig_jacobi: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  Workspace Wk(ws, ws_bytes);
  const int npad = (int)(n + (n & 1));
  double* cs = Wk.take<double>(npad + 2);
  double* norms = Wk.take<double>(4);
  k_set_identity<<<(unsigned)cdiv(n * n, 256), 256, 0, s>>>((int)n, W);
  GDR_LAUNCHED();
  int sweep = 0;
  cudaGraphExec_t sweep_exec = nullptr;
  bool try_graph = true;
  for (; sweep < max_sweeps; ++sweep) {
    double h[2];
    k_offdiag_norm<<<1, 1024, 0, s>>>((int)n, A, norms);
    GDR_LAUNCHED();
    GDR_CUDA(cudaMemcpyAsync(h, norms, 16, cudaMemcpyDeviceToHost, s));
    GDR_CUDA(cudaStreamSynchronize(s));
    if (h[0] <= tol * tol * h[1] || n == 1) break;
    // one sweep = 2 (n - 1) dependent launches of a few microseconds of work each: captured ONCE as a CUDA graph and
    // replayed per sweep (the launches of a replay cost ~1/4 of stream launches); falls back to plain launches when the
    // stream cannot be captured (it is already being captured by the caller)
    auto enqueue_sweep = [&]() {
      for (int rd = 0; rd < npad - 1; ++rd) {
        k_jacobi_angles<<<(unsigned)cdiv(npad / 2, 256), 256, 0, s>>>((int)n, npad, rd, A, cs);
        k_jacobi_apply<<<(unsigned)(npad / 2), 128, 0, s>>>((int)n, npad, rd, A, W, cs);
      }
    };
    if (!sweep_exec && try_graph && npad > 16) {
      cudaGraph_t graph = nullptr;
      if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        enqueue_sweep();
        const cudaError_t e = cudaStreamEndCapture(s, &graph);
        if (e != cudaSuccess || !graph || cudaGraphInstantiate(&sweep_exec, graph, 0) != cudaSuccess) sweep_exec = nullptr;
        if (graph) cudaGraphDestroy(graph);
      }
      if (!sweep_exec) {
        cudaGetLastError();
        try_graph = false;
      }
    }
    if (sweep_exec) {
      if (cudaGraphLaunch(sweep_exec, s) != cudaSuccess) {
        cudaGraphExecDestroy(sweep_exec);
        set_error("sym_eig_jacobi: graph launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        return GDR_ECUDA;
      }
    } else {
      enqueue_sweep();
    }
    count_launch(2 * (npad - 1));
    if (cudaGetLastError() != cudaSuccess) {
      if (sweep_exec) cudaGraphExecDestroy(sweep_exec);
      set_error("sym_eig_jacobi: launch failed");
      return GDR_ECUDA;
    }
  }
  if (sweep_exec) {
    cudaStreamSynchronize(s);
    cudaGraphExecDestroy(sweep_exec);
  }
  k_eig_order<<<1, 1024, 0, s>>>((int)n, A, evals, order);
  GDR_LAUNCHED();
  if (sweeps_out_host) *sweeps_out_host = sweep;
  return GDR_OK;
}

int gdr_dense_gather_cols(int64_t n, int64_t kcols, const double* W, const int32_t* order, double* Wk, gdr_stream_t stream) {
  GDR_CHECK_ARG(n > 0 && kcols > 0 && kcols <= n && W && order && Wk, "dense_gather_cols: bad arguments");
  k_gather_cols<<<(unsigned)cdiv(n * kcols, 256), 256, 0, (cudaStream_t)stream>>>((int)n, (int)kcols, W, order, Wk);
  GDR_LAUNCHED();
  return GDR_OK;
}

}  // extern "C"
