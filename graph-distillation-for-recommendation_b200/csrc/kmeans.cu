// kmeans.cu — stage 3: Lloyd k-means building blocks.
//
// Arithmetic follows scikit-learn's dense Lloyd iteration, the third-party code
// the reference calls at clustgdd_agent_transduct.py:102-105,
// clustgdd_agent_induct.py:131-136 and distill_recsys.py:172-180:
//   sklearn/cluster/_kmeans.py:1487-1493   mean-centring
//   sklearn/cluster/_k_means_lloyd.pyx:196-218  E-step + per-cluster sums
//   sklearn/cluster/_k_means_common.pyx:167-311 relocate / average / shift
//   sklearn/cluster/_k_means_common.pyx:94-124  inertia
// This file holds the exact-fp32 SIMT E-step (precision_mode 0, also the
// re-scoring kernel of the tensor-core path in kmeans_tc.cu), the deterministic
// M-step and the small reductions around them.
#include "common.cuh"
#include "comm.cuh"
#include <vector>

namespace gdr {

// implemented in kmeans_tc.cu
int64_t kmeans_assign_tc_total_ws_bytes(int64_t N, int64_t K, int64_t D);
int kmeans_assign_tc(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx, const float* C,
                     int64_t ldc, int32_t* labels, const int32_t* labels_prev,
                     int32_t* n_changed_dev, float* best_out, void* ws, int64_t ws_bytes,
                     cudaStream_t s);

// ----------------------------------------------------------------------------
// column mean / variance (fp64) and centring
// ----------------------------------------------------------------------------
constexpr int CC_ROWS_PER_BLOCK = 512;

__global__ void __launch_bounds__(256) k_colstats_partial(int64_t N, int D, const float* __restrict__ X,
                                                          int64_t ldx, double* __restrict__ part) {
  // block (32 x 8): x over columns, y over rows; each block covers CC_ROWS_PER_BLOCK rows.
  __shared__ double s_sum[8][33], s_sq[8][33];
  int64_t r0 = (int64_t)blockIdx.x * CC_ROWS_PER_BLOCK;
  int64_t r1 = min(N, r0 + CC_ROWS_PER_BLOCK);
  for (int c0 = 0; c0 < D; c0 += 32) {
    int c = c0 + threadIdx.x;
    double su = 0.0, sq = 0.0;
    if (c < D) {
      for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
        double x = (double)X[r * ldx + c];
        su += x;
        sq += x * x;
      }
    }
    s_sum[threadIdx.y][threadIdx.x] = su;
    s_sq[threadIdx.y][threadIdx.x] = sq;
    __syncthreads();
    if (threadIdx.y == 0 && c < D) {
      double a = 0.0, b = 0.0;
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        a += s_sum[y][threadIdx.x];
        b += s_sq[y][threadIdx.x];
      }
      part[((int64_t)blockIdx.x * D + c) * 2 + 0] = a;
      part[((int64_t)blockIdx.x * D + c) * 2 + 1] = b;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) k_colstats_final(int64_t N, int D, int nblocks,
                                                        const double* __restrict__ part,
                                                        float* __restrict__ mean_out,
                                                        double* __restrict__ var_col) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  double a = 0.0, b = 0.0;
  for (int i = 0; i < nblocks; ++i) {
    a += part[((int64_t)i * D + c) * 2 + 0];
    b += part[((int64_t)i * D + c) * 2 + 1];
  }
  double m = a / (double)N;
  double v = b / (double)N - m * m;
  mean_out[c] = (float)m;
  var_col[c] = v > 0.0 ? v : 0.0;
}

__global__ void k_var_mean(int D, const double* __restrict__ var_col, double* __restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double s = 0.0;
    for (int c = 0; c < D; ++c) s += var_col[c];
    out[0] = s / (double)D;
  }
}

__global__ void k_sub_rowvec(int64_t N, int D, int ldpad, const float* __restrict__ X, int64_t ldx,
                             const float* __restrict__ mean, float* __restrict__ out, int64_t ldo) {
  int64_t total = N * (int64_t)ldpad;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / ldpad;
    int c = (int)(i - r * ldpad);
    out[r * ldo + c] = c < D ? __fsub_rn(X[r * ldx + c], mean[c]) : 0.f;
  }
}

__global__ void k_add_rowvec(int64_t N, int D, float* __restrict__ X, int64_t ldx,
                             const float* __restrict__ v, float sign) {
  int64_t total = N * (int64_t)D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / D;
    int c = (int)(i - r * D);
    X[r * ldx + c] = __fadd_rn(X[r * ldx + c], __fmul_rn(sign, v[c]));
  }
}

// ----------------------------------------------------------------------------
// exact fp32 E-step (SIMT register-tiled GEMM with fused |c|^2 add + argmin)
// ----------------------------------------------------------------------------
constexpr int AS_BM = 128, AS_BN = 128, AS_BK = 16, AS_THREADS = 256;

__global__ void __launch_bounds__(256) k_row_sqnorm(int64_t K, int D, const float* __restrict__ C,
                                                    int64_t ldc, float* __restrict__ out) {
  // one warp per row, fixed-order shuffle reduction
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= K) return;
  float s = 0.f;
  for (int c = lane_id(); c < D; c += 32) {
    float x = C[row * ldc + c];
    s = fmaf(x, x, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane_id() == 0) out[row] = s;
}

__global__ void __launch_bounds__(AS_THREADS, 2)
k_assign_simt(int64_t N, int K, int D, const float* __restrict__ X, int64_t ldx,
              const float* __restrict__ C, int64_t ldc, const float* __restrict__ cnorm,
              int32_t* __restrict__ labels, const int32_t* __restrict__ labels_prev,
              int32_t* __restrict__ n_changed, float* __restrict__ best_out,
              const int32_t* __restrict__ rows, const int32_t* __restrict__ n_rows_dev) {
  // rows != nullptr: re-score only the listed rows (the tensor-core path's ambiguous set);
  // the list length lives on the device, surplus CTAs exit.
  __shared__ __align__(16) float As[AS_BK][AS_BM + 4];
  __shared__ __align__(16) float Bs[AS_BK][AS_BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * AS_BM;
  if (rows) {
    N = *n_rows_dev;
    if (row0 >= N) return;
  }

  float best[8];
  int bidx[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    best[i] = INFINITY;
    bidx[i] = 0;
  }
  // loader mapping: 128 rows x 16 k = 512 float4; thread -> (row = tid/4 + 64*h, k4 = tid%4)
  const int lrow = tid >> 2, lk4 = tid & 3;

  for (int j0 = 0; j0 < K; j0 += AS_BN) {
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < D; k0 += AS_BK) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        int r = lrow + 64 * h;
        int k = k0 + lk4 * 4;
        float4 xa = make_float4(0.f, 0.f, 0.f, 0.f), cb = xa;
        int64_t gr = row0 + r;
        if (gr < N && k < D) {
          int64_t xr = rows ? (int64_t)rows[gr] : gr;
          xa = *reinterpret_cast<const float4*>(X + xr * ldx + k);
          if (k + 1 >= D) xa.y = 0.f;
          if (k + 2 >= D) xa.z = 0.f;
          if (k + 3 >= D) xa.w = 0.f;
        }
        int gc = j0 + r;
        if (gc < K && k < D) {
          cb = *reinterpret_cast<const float4*>(C + (int64_t)gc * ldc + k);
          if (k + 1 >= D) cb.y = 0.f;
          if (k + 2 >= D) cb.z = 0.f;
          if (k + 3 >= D) cb.w = 0.f;
        }
        As[lk4 * 4 + 0][r] = xa.x;
        As[lk4 * 4 + 1][r] = xa.y;
        As[lk4 * 4 + 2][r] = xa.z;
        As[lk4 * 4 + 3][r] = xa.w;
        Bs[lk4 * 4 + 0][r] = cb.x;
        Bs[lk4 * 4 + 1][r] = cb.y;
        Bs[lk4 * 4 + 2][r] = cb.z;
        Bs[lk4 * 4 + 3][r] = cb.w;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < AS_BK; ++kk) {
        float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
        float4 a1 = *reinterpret_cast<const float4*>(&As[kk][64 + ty * 4]);
        float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
        float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
        float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = ed_chain(acc[i][j], a[i], b[j]);
      }
      __syncthreads();
    }
    // epilogue: d = |c|^2 - 2 x.c ; strict '<' keeps the first minimum (ascending j)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int col = j0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      if (col < K) {
        float cn = __ldg(cnorm + col);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float d = ed_finish(acc[i][j], cn);
          if (d < best[i]) {
            best[i] = d;
            bidx[i] = col;
          }
        }
      }
    }
  }
  // combine the 16 threads (tx) that share a row: (min value, lowest index)
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(0xffffffffu, best[i], o);
      int oi = __shfl_xor_sync(0xffffffffu, bidx[i], o);
      if (ob < best[i] || (ob == best[i] && oi < bidx[i])) {
        best[i] = ob;
        bidx[i] = oi;
      }
    }
  }
  int changed = 0;
  if (tx == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int r = i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4);
      int64_t gr = row0 + r;
      if (gr < N) {
        if (rows) gr = rows[gr];
        labels[gr] = bidx[i];
        if (best_out) best_out[gr] = best[i];
        if (labels_prev && labels_prev[gr] != bidx[i]) ++changed;
      }
    }
  }
  if (n_changed) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) changed += __shfl_xor_sync(0xffffffffu, changed, o);
    if (lane_id() == 0 && changed) atomicAdd(n_changed, changed);
  }
}

int launch_row_sqnorm(int64_t K, int D, const float* C, int64_t ldc, float* out, cudaStream_t s) {
  k_row_sqnorm<<<(unsigned)cdiv(K, 8), 256, 0, s>>>(K, D, C, ldc, out);
  GDR_LAUNCHED();
  return GDR_OK;
}

// Exact re-score of a short device-side row list.  grid = (row groups, centre slabs): a CTA
// keeps RF_ROWS listed rows in shared memory and each of its threads owns ONE centre of its
// slab; the centres are read through a TRANSPOSED copy CT[k][j] (consecutive threads ->
// consecutive addresses) and every loaded value feeds RF_ROWS chains.  Each (row, centre)
// distance is the SAME fp32 chain k_assign_simt evaluates — acc = fmaf(x_k, c_k, acc) for k
// ascending, then fmaf(-2, acc, |c|^2) — and the slabs are combined with a 64-bit atomicMin on
// (ordered distance bits << 32 | centre index): minimum distance, then lowest index, which is
// order-independent, so a re-scored row gets exactly the label of the full exact kernel.
constexpr int RF_THREADS = 128;
constexpr int RF_ROWS = 8;

__global__ void __launch_bounds__(RF_THREADS) k_refine_partial(int K, int D, const float* __restrict__ X,
                                                               int64_t ldx, const float* __restrict__ CT,
                                                               int64_t ldct, const float* __restrict__ cnorm,
                                                               const int32_t* __restrict__ rows,
                                                               const int32_t* __restrict__ n_rows_dev,
                                                               unsigned long long* __restrict__ packed) {
  extern __shared__ float s_mem[];   // [RF_ROWS][D] listed rows, then [D][RF_THREADS] centre slab
  float* s_x = s_mem;
  float* s_ct = s_mem + RF_ROWS * D;
  const int n_rows = *n_rows_dev;
  const int lane = threadIdx.x & 31;
  if ((int)blockIdx.x * RF_ROWS >= n_rows) return;   // no row group for this CTA
  // outer loop: centre slabs (staged once, all D loads per thread in flight together);
  // inner loop: the row groups of this CTA
  for (int j0 = blockIdx.y * RF_THREADS; j0 < K; j0 += gridDim.y * RF_THREADS) {
    const int j = j0 + threadIdx.x;
    const int jc = j < K ? j : K - 1;   // clamp the address; masked below
    __syncthreads();
#pragma unroll 32
    for (int k = 0; k < D; ++k) s_ct[k * RF_THREADS + threadIdx.x] = __ldg(CT + (int64_t)k * ldct + jc);
    const float cn = __ldg(cnorm + jc);
    for (int q0 = blockIdx.x * RF_ROWS; q0 < n_rows; q0 += gridDim.x * RF_ROWS) {
      const int nr = min(RF_ROWS, n_rows - q0);
      __syncthreads();
      // listed rows transposed to [k][RF_ROWS]: one k of all 8 rows is two broadcast 128-bit loads
      for (int t = threadIdx.x; t < RF_ROWS * D; t += RF_THREADS) {
        const int r = t / D, k = t - r * D;
        s_x[k * RF_ROWS + r] = r < nr ? X[(int64_t)rows[q0 + r] * ldx + k] : 0.f;
      }
      __syncthreads();
      float acc[RF_ROWS];
#pragma unroll
      for (int r = 0; r < RF_ROWS; ++r) acc[r] = 0.f;
      const float4* s_x4 = reinterpret_cast<const float4*>(s_x);
#pragma unroll 4
      for (int k = 0; k < D; ++k) {
        const float c = s_ct[k * RF_THREADS + threadIdx.x];
        const float4 xa = s_x4[2 * k], xb = s_x4[2 * k + 1];
        acc[0] = ed_chain(acc[0], xa.x, c);
        acc[1] = ed_chain(acc[1], xa.y, c);
        acc[2] = ed_chain(acc[2], xa.z, c);
        acc[3] = ed_chain(acc[3], xa.w, c);
        acc[4] = ed_chain(acc[4], xb.x, c);
        acc[5] = ed_chain(acc[5], xb.y, c);
        acc[6] = ed_chain(acc[6], xb.z, c);
        acc[7] = ed_chain(acc[7], xb.w, c);
      }
#pragma unroll
      for (int r = 0; r < RF_ROWS; ++r) {
        const float d = ed_finish(acc[r], cn);
        unsigned long long key = (j < K && d == d) ? rf_pack(d, j) : ~0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
          key = other < key ? other : key;
        }
        if (lane == 0 && r < nr) atomicMin(&packed[q0 + r], key);
      }
    }
  }
}

__global__ void __launch_bounds__(256) k_refine_commit(const int32_t* __restrict__ rows,
                                                       const int32_t* __restrict__ n_rows_dev,
                                                       const unsigned long long* __restrict__ packed,
                                                       int32_t* __restrict__ labels,
                                                       const int32_t* __restrict__ labels_prev,
                                                       int32_t* __restrict__ n_changed, float* __restrict__ best_out) {
  const int n_rows = *n_rows_dev;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n_rows; q += gridDim.x * blockDim.x) {
    const unsigned long long key = packed[q];
    const int64_t row = rows[q];
    int l = (int)(unsigned)(key & 0xffffffffull);
    if (key == ~0ull) l = 0;
    labels[row] = l;
    if (best_out) best_out[row] = rf_unpack(key);
    if (n_changed && labels_prev && labels_prev[row] != l) atomicAdd(n_changed, 1);
  }
}

// exact re-score of a device-side row list; CT = centres transposed [D][ldct], ldct >= K;
// packed[q] must be ~0 for every listed slot (k_tc_select initialises it).  max_rows only
// bounds the grid.
int launch_assign_simt_rows(int64_t max_rows, int64_t K, int64_t D, const float* X, int64_t ldx,
                            const float* CT, int64_t ldct, const float* cnorm, const int32_t* rows,
                            const int32_t* n_rows_dev, unsigned long long* packed, int32_t* labels,
                            const int32_t* labels_prev, int32_t* n_changed, float* best_out, cudaStream_t s) {
  size_t smem = ((size_t)RF_ROWS * D + (size_t)D * RF_THREADS) * 4;
  if (smem > 200 * 1024) {
    set_error("re-score kernel: D=%lld exceeds its shared-memory plan", (long long)D);
    return GDR_EUNSUPPORTED;
  }
  static PerDevice<size_t> smem_set_dev;
  size_t& smem_set = smem_set_dev.get();
  if (smem > 48 * 1024 && smem > smem_set) {
    GDR_CUDA(cudaFuncSetAttribute(k_refine_partial, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  // centre slabs along y (each staged once per CTA), row groups along x: about four CTAs per SM in total
  // (128 threads and <= 56 KB of shared memory each)
  const unsigned gy = (unsigned)std::min<int64_t>(cdiv(K, RF_THREADS), 1024);
  const unsigned gx = (unsigned)std::min<int64_t>(std::max<int64_t>(cdiv(max_rows, RF_ROWS), 1),
                                                  std::max<int64_t>(1, cdiv(4 * kSMs, gy)));
  k_refine_partial<<<dim3(gx, gy), RF_THREADS, smem, s>>>((int)K, (int)D, X, ldx, CT, ldct, cnorm, rows, n_rows_dev,
                                                          packed);
  GDR_LAUNCHED();
  k_refine_commit<<<64, 256, 0, s>>>(rows, n_rows_dev, packed, labels, labels_prev, n_changed, best_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

// M-step gather-sum: one CTA per cluster.  The member rows are staged through shared memory in
// chunks of R rows with fully parallel, coalesced 128-bit loads (8+ independent loads per thread
// in flight), then thread c adds column c of the staged rows IN ASCENDING ROW ORDER — one fp32
// chain per output element, exactly np.add.at / single-thread sklearn order — so the loads are
// parallel while the summation order stays sequential (bit-identical to the oracle).
// kCarry: each chain starts from sums[k][c] (the value at which the previous rank of a row partition ended it) instead
// of +0.0 and the result is written back in place; a CTA reads and writes only its own cluster's row.
template <bool kCarry>
__global__ void __launch_bounds__(256) k_gather_sum(int64_t K, int Dp4, int R,
                                                    const int32_t* __restrict__ mptr,
                                                    const uint32_t* __restrict__ ids,
                                                    const float* __restrict__ X, int64_t ldx,
                                                    float* __restrict__ sums, int64_t lds) {
  extern __shared__ __align__(16) float s_rows[];   // [R][Dp4]
  const int64_t k = blockIdx.x;
  const int b = mptr[k], e = mptr[k + 1];
  const int F4 = Dp4 >> 2;
  constexpr int MAXC = 4;                            // columns per thread: Dp4 <= 1024 per pass
  for (int c0 = 0; c0 < Dp4; c0 += 256 * MAXC) {
    const int w4 = min(F4 - (c0 >> 2), 64 * MAXC);   // float4 columns in this pass
    float acc[MAXC];
#pragma unroll
    for (int q = 0; q < MAXC; ++q) {
      const int c = threadIdx.x + 256 * q;
      acc[q] = kCarry && c < 4 * w4 ? sums[k * lds + c0 + c] : 0.f;
    }
    for (int i = b; i < e; i += R) {
      const int rc = min(R, e - i);
      for (int t = threadIdx.x; t < rc * w4; t += 256) {
        const int r = t / w4, c4 = t - r * w4;
        const float4 v = __ldg(reinterpret_cast<const float4*>(X + (int64_t)ids[i + r] * ldx + c0) + c4);
        *reinterpret_cast<float4*>(&s_rows[r * Dp4 + 4 * c4]) = v;
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < MAXC; ++q) {
        const int c = threadIdx.x + 256 * q;
        if (c < 4 * w4) {
          float a = acc[q];
          for (int r = 0; r < rc; ++r) a = __fadd_rn(a, s_rows[r * Dp4 + c]);
          acc[q] = a;
        }
      }
      __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < MAXC; ++q) {
      const int c = threadIdx.x + 256 * q;
      if (c < 4 * w4) sums[k * lds + c0 + c] = acc[q];
    }
  }
}

// ----------------------------------------------------------------------------
// M-step: membership lists (stable sort by label) + gather-sum through the SpMM
// ----------------------------------------------------------------------------
__global__ void k_label_keys(int64_t N, const int32_t* __restrict__ labels, uint64_t* __restrict__ keys,
                             uint32_t* __restrict__ ids) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N;
       i += (int64_t)gridDim.x * blockDim.x) {
    keys[i] = (uint64_t)(uint32_t)labels[i];
    ids[i] = (uint32_t)i;
  }
}

// rowptr[k] = first sorted position whose key >= k  (keys ascending), k in [0, K]
__global__ void k_bounds_from_sorted(int64_t N, int64_t K, const uint64_t* __restrict__ keys,
                                     int32_t* __restrict__ rowptr) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= N;
       i += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = i == 0 ? -1 : (int64_t)keys[i - 1];
    int64_t hi = i == N ? K : (int64_t)keys[i];
    if (hi > K) hi = K;
    for (int64_t k = lo + 1; k <= hi; ++k) rowptr[k] = (int32_t)i;
  }
}

__global__ void k_counts_from_rowptr(int64_t K, const int32_t* __restrict__ rowptr,
                                     int32_t* __restrict__ counts) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < K;
       i += (int64_t)gridDim.x * blockDim.x)
    counts[i] = rowptr[i + 1] - rowptr[i];
}

__global__ void k_label_hist(int64_t N, int64_t K, const int32_t* __restrict__ labels,
                             int32_t* __restrict__ counts, int32_t* __restrict__ status) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N;
       i += (int64_t)gridDim.x * blockDim.x) {
    int l = labels[i];
    if (l < 0 || l >= K) {
      if (status) atomicOr(status, 1);
    } else {
      atomicAdd(&counts[l], 1);  // integer: order-independent
    }
  }
}

// ----------------------------------------------------------------------------
// finalize: average, shift, empties
// ----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_average(int64_t K, int D, const float* __restrict__ sums,
                                                 int64_t lds, const int32_t* __restrict__ counts,
                                                 const float* __restrict__ C_old, int64_t ldo,
                                                 float* __restrict__ C_new, int64_t ldn,
                                                 double* __restrict__ shift_arr, int mean_mode) {
  int64_t k = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (k >= K) return;
  int cnt = counts[k];
  double sh = 0.0;
  if (cnt > 0) {
    float alpha = 1.0f / (float)cnt;  // sklearn multiplies by the fp32 reciprocal
    for (int c = lane_id(); c < D; c += 32) {
      float v = mean_mode ? __fdiv_rn(sums[k * lds + c], (float)cnt) : __fmul_rn(sums[k * lds + c], alpha);
      C_new[k * ldn + c] = v;
      if (C_old) {
        double d = (double)v - (double)C_old[k * ldo + c];
        sh += d * d;
      }
    }
  } else if (mean_mode) {
    for (int c = lane_id(); c < D; c += 32) C_new[k * ldn + c] = __int_as_float(0x7fc00000);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sh += __shfl_xor_sync(0xffffffffu, sh, o);
  if (lane_id() == 0) shift_arr[k] = sh;
}

// single block: total shift (fixed order), #empty, first argmax of counts; then the
// empty clusters take the centre of the largest cluster and their shift is added.
// sklearn's _average_centers (_k_means_common.pyx:274-295) does this IN PLACE while walking j upwards: an empty
// cluster j < argmax copies the argmax row BEFORE that row has been scaled (the raw sums), j > argmax the mean.
__global__ void __launch_bounds__(1024) k_finalize_tail(int64_t K, int D,
                                                        const float* __restrict__ sums, int64_t lds,
                                                        const int32_t* __restrict__ counts,
                                                        const float* __restrict__ C_old, int64_t ldo,
                                                        float* __restrict__ C_new, int64_t ldn,
                                                        double* __restrict__ shift_arr,
                                                        double* __restrict__ stats, int mean_mode) {
  __shared__ double s_d[1024];
  __shared__ int s_cnt[1024], s_idx[1024], s_emp[1024];
  int t = threadIdx.x;
  int bc = -1, bi = 0, ne = 0;
  for (int64_t k = t; k < K; k += 1024) {
    int c = counts[k];
    if (c > bc) {
      bc = c;
      bi = (int)k;
    }
    if (c == 0) ++ne;
  }
  s_cnt[t] = bc;
  s_idx[t] = bi;
  s_emp[t] = ne;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (t < o) {
      if (s_cnt[t + o] > s_cnt[t] || (s_cnt[t + o] == s_cnt[t] && s_idx[t + o] < s_idx[t])) {
        s_cnt[t] = s_cnt[t + o];
        s_idx[t] = s_idx[t + o];
      }
      s_emp[t] += s_emp[t + o];
    }
    __syncthreads();
  }
  const int amax = s_idx[0];
  const int n_empty = s_emp[0];
  if (!mean_mode && n_empty > 0) {
    // one warp per empty cluster (strided), copies row amax and recomputes its shift
    int w = t >> 5, l = t & 31;
    for (int64_t k = w; k < K; k += 32) {
      if (counts[k] != 0) continue;
      double sh = 0.0;
      for (int c = l; c < D; c += 32) {
        float v = k < amax ? sums[(int64_t)amax * lds + c] : C_new[(int64_t)amax * ldn + c];
        C_new[k * ldn + c] = v;
        if (C_old) {
          double d = (double)v - (double)C_old[k * ldo + c];
          sh += d * d;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sh += __shfl_xor_sync(0xffffffffu, sh, o);
      if (l == 0) shift_arr[k] = sh;
    }
    __syncthreads();
  }
  double s = 0.0;
  for (int64_t k = t; k < K; k += 1024) s += shift_arr[k];
  s_d[t] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (t < o) s_d[t] += s_d[t + o];
    __syncthreads();
  }
  if (t == 0) {
    stats[0] = s_d[0];
    stats[1] = (double)n_empty;
  }
}

// ----------------------------------------------------------------------------
// inertia / per-row distance to own centre
// ----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_row_dist(int64_t N, int D, const float* __restrict__ X,
                                                  int64_t ldx, const float* __restrict__ C, int64_t ldc,
                                                  const int32_t* __restrict__ labels,
                                                  float* __restrict__ dist_out,
                                                  double* __restrict__ block_part) {
  // one warp per row; fp32 squared differences, fixed-order shuffle tree
  __shared__ double s_w[8];
  int w = threadIdx.x >> 5;
  int64_t row = (int64_t)blockIdx.x * 8 + w;
  float s = 0.f;
  if (row < N) {
    int j = labels[row];
    for (int c = lane_id(); c < D; c += 32) {
      float d = __fsub_rn(X[row * ldx + c], C[(int64_t)j * ldc + c]);
      s = fmaf(d, d, s);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane_id() == 0) {
    if (row < N && dist_out) dist_out[row] = s;
    s_w[w] = row < N ? (double)s : 0.0;
  }
  __syncthreads();
  if (threadIdx.x == 0 && block_part) {
    double a = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) a += s_w[i];
    block_part[blockIdx.x] = a;
  }
}

__global__ void __launch_bounds__(1024) k_sum_f64(int64_t n, const double* __restrict__ in,
                                                  double* __restrict__ out) {
  __shared__ double s_d[1024];
  int t = threadIdx.x;
  double s = 0.0;
  for (int64_t i = t; i < n; i += 1024) s += in[i];
  s_d[t] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (t < o) s_d[t] += s_d[t + o];
    __syncthreads();
  }
  if (t == 0) out[0] = s_d[0];
}

// argmax of a float array (first index wins); two-stage, deterministic
__global__ void __launch_bounds__(256) k_argmax_part(int64_t n, const float* __restrict__ d,
                                                     float* __restrict__ pv, int32_t* __restrict__ pi) {
  __shared__ float sv[256];
  __shared__ int si[256];
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    float v = d[i];
    if (v > bv || (v == bv && (int)i < bi)) {
      bv = v;
      bi = (int)i;
    }
  }
  sv[threadIdx.x] = bv;
  si[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      float ov = sv[threadIdx.x + o];
      int oi = si[threadIdx.x + o];
      if (ov > sv[threadIdx.x] || (ov == sv[threadIdx.x] && oi < si[threadIdx.x])) {
        sv[threadIdx.x] = ov;
        si[threadIdx.x] = oi;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    pv[blockIdx.x] = sv[0];
    pi[blockIdx.x] = si[0];
  }
}

// moves sample far (argmax over the partials) from its cluster to `new_cluster`
__global__ void __launch_bounds__(256) k_relocate_one(int nparts, const float* __restrict__ pv,
                                                      const int32_t* __restrict__ pi, int D,
                                                      const float* __restrict__ X, int64_t ldx,
                                                      const int32_t* __restrict__ labels,
                                                      float* __restrict__ sums, int64_t lds,
                                                      int32_t* __restrict__ counts, int new_cluster,
                                                      float* __restrict__ dist) {
  __shared__ int s_far;
  if (threadIdx.x == 0) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = 0; i < nparts; ++i) {
      if (pv[i] > bv || (pv[i] == bv && pi[i] < bi)) {
        bv = pv[i];
        bi = pi[i];
      }
    }
    s_far = bi;
  }
  __syncthreads();
  int far = s_far;
  int old = labels[far];
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float x = X[(int64_t)far * ldx + c];
    sums[(int64_t)old * lds + c] = __fsub_rn(sums[(int64_t)old * lds + c], x);
    sums[(int64_t)new_cluster * lds + c] = x;
  }
  if (threadIdx.x == 0) {
    counts[new_cluster] = 1;
    counts[old] -= 1;
    dist[far] = -1.f;  // never picked again
  }
}

// ---- MiniBatchKMeans centre update (sklearn/cluster/_k_means_minibatch.pyx:56-110 update_center_dense) --------
// one warp per cluster, lanes over the feature columns; the batch is walked IN ORDER so that every centre element
// is the same fp32 chain as sklearn's:  acc = old * weight ; acc += x (members in batch order) ; weight += count ;
// acc *= 1 / weight.  A cluster without members in the batch copies its old centre.
__global__ void __launch_bounds__(256) k_minibatch_update(int64_t B, int64_t K, int D, const float* __restrict__ Xb,
                                                          int64_t ldx, const int32_t* __restrict__ labels,
                                                          const float* __restrict__ C_old, int64_t ldo,
                                                          float* __restrict__ C_new, int64_t ldn,
                                                          float* __restrict__ weight_sums) {
  const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c >= K) return;
  const int lane = lane_id();
  constexpr int MAXC = 8;                       // D <= 256 per pass
  for (int c0 = 0; c0 < D; c0 += 32 * MAXC) {
    float acc[MAXC];
    const float w = weight_sums[c];
#pragma unroll
    for (int q = 0; q < MAXC; ++q) {
      const int col = c0 + q * 32 + lane;
      acc[q] = col < D ? __fmul_rn(C_old[c * ldo + col], w) : 0.f;
    }
    int cnt = 0;
    for (int64_t s0 = 0; s0 < B; s0 += 32) {
      const int64_t s = s0 + lane;
      const unsigned hit = __ballot_sync(0xffffffffu, s < B && labels[s] == (int32_t)c);
      unsigned m = hit;
      while (m) {                               // members of this 32-sample window, ascending
        const int j = __ffs(m) - 1;
        m &= m - 1;
        const float* x = Xb + (s0 + j) * ldx;
#pragma unroll
        for (int q = 0; q < MAXC; ++q) {
          const int col = c0 + q * 32 + lane;
          if (col < D) acc[q] = __fadd_rn(acc[q], x[col]);
        }
      }
      cnt += __popc(hit);
    }
    if (cnt > 0) {
      const float wn = __fadd_rn(w, (float)cnt);     // wsum accumulates 1.0f per member: exact
      const float alpha = __fdiv_rn(1.0f, wn);
#pragma unroll
      for (int q = 0; q < MAXC; ++q) {
        const int col = c0 + q * 32 + lane;
        if (col < D) C_new[c * ldn + col] = __fmul_rn(acc[q], alpha);
      }
      __syncwarp();
      if (lane == 0 && c0 + 32 * MAXC >= D) weight_sums[c] = wn;
    } else {
#pragma unroll
      for (int q = 0; q < MAXC; ++q) {
        const int col = c0 + q * 32 + lane;
        if (col < D) C_new[c * ldn + col] = C_old[c * ldo + col];
      }
    }
  }
}

// ---- MiniBatchKMeans batch assembly on a row partition (gdr_minibatch_batch_dist) -----------------------------
// pack: the n batch positions this rank owns (order[0..n), batch order) -> rows of the compact buffer P [n][ldp],
// padding columns zero.  One warp per row.  A position whose row lies outside [row_lo, row_lo + n_local) (a plan that
// does not match the row blocks) packs a zero row instead of reading outside X.
__global__ void __launch_bounds__(256) k_mb_pack(int64_t n, int D, int ldp, const int64_t* __restrict__ idx,
                                                 const int32_t* __restrict__ order, int64_t row_lo, int64_t n_local,
                                                 const float* __restrict__ X, int64_t ldx, float* __restrict__ P) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n) return;
  const int64_t g = idx[order[r]] - row_lo;
  const bool own = g >= 0 && g < n_local;
  for (int c = lane_id(); c < ldp; c += 32) P[r * ldp + c] = (own && c < D) ? X[g * ldx + c] : 0.f;
}

// place: record k of the exchanged buffers (every rank's compact rows in rank order = the order of `order`) -> batch
// position order[k]: Xb row (ldb columns, zero beyond ldp) and, when labels travel, its label.  One warp per record.
__global__ void __launch_bounds__(256) k_mb_place(int64_t m, int ldp, const int32_t* __restrict__ order,
                                                  const float* __restrict__ P, const int32_t* __restrict__ Lp,
                                                  float* __restrict__ Xb, int64_t ldb, int32_t* __restrict__ labels_b) {
  const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= m) return;
  const int64_t j = order[k];
  for (int64_t c = lane_id(); c < ldb; c += 32) Xb[j * ldb + c] = c < ldp ? P[k * ldp + c] : 0.f;
  if (labels_b && lane_id() == 0) labels_b[j] = Lp[k];
}

// ---- distributed relocation (lloyd.cu: relocate_distributed) ----------------------------------
// candidate record: [dist, rank (int bits), old label (int bits), x[0..D)]
__global__ void __launch_bounds__(256) k_pick_candidate(int nparts, const float* __restrict__ pv,
                                                        const int32_t* __restrict__ pi, int D,
                                                        const float* __restrict__ X, int64_t ldx,
                                                        const int32_t* __restrict__ labels, float* __restrict__ dist,
                                                        float* __restrict__ rec, int rank) {
  __shared__ int s_far;
  __shared__ float s_val;
  if (threadIdx.x == 0) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = 0; i < nparts; ++i) {
      if (pv[i] > bv || (pv[i] == bv && pi[i] < bi)) {
        bv = pv[i];
        bi = pi[i];
      }
    }
    s_far = bi;
    s_val = bv;
  }
  __syncthreads();
  const int far = s_far;
  const float val = s_val;
  if (!(val >= 0.f) || far == 0x7fffffff) {   // no row left on this rank
    if (threadIdx.x == 0) rec[0] = -1.f;
    return;
  }
  for (int c = threadIdx.x; c < D; c += blockDim.x) rec[3 + c] = X[(int64_t)far * ldx + c];
  if (threadIdx.x == 0) {
    rec[0] = val;
    rec[1] = __int_as_float(rank);
    rec[2] = __int_as_float(labels[far]);
    dist[far] = -1.f;  // never picked again
  }
}

__global__ void k_fill_f32(int64_t n, float* __restrict__ p, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

// applies the global choice: the e-th empty cluster receives candidate order[e] (sequentially: a cluster may lose
// several rows and the fp32 subtraction order is part of the result)
__global__ void __launch_bounds__(256) k_relocate_apply(int ne, const int32_t* __restrict__ order,
                                                        const int32_t* __restrict__ empties, const float* __restrict__ allrec,
                                                        int D, float* __restrict__ sums, int64_t lds,
                                                        int32_t* __restrict__ counts) {
  for (int e = 0; e < ne; ++e) {
    const int j = order[e];
    if (j < 0) break;
    const float* r = allrec + (int64_t)j * (D + 3);
    const int old = __float_as_int(r[2]);
    const int nw = empties[e];
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
      const float x = r[3 + c];
      sums[(int64_t)old * lds + c] = __fsub_rn(sums[(int64_t)old * lds + c], x);
      sums[(int64_t)nw * lds + c] = x;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      counts[nw] = 1;
      counts[old] -= 1;
    }
    __syncthreads();
  }
}

// second pass of the variance: per-block sums of (x - mean) and (x - mean)^2
__global__ void __launch_bounds__(256) k_colvar_partial(int64_t N, int D, const float* __restrict__ X, int64_t ldx,
                                                        const double* __restrict__ mean, double* __restrict__ part) {
  __shared__ double s_sum[8][33], s_sq[8][33];
  int64_t r0 = (int64_t)blockIdx.x * CC_ROWS_PER_BLOCK;
  int64_t r1 = min(N, r0 + CC_ROWS_PER_BLOCK);
  for (int c0 = 0; c0 < D; c0 += 32) {
    int c = c0 + threadIdx.x;
    double su = 0.0, sq = 0.0;
    if (c < D) {
      const double m = mean[c];
      for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
        double x = (double)X[r * ldx + c] - m;
        su += x;
        sq += x * x;
      }
    }
    s_sum[threadIdx.y][threadIdx.x] = su;
    s_sq[threadIdx.y][threadIdx.x] = sq;
    __syncthreads();
    if (threadIdx.y == 0 && c < D) {
      double a = 0.0, b = 0.0;
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        a += s_sum[y][threadIdx.x];
        b += s_sq[y][threadIdx.x];
      }
      part[((int64_t)blockIdx.x * D + c) * 2 + 0] = a;
      part[((int64_t)blockIdx.x * D + c) * 2 + 1] = b;
    }
    __syncthreads();
  }
}

// params[0..D) = mean, params[D..2D) = scale (fp64); fp32 copies for the transform.
// sums2 == nullptr: first pass (mean only).
__global__ void k_scale_params(int64_t N, int D, const double* __restrict__ sums1, const double* __restrict__ sums2,
                               double* __restrict__ params, float* __restrict__ mean32, float* __restrict__ scale32) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  const double mean = sums1[c] / (double)N;
  params[c] = mean;
  mean32[c] = (float)mean;
  if (sums2) {
    const double var = sums2[D + c] / (double)N;
    // sklearn.preprocessing._data._is_constant_feature: var <= N*eps*var + (N*mean*eps)^2
    const double eps = 2.220446049250313e-16;
    const double bound = (double)N * eps * var + ((double)N * mean * eps) * ((double)N * mean * eps);
    double scale = sqrt(var);
    if (var <= bound) scale = 1.0;
    params[D + c] = scale;
    scale32[c] = (float)scale;
  }
}

__global__ void k_standardize(int64_t N, int D, const float* __restrict__ X, int64_t ldx, const float* __restrict__ mean,
                              const float* __restrict__ scale, float* __restrict__ out, int64_t ldo) {
  int64_t total = N * (int64_t)D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / D;
    int c = (int)(i - r * D);
    out[r * ldo + c] = __fdiv_rn(__fsub_rn(X[r * ldx + c], mean[c]), scale[c]);
  }
}

// fixed-order reduction of the per-block partials: out[c] = sum, out[D + c] = sum of squares
__global__ void __launch_bounds__(256) k_colstats_reduce(int D, int nblocks, const double* __restrict__ part,
                                                         double* __restrict__ out) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  double a = 0.0, b = 0.0;
  for (int i = 0; i < nblocks; ++i) {
    a += part[((int64_t)i * D + c) * 2 + 0];
    b += part[((int64_t)i * D + c) * 2 + 1];
  }
  out[c] = a;
  out[D + c] = b;
}

}  // namespace gdr

using namespace gdr;

namespace gdr {

int64_t relocate_candidates_ws_bytes(int64_t N) { return ws_need(N > 0 ? N : 1, 4) + 2 * ws_need(1024, 4) + 256; }

// this rank's `ne` farthest rows (distance to their own centre, largest first, ties by row order) as records
int relocate_candidates(int64_t N, int64_t D, const float* X, int64_t ldx, const float* C_old, int64_t ldc,
                        const int32_t* labels, int ne, int rank, float* rec, void* ws, int64_t ws_bytes, cudaStream_t s) {
  if (ws_bytes < relocate_candidates_ws_bytes(N)) {
    set_error("relocate_candidates: workspace too small");
    return GDR_EWORKSPACE;
  }
  const int64_t rec_w = D + 3;
  k_fill_f32<<<(unsigned)std::min<int64_t>(cdiv((int64_t)ne * rec_w, 256), 1024), 256, 0, s>>>((int64_t)ne * rec_w, rec, -1.f);
  GDR_LAUNCHED();
  if (N == 0) return GDR_OK;
  Workspace W(ws, ws_bytes);
  float* dist = W.take<float>(N);
  float* pv = W.take<float>(1024);
  int32_t* pi = W.take<int32_t>(1024);
  k_row_dist<<<(unsigned)cdiv(N, 8), 256, 0, s>>>(N, (int)D, X, ldx, C_old, ldc, labels, dist, nullptr);
  GDR_LAUNCHED();
  const int nparts = (int)std::min<int64_t>(1024, cdiv(N, 256));
  const int take = (int)std::min<int64_t>(ne, N);
  for (int e = 0; e < take; ++e) {
    k_argmax_part<<<nparts, 256, 0, s>>>(N, dist, pv, pi);
    GDR_LAUNCHED();
    k_pick_candidate<<<1, 256, 0, s>>>(nparts, pv, pi, (int)D, X, ldx, labels, dist, rec + (int64_t)e * rec_w, rank);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

int relocate_apply(int ne, const int32_t* order_dev, const int32_t* empties_dev, const float* allrec, int64_t D,
                   float* sums, int64_t lds, int32_t* counts, cudaStream_t s) {
  k_relocate_apply<<<1, 256, 0, s>>>(ne, order_dev, empties_dev, allrec, (int)D, sums, lds, counts);
  GDR_LAUNCHED();
  return GDR_OK;
}

// The membership lists of gdr_segment_sum: ids = the rows stably sorted by label, mptr[k] .. mptr[k + 1] = cluster k's
// range of them (labels outside [0, K) fall outside every range).  Workspace layout: segment_members_carve.
struct SegmentMembers {
  uint64_t* keys;
  uint32_t* ids;
  int32_t* mptr;
  void* sws;
  int64_t sws_bytes, off;
};

SegmentMembers segment_members_carve(void* ws, int64_t N, int64_t K) {
  Workspace W(ws, INT64_MAX);
  SegmentMembers m;
  m.keys = W.take<uint64_t>(N);
  m.ids = W.take<uint32_t>(N);
  m.mptr = W.take<int32_t>(K + 1);
  m.sws_bytes = sort_pairs_ws_bytes(N);
  m.sws = W.take<char>(m.sws_bytes);
  m.off = W.off;
  return m;
}

int segment_members(int64_t N, int64_t K, const int32_t* labels, const SegmentMembers& m, cudaStream_t s) {
  unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(N, 256), kSMs * 16));
  if (N > 0) {
    k_label_keys<<<grid, 256, 0, s>>>(N, labels, m.keys, m.ids);
    GDR_LAUNCHED();
    int bits = 1;
    while ((1ll << bits) < K) ++bits;
    int rc = sort_pairs(N, bits, m.keys, m.ids, m.sws, m.sws_bytes, s);
    if (rc) return rc;
  }
  k_bounds_from_sorted<<<grid, 256, 0, s>>>(N, K, m.keys, m.mptr);
  GDR_LAUNCHED();
  return GDR_OK;
}

// k_gather_sum over the membership lists: R rows of Dp4 floats are staged per step (48 KB of shared memory)
template <bool kCarry>
void gather_sum(int64_t K, int64_t D, const SegmentMembers& m, const float* X, int64_t ldx, float* sums, int64_t lds,
                cudaStream_t s) {
  const int Dp4 = (int)align_up(D, 4);
  const int R = (int)std::max<int64_t>(1, std::min<int64_t>(64, (48 * 1024) / ((int64_t)Dp4 * 4)));
  ProfileScope prof(PROF_SPMM + 1, s);
  k_gather_sum<kCarry><<<(unsigned)K, 256, (size_t)R * Dp4 * 4, s>>>(K, Dp4, R, m.mptr, m.ids, X, ldx, sums, lds);
}

}  // namespace gdr

extern "C" {

int64_t gdr_center_columns_ws_bytes(int64_t N, int64_t D) {
  int64_t nb = cdiv(N > 0 ? N : 1, CC_ROWS_PER_BLOCK);
  return ws_need(nb * D * 2, 8) + ws_need(D, 8) + 256;
}

int gdr_center_columns(int64_t N, int64_t D, const float* X, int64_t ldx, float* mean_out,
                       double* var_mean_out, float* Xc, int64_t ldxc, void* ws, int64_t ws_bytes,
                       gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && D > 0 && X && mean_out && ldx >= D, "center_columns: bad arguments");
  GDR_CHECK_ARG(!Xc || ldxc >= D, "center_columns: ldxc < D");
  if (ws_bytes < gdr_center_columns_ws_bytes(N, D)) {
    set_error("center_columns: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  int nb = (int)cdiv(N, CC_ROWS_PER_BLOCK);
  Workspace W(ws, ws_bytes);
  double* part = W.take<double>((int64_t)nb * D * 2);
  double* var_col = W.take<double>(D);
  k_colstats_partial<<<nb, dim3(32, 8), 0, s>>>(N, (int)D, X, ldx, part);
  GDR_LAUNCHED();
  k_colstats_final<<<(unsigned)cdiv(D, 256), 256, 0, s>>>(N, (int)D, nb, part, mean_out, var_col);
  GDR_LAUNCHED();
  if (var_mean_out) {
    k_var_mean<<<1, 32, 0, s>>>((int)D, var_col, var_mean_out);
    GDR_LAUNCHED();
  }
  if (Xc) {
    int ldpad = (int)std::min<int64_t>(ldxc, align_up(D, 4));
    int64_t total = N * ldpad;
    unsigned grid = (unsigned)std::min<int64_t>(cdiv(total, 256), kSMs * 16);
    k_sub_rowvec<<<grid, 256, 0, s>>>(N, (int)D, ldpad, X, ldx, mean_out, Xc, ldxc);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

// Column sums / sums of squares in fp64 (sums_out[0..D) = sum, [D..2D) = sum of squares) — the
// per-rank half of the mean/variance when rows are partitioned across GPUs.
int gdr_column_sums(int64_t N, int64_t D, const float* X, int64_t ldx, double* sums_out, void* ws,
                    int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && D > 0 && sums_out && ldx >= D, "column_sums: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  if (N == 0) {
    GDR_CUDA(cudaMemsetAsync(sums_out, 0, 2 * D * 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(X, "column_sums: null X");
  if (ws_bytes < gdr_center_columns_ws_bytes(N, D)) {
    set_error("column_sums: workspace too small");
    return GDR_EWORKSPACE;
  }
  int nb = (int)cdiv(N, CC_ROWS_PER_BLOCK);
  double* part = (double*)ws;
  k_colstats_partial<<<nb, dim3(32, 8), 0, s>>>(N, (int)D, X, ldx, part);
  GDR_LAUNCHED();
  k_colstats_reduce<<<(unsigned)cdiv(D, 256), 256, 0, s>>>((int)D, nb, part, sums_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

// StandardScaler(with_mean=True, with_std=True).fit_transform (distill_recsys.py:172):
// mean and population variance per column in fp64 (two passes: sum, then sum of squared
// deviations), scale = sqrt(var) with constant columns -> 1 (sklearn _is_constant_feature),
// out = fp32((x - fp32(mean)) / fp32(scale)) — bit-exact with sklearn on the golden vector.
int64_t gdr_standard_scale_ws_bytes(int64_t N, int64_t D) {
  return gdr_center_columns_ws_bytes(N, D) + 3 * ws_need(2 * D, 8) + 2 * ws_need(D, 4) + 256;
}

int gdr_standard_scale(int64_t N, int64_t D, const float* X, int64_t ldx, float* out, int64_t ldo,
                       double* mean_out /*nullable, f64[D]*/, double* scale_out /*nullable, f64[D]*/, void* ws,
                       int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && D > 0 && X && out && ldx >= D && ldo >= D, "standard_scale: bad arguments");
  if (ws_bytes < gdr_standard_scale_ws_bytes(N, D)) {
    set_error("standard_scale: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int nb = (int)cdiv(N, CC_ROWS_PER_BLOCK);
  Workspace W(ws, ws_bytes);
  double* part = (double*)W.take<char>(gdr_center_columns_ws_bytes(N, D));
  double* sums1 = W.take<double>(2 * D);
  double* sums2 = W.take<double>(2 * D);
  double* mean64 = W.take<double>(2 * D);  // [mean | scale]
  float* mean32 = W.take<float>(D);
  float* scale32 = W.take<float>(D);
  k_colstats_partial<<<nb, dim3(32, 8), 0, s>>>(N, (int)D, X, ldx, part);
  GDR_LAUNCHED();
  k_colstats_reduce<<<(unsigned)cdiv(D, 256), 256, 0, s>>>((int)D, nb, part, sums1);
  GDR_LAUNCHED();
  k_scale_params<<<(unsigned)cdiv(D, 256), 256, 0, s>>>(N, (int)D, sums1, nullptr, mean64, mean32, scale32);
  GDR_LAUNCHED();
  k_colvar_partial<<<nb, dim3(32, 8), 0, s>>>(N, (int)D, X, ldx, mean64, part);
  GDR_LAUNCHED();
  k_colstats_reduce<<<(unsigned)cdiv(D, 256), 256, 0, s>>>((int)D, nb, part, sums2);
  GDR_LAUNCHED();
  k_scale_params<<<(unsigned)cdiv(D, 256), 256, 0, s>>>(N, (int)D, sums1, sums2, mean64, mean32, scale32);
  GDR_LAUNCHED();
  int64_t total = N * D;
  k_standardize<<<(unsigned)std::min<int64_t>(cdiv(total, 256), kSMs * 16), 256, 0, s>>>(N, (int)D, X, ldx, mean32,
                                                                                      scale32, out, ldo);
  GDR_LAUNCHED();
  if (mean_out) GDR_CUDA(cudaMemcpyAsync(mean_out, mean64, D * 8, cudaMemcpyDeviceToDevice, s));
  if (scale_out) GDR_CUDA(cudaMemcpyAsync(scale_out, mean64 + D, D * 8, cudaMemcpyDeviceToDevice, s));
  return GDR_OK;
}

// Xc = X - mean (fp32 subtract, padding columns zeroed) — sklearn/_kmeans.py:1489
// second pass of StandardScaler on a row block: out[0..D) = sum (x - mean), out[D..2D) = sum (x - mean)^2 (fp64), so that
// the blocks of a row partition can be all-reduced (distill_recsys.py:172 on row-partitioned embeddings)
int gdr_column_moments(int64_t N, int64_t D, const float* X, int64_t ldx, const double* mean64, double* sums_out,
                       void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && D > 0 && mean64 && sums_out, "column_moments: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  if (N == 0) {
    GDR_CUDA(cudaMemsetAsync(sums_out, 0, 2 * D * 8, s));
    return GDR_OK;
  }
  GDR_CHECK_ARG(X && ldx >= D, "column_moments: null X");
  if (ws_bytes < gdr_center_columns_ws_bytes(N, D)) {
    set_error("column_moments: workspace too small");
    return GDR_EWORKSPACE;
  }
  const int nb = (int)cdiv(N, CC_ROWS_PER_BLOCK);
  double* part = (double*)ws;
  k_colvar_partial<<<nb, dim3(32, 8), 0, s>>>(N, (int)D, X, ldx, mean64, part);
  GDR_LAUNCHED();
  k_colstats_reduce<<<(unsigned)cdiv(D, 256), 256, 0, s>>>((int)D, nb, part, sums_out);
  GDR_LAUNCHED();
  return GDR_OK;
}

// out = fp32((x - mean) / scale) with given fp32 column parameters (StandardScaler.transform)
int gdr_standardize_apply(int64_t N, int64_t D, const float* X, int64_t ldx, const float* mean32, const float* scale32,
                          float* out, int64_t ldo, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && D > 0 && mean32 && scale32, "standardize_apply: bad arguments");
  if (N == 0) return GDR_OK;
  GDR_CHECK_ARG(X && out && ldx >= D && ldo >= D, "standardize_apply: null pointer");
  const int64_t total = N * D;
  k_standardize<<<(unsigned)std::min<int64_t>(cdiv(total, 256), kSMs * 16), 256, 0, (cudaStream_t)stream>>>(
      N, (int)D, X, ldx, mean32, scale32, out, ldo);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_center_apply(int64_t N, int64_t D, const float* X, int64_t ldx, const float* mean, float* Xc,
                     int64_t ldxc, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && D > 0 && mean && ldx >= D && ldxc >= D, "center_apply: bad arguments");
  if (N == 0) return GDR_OK;
  GDR_CHECK_ARG(X && Xc, "center_apply: null pointer");
  int ldpad = (int)std::min<int64_t>(ldxc, align_up(D, 4));
  int64_t total = N * ldpad;
  unsigned grid = (unsigned)std::min<int64_t>(cdiv(total, 256), kSMs * 16);
  k_sub_rowvec<<<grid, 256, 0, (cudaStream_t)stream>>>(N, (int)D, ldpad, X, ldx, mean, Xc, ldxc);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_add_row_vector(int64_t rows, int64_t D, float* X, int64_t ldx, const float* v, float sign,
                       gdr_stream_t stream) {
  GDR_CHECK_ARG(rows >= 0 && D >= 0, "add_row_vector: negative size");
  if (rows == 0 || D == 0) return GDR_OK;
  GDR_CHECK_ARG(X && v && ldx >= D, "add_row_vector: bad arguments");
  unsigned grid = (unsigned)std::min<int64_t>(cdiv(rows * D, 256), kSMs * 16);
  k_add_rowvec<<<grid, 256, 0, (cudaStream_t)stream>>>(rows, (int)D, X, ldx, v, sign);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_kmeans_assign_ws_bytes(int64_t N, int64_t K, int64_t D, int precision_mode) {
  int64_t b = ws_need(K, 4) + 256;
  if (precision_mode == 1) b = kmeans_assign_tc_total_ws_bytes(N, K, D);
  return b;
}

int gdr_kmeans_assign(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx, const float* C,
                      int64_t ldc, int32_t* labels, const int32_t* labels_prev,
                      int32_t* n_changed_dev, float* best_out, int precision_mode, void* ws,
                      int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && K > 0 && D > 0, "kmeans_assign: bad sizes");
  if (N == 0) return GDR_OK;
  GDR_CHECK_ARG(X && C && labels, "kmeans_assign: null pointer");
  GDR_CHECK_ARG(ldx % 4 == 0 && ldc % 4 == 0 && ldx >= D && ldc >= D &&
                    ((uintptr_t)X & 15) == 0 && ((uintptr_t)C & 15) == 0,
                "kmeans_assign: X/C need 16B alignment and ld %% 4 == 0");
  GDR_CHECK_ARG(K < (1ll << 31) && D < (1 << 20), "kmeans_assign: K or D too large");
  GDR_CHECK_ARG(precision_mode == 0 || precision_mode == 1, "kmeans_assign: precision_mode");
  if (ws_bytes < gdr_kmeans_assign_ws_bytes(N, K, D, precision_mode)) {
    set_error("kmeans_assign: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (precision_mode == 1) {
    return kmeans_assign_tc(N, K, D, X, ldx, C, ldc, labels, labels_prev, n_changed_dev, best_out,
                            ws, ws_bytes, s);
  }
  Workspace W(ws, ws_bytes);
  float* cnorm = W.take<float>(K);
  k_row_sqnorm<<<(unsigned)cdiv(K, 8), 256, 0, s>>>(K, (int)D, C, ldc, cnorm);
  GDR_LAUNCHED();
  {
    ProfileScope prof(PROF_ASSIGN, s);
    k_assign_simt<<<(unsigned)cdiv(N, AS_BM), AS_THREADS, 0, s>>>(N, (int)K, (int)D, X, ldx, C, ldc, cnorm,
                                                                 labels, labels_prev, n_changed_dev,
                                                                 best_out, nullptr, nullptr);
  }
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_segment_sum_ws_bytes(int64_t N, int64_t K, int64_t D) {
  (void)D;
  return ws_need(N, 8) + ws_need(N, 4) + ws_need(K + 1, 4) + sort_pairs_ws_bytes(N) + 256;
}

int gdr_segment_sum(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx,
                    const int32_t* labels, float* sums, int64_t lds, int32_t* counts, void* ws,
                    int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && K > 0 && D > 0, "segment_sum: bad sizes");
  GDR_CHECK_ARG(X && labels && sums, "segment_sum: null pointer");
  GDR_CHECK_ARG(ldx % 4 == 0 && lds % 4 == 0 && ldx >= align_up(D, 4) && lds >= align_up(D, 4) &&
                    ((uintptr_t)X & 15) == 0 && ((uintptr_t)sums & 15) == 0,
                "segment_sum: X/sums need 16B alignment and ld %% 4 == 0, ld >= D rounded to 4");
  GDR_CHECK_ARG(N < (1ll << 31), "segment_sum: N too large");
  if (ws_bytes < gdr_segment_sum_ws_bytes(N, K, D)) {
    set_error("segment_sum: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const SegmentMembers m = segment_members_carve(ws, N, K);
  if (int rc = segment_members(N, K, labels, m, s)) return rc;
  if (counts) {
    k_counts_from_rowptr<<<(unsigned)cdiv(K, 256), 256, 0, s>>>(K, m.mptr, counts);
    GDR_LAUNCHED();
  }
  gather_sum<false>(K, D, m, X, ldx, sums, lds, s);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_segment_sum_dist_ws_bytes(int64_t n_local, int64_t K, int64_t D) {
  (void)D;
  return ws_need(1, 4) + segment_members_carve(nullptr, n_local, K).off;   // [label status | members]
}

int gdr_segment_sum_dist(gdr_comm_t* comm, int64_t row_lo, int64_t n_local, int64_t K, int64_t D, const float* X,
                         int64_t ldx, const int32_t* labels, float* sums, int64_t lds, int32_t* counts, void* ws,
                         int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(comm, "segment_sum_dist: null communicator");
  const int world = comm->world, rank = comm->rank;
  cudaStream_t s = (cudaStream_t)stream;
  // local checks are decided collectively in comm_entry_check: an early return would leave the others in a collective
  int local_rc = GDR_OK;
  if (!(row_lo >= 0 && n_local >= 0 && n_local < (1ll << 31) && K > 0 && K < (1ll << 31) && D > 0 && sums && counts &&
        lds % 4 == 0 && lds >= align_up(D, 4) && ((uintptr_t)sums & 15) == 0 &&
        (n_local == 0 || (X && labels && ldx % 4 == 0 && ldx >= align_up(D, 4) && ((uintptr_t)X & 15) == 0)))) {
    set_error("segment_sum_dist: bad arguments (sizes, null pointer, or X/sums without 16B alignment and ld %% 4 == 0, "
              "ld >= D rounded to 4)");
    local_rc = GDR_EINVAL;
  } else if (!ws || ws_bytes < gdr_segment_sum_dist_ws_bytes(n_local, K, D)) {
    set_error("segment_sum_dist: workspace too small");
    local_rc = GDR_EWORKSPACE;
  }
  if (local_rc == GDR_OK) {
    // this rank's counts; a label outside [0, K) is this rank's GDR_ERANGE
    int32_t* status = (int32_t*)ws;
    int32_t bad = 0;
    int rc = gdr_label_histogram(n_local, K, labels, counts, status, stream);
    if (rc == GDR_OK && (cudaMemcpyAsync(&bad, status, 4, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                         cudaStreamSynchronize(s) != cudaSuccess)) {
      set_error("segment_sum_dist: read-back of the label check failed");
      rc = GDR_ECUDA;
    }
    if (rc == GDR_OK && bad) {
      set_error("segment_sum_dist: a label lies outside [0, %lld)", (long long)K);
      rc = GDR_ERANGE;
    }
    local_rc = rc;
  }
  std::vector<int64_t> row_off((size_t)world + 1);
  int rc = comm_entry_check(comm, s, "segment_sum_dist", local_rc, row_lo, n_local, -1, {K, D, lds}, "K, D or lds", 0,
                            row_off.data());
  if (rc != GDR_OK) return rc;
  if (row_off[world] >= (1ll << 31)) {
    set_error("segment_sum_dist: %lld rows in all, the counts need fewer than 2^31", (long long)row_off[world]);
    return GDR_EINVAL;
  }

  // sort before the receive, so that the ranks sort concurrently
  const SegmentMembers m = segment_members_carve((char*)ws + ws_need(1, 4), n_local, K);
  if ((rc = segment_members(n_local, K, labels, m, s))) return rc;
  // each chain of rank q continues where rank q - 1 ended it; rank 0 starts from +0.0, an empty rank hands on what it got
  const int64_t bytes = K * lds * 4;
  if (rank > 0) {
    if ((rc = comm_recv(comm, sums, bytes, rank - 1, s))) return rc;
  } else {
    GDR_CUDA(cudaMemsetAsync(sums, 0, bytes, s));
  }
  if (n_local > 0) {
    gather_sum<true>(K, D, m, X, ldx, sums, lds, s);
    GDR_LAUNCHED();
  }
  if (rank + 1 < world && (rc = comm_send(comm, sums, bytes, rank + 1, s))) return rc;
  // the last rank's sums are the result; the counts are exact int32 sums (fewer than 2^31 rows in all)
  if ((rc = comm_broadcast(comm, sums, bytes, world - 1, s))) return rc;
  return comm_allreduce_lloyd(comm, nullptr, 0, counts, K, s);
}

int gdr_kmeans_finalize(int64_t K, int64_t D, const float* sums, int64_t lds, const int32_t* counts,
                        const float* C_old, int64_t ldc_old, float* C_new, int64_t ldc_new,
                        double* stats_dev, int mean_mode, gdr_stream_t stream) {
  GDR_CHECK_ARG(K > 0 && D > 0 && sums && counts && C_new && stats_dev, "kmeans_finalize: bad arguments");
  GDR_CHECK_ARG(K <= (1 << 22), "kmeans_finalize: K too large for the shift scratch");
  cudaStream_t s = (cudaStream_t)stream;
  // shift scratch lives behind stats (caller provides f64[2 + K])
  double* shift_arr = stats_dev + 2;
  k_average<<<(unsigned)cdiv(K, 8), 256, 0, s>>>(K, (int)D, sums, lds, counts, C_old, ldc_old, C_new,
                                                ldc_new, shift_arr, mean_mode);
  GDR_LAUNCHED();
  k_finalize_tail<<<1, 1024, 0, s>>>(K, (int)D, sums, lds, counts, C_old, ldc_old, C_new, ldc_new, shift_arr,
                                     stats_dev, mean_mode);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_inertia_ws_bytes(int64_t N, int64_t D) {
  (void)D;
  return ws_need(cdiv(N > 0 ? N : 1, 8), 8) + 256;
}

int gdr_inertia(int64_t N, int64_t D, const float* X, int64_t ldx, const float* C, int64_t ldc,
                const int32_t* labels, double* out_dev, void* ws, int64_t ws_bytes,
                gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && D > 0 && X && C && labels && out_dev, "inertia: bad arguments");
  if (ws_bytes < gdr_inertia_ws_bytes(N, D)) {
    set_error("inertia: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  int64_t nb = cdiv(N, 8);
  double* part = (double*)ws;
  k_row_dist<<<(unsigned)nb, 256, 0, s>>>(N, (int)D, X, ldx, C, ldc, labels, nullptr, part);
  GDR_LAUNCHED();
  k_sum_f64<<<1, 1024, 0, s>>>(nb, part, out_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_kmeans_relocate_ws_bytes(int64_t N, int64_t K, int64_t D) {
  (void)D;
  (void)K;
  return ws_need(N, 4) + 2 * ws_need(1024, 4) + 256;
}

int gdr_kmeans_relocate(int64_t N, int64_t K, int64_t D, const float* X, int64_t ldx,
                        const float* C_old, int64_t ldc, const int32_t* labels, float* sums,
                        int64_t lds, int32_t* counts, void* ws, int64_t ws_bytes,
                        gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && K > 0 && D > 0 && X && C_old && labels && sums && counts,
                "kmeans_relocate: bad arguments");
  if (ws_bytes < gdr_kmeans_relocate_ws_bytes(N, K, D)) {
    set_error("kmeans_relocate: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<int32_t> h_counts(K);
  GDR_CUDA(cudaMemcpyAsync(h_counts.data(), counts, K * 4, cudaMemcpyDeviceToHost, s));
  GDR_CUDA(cudaStreamSynchronize(s));
  std::vector<int> empties;
  for (int64_t k = 0; k < K; ++k)
    if (h_counts[k] == 0) empties.push_back((int)k);
  if (empties.empty()) return GDR_OK;
  Workspace W(ws, ws_bytes);
  float* dist = W.take<float>(N);
  float* pv = W.take<float>(1024);
  int32_t* pi = W.take<int32_t>(1024);
  k_row_dist<<<(unsigned)cdiv(N, 8), 256, 0, s>>>(N, (int)D, X, ldx, C_old, ldc, labels, dist, nullptr);
  GDR_LAUNCHED();
  int nparts = (int)std::min<int64_t>(1024, cdiv(N, 256));
  // sklearn skips relocation when max(distances) == 0
  k_argmax_part<<<nparts, 256, 0, s>>>(N, dist, pv, pi);
  GDR_LAUNCHED();
  std::vector<float> h_pv(nparts);
  GDR_CUDA(cudaMemcpyAsync(h_pv.data(), pv, nparts * 4, cudaMemcpyDeviceToHost, s));
  GDR_CUDA(cudaStreamSynchronize(s));
  float mx = 0.f;
  for (float v : h_pv) mx = v > mx ? v : mx;
  if (mx == 0.f) return GDR_OK;
  for (size_t e = 0; e < empties.size(); ++e) {
    if (e > 0) {
      k_argmax_part<<<nparts, 256, 0, s>>>(N, dist, pv, pi);
      GDR_LAUNCHED();
    }
    k_relocate_one<<<1, 256, 0, s>>>(nparts, pv, pi, (int)D, X, ldx, labels, sums, lds, counts,
                                     empties[e], dist);
    GDR_LAUNCHED();
  }
  return GDR_OK;
}

int gdr_minibatch_update(int64_t B, int64_t K, int64_t D, const float* Xb, int64_t ldx, const int32_t* labels,
                         const float* C_old, int64_t ldc_old, float* C_new, int64_t ldc_new, float* weight_sums,
                         gdr_stream_t stream) {
  GDR_CHECK_ARG(B >= 0 && K > 0 && D > 0 && C_old && C_new && weight_sums && (B == 0 || (Xb && labels)),
                "minibatch_update: bad arguments");
  GDR_CHECK_ARG(C_old != C_new, "minibatch_update: in-place update is not supported");
  k_minibatch_update<<<(unsigned)cdiv(K * 32, 256), 256, 0, (cudaStream_t)stream>>>(B, K, (int)D, Xb, ldx, labels, C_old,
                                                                                   ldc_old, C_new, ldc_new, weight_sums);
  GDR_LAUNCHED();
  return GDR_OK;
}

int64_t gdr_minibatch_batch_dist_ws_bytes(int64_t m, int64_t K, int64_t D, int world) {
  (void)world;
  const int64_t ldp = align_up(D > 0 ? D : 1, 4);
  return ws_need(m * ldp, 4) + ws_need(m, 4) + ws_need(K > 0 ? K : 1, 4) + 256;
}

int gdr_minibatch_batch_dist(gdr_comm_t* comm, int64_t m, const int64_t* idx, const int32_t* order,
                             const int64_t* counts_host, int64_t row_lo, int64_t n_local, int64_t K, int64_t D,
                             const float* X_local, int64_t ldx, const float* C, int64_t ldc, float* Xb, int64_t ldb,
                             int32_t* labels_b, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  // every check is local and comes before the exchange; the caller agrees on the arguments once per fit
  GDR_CHECK_ARG(comm && counts_host && m >= 0 && m < (1ll << 31) && D > 0 && D < (1 << 20),
                "minibatch_batch_dist: bad arguments");
  const int world = comm->world, me = comm->rank;
  int64_t total = 0, off_me = 0;
  for (int p = 0; p < world; ++p) {
    GDR_CHECK_ARG(counts_host[p] >= 0, "minibatch_batch_dist: negative count for rank %d", p);
    if (p < me) off_me += counts_host[p];
    total += counts_host[p];
  }
  GDR_CHECK_ARG(total == m, "minibatch_batch_dist: the counts add up to %lld, not m = %lld", (long long)total,
                (long long)m);
  if (m == 0) return GDR_OK;
  const int64_t n_me = counts_host[me];
  GDR_CHECK_ARG(idx && order && Xb && ldb >= D, "minibatch_batch_dist: null idx / order / Xb or ldb < D");
  GDR_CHECK_ARG(row_lo >= 0 && n_local >= 0 && (n_me == 0 || (X_local && ldx >= D)),
                "minibatch_batch_dist: bad row block");
  if (C) {
    GDR_CHECK_ARG(labels_b && K > 0 && K < (1ll << 31) && ldc % 4 == 0 && ldc >= D && ((uintptr_t)C & 15) == 0,
                  "minibatch_batch_dist: C needs labels_b, 0 < K < 2^31, 16B alignment and ldc %% 4 == 0, ldc >= D");
  }
  if (!ws || ws_bytes < gdr_minibatch_batch_dist_ws_bytes(m, K, D, world)) {
    set_error("minibatch_batch_dist: workspace too small");
    return GDR_EWORKSPACE;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int ldp = (int)align_up(D, 4);
  Workspace W(ws, ws_bytes);
  float* P = W.take<float>(m * ldp);
  int32_t* L = W.take<int32_t>(m);
  float* cnorm = W.take<float>(K > 0 ? K : 1);
  if (n_me > 0) {
    k_mb_pack<<<(unsigned)cdiv(n_me * 32, 256), 256, 0, s>>>(n_me, (int)D, ldp, idx, order + off_me, row_lo, n_local,
                                                            X_local, ldx, P + off_me * ldp);
    GDR_LAUNCHED();
    if (C) {
      // the one-GPU E-step kernels (gdr_kmeans_assign, precision_mode 0) on the owned rows: k_assign_simt scans every
      // centre for each row tile, so a row's label does not depend on the rows that share the launch
      k_row_sqnorm<<<(unsigned)cdiv(K, 8), 256, 0, s>>>(K, (int)D, C, ldc, cnorm);
      GDR_LAUNCHED();
      k_assign_simt<<<(unsigned)cdiv(n_me, AS_BM), AS_THREADS, 0, s>>>(n_me, (int)K, (int)D, P + off_me * ldp, ldp, C,
                                                                       ldc, cnorm, L + off_me, nullptr, nullptr,
                                                                       nullptr, nullptr, nullptr);
      GDR_LAUNCHED();
    }
  }
  void* bufs[2] = {P, L};
  const int64_t row_bytes[2] = {(int64_t)ldp * 4, 4};
  if (int rc = comm_allgatherv_inplace(comm, C ? 2 : 1, bufs, row_bytes, counts_host, s)) return rc;
  k_mb_place<<<(unsigned)cdiv(m * 32, 256), 256, 0, s>>>(m, ldp, order, P, L, Xb, ldb, C ? labels_b : nullptr);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_label_histogram(int64_t N, int64_t K, const int32_t* labels, int32_t* counts,
                        int32_t* status_dev, gdr_stream_t stream) {
  GDR_CHECK_ARG(N >= 0 && K > 0 && counts, "label_histogram: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  GDR_CUDA(cudaMemsetAsync(counts, 0, K * 4, s));
  if (status_dev) GDR_CUDA(cudaMemsetAsync(status_dev, 0, 4, s));
  if (N == 0) return GDR_OK;
  GDR_CHECK_ARG(labels, "label_histogram: null labels");
  unsigned grid = (unsigned)std::min<int64_t>(cdiv(N, 256), kSMs * 16);
  k_label_hist<<<grid, 256, 0, s>>>(N, K, labels, counts, status_dev);
  GDR_LAUNCHED();
  return GDR_OK;
}

}  // extern "C"
