// common.cuh — shared helpers of libgdr_b200 (error plumbing, launch counting,
// workspace carving, small device utilities).  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/gdr.h"

namespace gdr {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define GDR_CHECK_ARG(cond, ...)                                   \
  do {                                                             \
    if (!(cond)) {                                                 \
      ::gdr::set_error(__VA_ARGS__);                               \
      return GDR_EINVAL;                                           \
    }                                                              \
  } while (0)

#define GDR_CUDA(call)                                                            \
  do {                                                                            \
    cudaError_t e__ = (call);                                                     \
    if (e__ != cudaSuccess) {                                                     \
      ::gdr::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call,               \
                       cudaGetErrorString(e__));                                  \
      return GDR_ECUDA;                                                           \
    }                                                                             \
  } while (0)

// after a kernel launch: bump the launch counter and surface launch errors
#define GDR_LAUNCHED()                                                            \
  do {                                                                            \
    ::gdr::count_launch();                                                        \
    cudaError_t e__ = cudaGetLastError();                                         \
    if (e__ != cudaSuccess) {                                                     \
      ::gdr::set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__,           \
                       cudaGetErrorString(e__));                                  \
      return GDR_ECUDA;                                                           \
    }                                                                             \
  } while (0)

// kernel kinds for gdr_profile_enable()
constexpr int PROF_ASSIGN = 1;  // the E-step main kernel (k_assign_tc / k_assign_simt over all rows)
constexpr int PROF_SPMM = 2;    // k_spmm (propagation hops and the M-step gather-sum)
struct ProfileScope {
  ProfileScope(int kind, cudaStream_t s);
  ~ProfileScope();
  void* stop_;
  cudaStream_t stream_;
};

constexpr int kSMs = 148;  // B200
#define GDR_MAX_RANKS 16      // ranks of one NVLink domain a symmetric buffer can span

// "done once" flags for per-device function attributes (cudaFuncSetAttribute is per device: a second
// GPU driven from the same process needs its own opt-in).  Usage: static PerDevice<bool> set; if (!set.get()) ...
template <typename T>
struct PerDevice {
  T v[64] = {};
  T& get() {
    int dev = 0;
    cudaGetDevice(&dev);
    return v[dev & 63];
  }
};

static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }
static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Bump allocator over the caller's workspace; every block 256-byte aligned.
struct Workspace {
  char* base;
  int64_t off;
  int64_t cap;
  Workspace(void* p, int64_t bytes) : base((char*)p), off(0), cap(bytes) {}
  template <typename T>
  T* take(int64_t n) {
    int64_t bytes = align_up(n * (int64_t)sizeof(T), 256);
    T* r = (T*)(base + off);
    off += bytes;
    return r;
  }
  bool ok() const { return off <= cap && (base != nullptr || off == 0); }
};
static inline int64_t ws_need(int64_t n, int64_t elem) { return align_up(n * elem, 256); }

// ---- internal primitives shared between translation units ------------------
// exclusive scan of int32 (n elements) -> out (n+1 elements, out[n] = total).
int64_t scan_ws_bytes(int64_t n);
int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, void* ws, int64_t ws_bytes,
                       cudaStream_t s);

int64_t sort_pairs_ws_bytes(int64_t n);
int sort_pairs(int64_t n, int key_bits, uint64_t* keys, uint32_t* vals, void* ws, int64_t ws_bytes,
               cudaStream_t s);
// same sort; the result is reported where the last pass left it (no copy back): *keys_sorted / *vals_sorted
int sort_pairs_ex(int64_t n, int key_bits, uint64_t* keys, uint32_t* vals, void* ws, int64_t ws_bytes,
                  uint64_t** keys_sorted, uint32_t** vals_sorted, cudaStream_t s);

// one stable pass on the digit [shift, shift + bits), bits in 7..11 (a stable partition); result in the workspace twins
int sort_pairs_digit(int64_t n, int shift, int bits, uint64_t* keys, uint32_t* vals, void* ws, int64_t ws_bytes,
                     uint64_t** keys_sorted, uint32_t** vals_sorted, int64_t* starts_dev, cudaStream_t s,
                     uint64_t* keys_dst = nullptr, uint32_t* vals_dst = nullptr);

// SpMM launcher shared by stage 2 and the k-means M-step (vals == nullptr -> 1.0,
// colidx32 gathers rows of X).
int spmm_launch(int64_t rows, int64_t F, const int32_t* rowptr, const int32_t* colidx,
                const float* vals, float alpha, const float* X, int64_t ldx, float* Y, int64_t ldy,
                float* T, int64_t ldt, float beta, cudaStream_t s);

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// The exact fp32 distance of the E-step, d(i, j) = fmaf(-2, acc, |c_j|^2) with acc = fmaf(x_k, c_jk, acc) for k
// ascending from acc = 0.  Every kernel that decides a label exactly (k_assign_simt, k_refine_partial,
// k_tc_cand_resolve) builds its distances from these two steps, so that they agree bit for bit.
__device__ __forceinline__ float ed_chain(float acc, float x, float c) { return fmaf(x, c, acc); }
__device__ __forceinline__ float ed_finish(float acc, float cnorm) { return fmaf(-2.f, acc, cnorm); }

// (distance, centre) as one 64-bit key whose unsigned order is (distance, then lowest index)
__device__ __forceinline__ unsigned long long rf_pack(float d, int j) {
  unsigned u = __float_as_uint(d);
  u = (u >> 31) ? ~u : (u | 0x80000000u);   // monotone map float -> uint32
  return ((unsigned long long)u << 32) | (unsigned)j;
}
__device__ __forceinline__ float rf_unpack(unsigned long long key) {
  unsigned u = (unsigned)(key >> 32);
  u = (u >> 31) ? (u & 0x7fffffffu) : ~u;
  return __uint_as_float(u);
}

__device__ __forceinline__ float4 ldg_nc_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
// gathered rows are re-used by other warps of the same SM only by chance, but
// they ARE re-used across SMs through L2: keep them on the default L1 path.
__device__ __forceinline__ float4 ldg_f4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}

}  // namespace gdr
