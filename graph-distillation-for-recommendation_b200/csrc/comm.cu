// comm.cu — the multi-GPU exchange steps of the path as C-ABI entry points (SURVEY §8b / §8e):
//   gdr_comm_init / gdr_comm_destroy      one NCCL communicator per process (one process per GPU)
//   gdr_allgather_rows                    stage 2: the propagated row block of every rank -> the full matrix
//   gdr_allreduce_centroids               stage 3: [K x ld sums | K counts + n_changed] in ONE grouped all-reduce
//   gdr_allgather_bytes / gdr_alltoallv   stage 1 / 4: degree vectors, edge buckets, (cell, count, sum) runs
// The reference is single-device, so nothing here restates it; these are the exchanges the row partition needs.
//
// NCCL is bound at RUN time (dlopen of the libnccl.so.2 already mapped by the host framework, else the system one):
// the library itself keeps no link-time dependency on NCCL and single-GPU users never load it.
#include "common.cuh"
#include "comm.cuh"
#include <dlfcn.h>
#include <mutex>
#include <string.h>
#include <algorithm>
#include <vector>

namespace gdr {

static NcclApi g_api;
static std::once_flag g_api_once;
static bool g_api_ok = false;
static char g_api_err[256] = "";

static void load_nccl() {
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    h = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);   // the copy the host framework (torch) already mapped
    if (h) break;
  }
  if (!h) {
    if (const char* p = getenv("GDR_NCCL_LIB")) h = dlopen(p, RTLD_NOW | RTLD_GLOBAL);
    for (const char* n : names) {
      if (h) break;
      h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    }
  }
  if (!h) {
    snprintf(g_api_err, sizeof(g_api_err), "cannot load libnccl.so.2 (%s); set GDR_NCCL_LIB", dlerror());
    return;
  }
#define GDR_SYM(field, name)                                                        \
  g_api.field = (decltype(g_api.field))dlsym(h, name);                              \
  if (!g_api.field) {                                                               \
    snprintf(g_api_err, sizeof(g_api_err), "libnccl lacks %s", name);               \
    return;                                                                         \
  }
  GDR_SYM(GetUniqueId, "ncclGetUniqueId")
  GDR_SYM(CommInitRank, "ncclCommInitRank")
  GDR_SYM(CommDestroy, "ncclCommDestroy")
  GDR_SYM(AllReduce, "ncclAllReduce")
  GDR_SYM(AllGather, "ncclAllGather")
  GDR_SYM(Send, "ncclSend")
  GDR_SYM(Recv, "ncclRecv")
  GDR_SYM(GroupStart, "ncclGroupStart")
  GDR_SYM(GroupEnd, "ncclGroupEnd")
  GDR_SYM(GetErrorString, "ncclGetErrorString")
  GDR_SYM(GetVersion, "ncclGetVersion")
#undef GDR_SYM
  g_api_ok = true;
}

const NcclApi* nccl_api() {
  std::call_once(g_api_once, load_nccl);
  if (!g_api_ok) {
    set_error("%s", g_api_err);
    return nullptr;
  }
  return &g_api;
}

#define GDR_NCCL(call)                                                                          \
  do {                                                                                          \
    ncclResult_t r__ = (call);                                                                  \
    if (r__ != ncclSuccess) {                                                                   \
      ::gdr::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, api->GetErrorString(r__));  \
      return GDR_ECUDA;                                                                         \
    }                                                                                           \
  } while (0)

int comm_allreduce_lloyd(gdr_comm* c, float* sums, int64_t n_floats, int32_t* ints, int64_t n_ints, cudaStream_t s) {
  if (!c || c->world == 1) return GDR_OK;
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  GDR_NCCL(api->GroupStart());
  if (n_floats > 0) GDR_NCCL(api->AllReduce(sums, sums, (size_t)n_floats, ncclFloat32, ncclSum, c->nccl, s));
  if (n_ints > 0) GDR_NCCL(api->AllReduce(ints, ints, (size_t)n_ints, ncclInt32, ncclSum, c->nccl, s));
  GDR_NCCL(api->GroupEnd());
  count_launch(1);
  return GDR_OK;
}

int comm_allreduce_f64(gdr_comm* c, double* buf, int64_t n, int op_max, cudaStream_t s) {
  if (!c || c->world == 1) return GDR_OK;
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  GDR_NCCL(api->AllReduce(buf, buf, (size_t)n, ncclFloat64, op_max ? ncclMax : ncclSum, c->nccl, s));
  count_launch(1);
  return GDR_OK;
}

int comm_allreduce_i64(gdr_comm* c, const int64_t* send, int64_t* recv, int64_t n, cudaStream_t s) {
  if (!c || c->world == 1) {
    if (send != recv && n > 0) GDR_CUDA(cudaMemcpyAsync(recv, send, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
    return GDR_OK;
  }
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  GDR_NCCL(api->AllReduce(send, recv, (size_t)n, ncclInt64, ncclSum, c->nccl, s));
  count_launch(1);
  return GDR_OK;
}

int comm_allgather(gdr_comm* c, const void* send, void* recv, int64_t bytes_per_rank, cudaStream_t s) {
  if (!c || c->world == 1) {
    if (send != recv && bytes_per_rank > 0)
      GDR_CUDA(cudaMemcpyAsync(recv, send, (size_t)bytes_per_rank, cudaMemcpyDeviceToDevice, s));
    return GDR_OK;
  }
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  GDR_NCCL(api->AllGather(send, recv, (size_t)bytes_per_rank, ncclInt8, c->nccl, s));
  count_launch(1);
  return GDR_OK;
}

int comm_send(gdr_comm* c, const void* buf, int64_t bytes, int peer, cudaStream_t s) {
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  GDR_NCCL(api->Send(buf, (size_t)bytes, ncclInt8, peer, c->nccl, s));
  count_launch(1);
  return GDR_OK;
}

int comm_recv(gdr_comm* c, void* buf, int64_t bytes, int peer, cudaStream_t s) {
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  GDR_NCCL(api->Recv(buf, (size_t)bytes, ncclInt8, peer, c->nccl, s));
  count_launch(1);
  return GDR_OK;
}

int comm_broadcast(gdr_comm* c, void* buf, int64_t bytes, int root, cudaStream_t s) {
  if (!c || c->world == 1) return GDR_OK;
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  GDR_NCCL(api->GroupStart());
  if (c->rank == root) {
    for (int p = 0; p < c->world; ++p)
      if (p != root) GDR_NCCL(api->Send(buf, (size_t)bytes, ncclInt8, p, c->nccl, s));
  } else {
    GDR_NCCL(api->Recv(buf, (size_t)bytes, ncclInt8, root, c->nccl, s));
  }
  GDR_NCCL(api->GroupEnd());
  count_launch(1);
  return GDR_OK;
}

int comm_allgatherv_inplace(gdr_comm* c, int n_bufs, void* const* bufs, const int64_t* row_bytes, const int64_t* counts,
                            cudaStream_t s) {
  if (!c || c->world == 1) return GDR_OK;
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  const int me = c->rank;
  int64_t off_me = 0;
  for (int p = 0; p < me; ++p) off_me += counts[p];
  GDR_NCCL(api->GroupStart());
  int64_t off = 0;
  for (int p = 0; p < c->world; ++p) {
    if (p != me) {
      for (int a = 0; a < n_bufs; ++a) {
        char* b = (char*)bufs[a];
        if (counts[me] > 0)
          GDR_NCCL(api->Send(b + off_me * row_bytes[a], (size_t)(counts[me] * row_bytes[a]), ncclInt8, p, c->nccl, s));
        if (counts[p] > 0)
          GDR_NCCL(api->Recv(b + off * row_bytes[a], (size_t)(counts[p] * row_bytes[a]), ncclInt8, p, c->nccl, s));
      }
    }
    off += counts[p];
  }
  GDR_NCCL(api->GroupEnd());
  count_launch(1);
  return GDR_OK;
}

int comm_entry_check(gdr_comm* c, cudaStream_t s, const char* call, int local_rc, int64_t row_lo, int64_t n_local,
                     int64_t n_global, std::initializer_list<int64_t> agreed, const char* agreed_names, int64_t extra,
                     int64_t* row_off, int64_t* extras) {
  GDR_CHECK_ARG(agreed.size() <= (size_t)kEntryAgreed, "%s: more than %d agreed words", call, kEntryAgreed);
  const int world = c->world;
  int64_t mine[kEntryWords] = {local_rc, row_lo, n_local, extra};
  std::copy(agreed.begin(), agreed.end(), mine + 4);
  std::vector<int64_t> all((size_t)world * kEntryWords);
  int64_t* row = c->entry + (int64_t)c->rank * kEntryWords;
  if (cudaMemcpyAsync(row, mine, sizeof(mine), cudaMemcpyHostToDevice, s) != cudaSuccess) {
    set_error("%s: copy of the argument check failed", call);
    return GDR_ECUDA;
  }
  if (int rc = comm_allgather(c, row, c->entry, sizeof(mine), s)) return rc;
  if (cudaMemcpyAsync(all.data(), c->entry, all.size() * 8, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    set_error("%s: read-back of the argument check failed", call);
    return GDR_ECUDA;
  }
  if (local_rc != GDR_OK) return local_rc;
  int64_t next_lo = 0;
  for (int r = 0; r < world; ++r) {
    const int64_t* m = &all[(size_t)r * kEntryWords];
    if (m[0] != GDR_OK) {
      set_error("%s: rank %d rejected its arguments", call, r);
      return GDR_EINVAL;
    }
    if (!std::equal(mine + 4, mine + kEntryWords, m + 4)) {
      set_error("%s: rank %d passed a different %s", call, r, agreed_names);
      return GDR_EINVAL;
    }
    if (row_lo >= 0 && m[1] != next_lo) {
      set_error("%s: the row block of rank %d does not follow the previous rank's", call, r);
      return GDR_EINVAL;
    }
    if (row_off) row_off[r] = next_lo;
    if (extras) extras[r] = m[3];
    next_lo += m[2];
  }
  if (n_global >= 0 && next_lo != n_global) {
    set_error("%s: the row blocks hold %lld rows, not %lld", call, (long long)next_lo, (long long)n_global);
    return GDR_EINVAL;
  }
  if (row_off) row_off[world] = next_lo;
  return GDR_OK;
}

}  // namespace gdr


// ---- symmetric buffers over CUDA IPC (one process per GPU, all GPUs of one NVLink domain) ----------------------
namespace gdr {

struct FlagPtrs {
  uint32_t* f[GDR_MAX_RANKS];
};
// every rank tells every peer "all my work enqueued before this kernel — including my stores into your copy — is done"
__global__ void k_symm_signal(FlagPtrs fp, int n, int rank, uint32_t epoch) {
  const int p = threadIdx.x;
  if (p < n) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(fp.f[p] + rank), "r"(epoch) : "memory");
  }
}

// ... and waits until every peer has said so
__global__ void k_symm_wait(const uint32_t* flag_local, int n, uint32_t epoch) {
  const int p = threadIdx.x;
  if (p < n) {
    uint32_t v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag_local + p) : "memory");
    } while ((int32_t)(v - epoch) < 0);
  }
  __syncthreads();
  __threadfence_system();
}

struct PutDst {
  float* dst[GDR_MAX_RANKS];
  int n;
};
// rows of `src` (ld floats each, ld % 4 == 0) -> the same rows of every destination (read once, n posted stores)
__global__ void k_symm_put_rows(int64_t n4, const float4* __restrict__ src, PutDst d) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(src + i);
    for (int p = 0; p < d.n; ++p) reinterpret_cast<float4*>(d.dst[p])[i] = v;
  }
}

// Variable scatter into the peers' copies: segment p = n_words[p] 4-byte words from src[p] to dst[p] (a peer-mapped
// address, 4-byte aligned).  Per segment: scalar head up to the first 16-byte boundary of the DESTINATION, 16-byte posted
// stores for the body (the source side is read as one 16-byte or four 4-byte loads), scalar tail.  Block b starts with
// segment (first + b) % n so that the ranks do not all pour into the same peer at the same time.
struct ScatterSegs {
  const uint32_t* src[GDR_MAX_RANKS];
  uint32_t* dst[GDR_MAX_RANKS];
  int64_t n_words[GDR_MAX_RANKS];
  int n, first;
};
__global__ void __launch_bounds__(256) k_symm_scatterv(ScatterSegs sg) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  for (int j = 0; j < sg.n; ++j) {
    const int p = (sg.first + (int)(blockIdx.x % (unsigned)sg.n) + j) % sg.n;
    const uint32_t* __restrict__ s = sg.src[p];
    uint32_t* __restrict__ d = sg.dst[p];
    const int64_t n = sg.n_words[p];
    if (n <= 0) continue;
    const int64_t h0 = (int64_t)(((16 - ((uintptr_t)d & 15)) & 15) >> 2), head = h0 < n ? h0 : n;
    const int64_t body = (n - head) >> 2, tail0 = head + (body << 2);
    if (tid < head) d[tid] = __ldg(s + tid);
    if (tid < n - tail0) d[tail0 + tid] = __ldg(s + tail0 + tid);
    const uint32_t* sb = s + head;
    uint4* db = reinterpret_cast<uint4*>(d + head);
    if (((uintptr_t)sb & 15) == 0) {
      const uint4* sv = reinterpret_cast<const uint4*>(sb);
      for (int64_t i = tid; i < body; i += nth) db[i] = __ldg(sv + i);
    } else if (((uintptr_t)sb & 7) == 0) {
      const uint2* sv = reinterpret_cast<const uint2*>(sb);
      for (int64_t i = tid; i < body; i += nth) {
        const uint2 a = __ldg(sv + 2 * i), b = __ldg(sv + 2 * i + 1);
        db[i] = make_uint4(a.x, a.y, b.x, b.y);
      }
    } else {
      for (int64_t i = tid; i < body; i += nth)
        db[i] = make_uint4(__ldg(sb + 4 * i), __ldg(sb + 4 * i + 1), __ldg(sb + 4 * i + 2), __ldg(sb + 4 * i + 3));
    }
  }
}

int symm_barrier(gdr_symm* sm, cudaStream_t s) {
  if (sm->comm->world == 1) return GDR_OK;
  const uint32_t e = ++sm->epoch;
  FlagPtrs fp;
  for (int p = 0; p < GDR_MAX_RANKS; ++p) fp.f[p] = p < sm->comm->world ? sm->flag_peer[p] : nullptr;
  k_symm_signal<<<1, 32, 0, s>>>(fp, sm->comm->world, sm->comm->rank, e);
  GDR_LAUNCHED();
  k_symm_wait<<<1, 32, 0, s>>>(sm->flag_local, sm->comm->world, e);
  GDR_LAUNCHED();
  return GDR_OK;
}

}  // namespace gdr

using namespace gdr;

extern "C" {

int gdr_comm_unique_id(void* id128_host) {
  GDR_CHECK_ARG(id128_host, "comm_unique_id: null output");
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  GDR_NCCL(api->GetUniqueId(&id));
  memcpy(id128_host, &id, sizeof(id));
  return GDR_OK;
}

int gdr_comm_init(gdr_comm_t** comm_out, const void* id128_host, int rank, int world) {
  GDR_CHECK_ARG(comm_out && world >= 1 && rank >= 0 && rank < world, "comm_init: bad arguments");
  gdr_comm* c = new gdr_comm();
  c->rank = rank;
  c->world = world;
  c->nccl = nullptr;
  c->entry = nullptr;
  GDR_CUDA(cudaGetDevice(&c->device));
  cudaError_t e = cudaMalloc((void**)&c->entry, (size_t)world * kEntryWords * 8);
  if (e != cudaSuccess) {
    set_error("comm_init: cudaMalloc of the entry-check buffer -> %s", cudaGetErrorString(e));
    cudaGetLastError();
    delete c;
    return GDR_ECUDA;
  }
  if (world > 1) {
    const NcclApi* api = nccl_api();
    if (!api || !id128_host) {
      gdr_comm_destroy(c);
      if (api) set_error("comm_init: null unique id");
      return api ? GDR_EINVAL : GDR_ECUDA;
    }
    ncclUniqueId id;
    memcpy(&id, id128_host, sizeof(id));
    ncclResult_t r = api->CommInitRank(&c->nccl, world, id, rank);
    if (r != ncclSuccess) {
      set_error("ncclCommInitRank -> %s", api->GetErrorString(r));
      c->nccl = nullptr;
      gdr_comm_destroy(c);
      return GDR_ECUDA;
    }
  }
  *comm_out = c;
  return GDR_OK;
}

int gdr_comm_destroy(gdr_comm_t* comm) {
  if (!comm) return GDR_OK;
  if (comm->nccl) {
    const NcclApi* api = nccl_api();
    if (api) api->CommDestroy(comm->nccl);
  }
  cudaFree(comm->entry);
  delete comm;
  return GDR_OK;
}

int gdr_comm_info(const gdr_comm_t* comm, int* rank_host, int* world_host, int* nccl_version_host) {
  GDR_CHECK_ARG(comm, "comm_info: null communicator");
  if (rank_host) *rank_host = comm->rank;
  if (world_host) *world_host = comm->world;
  if (nccl_version_host) {
    *nccl_version_host = 0;
    if (comm->world > 1) {
      const NcclApi* api = nccl_api();
      if (api) api->GetVersion(nccl_version_host);
    }
  }
  return GDR_OK;
}

int gdr_allgather_rows(gdr_comm_t* comm, const float* local, int64_t rows_per_rank, int64_t ld, float* full,
                       gdr_stream_t stream) {
  GDR_CHECK_ARG(comm && rows_per_rank >= 0 && ld > 0 && (rows_per_rank == 0 || (local && full)),
                "allgather_rows: bad arguments");
  return comm_allgather(comm, local, full, rows_per_rank * ld * 4, (cudaStream_t)stream);
}

int gdr_allgather_bytes(gdr_comm_t* comm, const void* local, int64_t bytes_per_rank, void* full, gdr_stream_t stream) {
  GDR_CHECK_ARG(comm && bytes_per_rank >= 0 && (bytes_per_rank == 0 || (local && full)), "allgather_bytes: bad arguments");
  return comm_allgather(comm, local, full, bytes_per_rank, (cudaStream_t)stream);
}

int gdr_allreduce_centroids(gdr_comm_t* comm, float* sums, int64_t n_floats, int32_t* ints, int64_t n_ints,
                            gdr_stream_t stream) {
  GDR_CHECK_ARG(comm && n_floats >= 0 && n_ints >= 0 && (n_floats == 0 || sums) && (n_ints == 0 || ints),
                "allreduce_centroids: bad arguments");
  return comm_allreduce_lloyd(comm, sums, n_floats, ints, n_ints, (cudaStream_t)stream);
}

int gdr_allreduce_f64(gdr_comm_t* comm, double* buf, int64_t n, int op_max, gdr_stream_t stream) {
  GDR_CHECK_ARG(comm && n >= 0 && (n == 0 || buf), "allreduce_f64: bad arguments");
  return comm_allreduce_f64(comm, buf, n, op_max, (cudaStream_t)stream);
}


int gdr_symm_create(gdr_comm_t* comm, int64_t bytes, gdr_symm_t** symm_out) {
  GDR_CHECK_ARG(comm && bytes > 0 && symm_out, "symm_create: bad arguments");
  GDR_CHECK_ARG(comm->world <= GDR_MAX_RANKS, "symm_create: world exceeds GDR_MAX_RANKS");
  const int world = comm->world, rank = comm->rank;
  const int64_t usable = align_up(bytes, 4096);
  gdr_symm* sm = new gdr_symm();
  memset(sm, 0, sizeof(*sm));
  sm->comm = comm;
  sm->bytes = usable;
  auto fail = [&](const char* what, cudaError_t e) {
    set_error("symm_create: %s -> %s", what, cudaGetErrorString(e));
    if (sm->local) cudaFree(sm->local);
    delete sm;
    cudaGetLastError();
    return GDR_ECUDA;
  };
  cudaError_t e = cudaMalloc((void**)&sm->local, (size_t)usable + 4096);
  if (e != cudaSuccess) {
    sm->local = nullptr;
    return fail("cudaMalloc", e);
  }
  if ((e = cudaMemset(sm->local + usable, 0, 4096)) != cudaSuccess) return fail("cudaMemset", e);
  sm->peer[rank] = sm->local;
  if (world > 1) {
    cudaIpcMemHandle_t mine;
    if ((e = cudaIpcGetMemHandle(&mine, sm->local)) != cudaSuccess) return fail("cudaIpcGetMemHandle", e);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    char *d_send = nullptr, *d_recv = nullptr;
    if ((e = cudaMalloc((void**)&d_send, 64)) != cudaSuccess) return fail("cudaMalloc", e);
    if ((e = cudaMalloc((void**)&d_recv, 64 * (size_t)world)) != cudaSuccess) return fail("cudaMalloc", e);
    cudaMemcpy(d_send, &mine, 64, cudaMemcpyHostToDevice);
    int rc = comm_allgather(comm, d_send, d_recv, 64, nullptr);       // also orders every rank's memset before any signal
    if (rc == GDR_OK && cudaStreamSynchronize(nullptr) != cudaSuccess) rc = GDR_ECUDA;
    std::vector<cudaIpcMemHandle_t> all((size_t)world);
    if (rc == GDR_OK) cudaMemcpy(all.data(), d_recv, 64 * (size_t)world, cudaMemcpyDeviceToHost);
    cudaFree(d_send);
    cudaFree(d_recv);
    if (rc != GDR_OK) {
      cudaFree(sm->local);
      delete sm;
      return rc;
    }
    for (int p = 0; p < world; ++p) {
      if (p == rank) continue;
      void* q = nullptr;
      if ((e = cudaIpcOpenMemHandle(&q, all[(size_t)p], cudaIpcMemLazyEnablePeerAccess)) != cudaSuccess) {
        for (int z = 0; z < p; ++z)
          if (z != rank && sm->peer[z]) cudaIpcCloseMemHandle(sm->peer[z]);
        return fail("cudaIpcOpenMemHandle (peer memory over NVLink unavailable)", e);
      }
      sm->peer[p] = (char*)q;
    }
  }
  sm->flag_local = (uint32_t*)(sm->local + usable);
  for (int p = 0; p < world; ++p) sm->flag_peer[p] = (uint32_t*)(sm->peer[p] + usable);
  *symm_out = sm;
  return GDR_OK;
}

int gdr_symm_destroy(gdr_symm_t* sm) {
  if (!sm) return GDR_OK;
  cudaDeviceSynchronize();
  for (int p = 0; p < sm->comm->world; ++p)
    if (p != sm->comm->rank && sm->peer[p]) cudaIpcCloseMemHandle(sm->peer[p]);
  // nobody may still be writing into this copy: a last collective orders every rank's close before the free
  if (sm->comm->world > 1 && sm->comm->nccl) {
    int32_t* d = nullptr;
    if (cudaMalloc((void**)&d, 4) == cudaSuccess) {
      cudaMemset(d, 0, 4);
      comm_allreduce_lloyd(sm->comm, nullptr, 0, d, 1, nullptr);
      cudaStreamSynchronize(nullptr);
      cudaFree(d);
    }
  }
  cudaFree(sm->local);
  cudaGetLastError();
  delete sm;
  return GDR_OK;
}

int gdr_symm_info(const gdr_symm_t* sm, void** local_ptr_host, int64_t* bytes_host) {
  GDR_CHECK_ARG(sm, "symm_info: null buffer");
  if (local_ptr_host) *local_ptr_host = sm->local;
  if (bytes_host) *bytes_host = sm->bytes;
  return GDR_OK;
}

int gdr_symm_barrier(gdr_symm_t* sm, gdr_stream_t stream) {
  GDR_CHECK_ARG(sm, "symm_barrier: null buffer");
  return symm_barrier(sm, (cudaStream_t)stream);
}

int gdr_symm_put_rows(gdr_symm_t* sm, int64_t dst_offset_bytes, const float* src, int64_t rows, int64_t ld,
                      int include_self, gdr_stream_t stream) {
  GDR_CHECK_ARG(sm && rows >= 0 && ld > 0 && ld % 4 == 0 && dst_offset_bytes >= 0 && dst_offset_bytes % 16 == 0,
                "symm_put_rows: bad arguments");
  if (rows == 0) return GDR_OK;
  GDR_CHECK_ARG(src && ((uintptr_t)src & 15) == 0, "symm_put_rows: src misaligned");
  GDR_CHECK_ARG(dst_offset_bytes + rows * ld * 4 <= sm->bytes, "symm_put_rows: destination range exceeds the buffer");
  PutDst d;
  d.n = 0;
  for (int p = 0; p < sm->comm->world; ++p)
    if (include_self || p != sm->comm->rank) d.dst[d.n++] = (float*)(sm->peer[p] + dst_offset_bytes);
  if (d.n == 0) return GDR_OK;
  const int64_t n4 = rows * ld / 4;
  const unsigned grid = (unsigned)std::min<int64_t>(cdiv(n4, 256), kSMs * 8);
  k_symm_put_rows<<<grid, 256, 0, (cudaStream_t)stream>>>(n4, (const float4*)src, d);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_symm_scatterv(gdr_symm_t* sm, const void* send, const int64_t* send_off_host, const int64_t* send_cnt_host,
                      const int64_t* dst_off_bytes_host, int64_t elem_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(sm && send_off_host && send_cnt_host && dst_off_bytes_host && elem_bytes > 0 && elem_bytes % 4 == 0,
                "symm_scatterv: bad arguments (elements are multiples of 4 bytes)");
  const int world = sm->comm->world;
  ScatterSegs sg;
  sg.n = world;
  sg.first = (sm->comm->rank + 1) % world;
  int64_t total = 0;
  for (int p = 0; p < world; ++p) {
    const int64_t cnt = send_cnt_host[p];
    GDR_CHECK_ARG(cnt >= 0 && send_off_host[p] >= 0 && dst_off_bytes_host[p] >= 0 && dst_off_bytes_host[p] % 4 == 0,
                  "symm_scatterv: bad segment");
    GDR_CHECK_ARG(dst_off_bytes_host[p] + cnt * elem_bytes <= sm->bytes, "symm_scatterv: destination range exceeds the buffer");
    sg.src[p] = reinterpret_cast<const uint32_t*>((const char*)send + send_off_host[p] * elem_bytes);
    sg.dst[p] = reinterpret_cast<uint32_t*>(sm->peer[p] + dst_off_bytes_host[p]);
    sg.n_words[p] = cnt * (elem_bytes / 4);
    total += sg.n_words[p];
  }
  if (total == 0) return GDR_OK;
  GDR_CHECK_ARG(send && ((uintptr_t)send & 3) == 0, "symm_scatterv: send misaligned");
  const unsigned grid = (unsigned)std::min<int64_t>(std::max<int64_t>(cdiv(total / 4 + 1, 256), 1), kSMs * 8);
  k_symm_scatterv<<<grid, 256, 0, (cudaStream_t)stream>>>(sg);
  GDR_LAUNCHED();
  return GDR_OK;
}

int gdr_alltoallv(gdr_comm_t* comm, const void* send, const int64_t* send_off_host, const int64_t* send_cnt_host,
                  void* recv, const int64_t* recv_off_host, const int64_t* recv_cnt_host, int64_t elem_bytes,
                  gdr_stream_t stream) {
  GDR_CHECK_ARG(comm && send_off_host && send_cnt_host && recv_off_host && recv_cnt_host && elem_bytes > 0,
                "alltoallv: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const int me = comm->rank;
  if (comm->world == 1) {
    if (send_cnt_host[0] > 0)
      GDR_CUDA(cudaMemcpyAsync((char*)recv + recv_off_host[0] * elem_bytes, (const char*)send + send_off_host[0] * elem_bytes,
                               (size_t)(send_cnt_host[0] * elem_bytes), cudaMemcpyDeviceToDevice, s));
    return GDR_OK;
  }
  const NcclApi* api = nccl_api();
  if (!api) return GDR_ECUDA;
  if (send_cnt_host[me] != recv_cnt_host[me]) {
    set_error("alltoallv: own block sizes differ");
    return GDR_EINVAL;
  }
  if (send_cnt_host[me] > 0)
    GDR_CUDA(cudaMemcpyAsync((char*)recv + recv_off_host[me] * elem_bytes, (const char*)send + send_off_host[me] * elem_bytes,
                             (size_t)(send_cnt_host[me] * elem_bytes), cudaMemcpyDeviceToDevice, s));
  GDR_NCCL(api->GroupStart());
  for (int p = 0; p < comm->world; ++p) {
    if (p == me) continue;
    if (send_cnt_host[p] > 0)
      GDR_NCCL(api->Send((const char*)send + send_off_host[p] * elem_bytes, (size_t)(send_cnt_host[p] * elem_bytes), ncclInt8, p,
                         comm->nccl, s));
    if (recv_cnt_host[p] > 0)
      GDR_NCCL(api->Recv((char*)recv + recv_off_host[p] * elem_bytes, (size_t)(recv_cnt_host[p] * elem_bytes), ncclInt8, p,
                         comm->nccl, s));
  }
  GDR_NCCL(api->GroupEnd());
  count_launch(1);
  return GDR_OK;
}

}  // extern "C"
