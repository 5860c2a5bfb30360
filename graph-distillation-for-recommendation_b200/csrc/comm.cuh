// comm.cuh — internal view of the communicator (comm.cu) for the distributed drivers.
#pragma once
#include <cuda_runtime.h>
#include <nccl.h>   // types and prototypes only: the functions are bound at run time (dlopen), never linked
#include <stdint.h>
#include <initializer_list>
#include "common.cuh"

struct gdr_comm {
  ncclComm_t nccl;
  int rank, world, device;
  int64_t* entry;   // [world][gdr::kEntryWords] gather buffer of gdr::comm_entry_check
};

// Symmetric buffer: the same allocation on every rank of the communicator, each rank holding peer-mapped (CUDA IPC over
// NVLink) pointers to all copies, plus one epoch flag per source rank for the stream-ordered barrier.
struct gdr_symm {
  gdr_comm* comm;
  char* local;
  char* peer[GDR_MAX_RANKS];       // peer[rank] == local
  int64_t bytes;                   // usable bytes (the flag page lies behind them)
  uint32_t* flag_local;            // [GDR_MAX_RANKS] epochs written by the peers
  uint32_t* flag_peer[GDR_MAX_RANKS];
  uint32_t epoch;
};

namespace gdr {

struct NcclApi {
  decltype(&ncclGetUniqueId) GetUniqueId;
  decltype(&ncclCommInitRank) CommInitRank;
  decltype(&ncclCommDestroy) CommDestroy;
  decltype(&ncclAllReduce) AllReduce;
  decltype(&ncclAllGather) AllGather;
  decltype(&ncclSend) Send;
  decltype(&ncclRecv) Recv;
  decltype(&ncclGroupStart) GroupStart;
  decltype(&ncclGroupEnd) GroupEnd;
  decltype(&ncclGetErrorString) GetErrorString;
  decltype(&ncclGetVersion) GetVersion;
};

const NcclApi* nccl_api();   // nullptr (+ error string) when libnccl cannot be loaded

// [sums f32 | ints i32] summed over the ranks as ONE grouped NCCL operation (no-op for world 1 / null comm)
int comm_allreduce_lloyd(gdr_comm* c, float* sums, int64_t n_floats, int32_t* ints, int64_t n_ints, cudaStream_t s);
int comm_allreduce_f64(gdr_comm* c, double* buf, int64_t n, int op_max, cudaStream_t s);
// int64 sums over the ranks, send -> recv (a copy for world 1 / null comm)
int comm_allreduce_i64(gdr_comm* c, const int64_t* send, int64_t* recv, int64_t n, cudaStream_t s);
int comm_allgather(gdr_comm* c, const void* send, void* recv, int64_t bytes_per_rank, cudaStream_t s);
// NCCL point-to-point: the matching comm_recv / comm_send runs on rank `peer` (world > 1 only)
int comm_send(gdr_comm* c, const void* buf, int64_t bytes, int peer, cudaStream_t s);
int comm_recv(gdr_comm* c, void* buf, int64_t bytes, int peer, cudaStream_t s);
// buf of rank `root` -> buf of every other rank, as one group of sends (no-op for world 1 / null comm)
int comm_broadcast(gdr_comm* c, void* buf, int64_t bytes, int root, cudaStream_t s);
// In-place variable all-gather of n_bufs arrays that share one row split: rows [off_p, off_p + counts[p]) of bufs[a]
// (row_bytes[a] bytes each, off_p = counts[0] + ... + counts[p-1]) go from rank p to the same rows of every other rank,
// as ONE group of NCCL sends and receives (no-op for world 1 / null comm).
int comm_allgatherv_inplace(gdr_comm* c, int n_bufs, void* const* bufs, const int64_t* row_bytes, const int64_t* counts,
                            cudaStream_t s);

// The collective entry check of the row-partitioned entry points (return codes: gdr.h, next to gdr_comm_init).  Every
// rank passes its verdict local_rc, its row block [row_lo, row_lo + n_local) (row_lo < 0 on every rank: the blocks
// follow one another by construction), the words every rank must pass alike (agreed_names names them in the message),
// one word `extra` the caller wants back from every rank, and n_global >= 0 when the blocks must cover n_global rows.
// On GDR_OK, row_off[0..world] (optional) = every rank's first global row and the total, extras[0..world) (optional) =
// every rank's extra word.  One H2D copy, one all-gather into c->entry, one read-back and a stream synchronisation.
constexpr int kEntryAgreed = 8, kEntryWords = 4 + kEntryAgreed;
int comm_entry_check(gdr_comm* c, cudaStream_t s, const char* call, int local_rc, int64_t row_lo, int64_t n_local,
                     int64_t n_global, std::initializer_list<int64_t> agreed, const char* agreed_names,
                     int64_t extra = 0, int64_t* row_off = nullptr, int64_t* extras = nullptr);

}  // namespace gdr
