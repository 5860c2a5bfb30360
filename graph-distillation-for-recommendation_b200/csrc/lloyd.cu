// lloyd.cu — the Lloyd loop of one k-means run as a single C-ABI call.
//
// Control flow of sklearn's _kmeans_single_lloyd (sklearn/cluster/_kmeans.py:630-758),
// the routine behind the reference's KMeans(...).fit() call sites
// (clustgdd_agent_transduct.py:105, clustgdd_agent_induct.py:134, distill_recsys.py:178):
//   repeat: E-step -> per-cluster sums -> relocate empties -> average -> centre shift
//   stop on identical labels (strict) or sum shift^2 <= tol; if not strict, one more E-step;
//   inertia of the final assignment.
// One iteration is ~25 short kernels; its body is captured ONCE per buffer parity into a CUDA
// graph (on an internal stream ordered after the caller's stream by events) and replayed, so
// the host issues one graph launch plus ONE 24-byte status read-back per iteration (the
// convergence test is a host decision in the reference as well).
#include "common.cuh"
#include "comm.cuh"
#include <algorithm>
#include <numeric>
#include <stdio.h>
#include <vector>

using namespace gdr;

namespace gdr {
int64_t kmeans_assign_tc_ws_bytes(int64_t N, int64_t K, int64_t D);
int64_t kmeans_tc_xsplit_bytes(int64_t N, int64_t D);
int g_lloyd_graph = 1;  // gdr_debug_set("lloyd_graph", 0) disables graph replay
bool profiling_enabled();
// kmeans.cu: distributed empty-cluster relocation (candidate records / application of the global choice)
int64_t relocate_candidates_ws_bytes(int64_t N);
int relocate_candidates(int64_t N, int64_t D, const float* X, int64_t ldx, const float* C_old, int64_t ldc,
                        const int32_t* labels, int ne, int rank, float* rec, void* ws, int64_t ws_bytes, cudaStream_t s);
int relocate_apply(int ne, const int32_t* order_dev, const int32_t* empties_dev, const float* allrec, int64_t D,
                   float* sums, int64_t lds, int32_t* counts, cudaStream_t s);
}  // namespace gdr

namespace {

struct LloydBuffers {
  int32_t* labels[2];
  float* centers[2];
  float* sums;
  int32_t* counts;
  int32_t* n_changed;
  double* stats;  // [2 + K]
  void* xsplit;   // tensor-core operand cache (mode 1)
  void* ws_assign;
  int64_t ws_assign_b;
  void* ws_seg;
  int64_t ws_seg_b;
  void* ws_misc;
  int64_t ws_misc_b;
};

int64_t carve(LloydBuffers* B, void* ws, int64_t N, int64_t K, int64_t D, int mode) {
  const int64_t ldc = align_up(D, 4);
  Workspace W(ws, INT64_MAX);
  auto take_bytes = [&](int64_t bytes) { return (void*)W.take<char>(bytes); };
  LloydBuffers tmp;
  LloydBuffers& b = B ? *B : tmp;
  const int64_t N_rows = N;
  N = N > 0 ? N : 1;   // a rank of the distributed run may own no rows: size the scratch for one
  (void)N_rows;
  b.labels[0] = W.take<int32_t>(N);
  b.labels[1] = W.take<int32_t>(N);
  b.centers[0] = W.take<float>(K * ldc);
  b.centers[1] = W.take<float>(K * ldc);
  b.sums = W.take<float>(K * ldc);
  b.counts = W.take<int32_t>(K + 1);   // [counts | n_changed] contiguous: one int32 all-reduce in the distributed run
  b.n_changed = b.counts + K;
  b.stats = W.take<double>(2 + K);
  b.xsplit = mode == 1 ? take_bytes(kmeans_tc_xsplit_bytes(N, D)) : nullptr;
  b.ws_assign_b = mode == 1 ? kmeans_assign_tc_ws_bytes(N, K, D) : gdr_kmeans_assign_ws_bytes(N, K, D, 0);
  b.ws_assign = take_bytes(b.ws_assign_b);
  b.ws_seg_b = gdr_segment_sum_ws_bytes(N, K, D);
  b.ws_seg = take_bytes(b.ws_seg_b);
  b.ws_misc_b = std::max(std::max(gdr_inertia_ws_bytes(N, D), gdr_kmeans_relocate_ws_bytes(N, K, D)),
                         relocate_candidates_ws_bytes(N));
  b.ws_misc = take_bytes(b.ws_misc_b);
  return W.off + 256;
}

struct HostStatus {
  double stats[2];
  int32_t n_changed;
  int32_t pad;
};

HostStatus* pinned_status() {
  static thread_local HostStatus* p = nullptr;
  if (!p && cudaHostAlloc((void**)&p, sizeof(HostStatus), cudaHostAllocDefault) != cudaSuccess) p = nullptr;
  return p;
}

// RAII for the internal stream / graphs so that every early return cleans up
struct GraphCtx {
  cudaStream_t gs = nullptr;
  cudaEvent_t ev = nullptr;
  cudaGraphExec_t exec[2] = {nullptr, nullptr};
  ~GraphCtx() {
    for (auto& e : exec)
      if (e) cudaGraphExecDestroy(e);
    if (ev) cudaEventDestroy(ev);
    if (gs) cudaStreamDestroy(gs);
  }
};

}  // namespace

namespace {

// Distributed _relocate_empty_clusters_dense (sklearn/_k_means_common.pyx:167-211): every rank proposes its n_empty
// farthest rows, the proposals are all-gathered, and all ranks apply the same global choice (largest distance first,
// ties by global row order) to the replicated, already reduced sums / counts.  Rare path: host-sorted.
int relocate_distributed(gdr_comm* comm, int64_t N, int64_t K, int64_t D, const float* Xc, int64_t ldx, const float* C_old,
                         int64_t ldw, const int32_t* labels, float* sums, int32_t* counts, void* ws, int64_t ws_bytes,
                         cudaStream_t s) {
  std::vector<int32_t> h_counts(K);
  GDR_CUDA(cudaMemcpyAsync(h_counts.data(), counts, K * 4, cudaMemcpyDeviceToHost, s));
  GDR_CUDA(cudaStreamSynchronize(s));
  std::vector<int32_t> empties;
  for (int64_t k = 0; k < K; ++k)
    if (h_counts[k] == 0) empties.push_back((int32_t)k);
  const int ne = (int)empties.size();
  if (ne == 0) return GDR_OK;
  const int world = comm->world;
  const int64_t rec_w = D + 3;
  float *rec = nullptr, *allrec = nullptr;
  int32_t* idx_dev = nullptr;
  GDR_CUDA(cudaMalloc(&rec, (size_t)ne * rec_w * 4));
  GDR_CUDA(cudaMalloc(&allrec, (size_t)ne * rec_w * 4 * world));
  GDR_CUDA(cudaMalloc(&idx_dev, (size_t)ne * 2 * 4));
  int rc = relocate_candidates(N, D, Xc, ldx, C_old, ldw, labels, ne, comm->rank, rec, ws, ws_bytes, s);
  if (rc == GDR_OK) rc = comm_allgather(comm, rec, allrec, (int64_t)ne * rec_w * 4, s);
  std::vector<float> h_dist((size_t)ne * world);
  if (rc == GDR_OK &&
      (cudaMemcpy2DAsync(h_dist.data(), 4, allrec, rec_w * 4, 4, (size_t)ne * world, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
       cudaStreamSynchronize(s) != cudaSuccess)) {
    set_error("relocate_distributed: read-back of the candidate distances failed");
    rc = GDR_ECUDA;
  }
  if (rc == GDR_OK) {
    std::vector<int32_t> order((size_t)ne * world);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return h_dist[a] > h_dist[b]; });
    if (h_dist[order[0]] > 0.f) {   // sklearn skips relocation when max(distances) == 0
      std::vector<int32_t> h_idx((size_t)ne * 2);
      for (int e = 0; e < ne; ++e) {
        h_idx[e] = h_dist[order[e]] < 0.f ? -1 : order[e];
        h_idx[ne + e] = empties[e];
      }
      if (cudaMemcpyAsync(idx_dev, h_idx.data(), (size_t)ne * 8, cudaMemcpyHostToDevice, s) != cudaSuccess) rc = GDR_ECUDA;
      if (rc == GDR_OK) rc = relocate_apply(ne, idx_dev, idx_dev + ne, allrec, D, sums, ldw, counts, s);
      if (cudaStreamSynchronize(s) != cudaSuccess && rc == GDR_OK) rc = GDR_ECUDA;
    }
  }
  cudaFree(rec);
  cudaFree(allrec);
  cudaFree(idx_dev);
  return rc;
}

// One Lloyd run.  comm == nullptr: the single-GPU loop.  With a communicator the rows are this rank's block of a
// row-partitioned X (N may be 0), the centres are replicated, and each iteration all-reduces
// [K x ld partial sums | K counts | n_changed] as ONE grouped NCCL operation inside the replayed CUDA graph; every
// rank then runs the identical finalise on identical data, so the replicated centres stay bit-identical across ranks
// and every rank takes the same convergence decision from its own 24-byte status read-back.
int lloyd_run(gdr_comm* comm, int64_t N, int64_t N_total, int64_t K, int64_t D, const float* Xc, int64_t ldx, float* C_inout,
              int64_t ldc, int32_t* labels_out, int max_iter, double tol_abs, int precision_mode,
              double* inertia_out_host, int32_t* n_iter_out_host, int32_t* info_out_host, int verbose,
              void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  const bool dist = comm != nullptr && comm->world > 1;
  cudaStream_t caller = (cudaStream_t)stream;
  HostStatus* hs = pinned_status();
  if (!hs) {
    set_error("kmeans_lloyd: cannot allocate the pinned status block");
    return GDR_ECUDA;
  }
  // Graph replay needs a capturable stream: run the whole loop on an internal stream that is
  // ordered after the caller's stream (and the caller's stream after it at the end).
  GraphCtx G;
  bool use_graph = g_lloyd_graph != 0 && !profiling_enabled() && max_iter >= (dist ? 5 : 3);
  // NCCL sets up its channels / buffers on the first collectives of a communicator (not capturable): the first
  // iteration of each buffer parity runs eagerly in the distributed loop and the capture starts after it
  const int first_graph_iter = dist ? 2 : 0;
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
  gdr_stream_t st = (gdr_stream_t)s;

  LloydBuffers B;
  carve(&B, ws, N, K, D, precision_mode);
  const int64_t ldw = align_up(D, 4);
  int rc;
  GDR_CUDA(cudaMemsetAsync(B.centers[0], 0, K * ldw * 4, s));
  GDR_CUDA(cudaMemsetAsync(B.centers[1], 0, K * ldw * 4, s));
  GDR_CUDA(cudaMemcpy2DAsync(B.centers[0], ldw * 4, C_inout, ldc * 4, D * 4, K, cudaMemcpyDeviceToDevice, s));
  if (N > 0) GDR_CUDA(cudaMemsetAsync(B.labels[1], 0xff, N * 4, s));  // labels_old = -1
  if (precision_mode == 1 && N > 0) {
    rc = gdr_kmeans_tc_prepare(N, D, Xc, ldx, B.xsplit, kmeans_tc_xsplit_bytes(N, D), st);
    if (rc) return rc;
  }
  auto assign = [&](const float* C, int32_t* lab, const int32_t* prev, int32_t* nchg) -> int {
    if (N == 0) return GDR_OK;
    if (precision_mode == 1)
      return gdr_kmeans_assign_tc(N, K, D, Xc, ldx, B.xsplit, C, ldw, lab, prev, nchg, nullptr, nullptr,
                                  B.ws_assign, B.ws_assign_b, st);
    return gdr_kmeans_assign(N, K, D, Xc, ldx, C, ldw, lab, prev, nchg, nullptr, 0, B.ws_assign, B.ws_assign_b, st);
  };
  // one iteration for buffer parity p (centres[p] -> centres[1-p], labels[p] new, labels[1-p] old),
  // ending with the status copy into pinned host memory
  auto enqueue_iteration = [&](int p) -> int {
    const int cur = p, nxt = 1 - p, lab_new = p, lab_old = 1 - p;
    GDR_CUDA(cudaMemsetAsync(B.n_changed, 0, 4, s));
    int r;
    if ((r = assign(B.centers[cur], B.labels[lab_new], B.labels[lab_old], B.n_changed))) return r;
    if (N > 0) {
      if ((r = gdr_segment_sum(N, K, D, Xc, ldx, B.labels[lab_new], B.sums, ldw, B.counts, B.ws_seg, B.ws_seg_b, st)))
        return r;
    } else {
      GDR_CUDA(cudaMemsetAsync(B.sums, 0, K * ldw * 4, s));
      GDR_CUDA(cudaMemsetAsync(B.counts, 0, K * 4, s));
    }
    if (dist && (r = comm_allreduce_lloyd(comm, B.sums, K * ldw, B.counts, K + 1, s))) return r;
    if ((r = gdr_kmeans_finalize(K, D, B.sums, ldw, B.counts, B.centers[cur], ldw, B.centers[nxt], ldw, B.stats, 0, st)))
      return r;
    GDR_CUDA(cudaMemcpyAsync(hs->stats, B.stats, 16, cudaMemcpyDeviceToHost, s));
    GDR_CUDA(cudaMemcpyAsync(&hs->n_changed, B.n_changed, 4, cudaMemcpyDeviceToHost, s));
    return GDR_OK;
  };
  auto run_iteration = [&](int p, int i) -> int {
    if (use_graph && i >= first_graph_iter) {
      if (!G.exec[p]) {
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
          int r = enqueue_iteration(p);
          cudaError_t e = cudaStreamEndCapture(s, &graph);
          if (r == GDR_OK && e == cudaSuccess && graph &&
              cudaGraphInstantiate(&G.exec[p], graph, 0) == cudaSuccess) {
            cudaGraphDestroy(graph);
          } else {
            if (graph) cudaGraphDestroy(graph);
            G.exec[p] = nullptr;
            cudaGetLastError();
            use_graph = false;  // capture not possible here: issue the launches directly
            if (r != GDR_OK) return r;
          }
        } else {
          cudaGetLastError();
          use_graph = false;
        }
      }
      if (use_graph && G.exec[p]) {
        GDR_CUDA(cudaGraphLaunch(G.exec[p], s));
        count_launch(1);
        return GDR_OK;
      }
    }
    return enqueue_iteration(p);
  };

  int p = 0;
  bool strict = false;
  int n_iter = 0, relocations = 0;
  for (int i = 0; i < max_iter; ++i) {
    n_iter = i + 1;
    if ((rc = run_iteration(p, i))) return rc;
    GDR_CUDA(cudaStreamSynchronize(s));
    double shift_tot = hs->stats[0];
    const int n_empty = (int)hs->stats[1];
    const int n_changed = hs->n_changed;
    const int cur = p, nxt = 1 - p;
    if (n_empty > 0) {
      // _relocate_empty_clusters_dense (sklearn/_k_means_common.pyx:167-211), then re-average
      ++relocations;
      if (dist)
        rc = relocate_distributed(comm, N, K, D, Xc, ldx, B.centers[cur], ldw, B.labels[p], B.sums, B.counts, B.ws_misc,
                                  B.ws_misc_b, s);
      else
        rc = gdr_kmeans_relocate(N, K, D, Xc, ldx, B.centers[cur], ldw, B.labels[p], B.sums, ldw, B.counts,
                                 B.ws_misc, B.ws_misc_b, st);
      if (rc) return rc;
      if ((rc = gdr_kmeans_finalize(K, D, B.sums, ldw, B.counts, B.centers[cur], ldw, B.centers[nxt], ldw, B.stats, 0,
                                    st)))
        return rc;
      GDR_CUDA(cudaMemcpyAsync(hs->stats, B.stats, 16, cudaMemcpyDeviceToHost, s));
      GDR_CUDA(cudaStreamSynchronize(s));
      shift_tot = hs->stats[0];
    }
    if (verbose && (!dist || comm->rank == 0))
      printf("Iteration %d, center shift %.6g, labels changed %d.\n", i, shift_tot, n_changed);
    if (n_changed == 0) {  // np.array_equal(labels, labels_old)  (:723-729)
      strict = true;
      p = 1 - p;  // centres[nxt] are current; labels[cur parity] stay the newest
      break;
    }
    p = 1 - p;
    if (shift_tot <= tol_abs) break;  // (:731-738)
  }
  // after the loop: centres[p] are the current centres, labels[1 - p] the newest labels
  // (max_iter == 0: centres[0], labels undefined -> the E-step below fills them)
  int32_t* labels = n_iter == 0 ? B.labels[0] : B.labels[1 - p];
  if (!strict) {
    // rerun the E-step so that the labels match the final centres (:742-754)
    if ((rc = assign(B.centers[p], labels, nullptr, nullptr))) return rc;
  }
  double* inertia_dev = B.stats;
  if (N > 0) {
    if ((rc = gdr_inertia(N, D, Xc, ldx, B.centers[p], ldw, labels, inertia_dev, B.ws_misc, B.ws_misc_b, st))) return rc;
  } else {
    GDR_CUDA(cudaMemsetAsync(inertia_dev, 0, 8, s));
  }
  if (dist && (rc = comm_allreduce_f64(comm, inertia_dev, 1, 0, s))) return rc;
  GDR_CUDA(cudaMemcpyAsync(hs->stats, inertia_dev, 8, cudaMemcpyDeviceToHost, s));
  if (N > 0) GDR_CUDA(cudaMemcpyAsync(labels_out, labels, N * 4, cudaMemcpyDeviceToDevice, s));
  GDR_CUDA(cudaMemcpy2DAsync(C_inout, ldc * 4, B.centers[p], ldw * 4, D * 4, K, cudaMemcpyDeviceToDevice, s));
  GDR_CUDA(cudaStreamSynchronize(s));
  if (s != caller) {
    // later work on the caller's stream must see our results (already complete: we synchronised)
    GDR_CUDA(cudaEventRecord(G.ev, s));
    GDR_CUDA(cudaStreamWaitEvent(caller, G.ev, 0));
  }
  if (inertia_out_host) *inertia_out_host = hs->stats[0];
  if (n_iter_out_host) *n_iter_out_host = n_iter;
  if (info_out_host) {
    info_out_host[0] = strict ? 1 : 0;
    info_out_host[1] = relocations;
  }
  (void)N_total;
  return GDR_OK;
}

}  // namespace

extern "C" {

int64_t gdr_kmeans_lloyd_ws_bytes(int64_t N, int64_t K, int64_t D, int precision_mode) {
  return carve(nullptr, nullptr, N, K, D, precision_mode);
}

int gdr_kmeans_lloyd(int64_t N, int64_t K, int64_t D, const float* Xc, int64_t ldx, float* C_inout,
                     int64_t ldc, int32_t* labels_out, int max_iter, double tol_abs, int precision_mode,
                     double* inertia_out_host, int32_t* n_iter_out_host, int32_t* info_out_host, int verbose,
                     void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(N > 0 && K > 0 && D > 0 && Xc && C_inout && labels_out && ws, "kmeans_lloyd: bad arguments");
  GDR_CHECK_ARG(N >= K, "kmeans_lloyd: n_samples=%lld should be >= n_clusters=%lld", (long long)N, (long long)K);
  GDR_CHECK_ARG(precision_mode == 0 || precision_mode == 1, "kmeans_lloyd: precision_mode");
  GDR_CHECK_ARG(max_iter >= 0, "kmeans_lloyd: max_iter");
  if (ws_bytes < gdr_kmeans_lloyd_ws_bytes(N, K, D, precision_mode)) {
    set_error("kmeans_lloyd: workspace too small");
    return GDR_EWORKSPACE;
  }
  return lloyd_run(nullptr, N, N, K, D, Xc, ldx, C_inout, ldc, labels_out, max_iter, tol_abs, precision_mode,
                   inertia_out_host, n_iter_out_host, info_out_host, verbose, ws, ws_bytes, stream);
}

int gdr_kmeans_lloyd_dist(gdr_comm_t* comm, int64_t N_local, int64_t N_total, int64_t K, int64_t D, const float* Xc_local,
                          int64_t ldx, float* C_inout, int64_t ldc, int32_t* labels_out, int max_iter, double tol_abs,
                          int precision_mode, double* inertia_out_host, int32_t* n_iter_out_host, int32_t* info_out_host,
                          int verbose, void* ws, int64_t ws_bytes, gdr_stream_t stream) {
  GDR_CHECK_ARG(comm && N_local >= 0 && K > 0 && D > 0 && C_inout && ws && (N_local == 0 || (Xc_local && labels_out)),
                "kmeans_lloyd_dist: bad arguments");
  GDR_CHECK_ARG(N_total >= K, "kmeans_lloyd_dist: n_samples=%lld should be >= n_clusters=%lld", (long long)N_total,
                (long long)K);
  GDR_CHECK_ARG(precision_mode == 0 || precision_mode == 1, "kmeans_lloyd_dist: precision_mode");
  GDR_CHECK_ARG(max_iter >= 0, "kmeans_lloyd_dist: max_iter");
  if (ws_bytes < gdr_kmeans_lloyd_ws_bytes(N_local, K, D, precision_mode)) {
    set_error("kmeans_lloyd_dist: workspace too small");
    return GDR_EWORKSPACE;
  }
  return lloyd_run(comm, N_local, N_total, K, D, Xc_local, ldx, C_inout, ldc, labels_out, max_iter, tol_abs, precision_mode,
                   inertia_out_host, n_iter_out_host, info_out_host, verbose, ws, ws_bytes, stream);
}

}  // extern "C"
