"""Row-partitioned multi-GPU execution of the distillation core (SURVEY §8e).

One process per GPU (``torch.distributed``; NCCL over NVLink on the B200 box, gloo in the CPU
tests).  Nodes are split into contiguous row blocks; the reference itself is single-device,
so nothing is ported here — the exchanges are the ones the algorithm needs:

  stage 2  all-gather of the propagated rows before each hop (every rank then runs the CSR
           SpMM on its own rows of A_hat against the full feature matrix).  The hop is pipelined
           over COLUMN SLABS of the feature matrix: slab s+1 is in flight on the collective's
           stream while the SpMM of slab s runs — different columns are independent fp32 chains,
           so the result stays bit-identical to the one-pass hop;
  stage 3  per Lloyd iteration ONE all-reduce of the [K x D] partial sums and ONE of the
           packed int32 [counts | n_changed]; every rank finalises identically, so the
           replicated centres stay bit-identical across ranks;
  means    the [K x D] per-cluster sums handed from rank to rank, each chain continued where the
           previous rank ended it, then sent to all (dist_cluster_means: the one-GPU bytes);
  sparsify all-gather of the degree vector and the logits; per radix pass of the top-k one all-reduce
           of the per-rank histograms, then one all-gather of the tie counts (dist_graph_sparse);
  stage 4  all-gather of the labels, local segmented edge counting, dense n x n all-reduce of
           (int32 counts, f32 sums), compaction back to CSR.

All arithmetic goes through an ``ops`` object.  ``CudaOps`` (default) calls libgdr_b200;
the CPU tests inject an oracle-backed stand-in so that the partition / packing / collective
logic is exercised with world_size 2 on gloo.  Integer outputs are independent of the
number of ranks; float outputs agree to the §8c tolerances (the all-reduce order changes
with the rank count).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from .kmeans import MiniBatchKMeans


@dataclass
class RowPartition:
    n: int
    world: int
    rank: int

    @property
    def rows_per(self) -> int:
        return (self.n + self.world - 1) // self.world

    def bounds(self, rank: Optional[int] = None) -> Tuple[int, int]:
        r = self.rank if rank is None else rank
        lo = min(self.n, r * self.rows_per)
        return lo, min(self.n, lo + self.rows_per)

    @property
    def lo(self) -> int:
        return self.bounds()[0]

    @property
    def hi(self) -> int:
        return self.bounds()[1]

    @property
    def n_local(self) -> int:
        lo, hi = self.bounds()
        return hi - lo


def _wire(t: torch.Tensor) -> torch.Tensor:
    """The tensor a collective is given for ``t``.  Row-padded matrices (``_dev.new_padded``: width f inside a
    leading dimension pad4(f)) are non-contiguous views whenever f % 4 != 0, which NCCL and gloo reject; the
    collective then runs on the padded base (same storage, all ld columns — the padding columns are zeros on every
    rank, so sums and gathers leave them zero)."""
    if t.is_contiguous():
        return t
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1]:
        ld, rows = t.stride(0), t.shape[0]
        have = t.untyped_storage().nbytes() // t.element_size() - t.storage_offset()
        if rows * ld <= have:
            return t.as_strided((rows, ld), (ld, 1))
    raise ValueError("collective on a non-contiguous tensor that is not a row-padded matrix")


class Comm:
    """Thin wrapper over torch.distributed (or a no-op for world size 1)."""

    def __init__(self, dist=None, group=None):
        self.dist, self.group = dist, group
        self.world = 1 if dist is None else dist.get_world_size(group)
        self.rank = 0 if dist is None else dist.get_rank(group)
        self.backend = None if dist is None else dist.get_backend(group)

    # -- the library's own communicator (gdr_comm_t: NCCL bound inside libgdr_b200) --------------------
    def lib_handle(self):
        """gdr_comm_t* of this group, created on first use (collective: every rank must call it at the same
        point).  Rank 0 draws the NCCL unique id through the C ABI, torch.distributed broadcasts the 128 bytes."""
        if getattr(self, "_lib_comm", None) is not None:
            return self._lib_comm
        import ctypes
        from . import _lib
        handle = ctypes.c_void_p()
        if self.dist is None or self.world == 1:
            _lib.call("gdr_comm_init", ctypes.addressof(handle), 0, 0, 1)
        else:
            if self.backend != "nccl":
                raise RuntimeError("the in-library communicator needs the nccl backend")
            idbuf = (ctypes.c_ubyte * 128)()
            if self.rank == 0:
                _lib.call("gdr_comm_unique_id", ctypes.addressof(idbuf))
            t = torch.tensor(list(bytes(idbuf)), dtype=torch.uint8, device=torch.device("cuda", torch.cuda.current_device()))
            src = self.dist.get_global_rank(self.group, 0) if self.group is not None else 0
            self.dist.broadcast(t, src=src, group=self.group)
            raw = bytes(t.cpu().tolist())
            idbuf = (ctypes.c_ubyte * 128).from_buffer_copy(raw)
            _lib.call("gdr_comm_init", ctypes.addressof(handle), ctypes.addressof(idbuf), self.rank, self.world)
        self._lib_comm = handle
        return handle

    def symm(self, nbytes: int):
        """Symmetric buffer of at least ``nbytes`` on every rank (gdr_symm_t: peer-mapped over NVLink), cached; returns
        (handle, local device pointer).  Collective.  Raises GdrError when peer memory is not available."""
        import ctypes
        from . import _lib
        cur = getattr(self, "_symm", None)
        if cur is not None and cur[2] >= nbytes:
            return cur[0], cur[1]
        if cur is not None:
            _lib.call("gdr_symm_destroy", cur[0])
            self._symm = None
        h = ctypes.c_void_p()
        _lib.call("gdr_symm_create", self.lib_handle(), int(nbytes), ctypes.addressof(h))
        ptr, size = ctypes.c_void_p(), ctypes.c_int64()
        _lib.call("gdr_symm_info", h, ctypes.addressof(ptr), ctypes.addressof(size))
        self._symm = (h, int(ptr.value), int(size.value))
        return h, int(ptr.value)

    def count_matrix(self, send_counts, device):
        """cnt[src][dst] = rows rank src sends to rank dst, on every rank (one small all-gather + read-back)."""
        sc = torch.tensor([int(c) for c in send_counts], dtype=torch.int64, device=device)
        mat = torch.empty(self.world * self.world, dtype=torch.int64, device=device)
        self.all_gather_rows(sc, mat)
        return mat.view(self.world, self.world).tolist()

    def symm_ok(self) -> bool:
        """True when exchanges can go through peer memory (NCCL process group on CUDA, peer access available).  The first
        call creates a small symmetric buffer to find out — collective, like every call that follows it."""
        global _P2P_BROKEN
        if self.dist is None or self.world <= 1 or self.backend != "nccl" or _P2P_BROKEN \
                or not getattr(self, "use_symm_exchange", True):
            return False
        if getattr(self, "_symm", None) is None:
            try:
                self.symm(1 << 20)
            except Exception as e:       # GdrError from gdr_symm_create: no peer access between these GPUs
                import warnings
                warnings.warn(f"peer memory unavailable ({e}); exchanges go through NCCL")
                _P2P_BROKEN = True
                return False
        return True

    def symm_exchange(self, arrays, cnt_mat):
        """Variable all-to-all of several arrays with the SAME row split, through the symmetric buffer (gdr_symm_scatterv:
        one kernel of posted NVLink stores per array, two stream-ordered barriers in all; no NCCL).  ``arrays[a]`` holds
        the rows for rank 0, 1, ... back to back; ``cnt_mat[src][dst]`` = rows rank src sends to rank dst (known to every
        rank).  Returns the received rows (source-rank order) as VIEWS of the symmetric buffer — valid until the next
        exchange or fused propagation on this communicator; clone what has to live longer."""
        return self._symm_exchange(arrays, cnt_mat, gather=False)

    def all_gather_symm(self, arrays, counts):
        """Concatenation over the ranks of every rank's 1-D block (``counts[r]`` rows from rank r), same transport."""
        w = self.world
        return self._symm_exchange(arrays, [[int(counts[s])] * w for s in range(w)], gather=True)

    def _symm_exchange(self, arrays, cnt_mat, gather):
        import ctypes
        from . import _lib
        w, me = self.world, self.rank
        srcs = [a.contiguous() for a in arrays]
        rowb = [a.element_size() * int(np.prod(a.shape[1:], dtype=np.int64)) for a in srcs]
        plan = exchange_plan(cnt_mat, me, rowb, gather)
        tot, regions, need = plan["rows_here"], plan["regions"], plan["bytes"]
        cur = getattr(self, "_symm", None)
        h, base = self.symm(max(need, cur[2] if cur is not None else 0))
        st = torch.cuda.current_stream().cuda_stream
        arr = ctypes.c_int64 * w
        sc, so_arr = arr(*plan["send_cnt"]), arr(*plan["send_off"])      # named: ctypes.addressof of a temporary dangles
        _lib.call("gdr_symm_barrier", h, st)              # every rank is done with what lay in the buffer
        for a, eb, dst in zip(srcs, rowb, plan["dst_off_bytes"]):
            do = arr(*dst)
            _lib.call("gdr_symm_scatterv", h, a.data_ptr() if a.numel() else 0, ctypes.addressof(so_arr), ctypes.addressof(sc),
                      ctypes.addressof(do), eb, st)
        _lib.call("gdr_symm_barrier", h, st)
        return [_device_view(base + reg, (tot,) + tuple(a.shape[1:]), a.dtype, a.device) for a, reg in zip(srcs, regions)]

    def close(self):
        """Destroys the library communicator (call before torch.distributed.destroy_process_group)."""
        if getattr(self, "_symm", None) is not None:
            from . import _lib
            _lib.call("gdr_symm_destroy", self._symm[0])
            self._symm = None
        h = getattr(self, "_lib_comm", None)
        if h is not None:
            from . import _lib
            _lib.call("gdr_comm_destroy", h)
            self._lib_comm = None

    def all_reduce(self, t: torch.Tensor, op: str = "sum") -> torch.Tensor:
        if self.dist is not None and self.world > 1:
            ops = {"sum": self.dist.ReduceOp.SUM, "max": self.dist.ReduceOp.MAX, "min": self.dist.ReduceOp.MIN}
            self.dist.all_reduce(_wire(t), op=ops[op], group=self.group)
        return t

    def all_gather_rows(self, local: torch.Tensor, out: torch.Tensor, async_op: bool = False):
        """out[(r*rows):(r+1)*rows] = local of rank r; all ranks pass equally shaped blocks.
        ``async_op``: returns a handle whose ``wait()`` orders the CURRENT stream after the
        collective (NCCL runs it on its own stream, so work enqueued before the wait overlaps)."""
        if self.dist is None or self.world == 1:
            out[: local.shape[0]].copy_(local)
            return _Done() if async_op else out
        lw, ow = _wire(local), _wire(out)
        if lw.dim() == 2 and lw.shape[1] != ow.shape[1]:
            raise ValueError("all_gather_rows: blocks of different leading dimension")
        if self.backend == "nccl":
            w = self.dist.all_gather_into_tensor(ow, lw, group=self.group, async_op=async_op)
        else:
            chunks = list(ow.chunk(self.world, dim=0))
            w = self.dist.all_gather(chunks, lw, group=self.group, async_op=async_op)
        return w if async_op else out


    def all_to_all_rows(self, send: torch.Tensor, send_counts, recv_counts=None) -> Tuple[torch.Tensor, list]:
        """Variable all-to-all along dim 0: ``send`` holds the rows for rank 0, 1, ... back to back
        (``send_counts[r]`` rows each).  Returns (received rows in source-rank order, recv_counts); ``recv_counts`` of an
        earlier exchange with the same counts can be passed in to skip the count exchange."""
        if self.dist is None or self.world == 1:
            n0 = int(send_counts[0])
            return send[:n0], [n0]
        if recv_counts is None:
            sc = torch.tensor([int(c) for c in send_counts], dtype=torch.int64, device=send.device)
            rc = torch.empty_like(sc)
            if self.backend == "nccl":
                self.dist.all_to_all_single(rc, sc, group=self.group)
            else:   # gloo has no all_to_all: gather the whole count matrix
                mat = [torch.empty_like(sc) for _ in range(self.world)]
                self.dist.all_gather(mat, sc, group=self.group)
                rc = torch.stack([m[self.rank] for m in mat])
            recv_counts = [int(c) for c in rc.tolist()]
        send = send[: int(sum(int(c) for c in send_counts))]
        out = torch.empty((sum(recv_counts),) + tuple(send.shape[1:]), dtype=send.dtype, device=send.device)
        if self.backend == "nccl":
            self.dist.all_to_all_single(out, send, recv_counts, [int(c) for c in send_counts], group=self.group)
        else:
            so = np.concatenate([[0], np.cumsum(send_counts)]).astype(np.int64)
            ro = np.concatenate([[0], np.cumsum(recv_counts)]).astype(np.int64)
            reqs = []
            for peer in range(self.world):
                if peer == self.rank:
                    out[ro[peer]:ro[peer + 1]].copy_(send[so[peer]:so[peer + 1]])
                    continue
                if recv_counts[peer]:
                    reqs.append(self.dist.irecv(out[ro[peer]:ro[peer + 1]], src=peer, group=self.group))
                if send_counts[peer]:
                    reqs.append(self.dist.isend(send[so[peer]:so[peer + 1]].contiguous(), dst=peer, group=self.group))
            for r in reqs:
                r.wait()
        return out, recv_counts

    def all_gather_var(self, local: torch.Tensor, counts) -> torch.Tensor:
        """Concatenation of every rank's 1-D ``local`` (``counts[r]`` elements from rank r)."""
        if self.dist is None or self.world == 1:
            return local
        if self.backend == "nccl" and local.is_cuda:
            # straight into place: one grouped send / recv set inside the library (gdr_alltoallv with the same block for
            # every peer), no padding to the largest piece and no concatenation pass
            import ctypes
            from . import _lib
            w = self.world
            arr = ctypes.c_int64 * w
            offs, tot = [], 0
            for c in counts:
                offs.append(tot)
                tot += int(c)
            out = torch.empty(tot, dtype=local.dtype, device=local.device)
            src = local.contiguous()
            so, sc = arr(*([0] * w)), arr(*([int(src.shape[0])] * w))
            ro, rc = arr(*offs), arr(*[int(c) for c in counts])
            _lib.call("gdr_alltoallv", self.lib_handle(), src.data_ptr(), ctypes.addressof(so), ctypes.addressof(sc), out.data_ptr(),
                      ctypes.addressof(ro), ctypes.addressof(rc), src.element_size(), torch.cuda.current_stream().cuda_stream)
            return out
        m = max(int(c) for c in counts)
        block = torch.zeros(m, dtype=local.dtype, device=local.device)
        block[: local.shape[0]] = local
        out = torch.empty(m * self.world, dtype=local.dtype, device=local.device)
        self.all_gather_rows(block, out)
        return torch.cat([out[r * m: r * m + int(counts[r])] for r in range(self.world)])


def exchange_plan(cnt_mat, me: int, row_bytes, gather: bool = False) -> dict:
    """Where rank ``me`` reads and writes in a symmetric-buffer exchange (pure host arithmetic; tests/test_parallel_gloo.py
    replays it for every rank of a world against a byte-level simulation).  ``cnt_mat[src][dst]`` rows go from src to dst;
    array a (``row_bytes[a]`` per row) occupies the SAME region of every rank's buffer, rows in source-rank order.
    ``gather``: every destination receives the sender's whole block (send offset 0)."""
    w = len(cnt_mat)
    tot = [sum(int(cnt_mat[s][d]) for s in range(w)) for d in range(w)]
    place = [sum(int(cnt_mat[s][p]) for s in range(me)) for p in range(w)]         # my rows' first row on rank p
    regions, need = [], 0
    for eb in row_bytes:
        if eb <= 0 or eb % 4:
            raise ValueError("symm_exchange: rows must be multiples of 4 bytes")
        regions.append(need)
        need += (max(tot) * eb + 255) // 256 * 256
    send_cnt = [int(cnt_mat[me][p]) for p in range(w)]
    send_off, acc = [], 0
    for p in range(w):
        send_off.append(0 if gather else acc)
        acc += send_cnt[p]
    return {"rows_here": tot[me], "regions": regions, "bytes": max(need, 256), "send_cnt": send_cnt, "send_off": send_off,
            "dst_off_bytes": [[reg + place[p] * eb for p in range(w)] for reg, eb in zip(regions, row_bytes)]}


class _DevWindow:
    """A window of a device allocation owned by the library, described by the CUDA array interface."""
    _TYPESTR = {torch.int64: "<i8", torch.int32: "<i4", torch.float32: "<f4", torch.float64: "<f8", torch.uint8: "|u1"}

    def __init__(self, ptr, shape, dtype):
        self.__cuda_array_interface__ = {"shape": tuple(int(v) for v in shape), "typestr": self._TYPESTR[dtype],
                                         "data": (int(ptr), False), "version": 2, "strides": None}


def _device_view(ptr: int, shape, dtype, device) -> torch.Tensor:
    """Tensor aliasing ``shape`` elements of ``dtype`` at device address ``ptr`` (no copy, no ownership)."""
    if int(np.prod(shape)) == 0:
        return torch.empty(tuple(shape), dtype=dtype, device=device)
    return torch.as_tensor(_DevWindow(ptr, shape, dtype), device=device)


class _Done:
    def wait(self):
        return True


# ------------------------------------------------------------------------------------------
# compute backend on the GPU
# ------------------------------------------------------------------------------------------
class CudaOps:
    """The kernels of libgdr_b200 behind the small interface the distributed drivers need."""

    def __init__(self, precision: str = "auto"):
        from . import _lib, coarsen, graph, kmeans, propagation
        from ._dev import new_padded, padded_rows, ptr, stream, workspace
        self._lib, self._g, self._km, self._pr, self._co = _lib, graph, kmeans, propagation, coarsen
        self.new_padded, self.padded_rows, self.ptr, self.stream, self.workspace = new_padded, padded_rows, ptr, stream, workspace
        self.precision = precision
        self._tc = None

    # -- stage 1 --
    def edges_route(self, row, col, n_rows, n_cols, rows_per, world, symmetrize):
        """This rank's (row, col) pairs [and their mirrors] -> keys (row << bits(n_cols)) | col tagged with the owner of the
        row, grouped by owner with one stable partition pass (gdr_edges_route).  Returns (keys int64, keys per owner,
        status: bit 0 = index out of range, bit 1 = the pair (0, 0) occurs)."""
        E = int(row.numel())
        dev = row.device
        m = E * (2 if symmetrize else 1)
        keys = torch.empty(max(m, 1), dtype=torch.int64, device=dev)
        meta = torch.zeros(130, dtype=torch.int64, device=dev)        # [owner starts 0..128 | status]
        ws = self.workspace(self._lib.query("gdr_edges_route_ws_bytes", E, int(symmetrize)), dev)
        self._lib.call("gdr_edges_route", E, self.ptr(row), self.ptr(col), int(n_rows), int(n_cols), int(symmetrize), int(rows_per),
                       int(world), self.ptr(keys), self.ptr(meta), self.ptr(meta[129:]), self.ptr(ws), ws.numel(), self.stream())
        h = meta.cpu().tolist()
        return keys, [int(h[r + 1] - h[r]) for r in range(world)], int(h[129]) & 0xFFFFFFFF

    def csr_from_keys(self, keys, row_lo, n_local, n_cols, binarize):
        """Keys received from every rank -> CSR of the local row block (gdr_csr_from_keys: keys-only sort + two-pass emit)."""
        m = int(keys.shape[0])
        dev = keys.device
        rowptr = torch.empty(n_local + 1, dtype=torch.int32, device=dev)
        colidx = torch.empty(max(m, 1), dtype=torch.int32, device=dev)
        vals = torch.empty(max(m, 1), dtype=torch.float32, device=dev)
        nnz = torch.zeros(1, dtype=torch.int64, device=dev)
        ws = self.workspace(self._lib.query("gdr_csr_from_keys_ws_bytes", m), dev)
        self._lib.call("gdr_csr_from_keys", m, self.ptr(keys) if m else 0, int(row_lo), int(n_local), int(n_cols), int(binarize),
                       self.ptr(rowptr), self.ptr(colidx), self.ptr(vals), self.ptr(nnz), self.ptr(ws), ws.numel(), self.stream())
        k = int(nnz.item())
        return self._g.CSR(rowptr, colidx[:k], vals[:k], (n_local, n_cols))

    def bucket_by_owner(self, src, dst, rows_per, world):
        """Edges (src, dst) reordered so that the edges of owner 0, 1, ... (owner = src // rows_per) are
        contiguous; returns ([E, 2] int64 rows, per-owner counts).  Stable radix sort on the owner id."""
        E = int(src.shape[0])
        dev = src.device
        owner = torch.div(src, rows_per, rounding_mode="floor")
        keys = owner.contiguous().view(torch.int64).clone()
        perm = torch.arange(E, dtype=torch.int32, device=dev)
        if E:
            ws = self.workspace(self._lib.query("gdr_sort_pairs_ws_bytes", E), dev)
            bits = max(1, int(world - 1).bit_length())
            self._lib.call("gdr_sort_pairs", E, bits, self.ptr(keys), self.ptr(perm), self.ptr(ws), ws.numel(), self.stream())
        counts = torch.bincount(owner, minlength=world)[:world].tolist()
        p = perm.long()
        return torch.stack([src[p], dst[p]], dim=1).contiguous(), counts

    def build_block_csr(self, rows_local, cols, n_local, n):
        """Binarised CSR of a row block (duplicates merged, columns sorted), global column ids."""
        return self._g.coo_to_csr(rows_local, cols, None, (n_local, n), symmetrize=False, binarize=True,
                                  device=rows_local.device)

    def block_degrees(self, A_blk, row_offset, add_identity):
        nl = A_blk.shape[0]
        dev = A_blk.device
        deg = torch.empty(nl, dtype=torch.float64, device=dev)
        rowptr_out = torch.empty(nl + 1, dtype=torch.int32, device=dev)
        ws = self.workspace(self._lib.query("gdr_sym_normalize_block_ws_bytes", nl), dev)
        self._lib.call("gdr_sym_normalize_block_degrees", nl, int(row_offset), self.ptr(A_blk.rowptr), self.ptr(A_blk.colidx),
                       self.ptr(A_blk.vals), int(add_identity), self.ptr(deg), self.ptr(rowptr_out), self.ptr(ws), ws.numel(),
                       self.stream())
        return deg, rowptr_out

    def block_fill(self, A_blk, row_offset, add_identity, deg_global, rowptr_out):
        nl = A_blk.shape[0]
        dev = A_blk.device
        cap = A_blk.nnz + nl
        colidx = torch.empty(cap, dtype=torch.int32, device=dev)
        vals = torch.empty(cap, dtype=torch.float32, device=dev)
        nnz_out = torch.zeros(1, dtype=torch.int64, device=dev)
        ws = self.workspace(256, dev)
        self._lib.call("gdr_sym_normalize_block_fill", nl, int(row_offset), self.ptr(A_blk.rowptr), self.ptr(A_blk.colidx),
                       self.ptr(A_blk.vals), int(add_identity), self.ptr(deg_global), self.ptr(rowptr_out), self.ptr(colidx),
                       self.ptr(vals), self.ptr(nnz_out), self.ptr(ws), ws.numel(), self.stream())
        m = int(nnz_out.item())
        return self._g.CSR(rowptr_out, colidx[:m], vals[:m], A_blk.shape)

    # -- bipartite (distill_recsys) --
    def build_block_csr_weighted(self, rows_local, cols, n_local, n_cols):
        """CSR of a row block with duplicate (row, col) lines SUMMED (distill_recsys.py:110-117), global column ids."""
        return self._g.coo_to_csr(rows_local, cols, None, (n_local, n_cols), symmetrize=False, binarize=False,
                                  device=rows_local.device)

    def row_sums(self, A):
        deg = torch.empty(A.shape[0], dtype=torch.float32, device=A.device)
        if A.shape[0]:
            self._lib.call("gdr_row_sums_f32", A.shape[0], self.ptr(A.rowptr), self.ptr(A.vals), self.ptr(deg), self.stream())
        return deg

    def bip_norm_block(self, A, deg_rows, deg_cols, eps):
        norm = torch.empty_like(A.vals)
        self._lib.call("gdr_bipartite_norm_block", A.shape[0], A.nnz, self.ptr(A.rowptr), self.ptr(A.colidx), self.ptr(A.vals),
                       self.ptr(deg_rows), self.ptr(deg_cols), float(eps), self.ptr(norm), self.stream())
        return self._g.CSR(A.rowptr, A.colidx, norm, A.shape)

    def column_moments(self, X, mean64):
        N, D = X.shape
        out = torch.zeros(2 * D, dtype=torch.float64, device=X.device)
        ws = self.workspace(self._lib.query("gdr_center_columns_ws_bytes", max(N, 1), D), X.device)
        self._lib.call("gdr_column_moments", N, D, self.ptr(X) if N else 0, X.stride(0) if N else D, self.ptr(mean64), self.ptr(out),
                       self.ptr(ws), ws.numel(), self.stream())
        return out

    def standardize_apply(self, X, mean32, scale32):
        N, D = X.shape
        out = self.new_padded(N, D, X.device)
        self._lib.call("gdr_standardize_apply", N, D, self.ptr(X) if N else 0, X.stride(0) if N else D, self.ptr(mean32),
                       self.ptr(scale32), self.ptr(out) if N else 0, out.stride(0) if N else D, self.stream())
        return out

    # -- stage 2 --
    def empty_rows(self, rows, f, like):
        return self.new_padded(rows, f, like.device, zero=True)

    def scale(self, x, a):
        out = self.new_padded(x.shape[0], x.shape[1], x.device)
        self._lib.call("gdr_scale_rows", x.shape[0], x.shape[1], float(a), self.ptr(x), x.stride(0), self.ptr(out),
                       out.stride(0), self.stream())
        return out

    def spmm(self, A_local, x_full, alpha, target, beta):
        y = self.new_padded(A_local.shape[0], x_full.shape[1], x_full.device)
        plan = A_local.spmm_plan()
        self._lib.call("gdr_spmm_prop_planned", A_local.shape[0], x_full.shape[1], self.ptr(A_local.rowptr),
                       self.ptr(A_local.colidx), self.ptr(A_local.vals), float(alpha), self.ptr(x_full), x_full.stride(0),
                       self.ptr(y), y.stride(0), self.ptr(target), 0 if target is None else target.stride(0), float(beta),
                       self.ptr(plan), plan.numel() - 1, self.stream())
        return y

    def remap_chunk_major(self, A, rows_per, cr, world):
        out = torch.empty_like(A.colidx)
        self._lib.call("gdr_remap_chunk_major", A.nnz, self.ptr(A.colidx), int(rows_per), int(cr), int(world), self.ptr(out),
                       self.stream())
        return self._g.CSR(A.rowptr, out, A.vals, A.shape)

    def slice_row_chunks(self, A, bounds):
        """Row blocks [bounds[k], bounds[k+1]) of a device CSR (views of colidx / vals), one host read for all cuts."""
        cuts = A.rowptr[torch.as_tensor(bounds, dtype=torch.int64, device=A.rowptr.device)].cpu().tolist()
        out = []
        for k in range(len(bounds) - 1):
            lo, hi, b, e = bounds[k], bounds[k + 1], int(cuts[k]), int(cuts[k + 1])
            out.append(self._g.CSR((A.rowptr[lo: hi + 1] - b).contiguous(), A.colidx[b:e], A.vals[b:e], (hi - lo, A.shape[1])))
        return out

    def spmm_rows(self, A_chunk, x_full, alpha, y, target, beta, r0):
        """Rows [r0, r0 + A_chunk.rows) of y (and of target):  y = (alpha*A_chunk) @ x_full ; target += beta * y."""
        rows, f = A_chunk.shape[0], x_full.shape[1]
        if rows == 0:
            return
        plan = A_chunk.spmm_plan()
        yo, to = y[r0: r0 + rows], None if target is None else target[r0: r0 + rows]
        self._lib.call("gdr_spmm_prop_planned", rows, f, self.ptr(A_chunk.rowptr), self.ptr(A_chunk.colidx),
                       self.ptr(A_chunk.vals), float(alpha), self.ptr(x_full), x_full.stride(0), self.ptr(yo), y.stride(0),
                       self.ptr(to), 0 if target is None else target.stride(0), float(beta), self.ptr(plan),
                       plan.numel() - 1, self.stream())

    def spmm_slab(self, A_local, x_slab, alpha, y, target, beta, c0):
        """y[:, c0:c0+w] = (alpha*A_local) @ x_slab ; target[:, c0:c0+w] += beta * that  (w = x_slab width;
        c0 a multiple of 4 floats so that every pointer stays 16-byte aligned)."""
        w = x_slab.shape[1]
        plan = A_local.spmm_plan()
        off = 4 * int(c0)
        self._lib.call("gdr_spmm_prop_planned", A_local.shape[0], w, self.ptr(A_local.rowptr), self.ptr(A_local.colidx),
                       self.ptr(A_local.vals), float(alpha), self.ptr(x_slab), x_slab.stride(0), self.ptr(y) + off,
                       y.stride(0), None if target is None else self.ptr(target) + off,
                       0 if target is None else target.stride(0), float(beta), self.ptr(plan), plan.numel() - 1,
                       self.stream())

    def prep_rows(self, x):
        return self.padded_rows(x.to(torch.float32))

    # -- stage 2, fused: the SpMM epilogue stores every output row straight into the peers' gathered operand --
    def p2p_layout(self, comm, part, f):
        ld = self._pad4(f)
        mat = (part.world * part.rows_per * ld * 4 + 255) // 256 * 256
        handle, base = comm.symm(2 * mat)
        return handle, base, ld, mat

    def p2p_distribute(self, comm, part, x):
        """Hop 0 of the fused propagation: this rank's rows of X into region 0 of every rank's symmetric buffer (one read,
        world posted NVLink stores per 16 bytes), then the barrier.  Enqueued on the CURRENT stream."""
        handle, base, ld, mat = self.p2p_layout(comm, part, x.shape[1])
        if x.stride(0) != ld:
            raise ValueError("p2p_distribute: rows must be padded to a multiple of 4 floats")
        self._lib.call("gdr_symm_barrier", handle, self.stream())      # nobody still reads region 0 of an earlier call
        self._lib.call("gdr_symm_put_rows", handle, int(part.rank * part.rows_per) * ld * 4,
                       self.ptr(x), x.shape[0], ld, 1, self.stream())
        self._lib.call("gdr_symm_barrier", handle, self.stream())

    def propagate_p2p(self, comm, part, A_local, x, target, T, alpha, one_minus, distributed=False):
        """Hops 1 .. T-1 with the all-gather fused into the SpMM epilogue (gdr_spmm_prop_mc): hop t reads the gathered
        matrix of region (t-1) & 1 and its rows land in region t & 1 of EVERY rank; one stream-ordered barrier per hop,
        no collective, no staging copy.  The last hop is a plain SpMM.  Returns the last hop's local rows."""
        handle, base, ld, mat = self.p2p_layout(comm, part, x.shape[1])
        n_local, f = x.shape
        if not distributed:
            self.p2p_distribute(comm, part, x)
        plan = A_local.spmm_plan()
        y = self.new_padded(n_local, f, x.device)
        for t in range(1, T):
            src = base + ((t - 1) & 1) * mat
            if t == T - 1:
                self._lib.call("gdr_spmm_prop_planned", n_local, f, self.ptr(A_local.rowptr), self.ptr(A_local.colidx),
                               self.ptr(A_local.vals), float(alpha), src, ld, self.ptr(y), y.stride(0), self.ptr(target),
                               target.stride(0), float(one_minus), self.ptr(plan), plan.numel() - 1, self.stream())
            else:
                self._lib.call("gdr_spmm_prop_mc", handle, (t & 1) * mat, ld, int(part.rank * part.rows_per), n_local, f,
                               self.ptr(A_local.rowptr), self.ptr(A_local.colidx), self.ptr(A_local.vals), float(alpha), src, ld,
                               0, 0, self.ptr(target), target.stride(0), float(one_minus), self.ptr(plan), plan.numel() - 1,
                               self.stream())
                self._lib.call("gdr_symm_barrier", handle, self.stream())
        return y

    # -- stage 3 --
    def column_sums(self, X):
        N, D = X.shape
        out = torch.zeros(2 * D, dtype=torch.float64, device=X.device)
        ws = self.workspace(self._lib.query("gdr_center_columns_ws_bytes", max(N, 1), D), X.device)
        self._lib.call("gdr_column_sums", N, D, self.ptr(X), X.stride(0), self.ptr(out), self.ptr(ws), ws.numel(), self.stream())
        return out

    def center(self, X, mean):
        N, D = X.shape
        Xc = self.new_padded(N, D, X.device)
        self._lib.call("gdr_center_apply", N, D, self.ptr(X), X.stride(0), self.ptr(mean), self.ptr(Xc), Xc.stride(0), self.stream())
        return Xc

    def prepare_kmeans(self, Xc, K):
        D = Xc.shape[1]
        use_tc = self.precision == "tc" or (self.precision == "auto" and D <= 128)
        self._tc = self._km.TcOperand(Xc) if (use_tc and Xc.shape[0] > 0) else None

    def centers_like(self, C, device):
        out = self.new_padded(C.shape[0], C.shape[1], device, zero=True)
        out.copy_(C)
        return out

    def assign(self, Xc, C, labels, labels_prev, n_changed):
        if Xc.shape[0] == 0:
            return
        self._km.assign_labels(Xc, C, labels, labels_prev=labels_prev, n_changed=n_changed, tc_operand=self._tc)

    def segment_sum(self, Xc, labels, K, sums, counts):
        if Xc.shape[0] == 0:
            sums.zero_()
            counts.zero_()
            return
        self._km.segment_sum(Xc, labels, K, sums=sums, counts=counts)

    def finalize(self, sums, counts, C_old, C_new):
        K, D = C_old.shape
        stats = torch.zeros(2 + K, dtype=torch.float64, device=C_old.device)
        self._lib.call("gdr_kmeans_finalize", K, D, self.ptr(sums), sums.stride(0), self.ptr(counts), self.ptr(C_old),
                       C_old.stride(0), self.ptr(C_new), C_new.stride(0), self.ptr(stats), 0, self.stream())
        s = stats[:2].cpu()
        return float(s[0]), int(s[1])

    def lloyd_native(self, comm, Xc, n_total, C0c, max_iter, tol_abs, verbose=False):
        """The whole Lloyd loop inside libgdr_b200 (gdr_kmeans_lloyd_dist): graph-replayed iterations with the packed
        all-reduce inside, one 24-byte status read-back per iteration.  Returns (labels, inertia, centres, n_iter)."""
        import ctypes
        n_local, D = Xc.shape
        K = C0c.shape[0]
        dev = C0c.device
        mode = 1 if (self.precision == "tc" or (self.precision == "auto" and D <= 128)) else 0
        centers = self.new_padded(K, D, dev, zero=True)
        centers.copy_(C0c)
        labels = torch.empty(max(n_local, 1), dtype=torch.int32, device=dev)[:n_local]
        ws = self.workspace(self._lib.query("gdr_kmeans_lloyd_ws_bytes", n_local, K, D, mode), dev)
        inertia, n_iter, info = ctypes.c_double(0.0), ctypes.c_int32(0), (ctypes.c_int32 * 2)()
        self._lib.call("gdr_kmeans_lloyd_dist", comm.lib_handle(), n_local, int(n_total), K, D,
                       self.ptr(Xc) if n_local else 0, Xc.stride(0) if n_local else self._pad4(D), self.ptr(centers),
                       centers.stride(0), self.ptr(labels) if n_local else 0, int(max_iter), float(tol_abs), mode,
                       ctypes.addressof(inertia), ctypes.addressof(n_iter), ctypes.addressof(info), int(bool(verbose)),
                       self.ptr(ws), ws.numel(), self.stream())
        self.last_info = (bool(info[0]), int(info[1]))
        return labels, float(inertia.value), centers, int(n_iter.value)

    def kmeans_plusplus_dist(self, comm, Xc, n_clusters, first, rand, n_trials):
        """k-means++ seeding of the row-partitioned Xc (gdr_kmeans_plusplus_dist; collective).  Returns the replicated
        centres [K, D] (padded rows) and their global row ids."""
        n_local, D = Xc.shape
        K = int(n_clusters)
        dev = Xc.device
        centers = self.new_padded(K, D, dev, zero=True)
        indices = torch.empty(K, dtype=torch.int64, device=dev)
        ws = self.workspace(self._lib.query("gdr_kmeans_plusplus_dist_ws_bytes", n_local, K, D, n_trials, comm.world), dev)
        self._lib.call("gdr_kmeans_plusplus_dist", comm.lib_handle(), n_local, K, D, self.ptr(Xc) if n_local else 0,
                       Xc.stride(0) if n_local else self._pad4(D), int(first), rand.ctypes.data, int(n_trials),
                       self.ptr(centers), centers.stride(0), self.ptr(indices), self.ptr(ws), ws.numel(), self.stream())
        return centers, indices

    @staticmethod
    def _pad4(d):
        return (int(d) + 3) // 4 * 4

    # -- truncated SVD (distill_recsys) --
    def gram_dist(self, comm, n_global, row_lo, A, B):
        """AᵀB of the row-partitioned fp64 A [n_local, p], B [n_local, r] (global rows row_lo .. row_lo + n_local of
        n_global), replicated with gdr_dense_gram's bits on the concatenated rows (gdr_dense_gram_dist; collective)."""
        n_local, p = A.shape
        r = B.shape[1]
        C = torch.empty((p, r), dtype=torch.float64, device=A.device)
        ws = self.workspace(self._lib.query("gdr_dense_gram_dist_ws_bytes", int(n_global), p, r, comm.world), A.device)
        self._lib.call("gdr_dense_gram_dist", comm.lib_handle(), int(n_global), int(row_lo), n_local, p, r,
                       self.ptr(A) if n_local else 0, A.stride(0) if n_local else p, self.ptr(B) if n_local else 0,
                       B.stride(0) if n_local else r, self.ptr(C), r, self.ptr(ws), ws.numel(), self.stream())
        return C

    def segment_sum_dist(self, comm, row_lo, X, labels, K):
        """segment_sum of the row-partitioned X (global rows row_lo .. row_lo + n_local) and int32 labels, replicated
        with gdr_segment_sum's bits on the concatenated rows (gdr_segment_sum_dist; collective).  Returns (sums [K, D]
        padded, counts int32 [K]).  A row count that differs between X and labels, or K <= 0, is this rank's rejection
        inside the collective entry check, so every rank fails together."""
        n_local, D = X.shape
        dev = X.device
        ok = labels.shape == (n_local,) and K > 0
        Kb = max(int(K), 1)
        sums = self.new_padded(Kb, D, dev, zero=True)
        counts = torch.zeros(Kb, dtype=torch.int32, device=dev)
        ws = self.workspace(self._lib.query("gdr_segment_sum_dist_ws_bytes", n_local, Kb, D), dev)
        self._lib.call("gdr_segment_sum_dist", comm.lib_handle(), int(row_lo), n_local, int(K), D,
                       self.ptr(X) if n_local else 0, X.stride(0) if n_local else sums.stride(0),
                       self.ptr(labels) if n_local and ok else 0, self.ptr(sums), sums.stride(0), self.ptr(counts),
                       self.ptr(ws), ws.numel(), self.stream())
        return sums, counts

    def minibatch_batch(self, comm, idx, row_off, X, C, Xb, labels_b):
        """Rows ``idx`` (numpy int64, the same on every rank) of the row-partitioned X into Xb on every rank, with their
        exact-fp32 labels against C when C is given (gdr_minibatch_batch_dist; a per-step collective)."""
        import ctypes
        m = int(idx.shape[0])
        n_local, D = X.shape
        K = int(C.shape[0]) if C is not None else 0
        dev = Xb.device
        order, counts = batch_plan(idx, row_off)
        idx_d = torch.from_numpy(idx).to(dev, non_blocking=True)
        order_d = torch.from_numpy(order).to(dev, non_blocking=True)
        key = (m, K, D)
        if getattr(self, "_mb_ws", (None,))[0] != key:
            self._mb_ws = (key, self.workspace(self._lib.query("gdr_minibatch_batch_dist_ws_bytes", m, K, D, comm.world), dev))
        ws = self._mb_ws[1]
        cnt = (ctypes.c_int64 * comm.world)(*[int(c) for c in counts])
        self._lib.call("gdr_minibatch_batch_dist", comm.lib_handle(), m, self.ptr(idx_d), self.ptr(order_d),
                       ctypes.addressof(cnt), int(row_off[comm.rank]), n_local, K, D, self.ptr(X) if n_local else 0,
                       X.stride(0) if n_local else self._pad4(D), self.ptr(C), C.stride(0) if C is not None else 0,
                       self.ptr(Xb), Xb.stride(0), self.ptr(labels_b) if C is not None else 0, self.ptr(ws), ws.numel(),
                       self.stream())
        return Xb

    def inertia(self, Xc, C, labels):
        out = torch.zeros(1, dtype=torch.float64, device=C.device)
        if Xc.shape[0] == 0:
            return out
        ws = self.workspace(self._lib.query("gdr_inertia_ws_bytes", Xc.shape[0], Xc.shape[1]), Xc.device)
        self._lib.call("gdr_inertia", Xc.shape[0], Xc.shape[1], self.ptr(Xc), Xc.stride(0), self.ptr(C), C.stride(0),
                       self.ptr(labels), self.ptr(out), self.ptr(ws), ws.numel(), self.stream())
        return out

    def row_dist(self, Xc, C, labels):
        return ((Xc - C[labels.long()]) ** 2).sum(dim=1)  # rare relocation path only

    # -- edge sparsification (between stages 3 and 4) --
    def er_lower_rows(self, A, deg, row_lo):
        """v/deg[row_lo + r] + v/deg[c] for the local block A with the global degree vector (gdr_er_lower_rows)."""
        er = torch.empty(max(A.nnz, 1), dtype=torch.float32, device=A.device)
        self._lib.call("gdr_er_lower_rows", A.shape[0], A.nnz, int(row_lo), self.ptr(A.rowptr), self.ptr(A.colidx),
                       self.ptr(A.vals), self.ptr(deg), self.ptr(er), self.stream())
        return er[: A.nnz]

    def cosine_reweight_rows(self, A, ebd, row_lo, eps=1e-8):
        """vals * cos(ebd[row_lo + r], ebd[c]) for the local block A, ``ebd`` global (gdr_edge_cosine_scale_rows)."""
        inv = torch.empty(ebd.shape[0], dtype=torch.float32, device=A.device)
        out = torch.empty(max(A.nnz, 1), dtype=torch.float32, device=A.device)
        self._lib.call("gdr_edge_cosine_scale_rows", A.shape[0], A.nnz, ebd.shape[1], int(row_lo), ebd.shape[0],
                       self.ptr(A.rowptr), self.ptr(A.colidx), self.ptr(A.vals), self.ptr(ebd), ebd.stride(0), float(eps),
                       self.ptr(inv), self.ptr(out), self.stream())
        return self._g.CSR(A.rowptr, A.colidx, out[: A.nnz], A.shape)

    def softmax_rows(self, x):
        from .sparsify import softmax_rows
        return softmax_rows(x)

    def sparsify_classes_dist(self, comm, A, row_lo, n_global, er, prob, k):
        """This rank's kept edges of every class (gdr_sparsify_classes_dist; collective).  ``A`` None: a rank without
        rows, which still joins.  ``prob`` None: one graph, weights ``er``.  Returns one local CSR per class (None for a
        rank without rows)."""
        C = 1 if prob is None else int(prob.shape[1])
        dev = er.device
        n_local, nnz = (0, 0) if A is None else (A.shape[0], A.nnz)
        cap = min(int(k), nnz)
        rowptr = torch.empty((C, n_local + 1), dtype=torch.int32, device=dev)
        colidx = torch.empty((C, max(cap, 1)), dtype=torch.int32, device=dev)
        vals = torch.empty((C, max(cap, 1)), dtype=torch.float32, device=dev)
        nnz_out = torch.zeros(C, dtype=torch.int64, device=dev)
        ws = self.workspace(self._lib.query("gdr_sparsify_classes_dist_ws_bytes", n_local, nnz, C, comm.world), dev)
        have = nnz > 0
        self._lib.call("gdr_sparsify_classes_dist", comm.lib_handle(), n_local, nnz, int(row_lo), int(n_global), C,
                       self.ptr(A.rowptr) if n_local else 0, self.ptr(A.colidx) if have else 0,
                       self.ptr(A.vals) if have else 0, self.ptr(er) if have else 0,
                       0 if prob is None else self.ptr(prob), 0 if prob is None else prob.stride(0), int(k),
                       self.ptr(rowptr), self.ptr(colidx) if have else 0, self.ptr(vals) if have else 0, self.ptr(nnz_out),
                       self.ptr(ws), ws.numel(), self.stream())
        if A is None:
            return [None] * C
        counts = nnz_out.tolist()
        return [self._g.CSR(rowptr[c], colidx[c, : counts[c]], vals[c, : counts[c]], A.shape) for c in range(C)]

    # -- stage 4 --
    def label_counts(self, labels, n):
        return self._co.label_counts(labels, n)

    def coarsen_route(self, A_local, labels_src, labels_dst, n, world, n_dst=None, src=None, dst=None):
        """Local edges -> (cell key | owner << 56, weight) pairs grouped by the owner rank of the coarse row (one stable
        partition pass, gdr_coarsen_route).  Returns (keys int64 [E], weights f32 [E] | None, pairs per owner); pairs of
        dropped diagonal cells sit behind the last owner's and are not sent."""
        n_dst = n if n_dst is None else n_dst
        dev = labels_dst.device
        if A_local is not None:
            E, w = A_local.nnz, A_local.vals
            args = (0, 0, A_local.shape[0], self.ptr(A_local.rowptr), self.ptr(A_local.colidx))
            drop = 1
        else:
            E, w = int(src.numel()), None
            args = (self.ptr(src), self.ptr(dst), 0, 0, 0)
            drop = 0
        keys = torch.empty(max(E, 1), dtype=torch.int64, device=dev)
        w_out = torch.empty(max(E, 1), dtype=torch.float32, device=dev) if w is not None else None
        starts = torch.zeros(129, dtype=torch.int64, device=dev)
        ws = self.workspace(self._lib.query("gdr_coarsen_route_ws_bytes", E), dev)
        self._lib.call("gdr_coarsen_route", E, *args, self.ptr(w), self.ptr(labels_src), self.ptr(labels_dst), int(n), int(n_dst),
                       drop, int(world), self.ptr(keys), self.ptr(w_out), self.ptr(starts), self.ptr(ws), ws.numel(), self.stream())
        st = starts.cpu().tolist()
        return keys, w_out, [int(st[r + 1] - st[r]) for r in range(world)]

    def cluster_stats(self, A_local, labels_local, n):
        """Per coarse row, over THIS rank's rows: (edges int32 [n], bit pattern of the largest |weight| int32 [n])
        (gdr_cluster_stats).  Summed / maxed over the ranks they fix the fixed-point step of coarse_merge_edges."""
        dev = labels_local.device
        nodes = torch.empty(n, dtype=torch.int32, device=dev)
        edges = torch.empty(n, dtype=torch.int32, device=dev)
        wmax = torch.empty(n, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        self._lib.call("gdr_cluster_stats", int(A_local.shape[0]), self.ptr(A_local.rowptr), self.ptr(A_local.vals),
                       self.ptr(labels_local), int(n), self.ptr(nodes), self.ptr(edges), self.ptr(wmax), self.ptr(status),
                       self.stream())
        return edges, wmax

    def coarse_merge_edges(self, keys, w, a_lo, n_rows, n, n_dst=None, stats=None):
        """Pairs received from every rank (source-rank order = global CSR order) -> CSR (rowptr, colidx, counts, wsum) of
        the coarse rows [a_lo, a_lo + n_rows).  With ``stats`` = the global (edges, max |w| bits) per coarse row and a
        coarse row that fits in shared memory: grouped by row, cells accumulated in shared memory — the sums are those of the
        single-GPU gdr_coarsen, bit for bit (gdr_coarse_merge_edges_dense).  Otherwise: stable sort by cell, run lengths,
        fp32 sums in CSR order (gdr_coarse_merge_edges)."""
        n_dst = n if n_dst is None else n_dst
        m = int(keys.shape[0])
        dev = keys.device
        rowptr = torch.empty(n_rows + 1, dtype=torch.int32, device=dev)
        colidx = torch.empty(max(m, 1), dtype=torch.int32, device=dev)
        counts = torch.empty(max(m, 1), dtype=torch.int32, device=dev)
        wsum = torch.empty(max(m, 1), dtype=torch.float32, device=dev) if w is not None else None
        nnz = torch.zeros(1, dtype=torch.int64, device=dev)
        dense = (stats is not None or w is None) and n_rows > 0 and \
            self._lib.query("gdr_coarse_merge_edges_dense_ok", int(n_rows), int(n_dst), int(w is not None))
        if dense:
            ws = self.workspace(self._lib.query("gdr_coarse_merge_edges_dense_ws_bytes", m, int(n_rows)), dev)
            self._lib.call("gdr_coarse_merge_edges_dense", m, self.ptr(keys) if m else 0,
                           self.ptr(w) if (m and w is not None) else 0, int(a_lo), int(n_rows), int(n), int(n_dst),
                           self.ptr(stats[0]) if stats is not None else 0, self.ptr(stats[1]) if stats is not None else 0,
                           self.ptr(rowptr), self.ptr(colidx), self.ptr(counts), self.ptr(wsum), self.ptr(nnz), self.ptr(ws),
                           ws.numel(), self.stream())
        else:
            ws = self.workspace(self._lib.query("gdr_coarse_merge_edges_ws_bytes", m), dev)
            self._lib.call("gdr_coarse_merge_edges", m, self.ptr(keys) if m else 0, self.ptr(w) if (m and w is not None) else 0,
                           int(a_lo), int(n_rows), int(n), int(n_dst), self.ptr(rowptr), self.ptr(colidx), self.ptr(counts),
                           self.ptr(wsum), self.ptr(nnz), self.ptr(ws), ws.numel(), self.stream())
        k = int(nnz.item())
        return rowptr, colidx[:k], counts[:k], (None if wsum is None else wsum[:k])

    def coarsen_records(self, A_local, labels_src, labels_dst, n, world, n_dst=None, src=None, dst=None):
        """Local edges -> sorted (cell, count, weight sum) records [m, 2] int64 (gdr_coarsen + gdr_coarse_records) and the
        number of records per owner rank of the key-range partition (coarse row a belongs to rank a // ceil(n / world)).
        Edges: the CSR ``A_local`` (graph_compress: weights summed, diagonal dropped) or the COO lines ``src`` / ``dst``
        (build_condensed_bipartite: plain line counts)."""
        n_dst = n if n_dst is None else n_dst
        if A_local is not None:
            rowptr, colidx, counts, wsum = self._co.coarsen_edges(labels_src, labels_dst, n, n_dst, csr=A_local,
                                                                  weights=A_local.vals, drop_diag=True)
        else:
            rowptr, colidx, counts, wsum = self._co.coarsen_edges(labels_src, labels_dst, n, n_dst, src=src, dst=dst)
        m = int(colidx.numel())
        rec = torch.empty((m, 2), dtype=torch.int64, device=labels_dst.device)
        if m:
            self._lib.call("gdr_coarse_records", n, n_dst, self.ptr(rowptr), self.ptr(colidx), self.ptr(counts), self.ptr(wsum),
                           self.ptr(rec), self.stream())
        cr = (n + world - 1) // world
        bounds = torch.tensor([min(n, r * cr) for r in range(world + 1)], dtype=torch.int64, device=rowptr.device)
        cuts = rowptr[bounds].cpu().tolist()
        return rec, [int(cuts[r + 1] - cuts[r]) for r in range(world)]

    def coarse_merge(self, rec, a_lo, n_rows, n, n_dst=None):
        """Records received from every rank -> CSR (rowptr, colidx, counts, wsum) of the coarse rows [a_lo, a_lo + n_rows)."""
        n_dst = n if n_dst is None else n_dst
        m = int(rec.shape[0])
        dev = rec.device
        rowptr = torch.empty(n_rows + 1, dtype=torch.int32, device=dev)
        colidx = torch.empty(max(m, 1), dtype=torch.int32, device=dev)
        counts = torch.empty(max(m, 1), dtype=torch.int32, device=dev)
        wsum = torch.empty(max(m, 1), dtype=torch.float32, device=dev)
        nnz = torch.zeros(1, dtype=torch.int64, device=dev)
        ws = self.workspace(self._lib.query("gdr_coarse_merge_ws_bytes", m), dev)
        self._lib.call("gdr_coarse_merge", m, self.ptr(rec) if m else 0, int(a_lo), int(n_rows), n, n_dst, self.ptr(rowptr),
                       self.ptr(colidx), self.ptr(counts), self.ptr(wsum), self.ptr(nnz), self.ptr(ws), ws.numel(), self.stream())
        k = int(nnz.item())
        return rowptr, colidx[:k], counts[:k], wsum[:k]

    def coarse_scale(self, rowptr, colidx, wsum, sizes, a_lo, n_rows):
        vals = torch.empty_like(wsum)
        if n_rows > 0 and wsum.numel():
            self._lib.call("gdr_coarsen_scale", n_rows, self.ptr(rowptr), self.ptr(colidx), self.ptr(wsum),
                           self.ptr(sizes[a_lo:]), self.ptr(sizes), self.ptr(vals), self.stream())
        return vals

    def csr_to_coo(self, rowptr, colidx, vals, n):
        return self._g.CSR(rowptr, colidx, vals, (n, n)).to_torch_coo()


# ------------------------------------------------------------------------------------------
# stage 1 (replicated build, local row slice)
# ------------------------------------------------------------------------------------------
def slice_rows(A, lo: int, hi: int):
    """Rows [lo, hi) of a device CSR as a CSR with global column ids (views, no copy of colidx/vals)."""
    from .graph import CSR
    b, e = int(A.rowptr[lo].item()), int(A.rowptr[hi].item())
    rowptr = (A.rowptr[lo: hi + 1] - A.rowptr[lo]).contiguous()
    return CSR(rowptr, A.colidx[b:e], A.vals[b:e], (hi - lo, A.shape[1]))


def build_local_adjacency(u, v, n: int, part: RowPartition, device):
    """Round-1 form of the distributed stage 1: the (small, one-off) CSR build + normalisation
    is replicated on every rank and each rank keeps its row block.  The exchange-based build
    (edges bucketed by owner, all-to-all of reversed edges, all-gather of degrees) is the
    listed next step (DESIGN.md §6)."""
    from .graph import coo_to_csr, sym_normalize
    A = sym_normalize(coo_to_csr(u, v, None, (n, n), symmetrize=True, binarize=True, device=device), 2)
    return slice_rows(A, part.lo, part.hi), A


def dist_build_adjacency(comm: Comm, part: RowPartition, u_slice: torch.Tensor, v_slice: torch.Tensor, n: int, ops=None,
                         self_loop_mode: int = 2, after_exchange=None):
    """Stage 1 on a row partition (SURVEY §8e): every rank holds a SLICE of the undirected pair list
    (utils_graphsaint.py:18-22 symmetrises it: adj + adj.T, values clipped to 1).  Each rank emits both
    directions of its pairs, buckets them by the owner of the source row, exchanges the buckets
    (all-to-all), builds the binarised CSR of its own rows, and — after an all-gather of the degree
    vector — normalises them (deep_robust_utils.py:180-207).  Returns the local rows of A_hat with global
    column ids; the block is bit-identical to the same rows of the single-device build.
    ``after_exchange``: called once the all-to-all of the keys has been enqueued — the place to start work that wants
    the NVLink fabric for itself (``prefetch_rows``) while the local sort / CSR emit runs."""
    ops = ops or CudaOps()
    sizes = [part.bounds(r)[1] - part.bounds(r)[0] for r in range(part.world)]
    if hasattr(ops, "edges_route"):
        # routing form: pack + one partition pass in the library, 8-byte keys over the wire, keys-only sort at the owner
        keys, counts, status = ops.edges_route(u_slice.to(torch.int64).contiguous(), v_slice.to(torch.int64).contiguous(), n, n,
                                               part.rows_per, part.world, True)
        if status & 1:
            raise ValueError("row/col index exceeds matrix dimensions")
        if self_loop_mode == 2:    # reference rule `if mx[0, 0] == 0: mx = mx + I`: a global decision
            has00 = torch.tensor([1 if status & 2 else 0], dtype=torch.int64, device=u_slice.device)
            add_identity = int(comm.all_reduce(has00, "max").item()) == 0
        else:
            add_identity = bool(self_loop_mode)
        if comm.symm_ok() and keys.is_cuda:
            # posted NVLink stores into the owners' symmetric buffers; copied out because the prefetch of X reuses the buffer
            recv = comm.symm_exchange([keys], comm.count_matrix(counts, keys.device))[0].clone()
        else:
            recv, _ = comm.all_to_all_rows(keys, counts)
        if after_exchange is not None:
            after_exchange()
        if part.n_local == 0:   # a rank past the end of a short matrix still joins the collectives
            comm.all_gather_var(torch.zeros(0, dtype=torch.float64, device=u_slice.device), sizes)
            return None
        A_blk = ops.csr_from_keys(recv, part.lo, part.n_local, n, True)
    else:
        src = torch.cat([u_slice, v_slice]).to(torch.int64)
        dst = torch.cat([v_slice, u_slice]).to(torch.int64)
        if src.numel() and (int(src.min()) < 0 or int(src.max()) >= n):
            raise ValueError("row/col index exceeds matrix dimensions")
        # reference rule `if mx[0, 0] == 0: mx = mx + I`: a global decision
        if self_loop_mode == 2:
            has00 = ((src == 0) & (dst == 0)).any().to(torch.int64).reshape(1)
            add_identity = int(comm.all_reduce(has00, "max").item()) == 0
        else:
            add_identity = bool(self_loop_mode)
        edges, counts = ops.bucket_by_owner(src, dst, part.rows_per, part.world)
        recv, _ = comm.all_to_all_rows(edges, counts)
        if part.n_local == 0:   # a rank past the end of a short matrix still joins the collectives
            comm.all_gather_var(torch.zeros(0, dtype=torch.float64, device=src.device), sizes)
            return None
        A_blk = ops.build_block_csr(recv[:, 0] - part.lo, recv[:, 1], part.n_local, n)
    deg_local, rowptr_out = ops.block_degrees(A_blk, part.lo, add_identity)
    deg = comm.all_gather_var(deg_local, sizes)
    return ops.block_fill(A_blk, part.lo, add_identity, deg, rowptr_out)


# ------------------------------------------------------------------------------------------
# stage 2
# ------------------------------------------------------------------------------------------
def slab_bounds(f: int, slabs: int):
    """Column slabs [c0, c1) of an f-wide matrix, every start a multiple of 4 floats."""
    f4 = (f + 3) // 4
    slabs = max(1, min(int(slabs), f4))
    per = (f4 + slabs - 1) // slabs
    out = []
    for s in range(slabs):
        c0, c1 = 4 * s * per, min(f, 4 * (s + 1) * per)
        if c0 < c1:
            out.append((c0, c1))
    return out


def default_slabs(world: int, f: int) -> int:
    """Pipeline depth of a hop.  Measured on B200 at config E (F = 100): 2 GPUs 19.1 ms (1 slab) vs 24.2 ms
    (3 slabs), 8 GPUs 8.7 ms vs 9.1 ms (2 slabs) — the narrower gathers of a slab cost the SpMM more than the
    hidden all-gather returns, so the default is the one-pass hop; ``slabs`` stays available per call."""
    return 1


def default_row_chunks(world: int) -> int:
    """Row chunks of the pipelined hop: the all-gather of chunk c overlaps the SpMM of chunks c+1.. (rows are
    independent, so nothing changes numerically and the SpMM keeps its full-width gathers).  Measured at config E:
    8 GPUs 8.49 ms (one pass) -> 7.94 ms (4 chunks); 4 GPUs 11.97 -> 11.75 ms; 2 GPUs 19.1 -> 20.8 ms (the all-gather is only 0.8 ms of a
    6.3 ms hop there and the extra launches / concurrent NCCL traffic cost more), hence 4 chunks from 4 ranks up."""
    return 4 if world >= 4 else 1


def describe(world: int, row_chunks: Optional[int] = None, hop: str = "auto") -> str:
    """One-line description of the exchanges, for bench.py's config.parallelism."""
    rc = default_row_chunks(world) if row_chunks is None else int(row_chunks)
    s2 = (f"stage 2: NCCL all-gather of the propagated rows per hop, pipelined over {rc} row chunk(s); " if hop == "nccl" or _P2P_BROKEN
          else "stage 2: hop fused with its all-gather (SpMM epilogue stores every row into all peers' gathered operand over "
               "NVLink, one stream-ordered barrier per hop; first distribution of X started under stage 1); ")
    xch = "all-to-all over NCCL" if _P2P_BROKEN else "posted NVLink stores into the owners' symmetric buffers"
    return (f"stage 1: pair slices routed to the owner of the row ({xch}), all-gather of degrees; " + s2 +
            "stage 3: one grouped all-reduce [sums | counts | n_changed] per Lloyd iteration inside the replayed CUDA graph; "
            f"stage 4: (cell, weight) pairs routed to the owner of the coarse row ({xch}), merged there in shared memory, result "
            "replicated on every rank")


_P2P_BROKEN = False      # set when peer memory turned out to be unavailable: the NCCL hop is used from then on


class PrefetchedRows:
    """Hop 0 of the fused propagation issued ahead of time (``prefetch_rows``): the feature rows are on their way into
    every rank's gathered operand while the caller does something else (stage 1) on the main stream."""

    def __init__(self, x, event):
        self.x, self.event = x, event


def prefetch_rows(comm: Comm, part: RowPartition, x_local: torch.Tensor, ops=None) -> Optional[PrefetchedRows]:
    """Starts distributing this rank's feature rows to all ranks on a side stream.  Hand the result to
    ``dist_propagate(prefetched=...)``.  Returns None when the fused hop is not available (the call is then a no-op)."""
    global _P2P_BROKEN
    ops = ops or CudaOps()
    if _P2P_BROKEN or comm.world == 1 or comm.backend != "nccl" or not hasattr(ops, "propagate_p2p"):
        return None
    x = ops.prep_rows(x_local)
    try:
        ops.p2p_layout(comm, part, x.shape[1])
    except Exception:
        _P2P_BROKEN = True
        return None
    side = getattr(comm, "_side_stream", None)
    if side is None:
        side = comm._side_stream = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.p2p_distribute(comm, part, x)
        ev = torch.cuda.Event()
        ev.record(side)
    x.record_stream(side)
    return PrefetchedRows(x, ev)


def dist_propagate(comm: Comm, part: RowPartition, A_local, x_local: torch.Tensor, prop_num: int, alpha: float,
                   ops=None, slabs: Optional[int] = None, row_chunks: Optional[int] = None, hop: str = "auto",
                   prefetched: Optional[PrefetchedRows] = None):
    """clustgdd_agent_transduct.py:59-65 on row-partitioned data.  Returns the local row blocks
    (prop_local, target_local).

    Each hop all-gathers the propagated rows and multiplies.  With ``slabs`` > 1 the feature
    columns are cut into slabs: all slab all-gathers are enqueued at once (asynchronously, in
    order) and the SpMM of slab s starts as soon as ITS gather has landed, so the transfer of
    the later slabs overlaps the arithmetic of the earlier ones.  Every output element of a row
    on the kernel's sequential path (<= 1024 non-zeros) is the same fp32 chain as in the one-pass
    hop, i.e. bit-identical; hub rows are summed as fixed-order partials whose grouping follows
    the slab width (deterministic, inside the 1e-5 contract)."""
    ops = ops or CudaOps()
    T = int(prop_num)
    if T < 1:
        raise ValueError("prop_num must be >= 1")
    global _P2P_BROKEN
    x = prefetched.x if prefetched is not None else ops.prep_rows(x_local)
    f = x.shape[1]
    one_minus = float(1.0 - alpha)
    target = ops.scale(x, one_minus)
    prop = x
    rows_per = part.rows_per
    # fused hop (default on NVLink): every hop's rows are stored by the SpMM epilogue straight into the gathered operand of
    # the next hop on every rank (peer memory); falls back to the NCCL all-gather hop when peer memory is unavailable
    want_p2p = hop in ("auto", "p2p") and slabs in (None, 1) and row_chunks in (None, 1) and T > 1 and part.world > 1 \
        and comm.backend == "nccl" and hasattr(ops, "propagate_p2p") and not _P2P_BROKEN
    if want_p2p:
        try:
            if prefetched is not None:
                torch.cuda.current_stream().wait_event(prefetched.event)
            return ops.propagate_p2p(comm, part, A_local, x, target, T, alpha, one_minus,
                                     distributed=prefetched is not None), target
        except Exception as e:       # GdrError from gdr_symm_create: no peer access between these GPUs
            if hop == "p2p" or prefetched is not None:
                raise
            import warnings
            warnings.warn(f"fused NVLink hop unavailable ({e}); using the NCCL all-gather hop")
            _P2P_BROKEN = True
    n_slabs = default_slabs(part.world, f) if slabs is None else int(slabs)
    n_chunks = default_row_chunks(part.world) if row_chunks is None else int(row_chunks)
    if n_slabs <= 1 and n_chunks > 1 and T > 2 and hasattr(ops, "spmm_rows"):
        return _propagate_row_chunks(comm, part, A_local, x, target, T, alpha, one_minus, ops, n_chunks)
    if n_slabs <= 1 or not hasattr(ops, "spmm_slab"):
        x_full = ops.empty_rows(rows_per * part.world, f, x)
        block = ops.empty_rows(rows_per, f, x)
        for _ in range(1, T):
            block[: prop.shape[0]].copy_(prop)
            comm.all_gather_rows(block, x_full)
            prop = ops.spmm(A_local, x_full, alpha, target, one_minus)
        return prop, target
    bounds = slab_bounds(f, n_slabs)
    send = [ops.empty_rows(rows_per, c1 - c0, x) for c0, c1 in bounds]
    full = [ops.empty_rows(rows_per * part.world, c1 - c0, x) for c0, c1 in bounds]
    bufs = [ops.empty_rows(prop.shape[0], f, x) for _ in range(2)]   # hop outputs, ping-pong
    for t in range(1, T):
        works = []
        for (c0, c1), sb, fb in zip(bounds, send, full):
            sb[: prop.shape[0], : c1 - c0].copy_(prop[:, c0:c1])
            works.append(comm.all_gather_rows(sb, fb, async_op=True))
        y = bufs[t & 1]
        for (c0, c1), fb, w in zip(bounds, full, works):
            w.wait()
            ops.spmm_slab(A_local, fb, alpha, y, target, one_minus, c0)
        prop = y
    return prop, target


def _propagate_row_chunks(comm, part, A_local, x, target, T, alpha, one_minus, ops, n_chunks):
    """Hops pipelined over ROW chunks of the local block.  As soon as the SpMM of chunk c has produced its rows of
    hop t, their all-gather (the input of hop t+1) starts on the collective's stream while the SpMM of chunk c+1
    runs.  The gathered matrix is kept CHUNK-MAJOR — row of node (rank r, local row i = c*cr + o) is
    c*world*cr + r*cr + o — so that every chunk's all-gather lands in one contiguous slab with no staging copy; the
    column indices of the local CSR are remapped to that layout once.  Rows are independent of each other, so the
    values are exactly those of the one-pass hop."""
    world, rows_per, n_local, f = part.world, part.rows_per, x.shape[0], x.shape[1]
    cr = (rows_per + n_chunks - 1) // n_chunks                      # chunk height, the same on every rank
    n_chunks = (rows_per + cr - 1) // cr
    A_perm = ops.remap_chunk_major(A_local, rows_per, cr, world)    # column ids -> rows of the chunk-major matrix
    bounds = [min(k * cr, n_local) for k in range(n_chunks + 1)]
    chunks = ops.slice_row_chunks(A_perm, bounds)
    full = [ops.empty_rows(n_chunks * world * cr, f, x) for _ in range(2)]
    ys = [ops.empty_rows(n_chunks * cr, f, x) for _ in range(2)]    # local rows padded to whole chunks
    ys[0][:n_local].copy_(x)
    for k in range(n_chunks):                                        # hop 1: nothing to overlap with yet
        comm.all_gather_rows(ys[0][k * cr:(k + 1) * cr], full[0][k * world * cr:(k + 1) * world * cr])
    for t in range(1, T):
        src, dst, y = full[(t - 1) & 1], full[t & 1], ys[t & 1]
        works = []
        for k, A_c in enumerate(chunks):
            ops.spmm_rows(A_c, src, alpha, y, target, one_minus, bounds[k])
            if t < T - 1:                                              # the last hop's output is not gathered
                works.append(comm.all_gather_rows(y[k * cr:(k + 1) * cr], dst[k * world * cr:(k + 1) * world * cr],
                                                  async_op=True))
        for w in works:
            w.wait()
    return ys[(T - 1) & 1][:n_local], target


# ------------------------------------------------------------------------------------------
# stage 3
# ------------------------------------------------------------------------------------------
def dist_kmeans_plusplus(comm: Comm, part: RowPartition, Xc_local: torch.Tensor, n_clusters: int, random_state,
                         ops=None, return_indices: bool = False):
    """k-means++ seeding (sklearn's ``_kmeans_plusplus``) of the row-partitioned ``Xc_local`` without gathering X.
    Collective.  ``part.n`` is the global row count; the ranks' blocks in rank order are the global rows.  The host
    draws are ``kmeans_init.kmeans_plusplus_device``'s (one ``choice``, then ``uniform(size=n_local_trials)`` per
    round), so every rank must pass the same ``random_state``; a mismatch raises GdrError on every rank.  With one rank
    the result is bit-identical to ``kmeans_plusplus_device``; with more, only the fp64 potentials are grouped by rank.
    Returns the replicated centres [K, D] (and their global row ids with ``return_indices``)."""
    from .kmeans_init import draw_plusplus
    ops = ops or CudaOps()
    if not hasattr(ops, "kmeans_plusplus_dist"):
        raise NotImplementedError(f"{type(ops).__name__} has no distributed k-means++ seeding")
    first, rand, n_trials = draw_plusplus(random_state, int(part.n), int(n_clusters))
    centers, indices = ops.kmeans_plusplus_dist(comm, Xc_local, n_clusters, first, rand, n_trials)
    return (centers, indices) if return_indices else centers


class DistKMeans:
    """Lloyd k-means on row-partitioned X with replicated centres.  ``init`` is an array identical on every rank,
    "k-means++" (greedy D^2 seeding of the centred rows, ``dist_kmeans_plusplus``) or "random" (the centred rows
    ``RandomState(random_state).permutation(N)[:K]``, copied from their owners).  A string init needs the same
    ``random_state`` (seed or RandomState) on every rank; one init per fit."""

    def __init__(self, n_clusters: int, init, max_iter: int = 300, tol: float = 1e-4, ops=None, comm: Comm = None,
                 verbose: bool = False, python_loop: bool = False, random_state=None):
        self.n_clusters, self.init, self.max_iter, self.tol = int(n_clusters), init, int(max_iter), tol
        self.random_state = random_state
        self.ops = ops or CudaOps()
        self.comm = comm or Comm()
        self.verbose = verbose
        self.python_loop = python_loop   # force the host-driven loop (any backend / injected ops); default: in-library loop

    def fit(self, X_local: torch.Tensor):
        ops, comm, K = self.ops, self.comm, self.n_clusters
        if isinstance(self.init, str):
            if self.init not in ("k-means++", "random"):
                raise ValueError(f"init should be 'k-means++', 'random' or an array, got {self.init!r}")
            if self.random_state is None:
                raise ValueError("a string init needs the same random_state on every rank")
            if not hasattr(ops, "kmeans_plusplus_dist"):
                raise NotImplementedError(f"{type(ops).__name__} has no distributed init {self.init!r}")
        X = ops.prep_rows(X_local)
        n_local, D = X.shape
        dev = X.device
        cnt = torch.tensor([n_local], dtype=torch.int64, device=dev)
        comm.all_reduce(cnt)
        N = int(cnt.item())
        if N < K:
            raise ValueError(f"n_samples={N} should be >= n_clusters={K}.")
        sums = ops.column_sums(X)
        comm.all_reduce(sums)
        m64 = sums[:D] / N
        var_mean = float(((sums[D:] / N - m64 * m64).clamp_min(0)).mean().item())
        mean = m64.to(torch.float32)
        tol_abs = 0.0 if self.tol == 0 else var_mean * float(self.tol)
        Xc = ops.center(X, mean)
        if isinstance(self.init, str):
            C0c = self._string_init(Xc, N)
        else:
            C0 = torch.as_tensor(np.asarray(self.init) if not isinstance(self.init, torch.Tensor) else self.init,
                                 dtype=torch.float32).to(dev)
            if tuple(C0.shape) != (K, D):
                raise ValueError("init has the wrong shape")
            C0c = ops.centers_like(C0 - mean, dev)
        if hasattr(ops, "lloyd_native") and (comm.world == 1 or comm.backend == "nccl") and not self.python_loop:
            lab, inertia, cen, n_iter = ops.lloyd_native(comm, Xc, N, C0c, self.max_iter, tol_abs, self.verbose)
            self.labels_ = lab
            self.cluster_centers_ = (cen + mean).contiguous()
            self.inertia_ = inertia
            self.n_iter_ = n_iter
            self._centers_centered, self._mean = cen, mean
            return self
        zeros = torch.zeros((K, D), dtype=torch.float32, device=dev)
        centers = [C0c, ops.centers_like(zeros, dev)]
        labels = [torch.full((n_local,), -1, dtype=torch.int32, device=dev) for _ in range(2)]
        psums = ops.centers_like(zeros, dev)
        ints = torch.zeros(K + 1, dtype=torch.int32, device=dev)   # [counts | n_changed]
        ops.prepare_kmeans(Xc, K)
        cur, nxt, ln, lo_ = 0, 1, 0, 1
        strict, n_iter = False, 0
        for i in range(self.max_iter):
            n_iter = i + 1
            ints.zero_()
            ops.assign(Xc, centers[cur], labels[ln], labels[lo_], ints[K:])
            ops.segment_sum(Xc, labels[ln], K, psums, ints[:K])
            comm.all_reduce(psums)       # K x D partial sums
            comm.all_reduce(ints)        # counts + changed-label count, exact
            shift_tot, n_empty = ops.finalize(psums, ints[:K], centers[cur], centers[nxt])
            n_changed = int(ints[K].item())
            if n_empty > 0:
                self._relocate(Xc, centers[cur], labels[ln], psums, ints[:K], part_lo=0)
                shift_tot, _ = ops.finalize(psums, ints[:K], centers[cur], centers[nxt])
            cur, nxt = nxt, cur
            if n_changed == 0:
                strict = True
                break
            if shift_tot <= tol_abs:
                break
            ln, lo_ = lo_, ln
        lab = labels[ln]
        if not strict:
            ops.assign(Xc, centers[cur], lab, None, None)
        inertia = ops.inertia(Xc, centers[cur], lab)
        comm.all_reduce(inertia)
        self.labels_ = lab
        self.cluster_centers_ = (centers[cur] + mean).contiguous()
        self.inertia_ = float(inertia.item())
        self.n_iter_ = n_iter
        self._centers_centered = centers[cur]
        self._mean = mean
        return self

    def _string_init(self, Xc, N):
        """Centred initial centres of a string init (replicated on every rank)."""
        from .kmeans import _check_random_state
        comm, ops, K = self.comm, self.ops, self.n_clusters
        rs = _check_random_state(self.random_state)
        if self.init == "k-means++":
            return dist_kmeans_plusplus(comm, RowPartition(N, comm.world, comm.rank), Xc, K, rs, ops=ops)
        # "random": every rank fills the chosen rows it owns; the owner's copy of each row is taken (never summed)
        n_local, D = Xc.shape
        dev = Xc.device
        cnt = torch.tensor([[n_local]], dtype=torch.int64, device=dev)
        counts = torch.empty((comm.world, 1), dtype=torch.int64, device=dev)
        comm.all_gather_rows(cnt, counts)
        offs = np.concatenate([[0], np.cumsum(counts.flatten().cpu().numpy())])
        seeds = rs.permutation(N)[:K]
        lo = int(offs[comm.rank])
        mine = np.nonzero((seeds >= lo) & (seeds < lo + n_local))[0]
        part = torch.zeros((K, D), dtype=torch.float32, device=dev)
        if mine.size:
            part[torch.from_numpy(mine).to(dev)] = Xc[torch.from_numpy(seeds[mine] - lo).to(dev)]
        allp = torch.empty((comm.world * K, D), dtype=torch.float32, device=dev)
        comm.all_gather_rows(part, allp)
        owner = np.searchsorted(offs, seeds, side="right") - 1
        return ops.centers_like(allp[torch.from_numpy(owner * K + np.arange(K)).to(dev)], dev)

    def _relocate(self, Xc, C_old, labels, sums, counts, part_lo):
        """_relocate_empty_clusters_dense across ranks: every rank proposes its n_empty farthest
        samples, the proposals are all-gathered and all ranks apply the same global choice to
        the (replicated, already reduced) sums / counts."""
        comm, ops = self.comm, self.ops
        empty = torch.nonzero(counts == 0).flatten()
        ne = int(empty.numel())
        if ne == 0:
            return
        D = Xc.shape[1]
        dev = Xc.device
        dist_local = ops.row_dist(Xc, C_old, labels) if Xc.shape[0] else torch.zeros(0, device=dev)
        k = min(ne, int(dist_local.numel()))
        rec = torch.full((ne, D + 3), -1.0, dtype=torch.float64, device=dev)  # [dist, rank, old label, row...]
        if k:
            val, idx = torch.topk(dist_local, k)
            rec[:k, 0] = val.double()
            rec[:k, 1] = float(comm.rank)
            rec[:k, 2] = labels[idx].double()
            rec[:k, 3:] = Xc[idx].double()
        allrec = torch.empty((ne * comm.world, D + 3), dtype=torch.float64, device=dev)
        comm.all_gather_rows(rec, allrec)
        order = torch.argsort(allrec[:, 0], descending=True, stable=True)
        if float(allrec[order[0], 0]) <= 0:
            return
        for e, j in zip(empty.tolist(), order[:ne].tolist()):
            if float(allrec[j, 0]) < 0:
                break
            old = int(allrec[j, 2].item())
            x = allrec[j, 3:].to(torch.float32)
            sums[old] -= x
            sums[e] = x
            counts[e] = 1
            counts[old] -= 1


def batch_plan(idx, row_off) -> Tuple[np.ndarray, np.ndarray]:
    """The host half of gdr_minibatch_batch_dist: ``order`` (int32) lists the batch positions of ``idx`` (global row
    ids) grouped by owning rank — rank order, ascending within a rank — and ``counts`` (int64 [world]) how many each
    rank owns.  ``row_off`` [world + 1] are the ranks' first global rows and the total (empty ranks repeat an offset).
    Pure numpy and stable, so every rank derives the same plan from the same draws."""
    idx = np.asarray(idx, dtype=np.int64)
    row_off = np.asarray(row_off, dtype=np.int64)
    world = row_off.shape[0] - 1
    if idx.size and (idx.min() < 0 or idx.max() >= row_off[-1]):
        raise ValueError(f"batch_plan: row ids must lie in [0, {int(row_off[-1])})")
    owner = np.searchsorted(row_off, idx, side="right") - 1
    order = np.argsort(owner, kind="stable").astype(np.int32)
    return order, np.bincount(owner, minlength=world).astype(np.int64)


def random_state_digest(rs: np.random.RandomState) -> int:
    """64-bit digest of a RandomState's whole state (equal states, equal digests), as a signed integer."""
    import hashlib
    name, keys, pos, has_gauss, cached = rs.get_state()
    h = hashlib.blake2b(digest_size=8)
    h.update(str(name).encode())
    h.update(np.ascontiguousarray(keys, dtype=np.uint32).tobytes())
    h.update(np.array([pos, has_gauss], dtype=np.int64).tobytes())
    h.update(np.float64(cached).tobytes())
    return int.from_bytes(h.digest(), "little", signed=True)


def _array_digest(a) -> int:
    import hashlib
    arr = np.ascontiguousarray(a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a), dtype=np.float32)
    h = hashlib.blake2b(digest_size=8)
    h.update(np.array(arr.shape, dtype=np.int64).tobytes())
    h.update(arr.tobytes())
    return int.from_bytes(h.digest(), "little", signed=True)


def _f64_bits(v) -> int:
    return int(np.float64(v).view(np.int64))


def _agree_on_entry(comm: Comm, device, what: str, err: Optional[Exception], n_local: int, *vals) -> np.ndarray:
    """The entry agreement of a row-partitioned fit: ONE all-gather of [verdict, n_local, vals...].  A rank whose own
    arguments were rejected raises its error, every other rank ValueError; so do all ranks when the vals differ.
    Returns the row offsets [world + 1] (the blocks in rank order)."""
    mine = torch.tensor([0 if err is None else 1, int(n_local)] + [int(v) for v in vals], dtype=torch.int64, device=device)
    allv = torch.empty(comm.world * mine.numel(), dtype=torch.int64, device=device)
    comm.all_gather_rows(mine, allv)
    allv = allv.view(comm.world, -1).cpu().numpy()
    if err is not None:
        raise err
    if allv[:, 0].any():
        raise ValueError(f"{what}: rank {int(np.nonzero(allv[:, 0])[0][0])} rejected its arguments")
    if not (allv[:, 2:] == allv[comm.rank, 2:]).all():
        raise ValueError(f"{what}: the ranks passed different arguments")
    return np.concatenate([[0], np.cumsum(allv[:, 1])]).astype(np.int64)


class DistMiniBatchKMeans(MiniBatchKMeans):
    """``MiniBatchKMeans`` on row-partitioned X: the one-GPU bytes for any number of ranks.

    Same constructor as ``MiniBatchKMeans`` plus ``comm`` and ``ops``; ``fit(X_local)`` takes this rank's contiguous row
    block (the blocks in rank order are X; any sizes, empty ones included).  The step loop is ``kmeans.minibatch_loop``,
    run on every rank with the same host draws: each batch (and the validation and init subsets) is assembled on every
    rank by gdr_minibatch_batch_dist — the owners pack and label their rows, one grouped exchange — and the centre update,
    the batch inertia and the reassignment then run replicated on identical data.  The init-subset k-means++ runs
    replicated.  The final E-step labels this rank's rows with the one-GPU kernel choice; its fp64 inertia is summed over
    the ranks.

    Collective.  At entry one all-gather checks N, K, D, batch_size, max_iter, max_no_improvement, init_size, n_init,
    the bits of tol and reassignment_ratio, compute_labels, the init kind, a digest of the RandomState and of an array
    init; a mismatch raises ValueError on every rank.  A string init needs ``random_state``.

    With tol = 0 the centres, every rank's labels (its slice of the one-GPU labels), n_steps_ and n_iter_ equal the
    one-GPU fit's; inertia_ is equal at one rank and within fp64 rounding of the rank grouping otherwise.  With tol > 0
    the tolerance comes from rank-grouped fp64 column sums.  Results: ``labels_`` int32 on the device (this rank's
    rows); ``cluster_centers_`` [K, D] on the device, ``inertia_``, ``n_iter_``, ``n_steps_`` replicated."""

    def __init__(self, n_clusters=8, *, init="k-means++", max_iter=100, batch_size=1024, verbose=0, compute_labels=True,
                 random_state=None, tol=0.0, max_no_improvement=10, init_size=None, n_init="auto",
                 reassignment_ratio=0.01, precision="auto", device=None, comm: Comm = None, ops=None):
        super().__init__(n_clusters=n_clusters, init=init, max_iter=max_iter, batch_size=batch_size, verbose=verbose,
                         compute_labels=compute_labels, random_state=random_state, tol=tol,
                         max_no_improvement=max_no_improvement, init_size=init_size, n_init=n_init,
                         reassignment_ratio=reassignment_ratio, precision=precision, device=device)
        self.comm = comm or Comm()
        self.ops = ops or CudaOps()

    def _entry_values(self, D: int):
        """(local error or None, the values every rank must pass alike)."""
        from .kmeans import _check_random_state
        err, kind, init_digest, rs_digest = None, 0, 0, 0
        try:
            self._mode(D)
            if isinstance(self.init, str):
                if self.init not in ("k-means++", "random"):
                    raise ValueError(f"init should be 'k-means++', 'random' or an array, got {self.init!r}")
                if self.random_state is None:
                    raise ValueError("a string init needs the same random_state on every rank")
                kind = 1 if self.init == "k-means++" else 2
            else:
                shape = tuple(self.init.shape) if isinstance(self.init, torch.Tensor) else np.shape(self.init)
                if tuple(shape) != (int(self.n_clusters), D):
                    raise ValueError(f"The shape of the initial centers {tuple(shape)} does not match "
                                     f"the number of clusters {self.n_clusters} / features {D}.")
                init_digest = _array_digest(self.init)
            if self.n_init != "auto" and int(self.n_init) <= 0:
                raise ValueError(f"n_init should be > 0, got {self.n_init} instead.")
            rs_digest = random_state_digest(_check_random_state(self.random_state))
            opt = lambda v: -1 if v is None else int(v)       # noqa: E731
            vals = (int(self.n_clusters), D, int(self.batch_size), int(self.max_iter), opt(self.max_no_improvement),
                    opt(self.init_size), -1 if self.n_init == "auto" else int(self.n_init), _f64_bits(self.tol),
                    _f64_bits(self.reassignment_ratio), int(bool(self.compute_labels)), kind, init_digest, rs_digest)
        except (ValueError, TypeError) as e:
            err, vals = (e if isinstance(e, ValueError) else ValueError(str(e))), (0,) * 13
        return err, vals

    def fit(self, X_local: torch.Tensor, y=None, sample_weight=None):
        from .kmeans import TcOperand, _check_random_state, minibatch_loop
        from ._dev import new_padded, pad4
        if sample_weight is not None:
            raise NotImplementedError("sample_weight is not supported (the reference never passes it)")
        ops, comm = self.ops, self.comm
        if not hasattr(ops, "minibatch_batch"):
            raise NotImplementedError(f"{type(ops).__name__} has no distributed mini-batch assembly")
        if not isinstance(X_local, torch.Tensor) or not X_local.is_cuda or X_local.dim() != 2:
            raise ValueError("X_local must be a 2-D CUDA tensor (this rank's rows)")
        X = ops.prep_rows(X_local)
        n_local, D = X.shape
        dev = X.device
        err, vals = self._entry_values(D)
        row_off = _agree_on_entry(comm, dev, "DistMiniBatchKMeans.fit", err, n_local, *vals)
        N = int(row_off[-1])
        self._check_fit_args(N)          # depends on agreed values only: raises on every rank alike
        rs = _check_random_state(self.random_state)
        bufs = {}

        def rows(idx):
            idx = np.arange(N, dtype=np.int64) if idx is None else idx
            out = new_padded(idx.shape[0], D, dev, zero=True)
            return ops.minibatch_batch(comm, idx, row_off, X, None, out, None)

        def assemble(idx, C, labels_b):
            if "Xb" not in bufs:
                bufs["Xb"] = new_padded(idx.shape[0], D, dev, zero=True)
            return ops.minibatch_batch(comm, idx, row_off, X, C, bufs["Xb"], labels_b)

        def var_mean():
            sums = ops.column_sums(X)
            comm.all_reduce(sums)
            m64 = sums[:D] / N
            return float(((sums[D:] / N - m64 * m64).clamp_min(0)).mean().item())

        centers, ewa = minibatch_loop(self, N, D, dev, rs, rows, assemble, var_mean)
        self._numpy_io = False
        self._centers_dev = centers
        self.n_features_in_ = D
        self.cluster_centers_ = centers.contiguous() if pad4(D) == D else centers.clone().contiguous()
        if self.compute_labels:
            mode = self._mode(D)
            labels = torch.empty(n_local, dtype=torch.int32, device=dev)
            if n_local:
                tc = TcOperand(X) if mode == 1 else None
                inertia = self._labels_inertia(X, centers, labels, mode=mode, tc=tc)
            else:
                inertia = torch.zeros(1, dtype=torch.float64, device=dev)
            comm.all_reduce(inertia)
            self.inertia_ = float(inertia.item())
            self._labels_dev = labels
            self.labels_ = labels
        else:
            self.inertia_ = (ewa if ewa is not None else 0.0) * N
        return self


# ------------------------------------------------------------------------------------------
# edge sparsification (between stages 3 and 4)
# ------------------------------------------------------------------------------------------
def dist_graph_sparse(comm: Comm, part: RowPartition, A_local, ratio: float, ebd_local: Optional[torch.Tensor] = None,
                      sp_type: str = "vanilla", ops=None):
    """``sparsify.graph_sparse`` (ClustGDD.graph_sparse, clustgdd_agent_transduct.py:131-232) on a row partition.
    Collective.  ``A_local`` is this rank's row block of A_hat with global column ids (``dist_build_adjacency``; None on a
    rank without rows, which still joins), ``ebd_local`` its rows of the logits.  Returns this rank's row blocks of the
    sparsified graphs as CSR with global column ids (None on a rank without rows): one for 'vanilla' / 'single' /
    'no_sp', one per class for 'attaw'.  The blocks concatenated in rank order are byte-identical to the one-GPU
    ``graph_sparse`` on the whole graph, for any number of ranks.  'rand' is not supported here: its draws are
    ``torch.randperm`` over the global edge list on the host generator."""
    if sp_type == "no_sp":
        return [A_local]
    if sp_type == "rand":
        raise NotImplementedError("sp_type='rand' has no row-partitioned form")
    if sp_type not in ("vanilla", "single", "attaw"):
        raise ValueError(f"unknown sp_type {sp_type!r}")
    if sp_type != "vanilla" and ebd_local is None:
        raise ValueError(f"sp_type={sp_type!r} needs ebd")
    ops = ops or CudaOps()
    if not hasattr(ops, "sparsify_classes_dist"):
        raise NotImplementedError(f"{type(ops).__name__} has no distributed sparsification")
    dev = ebd_local.device if ebd_local is not None else torch.device("cuda", torch.cuda.current_device())
    sizes = _block_sizes(part)
    nnz = torch.tensor([0 if A_local is None else A_local.nnz], dtype=torch.int64, device=dev)
    k = int(int(comm.all_reduce(nnz, "sum").item()) * ratio)     # graph_sparse's int(nedges * ratio)

    def global_er(A):
        # the degree vector of A's rows is needed at every column: row sums, all-gathered
        deg = comm.all_gather_var(ops.row_sums(A) if A is not None else torch.zeros(0, dtype=torch.float32, device=dev),
                                  sizes)
        return ops.er_lower_rows(A, deg, part.lo) if A is not None else torch.zeros(0, dtype=torch.float32, device=dev)

    if sp_type == "vanilla":
        return ops.sparsify_classes_dist(comm, A_local, part.lo, part.n, global_er(A_local), None, k)
    from ._dev import need_cuda
    e = need_cuda(ebd_local, "ebd").to(torch.float32).contiguous()
    if e.dim() != 2 or e.shape[0] != part.n_local:
        raise ValueError("ebd_local must be [rows of this rank, n_classes]")
    C = int(e.shape[1])
    ebd = comm.all_gather_var(e.reshape(-1), [s * C for s in sizes]).view(part.n, C)
    R = ops.cosine_reweight_rows(A_local, ebd, part.lo) if A_local is not None else None
    er = global_er(R)
    prob = ops.softmax_rows(ebd) if sp_type == "attaw" else None
    return ops.sparsify_classes_dist(comm, R, part.lo, part.n, er, prob, k)


# ------------------------------------------------------------------------------------------
# stage 4
# ------------------------------------------------------------------------------------------
def dist_graph_compress(comm: Comm, part: RowPartition, labels_local: torch.Tensor, A_local, ops=None, replicate: bool = True,
                        merge: str = "route", timing: Optional[dict] = None):
    """graph_compress (clustgdd_agent_transduct.py:234-250) for a row-partitioned A_hat.

    ``merge="route"`` (default): every local edge is sent once, as a (cell key, weight) pair, to the owner of its coarse
    row (a -> rank a // ceil(n / world); one stable partition pass + all-to-all); the owner sorts and reduces what it
    receives.  The exchange order is the global CSR order, so counts AND weight sums are bit-identical to the single-device
    result.  ``merge="records"``: every rank coarsens its local edges first and the (cell, count, sum) runs are exchanged and
    merged (sums added in source-rank order: deterministic, 1e-5 from the single-device sums).  O(local nnz) memory
    on every rank, no n x n array anywhere (config E: n^2 = 10^8 cells).  With ``replicate`` (default) the pieces are
    all-gathered, and every rank returns the reference's result: (adj_syn torch sparse COO n x n, merged integer cell
    counts).  Without it: this rank's coarse rows as (a_lo, rowptr, colidx, vals, counts).  ``timing``: a dict that receives
    the wall-clock milliseconds of every section (synchronising; tools/stage4_probe.py)."""
    import time as _time
    ops = ops or CudaOps()
    _t = [_time.perf_counter()]

    def mark(name):
        if timing is not None:
            if labels_local.is_cuda:
                torch.cuda.synchronize()
            now = _time.perf_counter()
            timing[name] = timing.get(name, 0.0) + (now - _t[0]) * 1e3
            _t[0] = now
    labels = _compress_labels(comm, part, labels_local, ops)
    mark("labels_allgather_sizes")
    return _dist_compress_graph(comm, ops, A_local, *labels, replicate, merge, mark)


def dist_graph_compress_list(comm: Comm, part: RowPartition, labels_local: torch.Tensor, A_local, adj_list_local,
                             ops=None, replicate: bool = True, merge: str = "route"):
    """graph_compress (clustgdd_agent_transduct.py:234-250) with the reference's shape: every graph of
    ``adj_list_local`` (this rank's row blocks, e.g. from ``dist_graph_sparse``) and ``A_local`` coarsened by the same
    labels.  Returns (compressed_list, adj_syn); each element is what ``dist_graph_compress`` returns for that graph.
    The labels all-gather, n and the cluster sizes are computed once per call."""
    ops = ops or CudaOps()
    labels = _compress_labels(comm, part, labels_local, ops)
    compressed = [_dist_compress_graph(comm, ops, a, *labels, replicate, merge) for a in adj_list_local]
    return compressed, _dist_compress_graph(comm, ops, A_local, *labels, replicate, merge)


def _compress_labels(comm: Comm, part: RowPartition, labels_local: torch.Tensor, ops):
    """(this rank's labels int32, all labels, n, cluster sizes): the per-call part of stage 4."""
    dev = labels_local.device
    rows_per, world = part.rows_per, part.world
    block = torch.full((rows_per,), -1, dtype=torch.int32, device=dev)
    block[: labels_local.shape[0]] = labels_local.to(torch.int32)
    gathered = torch.empty(rows_per * world, dtype=torch.int32, device=dev)
    comm.all_gather_rows(block, gathered)
    # drop the padding of every rank's block
    pieces = [gathered[r * rows_per: r * rows_per + (part.bounds(r)[1] - part.bounds(r)[0])] for r in range(world)]
    labels_all = torch.cat(pieces).contiguous()
    nmax = labels_all.max().to(torch.int64).reshape(1)
    n = int(comm.all_reduce(nmax, "max").item()) + 1
    sizes = ops.label_counts(labels_all, n)
    return labels_local.to(torch.int32).contiguous(), labels_all, n, sizes


def _dist_compress_graph(comm: Comm, ops, A_local, lab_l, labels_all, n, sizes, replicate, merge, mark=lambda name: None):
    """The per-graph part of stage 4: route (or records) exchange, merge, scale, and the replication."""
    world = comm.world
    cr = (n + world - 1) // world
    a_lo = min(n, comm.rank * cr)
    n_rows = min(n, a_lo + cr) - a_lo
    if merge == "route" and hasattr(ops, "coarsen_route"):
        # every edge goes to the owner of its coarse row once; the owner sorts + reduces (one sort per edge, sums in CSR order)
        keys, w, send_counts = ops.coarsen_route(A_local, lab_l, labels_all, n, world)
        stats = None
        if hasattr(ops, "cluster_stats"):
            # per-cluster (edges, max |w|) of the whole graph: the owner's shared-memory merge then rounds like one GPU does
            edges, wmax = ops.cluster_stats(A_local, lab_l, n)
            stats = (comm.all_reduce(edges, "sum"), comm.all_reduce(wmax, "max"))
        mark("route")
        if comm.symm_ok() and keys.is_cuda:
            recv_k, recv_w = comm.symm_exchange([keys, w], comm.count_matrix(send_counts, keys.device))
        else:
            recv_k, rc = comm.all_to_all_rows(keys, send_counts)
            recv_w, _ = comm.all_to_all_rows(w, send_counts, recv_counts=rc)
        mark("all_to_all")
        if stats is not None:
            rowptr, colidx, counts, wsum = ops.coarse_merge_edges(recv_k, recv_w, a_lo, n_rows, n, stats=stats)
        else:
            rowptr, colidx, counts, wsum = ops.coarse_merge_edges(recv_k, recv_w, a_lo, n_rows, n)
        mark("merge_edges")
    else:
        # local coarsening first, then (cell, count, sum) records by key range: less traffic when cells repeat a lot locally
        rec, send_counts = ops.coarsen_records(A_local, lab_l, labels_all, n, world)
        recv, _ = comm.all_to_all_rows(rec, send_counts)
        rowptr, colidx, counts, wsum = ops.coarse_merge(recv, a_lo, n_rows, n)
    vals = ops.coarse_scale(rowptr, colidx, wsum, sizes, a_lo, n_rows)
    mark("scale")
    if not replicate:
        return a_lo, rowptr, colidx, vals, counts
    if world == 1:
        return ops.csr_to_coo(rowptr, colidx, vals, n), counts
    rowptr_all, col_all, val_all, cnt_all = _replicate_coarse_rows(comm, n, rowptr, colidx, vals, counts)
    mark("replicate")
    out = ops.csr_to_coo(rowptr_all, col_all, val_all, n), cnt_all
    mark("to_coo")
    return out


def _replicate_coarse_rows(comm: Comm, n: int, rowptr, colidx, vals, counts):
    """All-gather of the key-range pieces (variable sizes) and their row pointers: every rank ends with the whole CSR."""
    world, dev = comm.world, rowptr.device
    cr = (n + world - 1) // world
    n_rows = int(rowptr.shape[0]) - 1
    nnz_mine = torch.tensor([int(colidx.shape[0])], dtype=torch.int64, device=dev)
    nnz_all = torch.empty(world, dtype=torch.int64, device=dev)
    comm.all_gather_rows(nnz_mine, nnz_all)
    nnz_list = [int(v) for v in nnz_all.tolist()]
    if comm.symm_ok() and colidx.is_cuda:
        # the three pieces stored straight into every rank's symmetric buffer (posted NVLink stores), then copied out of it
        col_all, val_all, cnt_all = (t.clone() for t in comm.all_gather_symm([colidx, vals, counts], nnz_list))
    else:
        col_all = comm.all_gather_var(colidx, nnz_list)
        val_all = comm.all_gather_var(vals, nnz_list)
        cnt_all = comm.all_gather_var(counts, nnz_list)
    rp_block = torch.zeros(cr + 1, dtype=torch.int32, device=dev)
    rp_block[: n_rows + 1] = rowptr
    rp_g = torch.empty(world * (cr + 1), dtype=torch.int32, device=dev)
    comm.all_gather_rows(rp_block, rp_g)
    rowptr_all = torch.empty(n + 1, dtype=torch.int32, device=dev)
    off = 0
    for r in range(world):
        lo = min(n, r * cr)
        rows_r = min(n, lo + cr) - lo
        if rows_r > 0:
            rowptr_all[lo: lo + rows_r] = rp_g[r * (cr + 1): r * (cr + 1) + rows_r] + off
        off += nnz_list[r]
    rowptr_all[n] = off
    return rowptr_all, col_all, val_all, cnt_all


# ------------------------------------------------------------------------------------------
# distill_recsys on a row partition: users and items each split over the ranks (SURVEY 8e)
# ------------------------------------------------------------------------------------------
def _block_sizes(part: RowPartition):
    return [part.bounds(r)[1] - part.bounds(r)[0] for r in range(part.world)]


def dist_build_interaction(comm: Comm, part_u: RowPartition, part_i: RowPartition, u_slice: torch.Tensor,
                           i_slice: torch.Tensor, ops=None):
    """build_interaction_matrix (distill_recsys.py:110-117) from a SLICE of the interaction lines per rank.  Returns
    (R_local, RT_local): the rows of R (users x items) of this rank's users and the rows of R^T of this rank's items,
    duplicate lines summed, global column ids — two all-to-alls of the lines, bucketed by the owner of u and of i."""
    ops = ops or CudaOps()
    nu, ni = part_u.n, part_i.n
    u = u_slice.to(torch.int64)
    i = i_slice.to(torch.int64)
    if u.numel() and (int(u.min()) < 0 or int(u.max()) >= nu or int(i.min()) < 0 or int(i.max()) >= ni):
        raise ValueError("row/col index exceeds matrix dimensions")
    if hasattr(ops, "edges_route"):
        ku, cu, st_u = ops.edges_route(u.contiguous(), i.contiguous(), nu, ni, part_u.rows_per, part_u.world, False)
        recv_u, _ = comm.all_to_all_rows(ku, cu)
        R_local = ops.csr_from_keys(recv_u, part_u.lo, part_u.n_local, ni, False)
        ki, ci, _ = ops.edges_route(i.contiguous(), u.contiguous(), ni, nu, part_i.rows_per, part_i.world, False)
        recv_i, _ = comm.all_to_all_rows(ki, ci)
        RT_local = ops.csr_from_keys(recv_i, part_i.lo, part_i.n_local, nu, False)
        return R_local, RT_local
    e_u, c_u = ops.bucket_by_owner(u, i, part_u.rows_per, part_u.world)
    recv_u, _ = comm.all_to_all_rows(e_u, c_u)
    R_local = ops.build_block_csr_weighted(recv_u[:, 0] - part_u.lo, recv_u[:, 1], part_u.n_local, ni)
    e_i, c_i = ops.bucket_by_owner(i, u, part_i.rows_per, part_i.world)
    recv_i, _ = comm.all_to_all_rows(e_i, c_i)
    RT_local = ops.build_block_csr_weighted(recv_i[:, 0] - part_i.lo, recv_i[:, 1], part_i.n_local, nu)
    return R_local, RT_local


def dist_bipartite_normalize(comm: Comm, part_u: RowPartition, part_i: RowPartition, R_local, RT_local, ops=None,
                             eps: float = 1e-8):
    """LightGCN edge norm (distill_recsys.py:329-335) for both row blocks: own row degrees, all-gather of the degree vector
    of the other side.  Same fp32 chains as the single-device build: values bit-identical.
    Returns (A_local [users x items], AT_local [items x users], deg_u_local, deg_i_local)."""
    ops = ops or CudaOps()
    deg_u_l, deg_i_l = ops.row_sums(R_local), ops.row_sums(RT_local)
    deg_u = comm.all_gather_var(deg_u_l, _block_sizes(part_u))
    deg_i = comm.all_gather_var(deg_i_l, _block_sizes(part_i))
    return (ops.bip_norm_block(R_local, deg_u_l, deg_i, eps), ops.bip_norm_block(RT_local, deg_i_l, deg_u, eps),
            deg_u_l, deg_i_l)


def dist_lightgcn_propagate(comm: Comm, part_u: RowPartition, part_i: RowPartition, A_local, AT_local,
                            u0_local: torch.Tensor, i0_local: torch.Tensor, num_layers: int, ops=None):
    """Forward of LightGCNCondensed.propagate (distill_recsys.py:337-353) on row-partitioned embeddings: per layer an
    all-gather of the item rows and of the user rows, then the two CSR SpMMs on the local rows (u <- A i, i <- A^T u,
    simultaneous update), output = mean over the L + 1 layers.  Row-wise independent: bit-identical to one device."""
    ops = ops or CudaOps()
    u, it = ops.prep_rows(u0_local), ops.prep_rows(i0_local)
    d = u.shape[1]
    u_acc, i_acc = ops.scale(u, 1.0), ops.scale(it, 1.0)
    ru, ri = part_u.rows_per, part_i.rows_per
    u_full, i_full = ops.empty_rows(ru * part_u.world, d, u), ops.empty_rows(ri * part_i.world, d, it)
    u_blk, i_blk = ops.empty_rows(ru, d, u), ops.empty_rows(ri, d, it)
    for _ in range(int(num_layers)):
        u_blk[: u.shape[0]].copy_(u)
        i_blk[: it.shape[0]].copy_(it)
        comm.all_gather_rows(u_blk, u_full)
        comm.all_gather_rows(i_blk, i_full)
        u_next = ops.spmm(A_local, i_full, 1.0, u_acc, 1.0)
        i_next = ops.spmm(AT_local, u_full, 1.0, i_acc, 1.0)
        u, it = u_next, i_next
    inv = 1.0 / float(num_layers + 1)
    return ops.scale(u_acc, inv), ops.scale(i_acc, inv)


def _same_on_every_rank(comm: Comm, device, what: str, *vals):
    """Raises ValueError on every rank unless every rank passed the same integers (one all-gather)."""
    mine = torch.tensor([int(v) for v in vals], dtype=torch.int64, device=device)
    allv = torch.empty(comm.world * mine.numel(), dtype=torch.int64, device=device)
    comm.all_gather_rows(mine, allv)
    if not bool((allv.view(comm.world, -1) == mine).all()):
        raise ValueError(f"{what}: the ranks passed different arguments")


def dist_truncated_svd(comm: Comm, part_u: RowPartition, part_i: RowPartition, R_local, RT_local, k: int, seed: int = 42,
                       block: int = None, n_blocks: int = None, ops=None):
    """svd.truncated_svd of the row-partitioned interaction matrix (R_local, RT_local as dist_build_interaction returns
    them) without gathering R.  Collective; every rank passes the same k, seed, block and n_blocks (checked: a mismatch
    raises ValueError on every rank).  The Krylov blocks Q and the products B = A Q stay row-partitioned: each SpMM runs
    on this rank's rows against its operand all-gathered in the padded equal-block layout, each Gram is
    gdr_dense_gram_dist, and the small (q b)² Ritz problem is solved on every rank from identical data.  Returns
    (U_local [this rank's users, k], S [k] descending, the same on every rank, V_local [this rank's items, k]), fp32
    on the device; the blocks in rank order are byte-identical to truncated_svd(R) for any number of ranks."""
    from .svd import krylov_ritz
    ops = ops or CudaOps()
    if not hasattr(ops, "gram_dist"):
        raise NotImplementedError(f"{type(ops).__name__} has no distributed Gram matrix")
    dev = R_local.device
    _same_on_every_rank(comm, dev, "dist_truncated_svd", part_u.n, part_i.n, k, seed, -1 if block is None else block,
                        -1 if n_blocks is None else n_blocks)
    # Krylov space on the smaller side (truncated_svd's choice): A maps it to the larger one
    if part_i.n <= part_u.n:
        A, At, p_s, p_o = R_local, RT_local, part_i, part_u
    else:
        A, At, p_s, p_o = RT_local, R_local, part_u, part_i

    def times(M, x_local, part):
        """This rank's rows of M X, X the whole matrix whose rows ``part`` splits (this rank holds x_local)."""
        f = x_local.shape[1]
        blk = ops.empty_rows(part.rows_per, f, x_local)
        blk[: x_local.shape[0]].copy_(x_local)
        full = ops.empty_rows(part.rows_per * part.world, f, x_local)      # row index = global id (equal blocks)
        comm.all_gather_rows(blk, full)
        return ops.spmm(M, full, 1.0, None, 0.0)

    Uo, S, Vs = krylov_ritz(p_s.n, slice(p_s.lo, p_s.hi), k, seed, block, n_blocks, dev,
                            lambda X, Y: ops.gram_dist(comm, p_s.n, p_s.lo, X, Y),
                            lambda X, Y: ops.gram_dist(comm, p_o.n, p_o.lo, X, Y),
                            lambda X: times(A, X, p_s), lambda Y: times(At, Y, p_o))
    return (Uo, S, Vs) if part_i.n <= part_u.n else (Vs, S, Uo)


def dist_compute_svd_embeddings(comm: Comm, part_u: RowPartition, part_i: RowPartition, R_local, RT_local, dim: int,
                                seed: int = 42, ops=None):
    """svd.compute_svd_embeddings (distill_recsys.py:124-155) on the row partition: (U sqrt(S), V sqrt(S)) of this
    rank's users and items from dist_truncated_svd, as fp32 DEVICE tensors (the input of dist_standard_scale), byte-
    identical to the rows of the one-GPU embeddings.  Collective; raises the reference's ValueError when no
    factorisation is possible, and ValueError on every rank when the ranks pass different dim or seed."""
    _same_on_every_rank(comm, R_local.device, "dist_compute_svd_embeddings", part_u.n, part_i.n, dim, seed)
    shape = (part_u.n, part_i.n)
    k = min(int(dim), min(shape) - 1)
    if k <= 0:
        raise ValueError(f"Cannot compute SVD with shape={tuple(shape)} and dim={dim}")
    U, S, V = dist_truncated_svd(comm, part_u, part_i, R_local, RT_local, k, seed=seed, ops=ops)
    sqrt_s = torch.sqrt(torch.clamp_min(S, 1e-12)).reshape(1, -1)
    return U * sqrt_s, V * sqrt_s


def dist_standard_scale(comm: Comm, x_local: torch.Tensor, ops=None):
    """StandardScaler().fit_transform (distill_recsys.py:172) on row-partitioned X: fp64 column sums and second moments
    about the mean are all-reduced (two passes, as sklearn's), result fp32((x - fp32(mean)) / fp32(scale))."""
    ops = ops or CudaOps()
    X = ops.prep_rows(x_local)
    n_local, D = X.shape
    cnt = torch.tensor([n_local], dtype=torch.int64, device=X.device)
    comm.all_reduce(cnt)
    N = int(cnt.item())
    s1 = ops.column_sums(X)
    comm.all_reduce(s1)
    mean64 = (s1[:D] / N).contiguous()
    s2 = ops.column_moments(X, mean64)
    comm.all_reduce(s2)
    var = s2[D:] / N
    eps = 2.220446049250313e-16                                   # sklearn _is_constant_feature
    bound = N * eps * var + (N * mean64 * eps) ** 2
    scale = torch.where(var <= bound, torch.ones_like(var), var.sqrt())
    return ops.standardize_apply(X, mean64.to(torch.float32).contiguous(), scale.to(torch.float32).contiguous())


def dist_kmeans_cluster(comm: Comm, part: RowPartition, X_local: torch.Tensor, n_clusters: int, seed: int,
                        minibatch: bool = True, batch_size: int = 2048, init="k-means++", ops=None):
    """kmeans.kmeans_cluster (distill_recsys.py:158-181) on a row partition: z-scores the columns
    (dist_standard_scale), then clusters with DistMiniBatchKMeans(n_clusters, random_state=seed, batch_size) when
    ``minibatch`` and more than 20 000 rows, else DistKMeans(init, random_state=seed) — the reference's rule (:173-178).
    K is capped to the global row count ``part.n``.  Collective.  Returns (this rank's labels int64, the centres
    [K, D] f32, the same on every rank), both on the device."""
    if n_clusters <= 0:
        raise ValueError("n_clusters must be > 0")
    N = int(part.n)
    K = max(1, min(int(n_clusters), N))
    ops = ops or CudaOps()
    Xs = dist_standard_scale(comm, X_local, ops=ops)
    if minibatch and N > 20000:
        km = DistMiniBatchKMeans(n_clusters=K, random_state=seed, batch_size=batch_size, n_init="auto", init=init,
                                 comm=comm, ops=ops)
    else:
        km = DistKMeans(K, init, random_state=seed, comm=comm, ops=ops)
    km.fit(Xs)
    return km.labels_.to(torch.int64), km.cluster_centers_


def dist_segment_sum(comm: Comm, part: RowPartition, X_local: torch.Tensor, labels_local: torch.Tensor, K: int, ops=None):
    """kmeans.segment_sum on a row partition: X_local [part.n_local, F] and labels_local [part.n_local] (int32 or int64)
    are this rank's rows of the features and labels, e.g. dist_propagate's padded blocks and DistKMeans.labels_ /
    dist_kmeans_cluster's labels.  Nothing is gathered: each fp32 chain runs over rank 0's members of its cluster, then
    continues on rank 1 from the value rank 0 ended it at, and so on (gdr_segment_sum_dist).  Collective.  Returns
    (sums [K, F] padded, counts int32 [K]), the same on every rank and byte-equal to segment_sum of the rows
    concatenated in rank order.  Raises ValueError on every rank when K <= 0, when the ranks pass different K or F, or
    when a label lies outside [0, K); the communicator stays usable."""
    from ._lib import GdrError
    ops = ops or CudaOps()
    if not hasattr(ops, "segment_sum_dist"):
        raise NotImplementedError(f"{type(ops).__name__} has no distributed segment sum")
    K = int(K)
    X = ops.prep_rows(X_local)
    lab = labels_local.to(X.device)
    if lab.dtype != torch.int32:
        lab = lab.clamp(-1, max(K, 0))      # out of int32 range stays out of [0, K) after the cast
    lab = lab.to(torch.int32).contiguous()
    try:
        return ops.segment_sum_dist(comm, part.lo, X, lab, K)
    except GdrError as e:
        if e.code in (-1, -4):              # GDR_EINVAL, GDR_ERANGE: rejected on every rank by the entry check
            raise ValueError(f"dist_segment_sum: {e}") from e
        raise


def dist_cluster_means(comm: Comm, part: RowPartition, features_local: torch.Tensor, labels_local: torch.Tensor,
                       n_clusters: int, ops=None) -> torch.Tensor:
    """kmeans.cluster_means (feat_syn, clustgdd_agent_transduct.py:116-127) of row-partitioned features and labels:
    [K, F], the same on every rank and byte-equal to cluster_means of the rows concatenated in rank order, NaN rows of
    empty clusters included.  Collective; the errors of dist_segment_sum."""
    from .kmeans import means_of_sums
    sums, counts = dist_segment_sum(comm, part, features_local, labels_local, n_clusters, ops=ops)
    return means_of_sums(sums, counts, empty_nan=True)


def dist_segment_mean_pool(comm: Comm, part: RowPartition, emb_local: torch.Tensor, assign_local: torch.Tensor,
                           n_segments: int, ops=None) -> torch.Tensor:
    """kmeans.segment_mean_pool (the teacher pooling of distill_recsys.py:623-636) of row-partitioned embeddings and
    assignments (e.g. u2cu from dist_kmeans_cluster): [n_segments, F], the same on every rank and byte-equal to the
    one-GPU pooling of the rows concatenated in rank order.  Collective; the errors of dist_segment_sum."""
    from .kmeans import means_of_sums
    sums, counts = dist_segment_sum(comm, part, emb_local, assign_local, n_segments, ops=ops)
    return means_of_sums(sums, counts, empty_nan=False)


def dist_build_condensed_bipartite(comm: Comm, part_u: RowPartition, part_i: RowPartition, u_slice: torch.Tensor,
                                   i_slice: torch.Tensor, u2cu_local: torch.Tensor, i2ci_local: torch.Tensor, num_cu: int,
                                   num_ci: int, ops=None, replicate: bool = True):
    """build_condensed_bipartite (distill_recsys.py:184-201): C[cu, ci] = number of train LINES (u, i) with
    u2cu[u] = cu, i2ci[i] = ci, duplicates counted.  The cluster maps (row-partitioned k-means labels) are all-gathered,
    every rank counts its slice of the lines, the (cell, count) runs are exchanged by key range and merged: integer
    counts, independent of the rank count.  Returns (rowptr, colidx, counts f32) of the whole num_cu x num_ci CSR
    (``replicate``) or (a_lo, rowptr, colidx, counts f32) of this rank's range of cu rows."""
    ops = ops or CudaOps()
    dev = u_slice.device
    world = comm.world

    def gather_map(part, local):
        block = torch.full((part.rows_per,), -1, dtype=torch.int32, device=dev)
        block[: local.shape[0]] = local.to(torch.int32)
        full = torch.empty(part.rows_per * world, dtype=torch.int32, device=dev)
        comm.all_gather_rows(block, full)
        return full            # padded layout index == global id (equal contiguous blocks)

    mu, mi = gather_map(part_u, u2cu_local), gather_map(part_i, i2ci_local)
    cr = (int(num_cu) + world - 1) // world
    a_lo = min(int(num_cu), comm.rank * cr)
    n_rows = min(int(num_cu), a_lo + cr) - a_lo
    if hasattr(ops, "coarsen_route"):
        keys, _, send_counts = ops.coarsen_route(None, mu, mi, int(num_cu), world, n_dst=int(num_ci),
                                                 src=u_slice.to(torch.int64).contiguous(), dst=i_slice.to(torch.int64).contiguous())
        recv_k, _ = comm.all_to_all_rows(keys, send_counts)
        rowptr, colidx, counts, _ = ops.coarse_merge_edges(recv_k, None, a_lo, n_rows, int(num_cu), n_dst=int(num_ci))
    else:
        rec, send_counts = ops.coarsen_records(None, mu, mi, int(num_cu), world, n_dst=int(num_ci),
                                               src=u_slice.to(torch.int64), dst=i_slice.to(torch.int64))
        recv, _ = comm.all_to_all_rows(rec, send_counts)
        rowptr, colidx, counts, _ = ops.coarse_merge(recv, a_lo, n_rows, int(num_cu), n_dst=int(num_ci))
    vals = counts.to(torch.float32)
    if not replicate:
        return a_lo, rowptr, colidx, vals
    if world == 1:
        return rowptr, colidx, vals
    rowptr_all, col_all, val_all, _ = _replicate_coarse_rows(comm, int(num_cu), rowptr, colidx, vals, counts)
    return rowptr_all, col_all, val_all
