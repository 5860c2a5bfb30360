"""Stage 4 — cluster-coarsened synthetic graph  P^T A P  by segmented edge counting.

Mirrors ``ClustGDD.graph_compress`` (clustgdd_agent_transduct.py:234-250,
clustgdd_agent_induct.py:258-274) and ``build_condensed_bipartite`` /
``condensed_csr_to_edge_index`` (distill_recsys.py:184-201, :387-395).  The reference
materialises a dense N x n one-hot (196 GB at the products shape); here every edge is
mapped to its (cluster, cluster) key, keys are radix-sorted and runs are counted/summed,
so memory is O(E) and counts are exact integers.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple, Union

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib
from ._dev import device_of, ptr, stream, to_device_f32, to_device_i64, workspace
from .graph import CSR


def label_counts(labels: torch.Tensor, n: int) -> torch.Tensor:
    """Cluster sizes (int32[n]); raises if a label falls outside [0, n)."""
    lab = labels.to(torch.int32).contiguous()
    counts = torch.empty(int(n), dtype=torch.int32, device=lab.device)
    status = torch.zeros(1, dtype=torch.int32, device=lab.device)
    _lib.call("gdr_label_histogram", lab.numel(), int(n), ptr(lab), ptr(counts), ptr(status), stream())
    if int(status.item()):
        raise ValueError("label outside [0, n_clusters)")
    return counts


def coarsen_edges(labels_src: torch.Tensor, labels_dst: torch.Tensor, n_src: int, n_dst: int, *,
                  src: torch.Tensor = None, dst: torch.Tensor = None, csr: CSR = None,
                  weights: torch.Tensor = None, drop_diag: bool = False):
    """Core of stage 4.  Edges given as COO (src, dst int64) or as a device CSR.
    Returns (rowptr int32[n_src+1], colidx int32[m], counts int32[m], wsum f32[m] | None)."""
    dev = labels_src.device
    ls = labels_src.to(torch.int32).contiguous()
    ld = labels_dst.to(torch.int32).contiguous()
    if csr is not None:
        E, n_rows = csr.nnz, csr.shape[0]
        p_src = p_dst = 0
        p_rp, p_ci = ptr(csr.rowptr), ptr(csr.colidx)
        w = weights
    else:
        E, n_rows = int(src.numel()), 0
        p_src, p_dst, p_rp, p_ci = ptr(src), ptr(dst), 0, 0
        w = weights
    cap = max(1, min(E, int(n_src) * int(n_dst)))
    rowptr = torch.empty(int(n_src) + 1, dtype=torch.int32, device=dev)
    colidx = torch.empty(cap, dtype=torch.int32, device=dev)
    counts = torch.empty(cap, dtype=torch.int32, device=dev)
    wsum = torch.empty(cap, dtype=torch.float32, device=dev) if w is not None else None
    nnz_out = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = workspace(_lib.query("gdr_coarsen_ws_bytes", E, int(n_src), int(n_dst)), dev)
    _lib.call("gdr_coarsen", E, p_src, p_dst, n_rows, p_rp, p_ci, ptr(w), ptr(ls), ptr(ld), int(n_src),
              int(n_dst), int(drop_diag), ptr(rowptr), ptr(colidx), ptr(counts), ptr(wsum), ptr(nnz_out),
              ptr(ws), ws.numel(), stream())
    m = int(nnz_out.item())
    return rowptr, colidx[:m], counts[:m], (None if wsum is None else wsum[:m])


def _compress_one(adj: Union[CSR, torch.Tensor], labels: torch.Tensor, n: int, sizes: torch.Tensor) -> torch.Tensor:
    A = adj if isinstance(adj, CSR) else CSR.from_torch_coo(adj)
    rowptr, colidx, _counts, wsum = coarsen_edges(labels, labels, n, n, csr=A, weights=A.vals, drop_diag=True)
    vals = torch.empty_like(wsum)
    if wsum.numel():
        _lib.call("gdr_coarsen_scale", n, ptr(rowptr), ptr(colidx), ptr(wsum), ptr(sizes), ptr(sizes),
                  ptr(vals), stream())
    S = CSR(rowptr, colidx, vals, (n, n))
    return S.to_torch_coo()


def graph_compress(cluster_labels: torch.Tensor, adj_norm, adj_list: Sequence) -> Tuple[List[torch.Tensor], torch.Tensor]:
    """clustgdd_agent_transduct.py:234-250.

    S[a, b] = sum_{i in a, j in b} A_ij / (n_a * n_b) for a != b (diagonal removed), returned as
    torch sparse COO n x n with n = cluster_labels.max() + 1 (trailing empty clusters shrink n,
    as in the reference).  One result per graph in ``adj_list`` plus one for ``adj_norm``.
    Every off-diagonal cell with at least one edge is stored: a cell whose weights cancel exactly
    (signed weights, e.g. ``graph_sparse`` outputs) is an explicit 0, where the reference's
    dense ``.to_sparse()`` drops it."""
    dev = adj_norm.device
    labels = cluster_labels.to(device=dev, dtype=torch.int32).contiguous()
    n = int(labels.max().item()) + 1
    sizes = label_counts(labels, n)
    compressed = [_compress_one(a, labels, n, sizes) for a in adj_list]
    adj_syn = _compress_one(adj_norm, labels, n, sizes)
    return compressed, adj_syn


def build_condensed_bipartite(train_u, train_i, u2cu, i2ci, num_cu: int, num_ci: int, device=None,
                              return_device: bool = False):
    """distill_recsys.py:184-201: C[cu, ci] = number of train lines (u, i) with u2cu[u] = cu and
    i2ci[i] = ci.  Returns scipy CSR float32 with integer-valued counts (duplicates counted)."""
    dev = device_of(device)
    u = to_device_i64(train_u, dev)
    i = to_device_i64(train_i, dev)
    mu = to_device_i64(u2cu, dev).to(torch.int32)
    mi = to_device_i64(i2ci, dev).to(torch.int32)
    if u.numel() and (int(u.max()) >= mu.numel() or int(i.max()) >= mi.numel() or int(u.min()) < 0 or int(i.min()) < 0):
        raise IndexError("train_u / train_i index outside the cluster maps")
    if mu.numel() and (int(mu.max()) >= num_cu or int(mu.min()) < 0):
        raise ValueError("row index exceeds matrix dimensions")
    if mi.numel() and (int(mi.max()) >= num_ci or int(mi.min()) < 0):
        raise ValueError("column index exceeds matrix dimensions")
    rowptr, colidx, counts, _ = coarsen_edges(mu, mi, int(num_cu), int(num_ci), src=u, dst=i)
    C = CSR(rowptr, colidx, counts.to(torch.float32), (int(num_cu), int(num_ci)))
    return C if return_device else C.to_scipy()


def condensed_csr_to_edge_index(C, device) -> Tuple[torch.Tensor, torch.Tensor]:
    """distill_recsys.py:387-395: CSR -> (edge_index int64 [2, E], edge_weight f32 [E])."""
    if isinstance(C, CSR):
        return C.coo_indices(), C.vals.clone()
    coo = C.tocoo()
    cu = torch.from_numpy(coo.row.astype(np.int64))
    ci = torch.from_numpy(coo.col.astype(np.int64))
    w = torch.from_numpy(coo.data.astype(np.float32))
    return torch.stack([cu, ci], dim=0).to(device), w.to(device)
