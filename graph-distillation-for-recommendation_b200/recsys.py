"""Bipartite LightGCN propagation on the GPU kernels (stages 1-2, bipartite form).

Forward semantics of ``LightGCNCondensed.propagate`` (distill_recsys.py:319-353):
    deg_u = sum_e w ; deg_i = sum_e w
    norm  = w / (sqrt(deg_u[cu] + 1e-8) * sqrt(deg_i[ci] + 1e-8))
    L layers of  u <- sum norm * i ,  i <- sum norm * u  (simultaneous), output = layer mean.
The two scatter-adds per layer become two CSR SpMMs (the cu x ci matrix and its
transpose); autograd stays with torch (``BipartitePropagate`` implements the backward
with the transposed SpMMs for the embedding inputs).
"""
from __future__ import annotations

from typing import Dict, Sequence, Tuple

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib
from ._dev import need_cuda, new_padded, padded_rows, ptr, stream, to_device_i64, workspace
from .graph import CSR, coo_to_csr
from .propagation import spmm


class BipartiteGraph:
    """Device CSR of the cu x ci weight matrix, its transpose, and the normalised values."""

    def __init__(self, edge_index: torch.Tensor, edge_weight: torch.Tensor, num_u: int, num_i: int,
                 eps: float = 1e-8):
        need_cuda(edge_index, "edge_index")
        self.num_u, self.num_i = int(num_u), int(num_i)
        W = coo_to_csr(edge_index[0], edge_index[1], edge_weight, (self.num_u, self.num_i),
                       device=edge_index.device)
        WT, t_perm = W.transpose()
        dev = W.device
        self.deg_u = torch.empty(self.num_u, dtype=torch.float32, device=dev)
        self.deg_i = torch.empty(self.num_i, dtype=torch.float32, device=dev)
        norm = torch.empty(W.nnz, dtype=torch.float32, device=dev)
        t_norm = torch.empty(W.nnz, dtype=torch.float32, device=dev)
        _lib.call("gdr_bipartite_normalize", self.num_u, self.num_i, W.nnz, ptr(W.rowptr), ptr(W.colidx),
                  ptr(W.vals), ptr(WT.rowptr), ptr(t_perm), float(eps), ptr(norm), ptr(t_norm),
                  ptr(self.deg_u), ptr(self.deg_i), stream())
        self.A = CSR(W.rowptr, W.colidx, norm, W.shape)        # users <- items
        self.AT = CSR(WT.rowptr, WT.colidx, t_norm, WT.shape)  # items <- users
        self.W = W


def lightgcn_propagate(graph: BipartiteGraph, u0: torch.Tensor, i0: torch.Tensor,
                       num_layers: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Forward of distill_recsys.py:337-353 (no autograd)."""
    u = padded_rows(u0.detach().to(torch.float32))
    it = padded_rows(i0.detach().to(torch.float32))
    d = u.shape[1]
    dev = u.device
    u_acc = new_padded(graph.num_u, d, dev)
    i_acc = new_padded(graph.num_i, d, dev)
    u_acc.copy_(u)
    i_acc.copy_(it)
    for _ in range(int(num_layers)):
        u_next = spmm(graph.A, it, accumulate_into=u_acc, beta=1.0)
        i_next = spmm(graph.AT, u, accumulate_into=i_acc, beta=1.0)
        u, it = u_next, i_next
    inv = 1.0 / float(num_layers + 1)
    u_out = new_padded(graph.num_u, d, dev)
    i_out = new_padded(graph.num_i, d, dev)
    _lib.call("gdr_scale_rows", graph.num_u, d, inv, ptr(u_acc), u_acc.stride(0), ptr(u_out), u_out.stride(0), stream())
    _lib.call("gdr_scale_rows", graph.num_i, d, inv, ptr(i_acc), i_acc.stride(0), ptr(i_out), i_out.stride(0), stream())
    return u_out, i_out


class RankformerGCNGraph:
    """CSR of the raw user-item interactions with the Rankformer GCN weights
    (Rankformer/code/rec.py:92-140): du / di = interaction counts clamped to >= 1,
    w1 = 1/du^alpha/di^beta (items -> users), w2 = 1/du^beta/di^alpha (users -> items).
    Duplicate (u, i) lines are summed into the CSR value, which is what scattering every line
    separately adds up to."""

    def __init__(self, u: torch.Tensor, i: torch.Tensor, num_users: int, num_items: int, alpha: float = 1.0,
                 beta: float = 0.0):
        need_cuda(u, "u")
        self.n, self.m = int(num_users), int(num_items)
        R = coo_to_csr(u, i, None, (self.n, self.m), device=u.device)
        RT, t_perm = R.transpose()
        dev = R.device
        self.deg_u = torch.empty(self.n, dtype=torch.float32, device=dev)
        self.deg_i = torch.empty(self.m, dtype=torch.float32, device=dev)
        w1 = torch.empty(R.nnz, dtype=torch.float32, device=dev)
        w2t = torch.empty(R.nnz, dtype=torch.float32, device=dev)
        scratch = torch.empty(max(R.nnz, 1), dtype=torch.float32, device=dev)
        _lib.call("gdr_bipartite_pow_normalize", self.n, self.m, R.nnz, ptr(R.rowptr), ptr(R.colidx), ptr(R.vals),
                  ptr(RT.rowptr), ptr(t_perm), float(alpha), float(beta), ptr(w1), ptr(w2t), ptr(self.deg_u),
                  ptr(self.deg_i), ptr(scratch), stream())
        self.A = CSR(R.rowptr, R.colidx, w1, R.shape)         # zu = A @ xi
        self.AT = CSR(RT.rowptr, RT.colidx, w2t, RT.shape)    # zi = AT @ xu


def rankformer_gcn_forward(graph: RankformerGCNGraph, x: torch.Tensor) -> torch.Tensor:
    """GCN.forward of Rankformer/code/rec.py:92-140: x = [users; items] -> [zu; zi]."""
    xu, xi = x[: graph.n], x[graph.n:]
    zu = spmm(graph.A, xi.contiguous())
    zi = spmm(graph.AT, xu.contiguous())
    return torch.cat([zu, zi], dim=0)


class BipartitePropagate(torch.autograd.Function):
    """Differentiable (w.r.t. the embeddings) wrapper: the backward of a layer-mean of
    alternating SpMMs is the same propagation with A and A^T swapped."""

    @staticmethod
    def forward(ctx, u0, i0, graph: BipartiteGraph, num_layers: int):
        ctx.graph, ctx.num_layers = graph, int(num_layers)
        return lightgcn_propagate(graph, u0, i0, num_layers)

    @staticmethod
    def backward(ctx, gu, gi):
        # out_u = mean_l U_l with U_{l+1} = A I_l, I_{l+1} = A^T U_l.  The adjoint recursion is
        # the same alternating propagation applied to (gu, gi) because [[0, A], [A^T, 0]] is symmetric.
        du, di = lightgcn_propagate(ctx.graph, gu.contiguous(), gi.contiguous(), ctx.num_layers)
        return du, di, None, None


# ---------------------------------------------------------------------------------------------------------------
# evaluation: full-ranking top-K and Recall / Precision / NDCG@K (distill_recsys.py:446-497 recall_at_k, called at
# :680 and :733; Rankformer/code/model.py:27-53).  The definitions are this library's (see include/gdr.h).
# ---------------------------------------------------------------------------------------------------------------
def _as_csr(m, shape, name: str, device) -> CSR:
    """gdr.CSR, torch sparse tensor or scipy sparse matrix -> device CSR of the given shape (duplicates summed)."""
    if isinstance(m, CSR):
        csr = m
    elif isinstance(m, torch.Tensor) and m.layout in (torch.sparse_coo, torch.sparse_csr):
        csr = CSR.from_torch_coo((m if m.layout == torch.sparse_coo else m.to_sparse_coo()).to(device))
    elif sp.issparse(m):
        csr = CSR.from_scipy(m, device=device)
    else:
        raise TypeError(f"{name} must be a gdr.CSR, a torch sparse tensor or a scipy sparse matrix")
    if tuple(csr.shape) != tuple(shape):
        raise ValueError(f"{name} has shape {tuple(csr.shape)}, expected {tuple(shape)}")
    if csr.device != device:
        raise ValueError(f"{name} lives on {csr.device}, the embeddings on {device}")
    return csr


def _rows_arg(rows, n_users: int, device):
    if rows is None:
        return None, n_users
    r = to_device_i64(rows, device).reshape(-1)
    return r, int(r.shape[0])


def recommend_topk(user_emb: torch.Tensor, item_emb: torch.Tensor, k: int, exclude=None,
                   rows=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Full-ranking top-k items per user: ``(scores [n_rows, k] f32, items [n_rows, k] int64)``.

    Row r is user ``rows[r]`` (user ids, int64; default: every user in order) and uses ``user_emb[rows[r]]`` and
    exclusion row ``rows[r]``.  The score of item j is the fp32 chain ``fmaf(u[t], i[t], acc)`` over t in order;
    items come by score descending, then item index ascending.  Items stored in ``exclude`` (n_users x n_items:
    a ``gdr.CSR``, torch sparse tensor or scipy sparse matrix, normally the training interactions) never appear;
    duplicate entries are summed by the CSR build and make no difference.  A row with fewer than k eligible items
    is padded with item -1 and score -inf.  The result is deterministic and identical on every run.
    Raises ValueError for non-finite embeddings or user ids out of range.  No autograd."""
    need_cuda(user_emb, "user_emb")
    need_cuda(item_emb, "item_emb")
    if user_emb.dim() != 2 or item_emb.dim() != 2 or user_emb.shape[1] != item_emb.shape[1]:
        raise ValueError("user_emb [n_users, d] and item_emb [n_items, d] need the same d")
    U = user_emb.detach().to(torch.float32).contiguous()
    I = item_emb.detach().to(torch.float32).contiguous()
    n_users, d = U.shape
    n_items = I.shape[0]
    k = int(k)
    if not 1 <= k <= n_items:
        raise ValueError(f"k={k} must lie in [1, n_items={n_items}]")
    dev = U.device
    if I.device != dev:
        raise ValueError("user_emb and item_emb must be on the same device")
    ex = None if exclude is None else _as_csr(exclude, (n_users, n_items), "exclude", dev)
    rows_d, n_rows = _rows_arg(rows, n_users, dev)
    scores = torch.empty((n_rows, k), dtype=torch.float32, device=dev)
    items = torch.empty((n_rows, k), dtype=torch.int32, device=dev)
    if n_rows == 0:
        return scores, items.long()
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = workspace(_lib.query("gdr_topk_scores_ws_bytes", n_rows, n_items, d, k), dev)
    _lib.call("gdr_topk_scores", n_rows, n_users, n_items, d, k, ptr(U), U.stride(0), ptr(rows_d), ptr(I), I.stride(0),
              ptr(ex.rowptr) if ex is not None else 0, ptr(ex.colidx) if ex is not None else 0,
              ptr(scores), k, ptr(items), k, ptr(status), ptr(ws), ws.numel(), stream())
    st = int(status.item())
    if st & 1:
        raise ValueError("recommend_topk: user_emb or item_emb holds a non-finite value")
    if st & 2:
        raise ValueError(f"recommend_topk: a user id in rows lies outside [0, {n_users})")
    return scores, items.long()


def ranking_metrics(items: torch.Tensor, test, ks: Sequence[int] = (20,), rows=None) -> Dict[str, float]:
    """Recall@K, Precision@K and NDCG@K of a top-k list (``recommend_topk``'s ``items``) against held-out items.

    ``test`` is the n_users x n_items test interaction matrix (``gdr.CSR``, torch sparse or scipy sparse; duplicates
    are summed by the CSR build and make no difference); n_items is taken from it.  ``rows`` must be the user ids
    the top-k list was computed for (default: row r is user r).  Per user with a non-empty test row and each K:
    hits = top-K items in the test row, recall = hits / |test_u|, precision = hits / K,
    ndcg = sum over hit ranks i < K of 1/log2(i+2) / sum_{i < min(K, |test_u|)} 1/log2(i+2).  Users with an empty
    test row are skipped (``n_skipped``).  Means are fp64 sums in ascending row order / ``n_eval``: deterministic.
    Every K must be <= k; all of them come from the one list, each reading a prefix of it."""
    need_cuda(items, "items")
    if items.dim() != 2:
        raise ValueError("items must be [n_rows, k]")
    dev = items.device
    n_rows, k = items.shape
    ks = [int(x) for x in ks]
    if not ks or any(not 1 <= x <= k for x in ks):
        raise ValueError(f"every K in ks must lie in [1, k={k}]")
    n_users = int(test.shape[0])
    tcsr = _as_csr(test, (n_users, int(test.shape[1])), "test", dev)
    rows_d, nr = _rows_arg(rows, n_users, dev)
    if nr != n_rows:
        raise ValueError(f"rows has {nr} entries, items has {n_rows} rows")
    if rows_d is not None and n_rows and bool(((rows_d < 0) | (rows_d >= n_users)).any()):
        raise ValueError(f"a user id in rows lies outside [0, {n_users})")
    it = items.to(torch.int32).contiguous()
    out = {}
    if n_rows == 0:
        for K in ks:
            out.update({f"recall@{K}": float("nan"), f"precision@{K}": float("nan"), f"ndcg@{K}": float("nan")})
        out.update(n_eval=0, n_skipped=0)
        return out
    sums = torch.zeros(3 * len(ks), dtype=torch.float64, device=dev)
    n_eval = torch.zeros(1, dtype=torch.int64, device=dev)
    ks_host = np.ascontiguousarray(ks, dtype=np.int32)
    ws = workspace(_lib.query("gdr_ranking_metrics_ws_bytes", n_rows, len(ks)), dev)
    _lib.call("gdr_ranking_metrics", n_rows, n_users, k, ptr(it), it.stride(0), ptr(rows_d), ptr(tcsr.rowptr),
              ptr(tcsr.colidx), len(ks), ks_host.ctypes.data, ptr(sums), ptr(n_eval), 0, ptr(ws), ws.numel(), stream())
    s = sums.cpu().numpy()
    ne = int(n_eval.item())
    for q, K in enumerate(ks):
        for m, name in enumerate(("recall", "precision", "ndcg")):
            out[f"{name}@{K}"] = float(s[3 * q + m] / ne) if ne else float("nan")
    out.update(n_eval=ne, n_skipped=n_rows - ne)
    return out
