"""Bipartite LightGCN propagation on the GPU kernels (stages 1-2, bipartite form).

Forward semantics of ``LightGCNCondensed.propagate`` (distill_recsys.py:319-353):
    deg_u = sum_e w ; deg_i = sum_e w
    norm  = w / (sqrt(deg_u[cu] + 1e-8) * sqrt(deg_i[ci] + 1e-8))
    L layers of  u <- sum norm * i ,  i <- sum norm * u  (simultaneous), output = layer mean.
The two scatter-adds per layer become two CSR SpMMs (the cu x ci matrix and its
transpose).  ``BipartitePropagate`` is differentiable w.r.t. the embeddings;
``LightGCNPropagate`` also w.r.t. the edge weights (the condensed model's trained weights),
on a graph that is built once and reweighted in place every step.  ``BPRSampler`` and ``bpr_loss`` are the rest of a
refinement step (triplet sampling, BPR loss and its gradient) on the device.
"""
from __future__ import annotations

from typing import Dict, Sequence, Tuple

import numpy as np
import scipy.sparse as sp
import torch
from torch.autograd.function import once_differentiable

from . import _lib
from ._dev import device_of, need_cuda, new_padded, pad4, padded_rows, ptr, stream, to_device_i64, workspace
from .graph import CSR, coo_to_csr
from .propagation import spmm


class BipartiteGraph:
    """Device CSR of the cu x ci weight matrix, its transpose, and the normalised values.

    ``set_edge_weight`` replaces the weights (in the order of ``edge_index``) and renormalises in place, keeping the
    sparsity pattern: the refinement loop builds the graph once and reweights it every step."""

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
        self.A = CSR(W.rowptr, W.colidx, norm, W.shape)        # users <- items
        self.AT = CSR(WT.rowptr, WT.colidx, t_norm, WT.shape)  # items <- users
        self.W = W
        self.eps = float(eps)
        self.t_perm = t_perm                # position in W of every entry of the transpose
        self._edge_index = edge_index
        self._edge_pos = None               # int32 [E]: CSR position of every input edge (first set_edge_weight)
        self._edge_pos_i64 = None
        self._normalize()

    def _normalize(self) -> None:
        """deg_u, deg_i, A.vals and AT.vals from W.vals (gdr_bipartite_normalize), into the existing buffers."""
        W = self.W
        _lib.call("gdr_bipartite_normalize", self.num_u, self.num_i, W.nnz, ptr(W.rowptr), ptr(W.colidx),
                  ptr(W.vals), ptr(self.AT.rowptr), ptr(self.t_perm), self.eps, ptr(self.A.vals), ptr(self.AT.vals),
                  ptr(self.deg_u), ptr(self.deg_i), stream())

    @property
    def num_edges(self) -> int:
        return int(self._edge_index.shape[1])

    def edge_positions(self) -> torch.Tensor:
        """int32 [E]: position in the CSR of every edge of ``edge_index`` (computed once, on first use).
        Raises ValueError when ``edge_index`` repeats a (u, i) pair: the CSR then holds their sum, and a weight per
        input edge has no entry of its own."""
        if self._edge_pos is None:
            E, W = self.num_edges, self.W
            if W.nnz != E:
                raise ValueError(f"edge_index repeats a (u, i) pair ({E} edges, {W.nnz} distinct pairs): per-edge "
                                 "weights need unique pairs")
            dev = W.device
            pos = torch.empty(E, dtype=torch.int32, device=dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            row = to_device_i64(self._edge_index[0], dev)
            col = to_device_i64(self._edge_index[1], dev)
            _lib.call("gdr_csr_locate", self.num_u, self.num_i, W.nnz, ptr(W.rowptr), ptr(W.colidx), E, ptr(row),
                      ptr(col), ptr(pos), ptr(status), stream())
            if int(status.item()):
                raise RuntimeError("edge_index holds a pair the graph does not store (was it modified in place?)")
            self._edge_pos, self._edge_pos_i64 = pos, pos.long()
        return self._edge_pos

    def set_edge_weight(self, edge_weight: torch.Tensor) -> None:
        """New edge weights, f32 [E] in the order of the ``edge_index`` the graph was built from: scattered to CSR
        order, then deg_u, deg_i, A.vals and AT.vals are recomputed in place (no sort, no transpose).  The result is
        bit-identical to a new ``BipartiteGraph(edge_index, edge_weight, ...)``.  No autograd (see
        ``LightGCNPropagate``)."""
        need_cuda(edge_weight, "edge_weight")
        w = edge_weight.detach().to(torch.float32).reshape(-1)
        if w.shape[0] != self.num_edges:
            raise ValueError(f"edge_weight has {w.shape[0]} entries, the graph {self.num_edges} edges")
        self.edge_positions()
        if self.num_edges:
            self.W.vals.index_copy_(0, self._edge_pos_i64, w)
        self._normalize()


def _layer_loop(A: CSR, AT: CSR, u0: torch.Tensor, i0: torch.Tensor, num_layers: int, keep: bool = False):
    """Layer loop of distill_recsys.py:337-353 on the normalised matrices A (users <- items) and AT.

    Returns (u_out, i_out, Xu, Xi).  With ``keep`` (and L > 0), Xu / Xi are the layers X_0 .. X_{L-1} stacked as
    [L, n, pad4(d)] f32 (zero padding columns), written by the SpMMs themselves; else None.  Keeping them changes
    no SpMM call: the outputs are the same bits either way."""
    u = padded_rows(u0.detach().to(torch.float32))
    it = padded_rows(i0.detach().to(torch.float32))
    n_u, n_i = A.shape
    d = u.shape[1]
    dev = u.device
    L = int(num_layers)
    Xu = Xi = None
    if keep and L > 0:
        alloc = torch.empty if pad4(d) == d else torch.zeros
        Xu = alloc((L, n_u, pad4(d)), dtype=torch.float32, device=dev)
        Xi = alloc((L, n_i, pad4(d)), dtype=torch.float32, device=dev)
        Xu[0, :, :d].copy_(u)
        Xi[0, :, :d].copy_(it)
        u, it = Xu[0, :, :d], Xi[0, :, :d]
    u_acc = new_padded(n_u, d, dev)
    i_acc = new_padded(n_i, d, dev)
    u_acc.copy_(u)
    i_acc.copy_(it)
    for l in range(L):
        keep_next = Xu is not None and l + 1 < L
        if A.nnz == 0:   # no edges: every propagated layer is zero (the SpMM entry point takes no empty CSR)
            u_next = Xu[l + 1, :, :d].zero_() if keep_next else new_padded(n_u, d, dev, zero=True)
            i_next = Xi[l + 1, :, :d].zero_() if keep_next else new_padded(n_i, d, dev, zero=True)
        else:
            u_next = spmm(A, it, out=Xu[l + 1, :, :d] if keep_next else None, accumulate_into=u_acc, beta=1.0)
            i_next = spmm(AT, u, out=Xi[l + 1, :, :d] if keep_next else None, accumulate_into=i_acc, beta=1.0)
        u, it = u_next, i_next
    inv = 1.0 / float(L + 1)
    u_out = new_padded(n_u, d, dev)
    i_out = new_padded(n_i, d, dev)
    _lib.call("gdr_scale_rows", n_u, d, inv, ptr(u_acc), u_acc.stride(0), ptr(u_out), u_out.stride(0), stream())
    _lib.call("gdr_scale_rows", n_i, d, inv, ptr(i_acc), i_acc.stride(0), ptr(i_out), i_out.stride(0), stream())
    return u_out, i_out, Xu, Xi


def lightgcn_propagate(graph: BipartiteGraph, u0: torch.Tensor, i0: torch.Tensor,
                       num_layers: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Forward of distill_recsys.py:337-353 (no autograd)."""
    u_out, i_out, _, _ = _layer_loop(graph.A, graph.AT, u0, i0, num_layers)
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


class LightGCNPropagate(torch.autograd.Function):
    """``u_out, i_out = LightGCNPropagate.apply(u0, i0, edge_weight, graph, num_layers)``: the condensed model's
    propagation (distill_recsys.py:319-353) differentiable w.r.t. the embeddings AND the edge weights.

    ``edge_weight`` is f32 [E] in the order of the graph's ``edge_index`` (``model.edge_weight()``); the forward
    reweights ``graph`` in place (``set_edge_weight``) and runs the layer loop of ``lightgcn_propagate`` (same bits).
    It keeps its own copy of the normalised values and degrees, so reweighting the graph again before ``backward``
    (a second forward, say) does not change this call's gradients.  Backward: the adjoint propagation gives
    d u0 / d i0 (the same calls as ``BipartitePropagate``), then gdr_lightgcn_edge_grad and
    gdr_bipartite_normalize_backward give d edge_weight.  Deterministic; no double backward."""

    @staticmethod
    def forward(ctx, u0, i0, edge_weight, graph: BipartiteGraph, num_layers: int):
        L = int(num_layers)
        if L < 0:
            raise ValueError("num_layers must be >= 0")
        if u0.dim() != 2 or i0.dim() != 2 or u0.shape[1] != i0.shape[1]:
            raise ValueError("u0 [num_u, d] and i0 [num_i, d] need the same d")
        if u0.shape[0] != graph.num_u or i0.shape[0] != graph.num_i:
            raise ValueError(f"u0 / i0 have {u0.shape[0]} / {i0.shape[0]} rows, the graph {graph.num_u} / {graph.num_i}")
        graph.set_edge_weight(edge_weight)
        A, AT = graph.A, graph.AT
        ctx.A = CSR(A.rowptr, A.colidx, A.vals.clone(), A.shape, _plan=A.spmm_plan())
        ctx.AT = CSR(AT.rowptr, AT.colidx, AT.vals.clone(), AT.shape, _plan=AT.spmm_plan())
        ctx.deg_u, ctx.deg_i = graph.deg_u.clone(), graph.deg_i.clone()
        ctx.graph, ctx.num_layers, ctx.w_dtype = graph, L, edge_weight.dtype
        u_out, i_out, ctx.Xu, ctx.Xi = _layer_loop(ctx.A, ctx.AT, u0, i0, L, keep=ctx.needs_input_grad[2])
        return u_out, i_out

    @staticmethod
    @once_differentiable
    def backward(ctx, gu, gi):
        need_w = ctx.needs_input_grad[2]
        du, di, Yu, Yi = _layer_loop(ctx.A, ctx.AT, gu.contiguous(), gi.contiguous(), ctx.num_layers, keep=need_w)
        dw = _edge_weight_grad(ctx, Yu, Yi, du.shape[1]).to(ctx.w_dtype) if need_w else None
        ctx.Xu = ctx.Xi = None
        return du, di, dw, None, None


def _edge_weight_grad(ctx, Yu, Yi, d: int) -> torch.Tensor:
    """dL/dw [E] in input edge order from the kept forward layers (ctx.Xu, ctx.Xi) and adjoint layers (Yu, Yi)."""
    g, A, AT, L = ctx.graph, ctx.A, ctx.AT, ctx.num_layers
    E, nnz = g.num_edges, A.nnz
    dev = A.device
    dw = torch.empty(E, dtype=torch.float32, device=dev)
    if E == 0:
        return dw
    G = torch.empty(nnz, dtype=torch.float32, device=dev)
    S_u = torch.empty(g.num_u, dtype=torch.float64, device=dev)
    _lib.call("gdr_lightgcn_edge_grad", g.num_u, g.num_i, nnz, ptr(A.rowptr), ptr(A.colidx), ptr(A.vals), L, d,
              ptr(ctx.Xu), ptr(ctx.Xi), ptr(Yu), ptr(Yi), pad4(d), 1.0 / float(L + 1), ptr(G), ptr(S_u), stream())
    ws = workspace(_lib.query("gdr_bipartite_normalize_backward_ws_bytes", g.num_i, nnz), dev)
    _lib.call("gdr_bipartite_normalize_backward", g.num_u, g.num_i, nnz, ptr(A.rowptr), ptr(A.colidx),
              ptr(AT.rowptr), ptr(g.t_perm), ptr(A.vals), ptr(ctx.deg_u), ptr(ctx.deg_i), g.eps, ptr(G), ptr(S_u), E,
              ptr(g.edge_positions()), ptr(dw), ptr(ws), ws.numel(), stream())
    return dw


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


def _map_arg(m, n_values: int, name: str, device) -> torch.Tensor:
    """user_map / item_map (torch or numpy, int32 or int64, 1-D) -> int64 device tensor; range checked on the device."""
    dt = m.dtype if isinstance(m, (torch.Tensor, np.ndarray)) else None
    if dt not in (torch.int32, torch.int64, np.dtype(np.int32), np.dtype(np.int64)):
        raise ValueError(f"{name} must be an int32 or int64 torch tensor or numpy array")
    if m.ndim != 1:
        raise ValueError(f"{name} must be 1-D")
    if n_values == 0 and m.shape[0]:
        raise ValueError(f"{name} has values but its embedding table has no rows")
    return to_device_i64(m, device)


def recommend_topk_condensed(user_emb: torch.Tensor, item_emb: torch.Tensor, k: int, user_map, item_map,
                             exclude=None, rows=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """``recommend_topk`` of a condensed model, from its cluster tables: ``(scores [n_rows, k] f32, items [n_rows, k]
    int64)``, byte-identical to ``recommend_topk(user_emb[user_map], item_emb[item_map], k, exclude, rows)``.

    ``user_emb`` [n_cu, d] and ``item_emb`` [n_ci, d] are the super-user and super-item rows (``LightGCNPropagate``'s
    outputs, say); ``user_map`` [n_users] and ``item_map`` [n_items] (``u2cu``, ``i2ci``: int32 or int64, torch or
    numpy) give every original user and item its row.  ``exclude`` (n_users x n_items) and ``rows`` are those of
    ``recommend_topk``, and item ids are original ids, so the result feeds ``ranking_metrics`` unchanged.  Only the
    n_cu x n_ci distinct scores are computed; rows whose ranking hits a tie of more than 32 clusters (a zero
    super-user) are finished on ``recommend_topk``'s exact path.  Raises ValueError for a non-finite value in a
    super-user row an evaluated row uses or in a super-item row with a member, for user ids or map values out of
    range, and for k outside [1, n_items].  Synchronises; no autograd."""
    need_cuda(user_emb, "user_emb")
    need_cuda(item_emb, "item_emb")
    if user_emb.dim() != 2 or item_emb.dim() != 2 or user_emb.shape[1] != item_emb.shape[1]:
        raise ValueError("user_emb [n_cu, d] and item_emb [n_ci, d] need the same d")
    U = user_emb.detach().to(torch.float32).contiguous()
    I = item_emb.detach().to(torch.float32).contiguous()
    dev = U.device
    if I.device != dev:
        raise ValueError("user_emb and item_emb must be on the same device")
    n_cu, d = U.shape
    n_ci = I.shape[0]
    um = _map_arg(user_map, n_cu, "user_map", dev)
    im = _map_arg(item_map, n_ci, "item_map", dev)
    n_users, n_items = int(um.shape[0]), int(im.shape[0])
    k = int(k)
    if not 1 <= k <= n_items:
        raise ValueError(f"k={k} must lie in [1, n_items={n_items}]")
    if d == 0:
        raise ValueError("the embeddings need d >= 1")
    ex = None if exclude is None else _as_csr(exclude, (n_users, n_items), "exclude", dev)
    rows_d, n_rows = _rows_arg(rows, n_users, dev)
    scores = torch.empty((n_rows, k), dtype=torch.float32, device=dev)
    items = torch.empty((n_rows, k), dtype=torch.int32, device=dev)
    if n_rows == 0:
        return scores, items.long()
    if n_users == 0:
        raise ValueError("recommend_topk_condensed: rows given but user_map is empty")
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = workspace(_lib.query("gdr_topk_condensed_ws_bytes", n_rows, n_users, n_items, n_cu, n_ci, d, k), dev)
    _lib.call("gdr_topk_condensed", n_rows, n_users, n_items, n_cu, n_ci, d, k, ptr(U), U.stride(0), ptr(I),
              I.stride(0), ptr(um), ptr(im), ptr(rows_d), ptr(ex.rowptr) if ex is not None else 0,
              ptr(ex.colidx) if ex is not None else 0, ptr(scores), k, ptr(items), k, ptr(status), ptr(ws), ws.numel(),
              stream())
    st = int(status.item())
    if st & 4:
        raise ValueError(f"recommend_topk_condensed: a user_map value outside [0, {n_cu}) or an item_map value "
                         f"outside [0, {n_ci})")
    if st & 2:
        raise ValueError(f"recommend_topk_condensed: a user id in rows lies outside [0, {n_users})")
    if st & 1:
        raise ValueError("recommend_topk_condensed: user_emb or item_emb holds a non-finite value in a used row")
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


# ---------------------------------------------------------------------------------------------------------------
# BPR training step (distill_recsys.py:684-733): device triplet sampler and the fused BPR loss + gradient
# ---------------------------------------------------------------------------------------------------------------
_BPR_MAX_BATCH = (1 << 31) // 3


class BPRSampler:
    """(user, positive, negative) triplets drawn on the device (``gdr_bpr_sample``).

    ``R`` is the n_users x n_items interaction matrix (``gdr.CSR`` with sorted, unique columns per row, a torch sparse
    tensor or a scipy sparse matrix; values are ignored: a positive is a distinct stored item), e.g.
    ``BipartiteGraph.W``, the condensed CSR of ``build_condensed_bipartite(..., return_device=True)`` or the full
    training CSR.  A user is eligible when 0 < deg(u) < n_items.  Triplet b of a step: user uniform over the eligible
    users, positive uniform over the user's row, negative uniform over the items outside it (the distribution of
    LightGCN's rejection sampler, drawn without rejection).  Random numbers: Philox4x32-10 keyed by ``seed`` with
    counter (b, step, j, 0), so a step is a pure function of (R, seed, step): identical on every run and every GPU,
    and any step can be regenerated on its own (``tests/bpr_ref.py`` mirrors it bit for bit).

    The constructor checks the columns and builds the eligible list once (a few synchronisations, at construction only); raises ValueError
    when no user is eligible.  ``sample`` does not synchronise."""

    def __init__(self, R, seed: int):
        if isinstance(R, CSR):
            dev = R.device
        elif isinstance(R, torch.Tensor) and R.is_cuda:
            dev = R.device
        else:
            dev = device_of(None)
        self.R = _as_csr(R, tuple(R.shape), "R", dev)
        self.seed = int(seed)
        if not 0 <= self.seed < 1 << 64:
            raise ValueError("seed must lie in [0, 2^64)")
        n_users, n_items = (int(x) for x in self.R.shape)
        rowptr, colidx = self.R.rowptr, self.R.colidx
        deg = (rowptr[1:] - rowptr[:-1]).to(torch.int64)
        if self.R.nnz:
            row = torch.repeat_interleave(torch.arange(n_users, device=dev), deg)
            c = colidx.to(torch.int64)
            bad = bool(((c < 0) | (c >= n_items)).any())
            if self.R.nnz > 1:
                bad |= bool(((c[1:] <= c[:-1]) & (row[1:] == row[:-1])).any())
            if bad:
                raise ValueError("R needs column indices in [0, n_items), sorted and unique inside each row")
        self.eligible = torch.nonzero((deg > 0) & (deg < n_items)).reshape(-1).to(torch.int32)
        self.n_eligible = int(self.eligible.shape[0])
        if self.n_eligible == 0:
            raise ValueError("no user is eligible for BPR sampling (every user has no item or every item)")

    def sample(self, batch_size: int, step: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """``(users, pos, neg)``: three int64 device tensors of length ``batch_size`` (in [1, 2^31/3]) for ``step``
        (in [0, 2^32))."""
        B, step = int(batch_size), int(step)
        if not 1 <= B <= _BPR_MAX_BATCH:
            raise ValueError(f"batch_size={B} must lie in [1, {_BPR_MAX_BATCH}]")
        if not 0 <= step < 1 << 32:
            raise ValueError(f"step={step} must lie in [0, 2^32)")
        R, dev = self.R, self.R.device
        out = torch.empty((3, B), dtype=torch.int64, device=dev)
        _lib.call("gdr_bpr_sample", R.shape[0], R.shape[1], ptr(R.rowptr), ptr(R.colidx), self.n_eligible,
                  ptr(self.eligible), self.seed, step, B, ptr(out[0]), ptr(out[1]), ptr(out[2]), stream())
        return out[0], out[1], out[2]


def _bpr_operand(x: torch.Tensor, name: str) -> torch.Tensor:
    need_cuda(x, name)
    if x.dim() != 2:
        raise ValueError(f"{name} must be [rows, d]")
    return padded_rows(x.detach().to(torch.float32))   # LightGCNPropagate's padded outputs pass without a copy


def _bpr_forward(U, I, users, pos, neg, want_gU: bool, want_gI: bool):
    Uf, If = _bpr_operand(U, "U"), _bpr_operand(I, "I")
    if Uf.shape[1] != If.shape[1]:
        raise ValueError("U [n_u, d] and I [n_i, d] need the same d")
    dev = Uf.device
    if If.device != dev:
        raise ValueError("U and I must be on the same device")
    n_u, d = Uf.shape
    n_i = If.shape[0]
    t = [to_device_i64(x, dev).reshape(-1) for x in (users, pos, neg)]
    B = int(t[0].shape[0])
    if t[1].shape[0] != B or t[2].shape[0] != B:
        raise ValueError("users, pos and neg need the same length")
    if B == 0:
        raise ValueError("bpr_loss needs at least one triplet")
    if B > _BPR_MAX_BATCH:
        raise ValueError(f"bpr_loss takes at most {_BPR_MAX_BATCH} triplets")
    if n_u == 0 or n_i == 0 or d == 0:
        raise ValueError("bpr_loss needs n_u, n_i and d >= 1")
    loss = torch.empty((), dtype=torch.float32, device=dev)
    gU = new_padded(n_u, d, dev) if want_gU else None
    gI = new_padded(n_i, d, dev) if want_gI else None
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = workspace(_lib.query("gdr_bpr_loss_ws_bytes", B, n_u, n_i), dev)
    _lib.call("gdr_bpr_loss", B, n_u, n_i, d, ptr(Uf), Uf.stride(0), ptr(If), If.stride(0), ptr(t[0]), ptr(t[1]),
              ptr(t[2]), ptr(loss), ptr(gU), gU.stride(0) if gU is not None else 0, ptr(gI),
              gI.stride(0) if gI is not None else 0, ptr(status), ptr(ws), ws.numel(), stream())
    st = int(status.item())
    if st & 1:
        raise ValueError(f"bpr_loss: a user id outside [0, {n_u}) or an item id outside [0, {n_i})")
    if st & 2:
        raise ValueError("bpr_loss: U or I holds a non-finite value in a row a triplet uses")
    return loss, gU, gI


class BPRLoss(torch.autograd.Function):
    """``loss = BPRLoss.apply(U, I, users, pos, neg)``: ``mean_b softplus(-x_b)`` with
    ``x_b = <U[u_b], I[p_b]> - <U[u_b], I[n_b]>`` (``-logsigmoid(x).mean()``), fused in ``gdr_bpr_loss``.

    ``U`` [n_u, d] and ``I`` [n_i, d] are typically ``LightGCNPropagate``'s outputs (padded strides are read in
    place); the triplets are int64 ids (``BPRSampler.sample``).  The forward computes the gradients too when an
    input needs them; backward scales them by the incoming scalar on the device (exact when it is 1).  Every sum has
    a fixed order: the loss and the gradients are bit-identical from run to run.  Raises ValueError for no triplets,
    ids out of range or a non-finite value in a used row (reading the status synchronises once per call).
    Once-differentiable.  No regularisation term: add it on the ego embeddings in torch."""

    @staticmethod
    def forward(ctx, U, I, users, pos, neg):
        loss, ctx.gU, ctx.gI = _bpr_forward(U, I, users, pos, neg, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        gU = ctx.gU * g if ctx.gU is not None else None
        gI = ctx.gI * g if ctx.gI is not None else None
        ctx.gU = ctx.gI = None
        return gU, gI, None, None, None


def bpr_loss(U: torch.Tensor, I: torch.Tensor, users, pos, neg) -> torch.Tensor:
    """``BPRLoss.apply(U, I, users, pos, neg)``: the fused BPR loss, differentiable w.r.t. ``U`` and ``I``."""
    return BPRLoss.apply(U, I, users, pos, neg)
