"""numpy model of the row-partitioned top-k of gdr_sparsify_classes_dist.

Each rank holds the weights of its own edges (the blocks in rank order are the global stored order).  Per radix pass
the ranks' 256-bin histograms of the candidates are summed (the all-reduce) and every rank picks the same byte, as
k_seld_pick does.  Once the threshold key T is fixed, each rank counts its ties (entries whose key equals T; the
all-gather) and rank p keeps every entry above T plus its first clamp(k_rem - sum_{q<p} ties_q, 0, ties_p) ties in
stored order.  Keys are the order-preserving image of the fp32 bits (f32_key in sparsify.cu), so NaN sorts above
+inf and -0.0 below +0.0.  The weights come from the oracle's functions on the whole graph, sliced by rank: the
row-block kernels read the same operands and give the same bits.
"""
import numpy as np


def f32_key(w):
    u = np.ascontiguousarray(w, dtype=np.float32).view(np.uint32)
    return np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def row_bounds(n, world):
    """RowPartition's blocks: ceil(n / world) rows each, the last ones short or empty."""
    per = (n + world - 1) // world
    return [min(n, r * per) for r in range(world)] + [n]


def select_dist(blocks, k):
    """Kept local indices of every rank's weight block for the global top-k (ties: first in global stored order)."""
    keys = [f32_key(w) for w in blocks]
    if k == 0:
        return [np.zeros(0, np.int64) for _ in keys]
    prefix, mask, k_rem = 0, 0, int(k)
    for shift in (24, 16, 8, 0):
        hist = np.zeros(256, np.int64)
        for u in keys:                                   # per-rank histograms, summed
            cand = u[(u & np.uint32(mask)) == np.uint32(prefix)]
            hist += np.bincount(((cand >> np.uint32(shift)) & np.uint32(0xFF)).astype(np.int64), minlength=256)
        d = 255
        while d > 0 and hist[d] < k_rem:
            k_rem -= int(hist[d])
            d -= 1
        prefix |= d << shift
        mask |= 0xFF << shift
    T = np.uint32(prefix)
    ties = [int((u == T).sum()) for u in keys]           # all-gathered
    out, before = [], 0
    for p, u in enumerate(keys):
        quota = min(max(k_rem - before, 0), ties[p])
        eq = np.flatnonzero(u == T)[:quota]
        out.append(np.sort(np.concatenate([np.flatnonzero(u > T), eq])).astype(np.int64))
        before += ties[p]
    return out


def select_global(w, k):
    """The kept indices as one array in global stored order (the one-GPU select under the same key order)."""
    u = f32_key(w)
    if k == 0:
        return np.zeros(0, np.int64)
    T = np.sort(u)[u.shape[0] - k]
    gt = np.flatnonzero(u > T)
    return np.sort(np.concatenate([gt, np.flatnonzero(u == T)[: k - gt.shape[0]]])).astype(np.int64)


def concat_kept(kept, edge_bounds):
    """Local kept indices of every rank -> global edge indices (rank p's edges start at edge_bounds[p])."""
    return np.concatenate([kept[p] + edge_bounds[p] for p in range(len(kept))]).astype(np.int64)


def graph_sparse_dist(oracle, rowptr, colidx, vals, ratio, bounds, ebd=None, sp_type="vanilla"):
    """Global kept edge indices of every graph dist_graph_sparse returns, for the row blocks ``bounds`` (rank r owns
    rows [bounds[r], bounds[r+1])), with k = int(total nnz * ratio) as graph_sparse computes it."""
    rowptr = np.asarray(rowptr, np.int64)
    nnz = int(np.asarray(vals).shape[0])
    k = int(nnz * ratio)
    eb = [int(rowptr[b]) for b in bounds]
    if sp_type == "vanilla":
        weights = [oracle.er_lower(rowptr, colidx, vals)]
    else:
        er, _ = oracle.attaw_er_lower(rowptr, colidx, vals, ebd)
        if sp_type == "single":
            weights = [er]
        else:
            P = oracle.softmax_rows(ebd)
            weights = [oracle.class_edge_weight(rowptr, colidx, er, P[:, c]) for c in range(P.shape[1])]
    return [concat_kept(select_dist([w[eb[p]: eb[p + 1]] for p in range(len(bounds) - 1)], k), eb) for w in weights], k
