"""CPU reference of stage 4's cell sums (csrc/graph.cu: gdr_coarsen, gdr_coarse_merge_edges[_dense], gdr_coarsen_scale):
exact per-cell counts and sums, the per-cluster fixed-point step of the shared-memory form, and the error bound each
form meets.  Test infrastructure only; the library never imports it.

Forms and their bounds, with u = 2^-24, S the exact cell sum and n the cell's edge count:
  shared-memory form  every term rounded to a multiple of the cluster's step q_a, summed exactly as a 64-bit integer,
                      converted through fp64 to fp32:   |got - S| <= n*q_a/2 + 2^-52*(|S| + n*q_a/2) + ulp32(...)/2.
                      Where n*q_a/2 <= ulp32(S)/4 this is within one ulp of fl32(S); for a cell small next to the
                      cluster's largest weight it is not (q_a is about 2^-48 of that weight, not of the cell).
  sort form           fp32 sums in a fixed order (sequential, or the 256-thread tree of k_long_runs):
                      |got - S| <= gamma_{n-1} * sum |w|.
  coarsen_scale       fl(fl(s * fl(1/n_a)) * fl(1/n_b)): four roundings on top of the cell's error."""
import math

import numpy as np

U = 2.0 ** -24
SMEM_BYTES = 200 * 1024          # dynamic shared memory of one coarse row (cd_applicable)


def step(wmax, n_edges) -> int:
    """Exponent e of the fixed-point step q_a = 2^e of a cluster whose nodes' adjacency rows hold n_edges edges
    (diagonal included, as k_cd_stats counts them) of largest |w| wmax: wmax < 2^ew, n_edges < 2^ee, e = ew + ee - 62."""
    ew = int(np.frexp(np.float32(wmax))[1])
    ee = int(np.frexp(float(max(int(n_edges), 1)))[1])
    return ew + ee - 62


def cluster_stats(rowptr, w, labels, n_src):
    """(edges int64 [n_src], max |w| float32 [n_src]) over the adjacency rows of each cluster's nodes (k_cd_stats)."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    labels = np.asarray(labels, dtype=np.int64)
    edges = np.bincount(labels, weights=np.diff(rowptr), minlength=n_src).astype(np.int64)
    wmax = np.zeros(n_src, dtype=np.float32)
    rows = np.repeat(np.arange(rowptr.shape[0] - 1), np.diff(rowptr))
    np.maximum.at(wmax, labels[rows], np.abs(np.asarray(w, dtype=np.float32)))
    return edges, wmax


def steps(rowptr, w, labels, n_src):
    """q_a (float64 [n_src]) of every cluster."""
    edges, wmax = cluster_stats(rowptr, w, labels, n_src)
    return np.array([2.0 ** step(m, e) for m, e in zip(wmax, edges)])


def cells(a, b, w=None, drop_diag=False):
    """Edges grouped by cell (a[e], b[e]), cells in (a, b) order.  Returns a dict of arrays: a, b, count, and with
    weights sum (math.fsum of the fp32 weights: the exact sum correctly rounded to fp64), abs_sum (sum |w|)."""
    a = np.asarray(a, dtype=np.int64)
    b = np.asarray(b, dtype=np.int64)
    keep = a != b if drop_diag else np.ones(a.shape, dtype=bool)
    a, b = a[keep], b[keep]
    order = np.lexsort((b, a))
    a, b = a[order], b[order]
    head = np.ones(a.shape, dtype=bool)
    head[1:] = (a[1:] != a[:-1]) | (b[1:] != b[:-1])
    starts = np.flatnonzero(head)
    out = {"a": a[starts], "b": b[starts], "count": np.diff(np.append(starts, a.shape[0]))}
    if w is not None:
        ws = np.asarray(w, dtype=np.float32)[keep][order].astype(np.float64)
        groups = np.split(ws, starts[1:]) if ws.size else []
        out["sum"] = np.array([math.fsum(g) for g in groups], dtype=np.float64)
        out["abs_sum"] = np.array([math.fsum(np.abs(g)) for g in groups], dtype=np.float64)
    return out


def csr_cells(rowptr, colidx, w, labels_src, labels_dst, drop_diag=False):
    """cells() of a CSR adjacency: cell (labels_src[row], labels_dst[col])."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    rows = np.repeat(np.arange(rowptr.shape[0] - 1), np.diff(rowptr))
    return cells(np.asarray(labels_src)[rows], np.asarray(labels_dst)[np.asarray(colidx, dtype=np.int64)], w, drop_diag)


def ulp32(x):
    """Spacing of fp32 in the binade of |x| (2^-149 at and below the subnormals)."""
    x = np.abs(np.asarray(x, dtype=np.float64))
    e = np.frexp(x)[1]                                   # x = m * 2^e, m in [0.5, 1)
    return np.where(x > 0, np.ldexp(1.0, np.maximum(e - 24, -149)), 2.0 ** -149)


def gamma(k):
    k = np.asarray(k, dtype=np.float64)
    return k * U / (1.0 - k * U)


def dense_bound(S, count, q):
    """|got - S| of the shared-memory form.  n*q/2: the terms' rounding to multiples of q; 2^-52 (|S| + n*q/2): the
    conversion of the 64-bit integer to fp64; then one rounding to fp32, in the binade of the largest value the fp64
    intermediate can take (it may lie in the binade above S)."""
    S = np.abs(np.asarray(S, dtype=np.float64))
    fx = np.asarray(count, dtype=np.float64) * np.asarray(q, dtype=np.float64) / 2
    pre = fx + 2.0 ** -52 * (S + fx)
    return pre + ulp32(S + pre) / 2


def one_ulp_regime(S, count, q):
    """Cells for which the shared-memory result is within one ulp of fl32(S): n*q/2 <= ulp32(S)/4."""
    return np.asarray(count, dtype=np.float64) * np.asarray(q, dtype=np.float64) / 2 <= ulp32(S) / 4


def sort_bound(count, abs_sum):
    """|got - S| of the sort form: any fixed order of n fp32 additions (depth <= n - 1)."""
    return gamma(np.maximum(np.asarray(count) - 1, 0)) * np.asarray(abs_sum, dtype=np.float64)


def scale_bound(cell_bound, S, n_a, n_b):
    """|got - S / (n_a n_b)| of gdr_coarsen_scale applied to a cell sum within cell_bound of S: the reciprocals and the
    two products round four times (plus two subnormal steps where the value underflows)."""
    nn = np.asarray(n_a, dtype=np.float64) * np.asarray(n_b, dtype=np.float64)
    S = np.abs(np.asarray(S, dtype=np.float64))
    return (cell_bound + gamma(4) * (S + cell_bound)) / nn + 2.0 ** -148


def fixed_point_sum(w, e):
    """The shared-memory form's arithmetic for one cell with step 2^e: round(w / q) to nearest even per term, an exact
    integer sum, (double) of the integer times q, then (float)."""
    terms = [int(np.rint(np.float64(x) * 2.0 ** (-e))) for x in np.asarray(w, dtype=np.float32)]
    return np.float32(float(sum(terms)) * 2.0 ** e)
