"""numpy model of the per-cluster sums on a row partition (gdr_segment_sum_dist, csrc/kmeans.cu) and of the one-GPU
order it reproduces (gdr_segment_sum).

One GPU: every output element is one fp32 chain from +0.0 over the cluster's members in ascending row order.

Partition: the ranks' row blocks, in rank order, are the global row order.  Rank 0 starts every chain from +0.0; rank
q > 0 receives the sums rank q - 1 ended with and continues each chain over its own members of the cluster, in
ascending row order; an empty rank hands on what it received.  The last rank's sums are the result.  The counts are
the sum of the ranks' histograms.
"""
import numpy as np


def chain(sums, X, labels):
    """sums continued over the rows of X in order: row i is added to the chain of cluster labels[i] (fp32)."""
    sums = sums.copy()
    for x, l in zip(X, labels):
        sums[l] = sums[l] + x
    return sums


def segment_sum_dist(blocks_X, blocks_lab, K):
    """The partitioned protocol over the ranks' blocks (rank order = row order).  Returns (sums, counts, messages):
    messages[q] are the sums rank q hands to rank q + 1 (the last one's are the result)."""
    D = blocks_X[0].shape[1]
    sums = np.zeros((K, D), dtype=np.float32)           # rank 0 starts from +0.0
    counts = np.zeros(K, dtype=np.int64)
    messages = []
    for X, lab in zip(blocks_X, blocks_lab):
        assert X.dtype == np.float32 and X.shape[0] == lab.shape[0]
        if X.shape[0] > 0:
            sums = chain(sums, X, lab)
        counts += np.bincount(lab, minlength=K)
        messages.append(sums)
    return sums, counts.astype(np.int32), messages


def restarted_per_rank(blocks_X, blocks_lab, K):
    """The order a partition would give without the hand-off: each rank chains from +0.0 and the ranks' sums are added
    in rank order (negative control)."""
    D = blocks_X[0].shape[1]
    total = np.zeros((K, D), dtype=np.float32)
    for X, lab in zip(blocks_X, blocks_lab):
        total = total + chain(np.zeros((K, D), dtype=np.float32), X, lab)
    return total


def cut(X, cuts):
    """The blocks [cuts[q], cuts[q + 1]) of X."""
    return [X[a:b] for a, b in zip(cuts[:-1], cuts[1:])]


def equal_cuts(N, world):
    """parallel.RowPartition's blocks: cdiv(N, world) rows per rank, the last ones short or empty."""
    rows_per = -(-N // world)
    return [min(N, r * rows_per) for r in range(world)] + [N]
