"""numpy model of the Gram matrix on a row partition (gdr_dense_gram_dist, csrc/svd.cu) and of the one-GPU order it
reproduces (gdr_dense_gram).

One GPU: min(16, cdiv(N, 2048)) contiguous slabs of cdiv(N, slabs) rows; every output element of a slab is one chain
over the slab's rows in order, from 0.0, taken GR rows per step with zero rows padding the last step; the slab partials
are added in slab order from 0.0.

Partition: each rank cuts its rows at the same slab boundaries.  A segment that starts its slab chains from 0.0; the
first segment may continue a slab begun on an earlier rank and chains from the carry, the accumulators that rank's
segment of the slab ended with.  A rank adds the slabs that end on it, in order, to the running sum it receives and
hands (carry, running sum) to the next rank; an empty rank hands on what it received.  The last rank's sum is C.

Both arms take the chain step from ``step`` (an fp64 product added to the accumulator), so that a comparison checks
how the chains are split across ranks, not the arithmetic of one step.
"""
import numpy as np

GRAM_MAX_SLABS = 16
SLAB_MIN_ROWS = 2048
GR = 32


def slab_geometry(N):
    """(slabs, rows per slab) of an N-row Gram."""
    slabs = max(1, min(GRAM_MAX_SLABS, -(-N // SLAB_MIN_ROWS)))
    return slabs, -(-N // slabs)


def step(acc, a, b):
    return acc + a[:, None] * b[None, :]


def chain(acc, A, B):
    """acc continued over the rows of A and B in order, GR rows per step, zero rows padding the last step."""
    pad = (-A.shape[0]) % GR
    A = np.concatenate([A, np.zeros((pad, A.shape[1]))])
    B = np.concatenate([B, np.zeros((pad, B.shape[1]))])
    for g in range(A.shape[0]):
        acc = step(acc, A[g], B[g])
    return acc


def gram_one(A, B):
    """gdr_dense_gram's order on all N rows."""
    N = A.shape[0]
    slabs, rows_per = slab_geometry(N)
    zero = np.zeros((A.shape[1], B.shape[1]))
    parts = [chain(zero, A[z * rows_per: min(N, (z + 1) * rows_per)], B[z * rows_per: min(N, (z + 1) * rows_per)])
             for z in range(slabs)]
    total = zero
    for P in parts:
        total = total + P
    return total


def segments(N, lo, hi):
    """The rows [lo, hi) of one rank cut at the slab boundaries: (a, b, starts_slab, ends_slab) per segment."""
    _, rows_per = slab_geometry(N)
    out, a = [], lo
    while a < hi:
        z0 = a // rows_per * rows_per
        z1 = min(N, z0 + rows_per)
        b = min(hi, z1)
        out.append((a, b, a == z0, b == z1))
        a = b
    return out


def gram_dist(blocks_A, blocks_B):
    """The partitioned protocol over the ranks' row blocks (rank order = row order).  Returns C and the messages
    (carry, running sum) each rank hands to the next."""
    N = sum(a.shape[0] for a in blocks_A)
    zero = np.zeros((blocks_A[0].shape[1], blocks_B[0].shape[1]))
    carry, total = None, zero            # what rank 0 starts from: no carry, a running sum of 0.0
    messages, lo = [], 0
    for A, B in zip(blocks_A, blocks_B):
        hi = lo + A.shape[0]
        done, carry_out = [], None
        for a, b, starts, ends in segments(N, lo, hi):
            if not starts:
                assert carry is not None, "a segment continues a slab that no earlier rank began"
            acc = chain(zero if starts else carry, A[a - lo: b - lo], B[a - lo: b - lo])
            if ends:
                done.append(acc)
            else:
                carry_out = acc
        if hi > lo:
            for P in done:
                total = total + P
            carry = carry_out
        messages.append((carry, total))
        lo = hi
    return total, messages


def equal_blocks(X, world):
    """parallel.RowPartition's blocks: cdiv(N, world) rows per rank, the last ones short or empty."""
    N = X.shape[0]
    rows_per = -(-N // world)
    return [X[min(N, r * rows_per): min(N, (r + 1) * rows_per)] for r in range(world)]
