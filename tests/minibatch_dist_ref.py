"""numpy model of one mini-batch assembly on a row partition (gdr_minibatch_batch_dist): the plan (parallel.batch_plan),
each owner packing its positions in batch order and labelling the packed rows, the exchange that hands every rank all
packed blocks in rank order, and the placement of record k at batch position order[k]."""
import numpy as np


def split_rows(X, row_off):
    """The row blocks of X that the ranks hold."""
    return [X[row_off[r]:row_off[r + 1]] for r in range(len(row_off) - 1)]


def assemble(blocks, row_off, idx, order, counts, label_fn=None):
    """What every rank holds after the call: (Xb, labels_b or None).  ``label_fn`` maps packed rows to their labels;
    it is applied per owner, to that owner's packed rows only."""
    world = len(blocks)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    packed, labels = [], []
    for r in range(world):
        pos = order[offs[r]:offs[r + 1]]
        rows = blocks[r][idx[pos] - row_off[r]]                  # pack: the owner's rows, batch order
        packed.append(rows)
        if label_fn is not None:
            labels.append(label_fn(rows) if len(rows) else np.zeros(0, np.int32))
    recv = np.concatenate(packed)                                # exchange: every block, rank order
    Xb = np.empty_like(recv)
    Xb[order] = recv                                             # place: record k -> position order[k]
    lab = None
    if label_fn is not None:
        lab = np.empty(len(idx), np.int32)
        lab[order] = np.concatenate(labels)
    return Xb, lab


def nearest(C):
    """Per-row label function: index of the nearest centre (first on ties), fp64."""
    def fn(rows):
        d = ((rows[:, None, :].astype(np.float64) - C[None, :, :].astype(np.float64)) ** 2).sum(-1)
        return d.argmin(1).astype(np.int32)
    return fn
