"""numpy model of the row-partitioned k-means++ of gdr_kmeans_plusplus_dist.

The global rows are the ranks' blocks in rank order.  Per round every rank knows the per-rank totals T_r of the
current ``closest``; the owner of draw l is the first rank with rows and P_r + T_r >= u_l * pot (P_r, pot: rank-order
fp64 sums of the T_r); the owner searches its fp64 block prefix (blocks of 1024 rows) and then the rows of the block,
starting from P_r; a draw no row reaches is clipped to global row N_total - 1.  Each rank scores every candidate over
its own rows (fp32 min, fp64 block sums), the per-candidate rank totals are added in rank order and the first argmin
wins.  The fp32 distances are computed in fp64 and rounded (the device's fsub/fma chains differ in the last bit on
some rows); the fp64 sums are taken sequentially where the device uses fixed trees.  The model therefore checks the
protocol (ownership, boundaries, clipping, empty ranks), not the device's bits.
"""
import numpy as np

ROWS_PER_BLOCK = 1024


def sqdist(X, c):
    d = X.astype(np.float64) - np.asarray(c, dtype=np.float64)[None]
    return (d * d).sum(1).astype(np.float32)


def _block_sums(v):
    return np.array([v[b:b + ROWS_PER_BLOCK].astype(np.float64).sum() for b in range(0, len(v), ROWS_PER_BLOCK)],
                    dtype=np.float64)


def _total(bs):
    t = 0.0
    for x in bs:
        t += x
    return t


def draws(random_state, n_total, K):
    """The host draws, in sklearn's order: (first centre, [K-1, n_trials] uniforms)."""
    L = 2 + int(np.log(K))
    first = int(random_state.choice(n_total, p=np.full(n_total, 1.0 / n_total)))
    rand = np.array([random_state.uniform(size=L) for _ in range(K - 1)]).reshape(K - 1, L)
    return first, rand


def kpp_dist(blocks, K, first, rand):
    """blocks: the ranks' row blocks (2-D arrays, possibly empty).  Returns the K global row ids."""
    sizes = [b.shape[0] for b in blocks]
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    n_total = int(off[-1])
    world = len(blocks)
    X = np.concatenate(blocks)

    def pass_over(Xr, cl, cand):
        return sqdist(Xr, cand) if cl is None else np.minimum(cl, sqdist(Xr, cand))

    closest, T = [], []
    for r in range(world):
        c = pass_over(blocks[r], None, X[first])
        closest.append(c)
        T.append(_total(_block_sums(c)))
    idx = [first]
    for c_i in range(1, K):
        pot = 0.0
        for t in T:
            pot += t
        cand = []
        for u in rand[c_i - 1]:
            thr = u * pot
            owner, P = -1, 0.0
            for r in range(world):
                if sizes[r] and P + T[r] >= thr:
                    owner = r
                    break
                P += T[r]
            g = n_total - 1
            if owner >= 0:
                bs = _block_sums(closest[owner])
                bprefix = np.concatenate([[0.0], np.cumsum(bs)])
                hit = np.nonzero(P + bprefix[1:] >= thr)[0]
                if hit.size:
                    b = int(hit[0])
                    r0 = b * ROWS_PER_BLOCK
                    run = P + bprefix[b] + np.cumsum(closest[owner][r0:r0 + ROWS_PER_BLOCK].astype(np.float64))
                    rows = np.nonzero(run >= thr)[0]
                    if rows.size:
                        g = int(off[owner] + r0 + rows[0])
            cand.append(g)
        cols, S = [], np.zeros((world, len(cand)))
        for r in range(world):
            cr = [pass_over(blocks[r], closest[r], X[j]) for j in cand]
            cols.append(cr)
            S[r] = [_total(_block_sums(v)) for v in cr]
        pots = []
        for l in range(len(cand)):
            s = S[0, l]
            for r in range(1, world):
                s += S[r, l]
            pots.append(s)
        best = 0
        for l in range(1, len(cand)):
            if pots[l] < pots[best]:
                best = l
        idx.append(cand[best])
        closest = [cols[r][best] for r in range(world)]
        T = [_total(_block_sums(v)) for v in closest]
    return np.array(idx, dtype=np.int64)


def row_blocks(X, world):
    """RowPartition's blocks: ceil(n / world) rows per rank, the last ones short or empty."""
    n = X.shape[0]
    per = -(-n // world)
    return [X[min(n, r * per):min(n, (r + 1) * per)] for r in range(world)]
