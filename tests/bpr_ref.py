"""numpy reference of gdr_bpr_sample (csrc/bpr.cu): Philox4x32-10, the complement select and the triplet sampler,
bit for bit.  Vectorised over the triplets of a step."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: 4 arrays (or ints) of 32-bit words, key: 2 ints -> 4 uint64 arrays holding 32-bit words."""
    c = [np.asarray(x, dtype=np.uint64) & MASK32 for x in ctr]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]   # < 2^64: no wrap
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1),
             p0 & MASK32]
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return c


def draw_below(lo, hi, n):
    """umulhi64((hi << 32) | lo, n) for n < 2^32, as int64."""
    n = np.asarray(n, dtype=np.uint64)
    assert (n < np.uint64(1 << 32)).all()
    t = ((lo * n) >> np.uint64(32)) + hi * n   # < 2^64: hi, lo < 2^32, n < 2^32
    return (t >> np.uint64(32)).astype(np.int64)


def complement_select(cols, r):
    """The r-th item (0-based) outside the sorted, unique row ``cols``: r + #{t : c_t - t <= r}."""
    cols = np.asarray(cols, dtype=np.int64)
    return int(r) + int(np.searchsorted(cols - np.arange(len(cols)), r, side="right"))


def eligible_users(rowptr, n_items):
    deg = np.diff(rowptr)
    return np.nonzero((deg > 0) & (deg < n_items))[0].astype(np.int64)


def sample(rowptr, colidx, n_items, seed, step, batch):
    """(users, pos, neg) int64 [batch] of gdr.BPRSampler(R, seed).sample(batch, step)."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    colidx = np.asarray(colidx, dtype=np.int64)
    elig = eligible_users(rowptr, n_items)
    if len(elig) == 0:
        raise ValueError("no eligible user")
    key = (seed & 0xFFFFFFFF, seed >> 32)
    b = np.arange(batch, dtype=np.uint64)
    z = np.zeros(batch, dtype=np.uint64)
    w = philox4x32_10((b, z + np.uint64(step), z, z), key)
    v = philox4x32_10((b, z + np.uint64(step), z + np.uint64(1), z), key)
    users = elig[draw_below(w[0], w[1], len(elig))]
    start = rowptr[users]
    deg = rowptr[users + 1] - start
    pos = colidx[start + draw_below(w[2], w[3], deg)]
    r = draw_below(v[0], v[1], n_items - deg)
    lo, hi = np.zeros(batch, dtype=np.int64), deg.copy()   # vectorised binary search of the complement select
    while (lo < hi).any():
        act = lo < hi
        mid = (lo + hi) >> 1
        ok = act & (colidx[np.where(act, start + mid, 0)] - mid <= r)
        lo = np.where(ok, mid + 1, lo)
        hi = np.where(act & ~ok, mid, hi)
    return users, pos, r + lo
