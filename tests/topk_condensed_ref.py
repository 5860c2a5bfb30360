"""numpy mirror of gdr.recommend_topk_condensed's cluster walk (topk_condensed.cu): the distinct scores S[g, c], the
per-group prefix of clusters (member count reaching min(n_items, k + max |exclusion row|), whole tie runs), then per
row the prefix one tie run at a time, members of a run merged by item id, excluded items skipped, stop at k.  Rows that
meet a tie run of more than 32 clusters before they have k items are finished by topk_ref on their expanded row, as
the library finishes them on the exact path.  Test infrastructure only; the library never imports it."""
import numpy as np

import topk_ref

MAX_RUN = 32


def cluster_scores(Ucl, Icl, groups, has_members):
    """S[g, c] for g in groups: the exact fmaf chain (topk_ref with k = n_ci), -0 reported as +0.  Rows of clusters
    without members are zeroed first (they may hold NaN and are never read)."""
    I = np.array(Icl, dtype=np.float32, copy=True)
    I[~has_members] = 0
    s, it = topk_ref.topk(Ucl, I, I.shape[0], rows=np.asarray(groups, dtype=np.int64))
    S = np.empty_like(s)
    np.put_along_axis(S, it.astype(np.int64), s, axis=1)
    return S


def topk_condensed(Ucl, Icl, k, u2cu, i2ci, ex_rowptr=None, ex_colidx=None, rows=None):
    """(scores [n_rows, k] f32, items [n_rows, k] int32, fallback row indices) of the cluster walk."""
    u2cu = np.asarray(u2cu, dtype=np.int64)
    i2ci = np.asarray(i2ci, dtype=np.int64)
    n_users, n_items, n_ci = len(u2cu), len(i2ci), Icl.shape[0]
    users = np.arange(n_users) if rows is None else np.asarray(rows, dtype=np.int64)
    n_rows = len(users)
    m = np.bincount(i2ci, minlength=n_ci)
    members = [np.flatnonzero(i2ci == c) for c in range(n_ci)]   # ascending item ids

    def excl(u):
        return set() if ex_rowptr is None else set(np.asarray(ex_colidx[ex_rowptr[u]:ex_rowptr[u + 1]]).tolist())

    groups = sorted(set(u2cu[users].tolist()))
    S = cluster_scores(Ucl, Icl, groups, m > 0) if groups else None
    slot = {g: i for i, g in enumerate(groups)}
    deg = np.zeros(n_users, np.int64) if ex_rowptr is None else np.diff(np.asarray(ex_rowptr, dtype=np.int64))
    need = {g: 0 for g in groups}
    for u in users:
        need[u2cu[u]] = max(need[u2cu[u]], int(deg[u]))
    prefix = {}
    for g in groups:
        ng = min(n_items, k + need[g])
        s = S[slot[g]].astype(np.float64)
        cl = [c for c in sorted(range(n_ci), key=lambda c: (-s[c], c)) if m[c] > 0]
        cum, cut = 0, len(cl)
        for i, c in enumerate(cl):
            cum += m[c]
            if cum >= ng:
                cut = i + 1
                while cut < len(cl) and s[cl[cut]] == s[c]:   # the whole tie run at the boundary
                    cut += 1
                break
        prefix[g] = cl[:cut]

    scores = np.full((n_rows, k), -np.inf, dtype=np.float32)
    items = np.full((n_rows, k), -1, dtype=np.int32)
    fallback = []
    for r, u in enumerate(users):
        g = u2cu[u]
        s, P, ex = S[slot[g]], prefix[g], excl(u)
        out, p, fb = [], 0, False
        while len(out) < k and p < len(P):
            L = 1
            while p + L < len(P) and s[P[p + L]] == s[P[p]]:
                L += 1
            if L > MAX_RUN:
                fb = True
                break
            run = np.sort(np.concatenate([members[c] for c in P[p:p + L]]))
            for j in run:
                if len(out) == k:
                    break
                if int(j) not in ex:
                    out.append((s[P[p]], j))
            p += L
        if fb:
            fallback.append(r)
            continue
        for i, (sc, j) in enumerate(out):
            scores[r, i] = sc
            items[r, i] = j
    if fallback:
        fr = np.asarray(fallback)
        fs, fi = topk_ref.topk(Ucl[u2cu], Icl[i2ci], k, ex_rowptr, ex_colidx, users[fr])
        scores[fr], items[fr] = fs, fi
    return scores, items, fallback
