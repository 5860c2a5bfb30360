#!/usr/bin/env python
"""CPU estimate (numpy only) of the candidate second level of the two-level tensor-core screen: the level-1 score and
radius of k_split_tf32 / k_tc_select1 on a row sample, the share of rows level 1 leaves undecided, how many centres the
seeded candidate pass records per row and column half, how many survive the final filter, and the overflow rate per
list capacity.  Data: config-shaped z-scored rows (synth.features, seed 17) and centres after one Lloyd update from
random rows, as tests/test_gpu_tc.py::test_tc_full_size_labels_equal_exact_kernel.
    python tools/cand_estimate.py [E|B] [D] [sample rows]"""
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAND = 2.0 ** -15


def tf32(a):
    """cvt.rna.tf32.f32: round to 10 explicit significand bits, ties away from zero."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_up(v):
    """smallest TF32 value >= v"""
    u = np.ascontiguousarray(v, dtype=np.float32).view(np.uint32).copy()
    pos = v >= 0
    u[pos] = (u[pos] + np.uint32(0x1FFF)) & np.uint32(0xFFFFE000)
    u[~pos] &= np.uint32(0xFFFFE000)
    return u.view(np.float32)


def augment(X, C):
    """First-level operands of k_split_tf32 (aug_mode 1 for rows, 2 for centres) and the per-row / per-centre norms."""
    X = X.astype(np.float32)
    C = C.astype(np.float32)
    xh, ch = tf32(X), tf32(C)
    xn = np.sqrt((X.astype(np.float64) ** 2).sum(1)).astype(np.float32)
    xd = np.sqrt(((X - xh).astype(np.float64) ** 2).sum(1)).astype(np.float32)
    c2 = (C.astype(np.float64) ** 2).sum(1).astype(np.float32)
    cn = np.sqrt(c2)
    cd = np.sqrt(((C - ch).astype(np.float64) ** 2).sum(1)).astype(np.float32)
    ones = np.ones_like(xn)
    x1 = np.concatenate([xh, tf32_up(1.001 * xd)[:, None], tf32_up(1.001 * xn)[:, None], ones[:, None], ones[:, None]], 1)
    w = (-0.5 * c2 * (1 - BAND)).astype(np.float32)
    p = tf32(w)
    q = tf32_up(w - p)
    c1 = np.concatenate([ch, tf32_up(1.001 * cn)[:, None], tf32_up(1.001 * (cd + BAND * cn))[:, None], p[:, None], q[:, None]], 1)
    return x1, c1, dict(xn=xn, xd=xd, c2=c2, cn=cn, cd=cd, cm=np.float32(cn.max()), cdm=np.float32(cd.max()))


def tolmax(xn, xd, cm, cdm):
    return 1.001 * (2.02 * (xd * cm + xn * (cdm + BAND * cm) + 2.0 ** -16 * cm * cm) + BAND * xn * cm +
                    2.0 ** -20 * (xn * cm + cm * cm))


def tol(xn, xd, cn, cd, c2, cm, s):
    """k_tc_select1's tol(i, l) with |s| for its last term"""
    E = xd * cn + xn * (cd + BAND * cn)
    return 2.02 * (E + 2.0 ** -16 * c2) + BAND * xn * cm + 2.0 ** -21 * np.abs(s)


def screen(X, C, perturb=None):
    """Model of level 1, the candidate pass and the final filter on rows X against centres C.
    Returns per row: undecided (bool), recorded count per column half [n, 2], kept (bool [n, K]) and the negated
    scores d [n, K].  perturb(d, acc_bound) may move each modelled score within the accumulation allowance."""
    x1, c1, m = augment(X, C)
    d = -(x1.astype(np.float64) @ c1.T.astype(np.float64))               # negated scores, exact accumulation
    bound = (X.shape[1] + 4) * 2.0 ** -23 * np.outer(m["xn"], m["cn"])   # TMEM accumulation allowance
    if perturb is not None:
        d = perturb(d, bound)
    n, K = d.shape
    l = d.argmin(1)
    b = d[np.arange(n), l]
    d2 = d.copy()
    d2[np.arange(n), l] = np.inf
    s2 = d2.min(1)
    xn, xd = m["xn"].astype(np.float64), m["xd"].astype(np.float64)
    t1 = tol(xn, xd, m["cn"][l], m["cd"][l], m["c2"][l], m["cm"], np.maximum(np.abs(b), np.where(np.isinf(s2), 0, np.abs(s2))))
    undecided = ~(s2 - b > t1)
    tm = tolmax(xn, xd, np.float64(m["cm"]), np.float64(m["cdm"]))
    slack = 2.0 ** -18 * (xn * m["cm"] + m["cm"] ** 2)
    limit = (b + slack + tm)[:, None]
    rec = d < limit
    col = np.arange(K) % 256 >= 128
    counts = np.stack([(rec & ~col).sum(1), (rec & col).sum(1)], 1)
    tl = tol(xn[:, None], xd[:, None], m["cn"][l][:, None], m["cd"][l][:, None], m["c2"][l][:, None], m["cm"],
             np.maximum(np.abs(b)[:, None], np.abs(d)))
    kept = rec & ~(d - b[:, None] > tl)
    return undecided, counts, kept, d


def _synth():
    spec = importlib.util.spec_from_file_location("synth", os.path.join(ROOT, "graph-distillation-for-recommendation_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def lloyd_update(X, C, chunk=16384):
    cn = (C * C).sum(1)
    K = C.shape[0]
    lab = np.empty(X.shape[0], np.int64)
    for s in range(0, X.shape[0], chunk):
        lab[s:s + chunk] = (cn[None, :] - 2 * X[s:s + chunk] @ C.T).argmin(1)
    sums = np.zeros_like(C, dtype=np.float64)
    np.add.at(sums, lab, X)
    cnt = np.bincount(lab, minlength=K)
    return (sums / np.maximum(cnt, 1)[:, None]).astype(np.float32)


def main():
    synth = _synth()
    name = sys.argv[1] if len(sys.argv) > 1 else "E"
    cfg = synth.CONFIGS[name]
    n, K = cfg["n"], cfg["k"]
    D = int(sys.argv[2]) if len(sys.argv) > 2 else cfg["f"]
    S = int(sys.argv[3]) if len(sys.argv) > 3 else 20000
    X = synth.features(n, D, seed=17).astype(np.float32)
    X -= X.mean(0)
    C = X[np.random.RandomState(3).permutation(n)[:K]].copy()
    C = lloyd_update(X, C)
    Xs = X[np.random.RandomState(5).permutation(n)[:S]]
    und, cnt, kept = [], [], []
    for s in range(0, S, 1000):
        u, c, k, _ = screen(Xs[s:s + 1000], C)
        und.append(u)
        cnt.append(c[u])
        kept.append(k[u].sum(1))
    und, cnt, kept = np.concatenate(und), np.concatenate(cnt), np.concatenate(kept)
    tot = cnt.sum(1)
    print(f"config {name}: N = {n}, D = {D}, K = {K}; sample of {S} rows, centres after one Lloyd update")
    print(f"undecided after level 1: {und.mean() * 100:.2f} % ({und.sum()} rows)")
    edges = [0, 1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64, 128, 1 << 30]
    for what, v in (("recorded per row (both halves)", tot), ("recorded per column half (max of the two)", cnt.max(1)),
                    ("kept after the final filter", kept)):
        h = np.histogram(v, bins=edges)[0]
        print(f"{what}: mean {v.mean():.2f}, p50 {np.percentile(v, 50):.0f}, p99 {np.percentile(v, 99):.0f}, "
              f"p99.9 {np.percentile(v, 99.9):.0f}, max {v.max()}")
        print("   " + "  ".join(f"[{edges[i]},{edges[i + 1] if edges[i + 1] < 1 << 29 else 'inf'}): {h[i]}" for i in range(len(h)) if h[i]))
    for cap in (16, 32, 64):
        print(f"overflow (either half > {cap}): {(cnt.max(1) > cap).mean() * 100:.3f} % of undecided rows")


if __name__ == "__main__":
    main()
