"""recommend_topk_condensed on the GPU: every case byte-identical to recommend_topk on the expanded tables
(user_emb[user_map], item_emb[item_map]) under both of its forced paths, and to the CPU reference (topk_ref) on the
rows it checks.  Tie-heavy cluster tables, the fallback for long tie runs, NaN in an empty super-item, padding, rows
subsets, identity maps, and the full Yelp2018 / Amazon-book shapes with k-means maps."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import topk_ref
from conftest import golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def gdr():
    import gdr as g
    assert torch.cuda.is_available()
    return g


class debug_key:
    """gdr_debug_set(key, value) inside the block, automatic (0) after."""

    def __init__(self, key, value):
        self.key, self.value = key, value

    def __enter__(self):
        from gdr import _lib
        _lib.call("gdr_debug_set", self.key, self.value)

    def __exit__(self, *exc):
        from gdr import _lib
        _lib.call("gdr_debug_set", self.key, 0)


def fallback_rows():
    from gdr import _lib
    v = ctypes.c_int64(0)
    _lib.call("gdr_debug_get", b"topk_condensed_fallback_rows", ctypes.addressof(v))
    return v.value


def _same(a, b):
    sa, ia = a
    sb, ib = b
    assert ia.dtype == ib.dtype == torch.int64 and sa.dtype == sb.dtype == torch.float32
    assert torch.equal(ia, ib), "items differ"
    assert torch.equal(sa.view(torch.int32), sb.view(torch.int32)), "scores are not bit-identical"


def check(gdr, Ucl, Icl, k, u2cu, i2ci, R=None, rows=None, ref_rows=None):
    """The condensed call against the expanded call under both forced paths and against topk_ref on ref_rows (output
    row indices; default all).  Returns (scores, items, fallback rows of the condensed call)."""
    Ut, It = torch.as_tensor(Ucl).to(DEV), torch.as_tensor(Icl).to(DEV)
    ex = None if R is None else gdr.CSR.from_scipy(R, device=DEV)
    rows_t = None if rows is None else torch.as_tensor(rows).to(DEV)
    got = gdr.recommend_topk_condensed(Ut, It, k, u2cu, i2ci, exclude=ex, rows=rows_t)
    n_fb = fallback_rows()
    um, im = torch.as_tensor(np.asarray(u2cu)).long().to(DEV), torch.as_tensor(np.asarray(i2ci)).long().to(DEV)
    Ue, Ie = Ut[um], It[im]
    for path in (1, 2):
        if path == 2 and (Ut.shape[1] > 128 or k > 256):
            continue
        with debug_key(b"topk_path", path):
            _same(got, gdr.recommend_topk(Ue, Ie, k, exclude=ex, rows=rows_t))
    users = np.arange(len(u2cu)) if rows is None else np.asarray(rows, dtype=np.int64)
    sel = np.arange(len(users)) if ref_rows is None else np.asarray(ref_rows)
    if len(sel):
        rs_, ri = topk_ref.topk(Ue.cpu().numpy(), Ie.cpu().numpy(), k, None if R is None else R.indptr,
                                None if R is None else R.indices, users[sel])
        np.testing.assert_array_equal(got[1].cpu().numpy()[sel], ri)
        assert np.array_equal(got[0].cpu().numpy()[sel].view(np.uint32), rs_.view(np.uint32))
    return got[0], got[1], n_fb


def _golden():
    g = golden("recsys_ali_subset.npz")
    u2cu, i2ci = g["u2cu"], g["i2ci"]
    R = sp.csr_matrix((np.ones(len(g["r_indices"]), np.float32), g["r_indices"], g["r_indptr"]),
                      shape=(len(u2cu), len(i2ci)))
    return u2cu, i2ci, R


@pytest.mark.parametrize("d", [1, 7, 64, 100, 200])
def test_golden_maps(gdr, d):
    u2cu, i2ci, R = _golden()
    rs = np.random.RandomState(d)
    Ucl = rs.standard_normal((int(u2cu.max()) + 1, d)).astype(np.float32)
    Icl = rs.standard_normal((int(i2ci.max()) + 1, d)).astype(np.float32)
    sample = rs.choice(len(u2cu), 150, replace=False)
    for k in (1, 20, 100):
        check(gdr, Ucl, Icl, k, u2cu, i2ci, R, ref_rows=sample)
        # int64 torch maps and a rows subset give the same rows
        rows = rs.choice(len(u2cu), 500, replace=False).astype(np.int64)
        s, it, _ = check(gdr, Ucl, Icl, k, torch.from_numpy(u2cu.astype(np.int64)), i2ci, R, rows=rows, ref_rows=[])
        s_all, it_all = gdr.recommend_topk_condensed(torch.from_numpy(Ucl).to(DEV), torch.from_numpy(Icl).to(DEV), k,
                                                     u2cu, i2ci, exclude=R)
        r_t = torch.from_numpy(rows).to(DEV)
        assert torch.equal(it, it_all[r_t]) and torch.equal(s, s_all[r_t])


def _tie_tables(seed, n_users=400, n_items=700, n_cu=12, n_ci=60, d=6):
    rs = np.random.RandomState(seed)
    Ucl = rs.randint(-2, 3, (n_cu, d)).astype(np.float32)   # integer entries: exact scores, many ties
    Icl = rs.randint(-2, 3, (n_ci, d)).astype(np.float32)
    Ucl[0] = 0                     # a zero super-user: every cluster ties (fallback)
    Ucl[1] = -0.0
    Ucl[2, :3] = -0.0
    Icl[3] = Icl[2]                # the same vector for distinct clusters
    Icl[5] = Icl[2]
    Icl[-3] = -0.0
    u2cu = rs.randint(0, n_cu, n_users)
    u2cu[:4] = [0, 1, 2, 0]
    i2ci = rs.randint(0, n_ci - 2, n_items)   # clusters n_ci - 2 and n_ci - 1 are empty
    i2ci[i2ci == 7] = 8
    i2ci[11] = 7                   # a cluster of one item
    R = sp.random(n_users, n_items, density=0.03, format="csr", random_state=rs, dtype=np.float32).tolil()
    R[5, :] = 1.0                  # user 5 keeps 6 items (padding)
    R[5, :6] = 0.0
    R[6, :600] = 1.0               # heavy exclusion
    R = R.tocsr()
    R.eliminate_zeros()
    R.sort_indices()
    return Ucl, Icl, u2cu, i2ci, R


@pytest.mark.parametrize("seed", [0, 1])
def test_ties_fallback_and_padding(gdr, seed):
    Ucl, Icl, u2cu, i2ci, R = _tie_tables(seed)
    for k in (1, 20, 100, 700):
        s, it, n_fb = check(gdr, Ucl, Icl, k, u2cu, i2ci, R)
        assert n_fb > 0   # the zero super-user's rows
        if k >= 20:
            assert (it[5, 6:] == -1).all() and torch.isinf(s[5, 6:]).all()
        check(gdr, Ucl, Icl, k, u2cu, i2ci)
    # NaN in an empty super-item is never read
    Icl2 = Icl.copy()
    Icl2[-1] = np.nan
    s, it, _ = check(gdr, Ucl, Icl2, 20, u2cu, i2ci, R)
    _same((s, it), gdr.recommend_topk_condensed(torch.from_numpy(Ucl).to(DEV), torch.from_numpy(Icl).to(DEV), 20,
                                                u2cu, i2ci, exclude=R))


def test_forced_fallback_equals_normal_run(gdr):
    for Ucl, Icl, u2cu, i2ci, R in (_tie_tables(3), _tie_tables(4, n_cu=40, n_ci=9, d=3)):
        Ut, It = torch.from_numpy(Ucl).to(DEV), torch.from_numpy(Icl).to(DEV)
        for k in (3, 50):
            a = gdr.recommend_topk_condensed(Ut, It, k, u2cu, i2ci, exclude=R)
            assert fallback_rows() < len(u2cu)
            with debug_key(b"topk_condensed_path", 1):
                b = gdr.recommend_topk_condensed(Ut, It, k, u2cu, i2ci, exclude=R)
                assert fallback_rows() == len(u2cu)
            _same(a, b)


def test_rows_repeats_subset_and_empty(gdr):
    Ucl, Icl, u2cu, i2ci, R = _tie_tables(5)
    rows = np.array([5, 5, 0, 3, 399, 6, 5, 17], dtype=np.int64)
    check(gdr, Ucl, Icl, 20, u2cu, i2ci, R, rows=rows)
    s, it = gdr.recommend_topk_condensed(torch.from_numpy(Ucl).to(DEV), torch.from_numpy(Icl).to(DEV), 20, u2cu,
                                         i2ci, exclude=R, rows=np.zeros(0, np.int64))
    assert s.shape == (0, 20) and it.shape == (0, 20) and it.dtype == torch.int64


def test_identity_maps_equal_plain_topk(gdr):
    rs = np.random.RandomState(11)
    U = rs.standard_normal((300, 33)).astype(np.float32)
    I = rs.standard_normal((1000, 33)).astype(np.float32)
    R = sp.random(300, 1000, density=0.05, format="csr", random_state=rs, dtype=np.float32)
    R.sort_indices()
    for k in (1, 20, 100):
        s, it, n_fb = check(gdr, U, I, k, np.arange(300, dtype=np.int32), np.arange(1000), R, ref_rows=np.arange(40))
        assert n_fb == 0
        _same((s, it), gdr.recommend_topk(torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV), k, exclude=R))


def test_errors(gdr):
    Ucl, Icl, u2cu, i2ci, R = _tie_tables(6)
    Ut, It = torch.from_numpy(Ucl).to(DEV), torch.from_numpy(Icl).to(DEV)
    used_ci = int(i2ci[0])
    bad_I = It.clone()
    bad_I[used_ci, 2] = float("nan")
    with pytest.raises(ValueError, match="non-finite"):
        gdr.recommend_topk_condensed(Ut, bad_I, 20, u2cu, i2ci, exclude=R)
    bad_U = Ut.clone()
    bad_U[int(u2cu[7]), 0] = float("inf")
    with pytest.raises(ValueError, match="non-finite"):
        gdr.recommend_topk_condensed(bad_U, It, 20, u2cu, i2ci, exclude=R)
    # a non-finite super-user that no evaluated row uses is not read (as in the expanded call)
    rows = np.flatnonzero(u2cu != u2cu[7])
    check(gdr, bad_U.cpu().numpy(), Icl, 20, u2cu, i2ci, R, rows=rows, ref_rows=[])
    for um, im in ((np.where(u2cu == 3, Ucl.shape[0], u2cu), i2ci), (u2cu, np.where(i2ci == 4, -1, i2ci))):
        with pytest.raises(ValueError, match="outside"):
            gdr.recommend_topk_condensed(Ut, It, 20, um, im, exclude=R)
    with pytest.raises(ValueError, match="outside"):
        gdr.recommend_topk_condensed(Ut, It, 20, u2cu, i2ci, exclude=R, rows=np.array([0, len(u2cu)]))
    for k in (0, len(i2ci) + 1):
        with pytest.raises(ValueError):
            gdr.recommend_topk_condensed(Ut, It, k, u2cu, i2ci)
    with pytest.raises(ValueError):   # exclusion shape must be n_users x n_items
        gdr.recommend_topk_condensed(Ut, It, 5, u2cu[:-1], i2ci, exclude=R)
    with pytest.raises(ValueError):   # maps must be integers
        gdr.recommend_topk_condensed(Ut, It, 5, u2cu.astype(np.float32), i2ci)


def condensed_workload(gdr, name, dev, d=64, L=2):
    """The condensed model at the Yelp2018 (C) / Amazon-book (D) shape: bench.py's seeds and synthetic interactions,
    gdr.kmeans_cluster maps at a 10 % rate (as tools/lightgcn_grad_bench.py), condensed tables from a seeded
    LightGCNPropagate forward.  Returns (Ucl, Icl, u2cu, i2ci, R = the training CSR)."""
    from gdr import synth
    cfg = synth.BIPARTITE[name]
    seed = 1234 + {"C": 2, "D": 3}[name]
    n_u, n_i = cfg["users"], cfg["items"]
    u, i = synth.bipartite_interactions(n_u, n_i, cfg["inter"], seed)
    rs = np.random.RandomState(seed + 100)
    emb_u = (rs.standard_normal((n_u, d)) * 0.1).astype(np.float32)
    emb_i = (rs.standard_normal((n_i, d)) * 0.1).astype(np.float32)
    ncu, nci = int(np.ceil(n_u * 0.1)), int(np.ceil(n_i * 0.1))
    u2cu, _ = gdr.kmeans_cluster(emb_u, ncu, seed=42, init="random", device=dev)
    i2ci, _ = gdr.kmeans_cluster(emb_i, nci, seed=42, init="random", device=dev)
    C = gdr.build_condensed_bipartite(u, i, u2cu, i2ci, ncu, nci, device=dev, return_device=True)
    ei, ew = gdr.condensed_csr_to_edge_index(C, dev)
    graph = gdr.BipartiteGraph(ei, ew, ncu, nci)
    rs = np.random.RandomState(7)
    u0 = torch.from_numpy((rs.standard_normal((ncu, d)) * 0.1).astype(np.float32)).to(dev)
    i0 = torch.from_numpy((rs.standard_normal((nci, d)) * 0.1).astype(np.float32)).to(dev)
    with torch.no_grad():
        Ucl, Icl = gdr.LightGCNPropagate.apply(u0, i0, ew, graph, L)
    R = gdr.coo_to_csr(u, i, None, (n_u, n_i), device=dev)
    return Ucl, Icl, u2cu, i2ci, R


@pytest.mark.parametrize("name", ["C", "D"])
def test_full_size_kmeans_maps(gdr, name):
    Ucl, Icl, u2cu, i2ci, R = condensed_workload(gdr, name, DEV)
    um, im = torch.from_numpy(u2cu).to(DEV), torch.from_numpy(i2ci).to(DEV)
    got = gdr.recommend_topk_condensed(Ucl, Icl, 20, um, im, exclude=R)
    again = gdr.recommend_topk_condensed(Ucl, Icl, 20, um, im, exclude=R)
    _same(got, again)
    assert (got[1] >= 0).all()
    Ue, Ie = Ucl[um].contiguous(), Icl[im].contiguous()
    for path in (1, 2):
        with debug_key(b"topk_path", path):
            _same(got, gdr.recommend_topk(Ue, Ie, 20, exclude=R))
    sample = np.random.RandomState(3).choice(len(u2cu), 48, replace=False).astype(np.int64)
    Rs = R.to_scipy()
    rs_, ri = topk_ref.topk(Ue.cpu().numpy(), Ie.cpu().numpy(), 20, Rs.indptr, Rs.indices, sample)
    np.testing.assert_array_equal(got[1].cpu().numpy()[sample], ri)
    assert np.array_equal(got[0].cpu().numpy()[sample].view(np.uint32), rs_.view(np.uint32))
    # the result feeds ranking_metrics unchanged
    from gdr import synth
    cfg = synth.BIPARTITE[name]
    tu, ti = synth.bipartite_interactions(cfg["users"], cfg["items"], 200000, 1234 + {"C": 2, "D": 3}[name] + 1)
    T = sp.csr_matrix((np.ones(len(tu), np.float32), (tu, ti)), shape=(cfg["users"], cfg["items"]))
    T.sum_duplicates()
    T.sort_indices()
    expanded = gdr.recommend_topk(Ue, Ie, 20, exclude=R)
    assert gdr.ranking_metrics(got[1], T, ks=(1, 20)) == gdr.ranking_metrics(expanded[1], T, ks=(1, 20))
