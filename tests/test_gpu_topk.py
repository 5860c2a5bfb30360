"""Full-ranking top-K recommendation and Recall / Precision / NDCG@K on the GPU: bit-exact items and scores against
the CPU reference (topk_ref.c, the same fmaf chain), the tie-heavy rows of a condensed model, full-size runs at the
Yelp2018 / Amazon-book shapes, and agreement with an fp32 torch product outside the rounding band."""
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


class forced_path:
    """gdr_debug_set("topk_path"): 1 exact SIMT path, 2 tensor-core screen (d <= 128); restored to automatic after."""

    def __init__(self, path):
        self.path = path

    def __enter__(self):
        from gdr import _lib
        _lib.call("gdr_debug_set", b"topk_path", self.path)

    def __exit__(self, *exc):
        from gdr import _lib
        _lib.call("gdr_debug_set", b"topk_path", 0)


def overflow_rows():
    import ctypes
    from gdr import _lib
    v = ctypes.c_int64(0)
    _lib.call("gdr_debug_get", b"topk_overflow_rows", ctypes.addressof(v))
    return v.value


def _data(n_users, n_items, d, seed):
    rs = np.random.RandomState(seed)
    U = rs.standard_normal((n_users, d)).astype(np.float32)
    I = rs.standard_normal((n_items, d)).astype(np.float32)
    U[0] = 0          # zero users tie across the whole row
    U[5] = 0
    I[20] = I[10]     # equal item rows tie everywhere
    I[n_items - 1] = I[10]
    # ~5% of the items per user excluded; user 3 keeps only 10 items (fewer than k: padding)
    R = sp.random(n_users, n_items, density=0.05, format="csr", random_state=rs, dtype=np.float32)
    R = R.tolil()
    R[3, :] = 1.0
    R[3, :10] = 0.0
    R = R.tocsr()
    R.eliminate_zeros()
    R.sort_indices()
    rows = np.concatenate([[0, 3, 5, 3], rs.randint(0, n_users, 93)]).astype(np.int64)
    return U, I, R, rows


def _check(gdr, U, I, k, R=None, rows=None):
    ex = None if R is None else gdr.CSR.from_scipy(R, device=DEV)
    s, it = gdr.recommend_topk(torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV), k, exclude=ex,
                               rows=None if rows is None else torch.from_numpy(rows).to(DEV))
    rs_, ri = topk_ref.topk(U, I, k, None if R is None else R.indptr, None if R is None else R.indices, rows)
    assert it.dtype == torch.int64 and s.dtype == torch.float32
    np.testing.assert_array_equal(it.cpu().numpy(), ri)
    assert np.array_equal(s.cpu().numpy().view(np.uint32), rs_.view(np.uint32)), "scores are not bit-identical"
    return s, it


@pytest.mark.parametrize("path", [1, 2])
@pytest.mark.parametrize("n_items", [1000, 5003])
@pytest.mark.parametrize("d", [1, 7, 47, 64, 100, 128, 200])
def test_topk_bit_exact_against_reference(gdr, d, n_items, path):
    if path == 2 and d > 128:
        pytest.skip("the tensor-core screen covers d <= 128")
    U, I, R, rows = _data(300, n_items, d, seed=d * 7 + n_items)
    with forced_path(path):
        for k in (1, 20, 100):
            _check(gdr, U, I, k)
            _, it = _check(gdr, U, I, k, R)
            if path == 2:
                assert overflow_rows() >= 2   # the two zero users tie across the whole row
            _check(gdr, U, I, k, R, rows)
            if k > 10:   # user 3 has 10 eligible items
                assert (it[3, 10:] == -1).all()


def test_tensor_core_path_rejects_wide_d(gdr):
    U, I, _, _ = _data(50, 300, 200, seed=3)
    with forced_path(2), pytest.raises(gdr.GdrError):
        gdr.recommend_topk(torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV), 5)


def test_topk_exclusion_formats_agree(gdr):
    U, I, R, rows = _data(200, 1000, 16, seed=1)
    Ut, It = torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV)
    ref = gdr.recommend_topk(Ut, It, 20, exclude=gdr.CSR.from_scipy(R, device=DEV))
    coo = R.tocoo()
    idx = torch.from_numpy(np.stack([coo.row, coo.col]).astype(np.int64))
    dup = torch.sparse_coo_tensor(torch.cat([idx, idx], 1), torch.ones(2 * coo.nnz), R.shape).to(DEV)   # duplicates
    for ex in (R, dup):
        s, it = gdr.recommend_topk(Ut, It, 20, exclude=ex)
        assert torch.equal(s, ref[0]) and torch.equal(it, ref[1])


def test_topk_condensed_model_ties(gdr):
    """Embeddings expanded through the stored user -> cluster / item -> cluster maps of a condensed model: whole
    groups of users and items share one vector, so scores tie in long runs."""
    g = golden("recsys_ali_subset.npz")
    u2cu, i2ci = g["u2cu"], g["i2ci"]
    rs = np.random.RandomState(5)
    Ucl = rs.standard_normal((int(u2cu.max()) + 1, 64)).astype(np.float32)
    Icl = rs.standard_normal((int(i2ci.max()) + 1, 64)).astype(np.float32)
    U, I = Ucl[u2cu], Icl[i2ci]
    R = sp.csr_matrix((np.ones(len(g["r_indices"]), np.float32), g["r_indices"], g["r_indptr"]), shape=(len(u2cu), len(i2ci)))
    rows = rs.choice(len(u2cu), 600, replace=False).astype(np.int64)
    for path in (1, 2):
        with forced_path(path):
            for k in (20, 100):
                _check(gdr, U, I, k, R, rows)


def test_topk_rejects_non_finite_and_bad_rows(gdr):
    U, I, _, _ = _data(50, 300, 8, seed=2)
    for bad in ("U", "I"):
        U2, I2 = U.copy(), I.copy()
        (U2 if bad == "U" else I2)[7, 3] = np.nan if bad == "U" else np.inf
        for path in (1, 2):
            with forced_path(path), pytest.raises(ValueError, match="non-finite"):
                gdr.recommend_topk(torch.from_numpy(U2).to(DEV), torch.from_numpy(I2).to(DEV), 5)
    with pytest.raises(ValueError, match="outside"):
        gdr.recommend_topk(torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV), 5,
                           rows=torch.tensor([1, 50], device=DEV))
    with pytest.raises(ValueError):
        gdr.recommend_topk(torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV), 301)


def _zscore(x):
    return ((x - x.mean(0)) / x.std(0)).astype(np.float32)


def _bench_inputs(gdr, name):
    from gdr import synth
    cfg = synth.BIPARTITE[name]
    seed = 1234 + {"C": 2, "D": 3}[name]   # bench.py's seeds
    u, i = synth.bipartite_interactions(cfg["users"], cfg["items"], cfg["inter"], seed)
    rs = np.random.RandomState(seed + 100)
    U = _zscore(0.1 * rs.standard_normal((cfg["users"], 64)))
    I = _zscore(0.1 * rs.standard_normal((cfg["items"], 64)))
    R = gdr.coo_to_csr(u, i, None, (cfg["users"], cfg["items"]), device=DEV)
    return U, I, R, seed


@pytest.mark.parametrize("name", ["C", "D"])
def test_topk_full_size(gdr, name):
    U, I, R, seed = _bench_inputs(gdr, name)
    Ut, It = torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV)
    with forced_path(2):
        s, it = gdr.recommend_topk(Ut, It, 20, exclude=R)
        s2, it2 = gdr.recommend_topk(Ut, It, 20, exclude=R)
    assert torch.equal(it, it2) and torch.equal(s, s2), "two runs differ"
    with forced_path(1):
        se, ie = gdr.recommend_topk(Ut, It, 20, exclude=R)
    assert torch.equal(it, ie) and torch.equal(s, se), "tensor-core and exact paths differ"
    assert (it >= 0).all()
    sample = np.random.RandomState(seed).choice(U.shape[0], 48, replace=False).astype(np.int64)
    Rs = R.to_scipy()
    rs_, ri = topk_ref.topk(U, I, 20, Rs.indptr, Rs.indices, sample)
    np.testing.assert_array_equal(it[torch.from_numpy(sample).to(DEV)].cpu().numpy(), ri)
    assert np.array_equal(s[torch.from_numpy(sample).to(DEV)].cpu().numpy().view(np.uint32), rs_.view(np.uint32))


def test_topk_agrees_with_torch_outside_rounding_band(gdr):
    """fp32 cuBLAS (TF32 off) + masked_fill + topk picks the same set wherever the exact k-th and (k+1)-th scores
    differ by more than 2^-15 |u| max|i|."""
    U, I, R, _ = _bench_inputs(gdr, "C")
    U, I = U[:6000], I
    R = gdr.CSR.from_scipy(R.to_scipy()[:6000], device=DEV)
    k = 20
    Ut, It = torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV)
    s, it = gdr.recommend_topk(Ut, It, k + 1, exclude=R)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        S = Ut @ It.T
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    S[R.coo_indices()[0], R.coo_indices()[1]] = -float("inf")
    _, ti = torch.topk(S, k, dim=1)
    band = 2.0 ** -15 * Ut.norm(dim=1) * It.norm(dim=1).max()
    clear = (s[:, k - 1] - s[:, k]) > band
    assert clear.float().mean() > 0.5
    ours = torch.sort(it[:, :k], dim=1).values
    theirs = torch.sort(ti, dim=1).values
    assert torch.equal(ours[clear], theirs[clear])


def test_metrics_against_reference(gdr):
    U, I, R, seed = _bench_inputs(gdr, "C")
    from gdr import synth
    n_users, n_items = U.shape[0], I.shape[0]
    tu, ti = synth.bipartite_interactions(n_users, n_items, 200000, seed + 1)
    T = sp.csr_matrix((np.ones(len(tu), np.float32), (tu, ti)), shape=(n_users, n_items))
    T.sum_duplicates()
    T.sort_indices()
    Ut, It = torch.from_numpy(U).to(DEV), torch.from_numpy(I).to(DEV)
    _, it = gdr.recommend_topk(Ut, It, 20, exclude=R)
    ks = (1, 5, 20)
    got = gdr.ranking_metrics(it, T, ks=ks)
    want = topk_ref.metrics(it.cpu().numpy(), T.indptr, T.indices, ks)
    assert got["n_eval"] == want["n_eval"] and got["n_skipped"] == want["n_skipped"] and got["n_skipped"] > 0
    for key in want:
        if "@" in key:
            assert got[key] == pytest.approx(want[key], rel=1e-12, abs=0), key
    assert got == gdr.ranking_metrics(it, gdr.CSR.from_scipy(T, device=DEV), ks=ks)   # deterministic
    # a subset of users through `rows`
    rows = np.arange(0, n_users, 7, dtype=np.int64)
    _, itr = gdr.recommend_topk(Ut, It, 20, exclude=R, rows=rows)
    got_r = gdr.ranking_metrics(itr, T, ks=(20,), rows=rows)
    want_r = topk_ref.metrics(itr.cpu().numpy(), T.indptr, T.indices, (20,), rows=rows)
    for key in ("recall@20", "precision@20", "ndcg@20"):
        assert got_r[key] == pytest.approx(want_r[key], rel=1e-12, abs=0), key
