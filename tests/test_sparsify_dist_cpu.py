"""The row-partitioned top-k protocol of gdr_sparsify_classes_dist (numpy model in sparsify_dist_ref.py) against the
one-GPU selection, oracle.topk_edges, at worlds 1-8: the golden graph for every sp_type the partition supports, ties
across one or several rank boundaries, k = 0 and k = nnz, empty ranks, NaN and signed zeros."""
import numpy as np
import pytest

from conftest import golden
import sparsify_dist_ref as ref

WORLDS = [1, 2, 3, 4, 5, 6, 7, 8]


def _golden_csr():
    g = golden("sparsify.npz")
    n = int(g["n"])
    rp = np.zeros(n + 1, np.int64)
    np.add.at(rp, g["src"] + 1, 1)
    return g, n, np.cumsum(rp).astype(np.int32), g["dst"].astype(np.int32), g["val"]


def _split(w, cuts):
    """Weights of the edge blocks [cuts[p], cuts[p+1])."""
    return [w[cuts[p]: cuts[p + 1]] for p in range(len(cuts) - 1)]


def _dist(w, cuts, k):
    return ref.concat_kept(ref.select_dist(_split(w, cuts), k), cuts)


@pytest.mark.parametrize("sp_type", ["vanilla", "single", "attaw"])
@pytest.mark.parametrize("world", WORLDS)
def test_golden_graph_every_world_size(oracle, sp_type, world):
    g, n, rp, ci, va = _golden_csr()
    ratio = float(g["ratio"])
    kept, k = ref.graph_sparse_dist(oracle, rp, ci, va, ratio, ref.row_bounds(n, world), ebd=g["ebd"], sp_type=sp_type)
    one = oracle.graph_sparse(rp, ci, va, ratio, ebd=g["ebd"], sp_type=sp_type)
    assert len(kept) == len(one) == (int(g["C"]) if sp_type == "attaw" else 1)
    er = oracle.er_lower(rp, ci, va) if sp_type == "vanilla" else oracle.attaw_er_lower(rp, ci, va, g["ebd"])[0]
    P = oracle.softmax_rows(g["ebd"])
    for c, idx in enumerate(kept):
        w = er if sp_type != "attaw" else oracle.class_edge_weight(rp, ci, er, P[:, c])
        np.testing.assert_array_equal(idx, oracle.topk_edges(w, k))
        # and the rebuilt CSR is the oracle's graph_sparse output
        rpo, cio, _ = oracle.filter_csr(rp, ci, va, idx)
        np.testing.assert_array_equal(rpo, one[c][0])
        np.testing.assert_array_equal(cio, one[c][1])


@pytest.mark.parametrize("world", WORLDS)
def test_all_weights_equal_quota_crosses_rank_boundaries(oracle, world):
    w = np.full(1000, 0.25, np.float32)
    cuts = ref.row_bounds(1000, world)
    for k in (1, 137, 499, 500, 501, 999, 1000):
        got = _dist(w, cuts, k)
        np.testing.assert_array_equal(got, oracle.topk_edges(w, k))
        assert got.tolist() == list(range(k))            # the first k in stored order, whatever the ranks


@pytest.mark.parametrize("world", WORLDS)
def test_ties_straddling_one_boundary(oracle, world):
    rng = np.random.RandomState(3)
    w = rng.rand(800).astype(np.float32)
    cuts = ref.row_bounds(800, world)
    b = cuts[1] if world > 1 else 400
    w[max(0, b - 20): b + 20] = np.float32(0.5)          # 40 ties around the first boundary
    above = int((w > 0.5).sum())
    for k in (above + 1, above + 15, above + 20, above + 21, above + 39, above + 40, above + 41):
        np.testing.assert_array_equal(_dist(w, cuts, k), oracle.topk_edges(w, k))


@pytest.mark.parametrize("world", WORLDS)
def test_k_zero_and_k_nnz(oracle, world):
    w = np.random.RandomState(4).randn(321).astype(np.float32)
    cuts = ref.row_bounds(321, world)
    assert _dist(w, cuts, 0).shape == (0,)
    np.testing.assert_array_equal(_dist(w, cuts, 321), np.arange(321))
    np.testing.assert_array_equal(_dist(w, cuts, 321), oracle.topk_edges(w, 321))


def test_empty_ranks_and_ranks_without_edges(oracle):
    g, n, rp, ci, va = _golden_csr()
    er = oracle.er_lower(rp, ci, va)
    k = int(va.shape[0] * float(g["ratio"]))
    nz = int(rp[n])
    # rows per rank: none, some, none, rows whose edges were all given to the neighbours (same cut twice), the rest
    cuts = [0, 0, 1200, 1200, 1200, 3000, nz, nz]
    np.testing.assert_array_equal(_dist(er, cuts, k), oracle.topk_edges(er, k))
    # more ranks than edges
    w = er[:5]
    np.testing.assert_array_equal(_dist(w, [0, 1, 2, 3, 4, 5, 5, 5], 3), oracle.topk_edges(w, 3))


@pytest.mark.parametrize("world", WORLDS)
def test_nan_sorts_above_inf(world):
    w = np.random.RandomState(5).randn(500).astype(np.float32)
    w[[7, 100, 101, 333]] = np.nan
    w[[8, 250]] = np.inf
    cuts = ref.row_bounds(500, world)
    for k in (1, 3, 4, 5, 6, 7, 50):
        got = _dist(w, cuts, k)
        np.testing.assert_array_equal(got, ref.select_global(w, k))
        assert set([7, 100, 101, 333][:k]) <= set(got.tolist())
        if k >= 6:
            assert {8, 250} <= set(got.tolist())


@pytest.mark.parametrize("world", WORLDS)
def test_negative_zero_below_positive_zero(world):
    w = np.zeros(60, np.float32)
    w[::2] = -0.0
    w[:10] = -1.0
    cuts = ref.row_bounds(60, world)
    for k in (10, 25, 26, 40, 50, 60):
        got = _dist(w, cuts, k)
        np.testing.assert_array_equal(got, ref.select_global(w, k))
        pos, neg = list(range(11, 60, 2)), list(range(10, 60, 2))   # +0.0 ranks above -0.0
        assert got.tolist() == sorted(pos[:k] + neg[: max(0, k - 25)] + list(range(max(0, k - 50))))


def test_one_rank_model_is_the_oracle_select(oracle):
    rng = np.random.RandomState(6)
    for _ in range(20):
        w = rng.choice(np.float32([-2, -1, 0.5, 1, 3]), size=200)
        k = int(rng.randint(0, 201))
        np.testing.assert_array_equal(ref.select_global(w, k), oracle.topk_edges(w, k))
        np.testing.assert_array_equal(ref.select_dist([w], k)[0], oracle.topk_edges(w, k))
