"""The row-partitioned k-means++ protocol (numpy model in kpp_dist_ref.py) against sklearn's golden picks and on the
cases where the rank structure shows: empty ranks, a rank with zero potential, a threshold on a rank boundary, the
clip rule, K = 1 and K = N."""
import numpy as np
import pytest

from conftest import golden
import kpp_dist_ref as ref


@pytest.mark.parametrize("k", [25, 60, 200])
@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 6, 7, 8])
def test_golden_picks_every_world_size(k, world):
    g = golden("kmeans_plusplus.npz")
    X = g["x"]
    first, rand = ref.draws(np.random.RandomState(int(g[f"k{k}_seed"])), X.shape[0], k)
    got = ref.kpp_dist(ref.row_blocks(X, world), k, first, rand)
    np.testing.assert_array_equal(got, g[f"k{k}_indices"])


def test_empty_ranks():
    g = golden("kmeans_plusplus.npz")
    X = g["x"]
    first, rand = ref.draws(np.random.RandomState(int(g["k60_seed"])), X.shape[0], 60)
    blocks = [X[:0], X[:1500], X[:0], X[1500:1501], X[1501:], X[:0]]
    np.testing.assert_array_equal(ref.kpp_dist(blocks, 60, first, rand), g["k60_indices"])
    # more ranks than rows
    Xs = X[:5]
    first, rand = ref.draws(np.random.RandomState(3), 5, 5)
    one = ref.kpp_dist([Xs], 5, first, rand)
    assert sorted(one) == list(range(5))
    np.testing.assert_array_equal(ref.kpp_dist(ref.row_blocks(Xs, 8), 5, first, rand), one)


def test_rank_with_zero_potential():
    # rank 1 holds copies of the first centre: T_1 = 0 after the start-up, its rows are never drawn again
    rng = np.random.RandomState(5)
    A = rng.randn(300, 3).astype(np.float32)
    B = np.repeat(A[:1], 200, axis=0)
    C = rng.randn(250, 3).astype(np.float32)
    X = np.concatenate([A, B, C])
    first = 0
    rand = np.random.RandomState(6).uniform(size=(19, 4))
    blocks = [A, B, C]
    got = ref.kpp_dist(blocks, 20, first, rand)
    np.testing.assert_array_equal(got, ref.kpp_dist([X], 20, first, rand))
    assert not np.any((got[1:] >= 300) & (got[1:] < 500))


def test_threshold_on_a_rank_boundary():
    # distances to the first centre (row 0): [0, 4, 0 | 0, 4, 4, 4], pot = 16; u = 0.25 puts the threshold exactly on
    # P_1 = 4: the first rank whose prefix reaches it (rank 0) owns the draw and its row 1 is the first to reach it
    X = np.array([[0.0], [2.0], [0.0], [0.0], [2.0], [2.0], [2.0]], dtype=np.float32)
    rand = np.array([[0.25, 0.25, 0.25]])
    for blocks in ([X], [X[:3], X[3:]], [X[:3], X[3:3], X[3:]]):
        assert ref.kpp_dist(blocks, 2, 0, rand).tolist() == [0, 1]


def test_clip_rule():
    # a draw above the total potential is reached by no row: np.clip puts it on the last global row, also when the
    # last rank is empty
    X = np.arange(10, dtype=np.float32)[:, None]
    rand = np.array([[1.0 + 2.0 ** -40, 1.0 + 2.0 ** -40, 1.0 + 2.0 ** -40]])
    for blocks in ([X], ref.row_blocks(X, 3), [X[:4], X[4:], X[:0]]):
        assert ref.kpp_dist(blocks, 2, 3, rand).tolist() == [3, 9]


def test_k_one_and_k_n():
    rng = np.random.RandomState(9)
    X = rng.randn(40, 4).astype(np.float32)
    first, rand = ref.draws(np.random.RandomState(10), 40, 1)
    for w in (1, 3, 8):
        assert ref.kpp_dist(ref.row_blocks(X, w), 1, first, rand).tolist() == [first]
    first, rand = ref.draws(np.random.RandomState(11), 40, 40)
    one = ref.kpp_dist([X], 40, first, rand)
    assert sorted(one.tolist()) == list(range(40))
    for w in (2, 3, 8):
        np.testing.assert_array_equal(ref.kpp_dist(ref.row_blocks(X, w), 40, first, rand), one)


def test_dist_kmeans_string_init_arguments():
    import torch
    from gdr import parallel as par
    X = torch.zeros((10, 2))
    with pytest.raises(ValueError):
        par.DistKMeans(3, "k-means++", ops=object()).fit(X)       # random_state is required
    with pytest.raises(ValueError):
        par.DistKMeans(3, "kmeans++", random_state=0, ops=object()).fit(X)
    for init in ("k-means++", "random"):
        with pytest.raises(NotImplementedError):
            par.DistKMeans(3, init, random_state=0, ops=object()).fit(X)
    with pytest.raises(NotImplementedError):
        par.dist_kmeans_plusplus(par.Comm(), par.RowPartition(10, 1, 0), X, 3, np.random.RandomState(0), ops=object())
