"""The per-cluster sums on a row partition (numpy model in segment_sum_dist_ref.py): bit-equal to the one-GPU order
(oracle.segment_sum) at worlds 1-8, with equal blocks, arbitrary cuts, empty and trailing-empty ranks, a cluster whose
members span every rank, rows of -0.0 and more clusters than rows."""
import numpy as np
import pytest

import segment_sum_dist_ref as ref


def _data(N, D=5, K=7, seed=0):
    rs = np.random.RandomState(seed + 31 * N + K)
    # magnitudes spread over many binades: a chain cut or re-associated anywhere changes the last bits
    X = (rs.standard_normal((N, D)) * np.exp(rs.uniform(-10, 10, (N, 1)))).astype(np.float32)
    lab = rs.randint(0, K, N).astype(np.int32)
    return X, lab


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.int32)


def _check(oracle, X, lab, K, cuts):
    sums, counts, msgs = ref.segment_sum_dist(ref.cut(X, cuts), ref.cut(lab, cuts), K)
    s1, c1 = oracle.segment_sum(X, lab, K)
    np.testing.assert_array_equal(_bits(sums), _bits(s1))
    np.testing.assert_array_equal(counts, c1)
    return msgs


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("N", [1, 5, 64, 999, 4000])
def test_equal_blocks_bit_equal_to_one_gpu(oracle, N, world):
    X, lab = _data(N)
    _check(oracle, X, lab, 7, ref.equal_cuts(N, world))


@pytest.mark.parametrize("cuts", [[0, 0, 700, 700, 2900, 3001], [0, 1, 2, 2049, 3000, 3001], [0, 3001, 3001, 3001],
                                  [0, 0, 0, 3001], [0, 17, 1500, 1501, 2222, 2223, 2800, 3001]])
def test_arbitrary_cuts(oracle, cuts):
    X, lab = _data(3001, K=40)
    _check(oracle, X, lab, 40, cuts)


def test_empty_and_trailing_empty_ranks(oracle):
    N, world = 5, 4                           # blocks of 2 rows: rank 3 holds none
    X, lab = _data(N, K=3)
    cuts = ref.equal_cuts(N, world)
    assert np.diff(cuts).tolist() == [2, 2, 1, 0]
    msgs = _check(oracle, X, lab, 3, cuts)
    np.testing.assert_array_equal(_bits(msgs[3]), _bits(msgs[2]))   # the empty rank hands on what it received
    N, world = 10, 8                          # blocks of 2 rows: ranks 5, 6 and 7 hold none
    X, lab = _data(N, K=4)
    cuts = ref.equal_cuts(N, world)
    assert np.diff(cuts).tolist() == [2, 2, 2, 2, 2, 0, 0, 0]
    _check(oracle, X, lab, 4, cuts)
    _check(oracle, X, lab, 4, [0, 0, 3, 3, 3, 7, 10, 10, 10])       # empty ranks in front and in the middle too


@pytest.mark.parametrize("world", [2, 3, 4, 5, 6, 7, 8])
def test_one_cluster_through_every_rank(oracle, world):
    N = 800
    X, lab = _data(N, K=5)
    lab[::97] = 4                            # cluster 4: a few members in every block
    cuts = ref.equal_cuts(N, world)
    assert all((lab[a:b] == 4).any() for a, b in zip(cuts[:-1], cuts[1:]))
    _check(oracle, X, lab, 5, cuts)


def test_negative_zero_rows(oracle):
    X, lab = _data(200, K=6)
    X[lab == 2] = -0.0                        # a cluster of -0.0 rows sums to +0.0 from +0.0, on every rank
    X[::3, 1] = -0.0
    for world in range(1, 9):
        sums, _, _ = ref.segment_sum_dist(ref.cut(X, ref.equal_cuts(200, world)),
                                          ref.cut(lab, ref.equal_cuts(200, world)), 6)
        assert not np.signbit(sums[2]).any()
        _check(oracle, X, lab, 6, ref.equal_cuts(200, world))


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_more_clusters_than_rows(oracle, world):
    X, lab = _data(13, K=50)
    _check(oracle, X, lab, 50, ref.equal_cuts(13, world))
    X, lab = _data(3, K=10)
    _check(oracle, X, lab, 10, ref.equal_cuts(3, world))


def test_restarting_the_chain_at_a_rank_boundary_changes_the_bits(oracle):
    """Negative control: each rank chaining from +0.0, with the ranks' sums added in rank order, gives other bits, so
    the tests above do see how the chains are split."""
    N, K = 999, 7
    X, lab = _data(N, K=K)
    blocks = ref.equal_cuts(N, 8)
    got = ref.restarted_per_rank(ref.cut(X, blocks), ref.cut(lab, blocks), K)
    s1, _ = oracle.segment_sum(X, lab, K)
    assert not np.array_equal(_bits(got), _bits(s1))
