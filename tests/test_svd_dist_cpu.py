"""The Gram matrix on a row partition (numpy model in svd_dist_ref.py): bit-equal to the one-GPU slab order at worlds
1-8, including one slab through every rank, slabs spanning several ranks, empty ranks and uneven last blocks."""
import numpy as np
import pytest

import svd_dist_ref as ref


def _data(N, p=3, r=2, seed=0):
    rs = np.random.RandomState(seed + N)
    # magnitudes spread over many binades: a chain cut or re-associated anywhere changes the last bits
    A = rs.standard_normal((N, p)) * np.exp(rs.uniform(-8, 8, (N, 1)))
    B = rs.standard_normal((N, r)) * np.exp(rs.uniform(-8, 8, (N, 1)))
    return A, B


def _bits(x):
    return np.ascontiguousarray(x).view(np.int64)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("N", [1, 10, 1500, 2047, 2048, 2049, 16 * 2048 - 1, 16 * 2048 + 1])
def test_equal_blocks_bit_equal_to_one_gpu(N, world):
    A, B = _data(N)
    C, _ = ref.gram_dist(ref.equal_blocks(A, world), ref.equal_blocks(B, world))
    np.testing.assert_array_equal(_bits(C), _bits(ref.gram_one(A, B)))


def test_one_gpu_model_is_the_gram():
    A, B = _data(5003)
    np.testing.assert_allclose(ref.gram_one(A, B), A.T @ B, rtol=1e-12, atol=1e-12 * np.abs(A.T @ B).max())


def test_one_slab_through_every_rank():
    N, world = 1500, 8
    assert ref.slab_geometry(N) == (1, 1500)
    A, B = _data(N)
    C, msgs = ref.gram_dist(ref.equal_blocks(A, world), ref.equal_blocks(B, world))
    # no rank before the last completes the slab: the running sum stays 0.0 and the carry travels
    assert all(not m[1].any() and m[0] is not None for m in msgs[:-1])
    np.testing.assert_array_equal(_bits(C), _bits(ref.gram_one(A, B)))


def test_slab_spanning_four_ranks():
    N, world = 2049, 8                        # 2 slabs of 1025 rows, blocks of 257: slab 0 covers ranks 0-3
    blocks = [(r * 257, min(N, (r + 1) * 257)) for r in range(world)]
    spanned = [r for r, (lo, hi) in enumerate(blocks) if any(a < 1025 for a, _, _, _ in ref.segments(N, lo, hi))]
    assert spanned == [0, 1, 2, 3]
    A, B = _data(N)
    C, _ = ref.gram_dist(ref.equal_blocks(A, world), ref.equal_blocks(B, world))
    np.testing.assert_array_equal(_bits(C), _bits(ref.gram_one(A, B)))


def test_empty_trailing_ranks():
    N, world = 10, 8                          # blocks of 2 rows: ranks 5, 6 and 7 hold none
    A, B = _data(N)
    bA = ref.equal_blocks(A, world)
    assert [a.shape[0] for a in bA] == [2, 2, 2, 2, 2, 0, 0, 0]
    C, msgs = ref.gram_dist(bA, ref.equal_blocks(B, world))
    assert all(np.array_equal(_bits(m[1]), _bits(C)) for m in msgs[4:])
    np.testing.assert_array_equal(_bits(C), _bits(ref.gram_one(A, B)))


@pytest.mark.parametrize("cuts", [[0, 0, 700, 700, 4100, 4100], [0, 1, 2, 2049, 6000, 6001], [0, 6001, 6001, 6001],
                                  [0, 0, 0, 6001], [0, 2048, 4096, 5000, 6001]])
def test_arbitrary_and_empty_blocks(cuts):
    A, B = _data(6001)
    cuts = cuts + [6001] if cuts[-1] != 6001 else cuts
    bA = [A[a:b] for a, b in zip(cuts[:-1], cuts[1:])]
    bB = [B[a:b] for a, b in zip(cuts[:-1], cuts[1:])]
    C, _ = ref.gram_dist(bA, bB)
    np.testing.assert_array_equal(_bits(C), _bits(ref.gram_one(A, B)))


def test_uneven_last_block():
    N, world = 16 * 2048 + 1, 4               # blocks of 8193 rows, the last of 8190
    A, B = _data(N)
    bA = ref.equal_blocks(A, world)
    assert bA[-1].shape[0] < bA[0].shape[0]
    C, _ = ref.gram_dist(bA, ref.equal_blocks(B, world))
    np.testing.assert_array_equal(_bits(C), _bits(ref.gram_one(A, B)))


def test_restarting_the_chain_at_a_rank_boundary_changes_the_bits():
    """Negative control: each rank's block chained from 0.0 and the blocks added in rank order (no carry) gives other
    bits, so the tests above do see how the chains are split."""
    N, world = 2049, 8
    A, B = _data(N)
    zero = np.zeros((3, 2))
    total = zero
    for a, b in zip(ref.equal_blocks(A, world), ref.equal_blocks(B, world)):
        total = total + ref.chain(zero, a, b)
    assert not np.array_equal(_bits(total), _bits(ref.gram_one(A, B)))
