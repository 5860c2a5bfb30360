"""CPU checks of the mini-batch assembly on a row partition: parallel.batch_plan with the numpy model of pack ->
rank-order exchange -> place (tests/minibatch_dist_ref.py) reproduces X[idx] and puts every row's label at its
position, for worlds 1-8, random and empty row blocks, duplicate ids, ids on block boundaries, all ids on one rank and
a batch of one.  Also: the RandomState digest separates different states and matches equal ones."""
import numpy as np
import pytest

from minibatch_dist_ref import assemble, nearest, split_rows


def _plan():
    from gdr import parallel as par
    return par.batch_plan


def _random_offsets(rs, N, world, n_empty=0):
    cuts = np.sort(rs.randint(0, N + 1, world - 1))
    if n_empty:
        for r in rs.choice(world, size=min(n_empty, world - 1), replace=False):
            if 0 < r < world:
                cuts[r - 1] = cuts[r - 2] if r >= 2 else 0
        cuts = np.sort(cuts)
    return np.concatenate([[0], cuts, [N]]).astype(np.int64)


def _check(X, row_off, idx, C=None):
    order, counts = _plan()(idx, row_off)
    assert order.dtype == np.int32 and counts.dtype == np.int64
    assert counts.shape == (len(row_off) - 1,) and counts.sum() == len(idx)
    # grouped by owner in rank order, ascending within an owner
    owner = np.searchsorted(row_off, idx, side="right") - 1
    assert np.all(np.diff(owner[order]) >= 0)
    offs = np.concatenate([[0], np.cumsum(counts)])
    for r in range(len(counts)):
        seg = order[offs[r]:offs[r + 1]]
        assert np.all(np.diff(seg) > 0)
        assert np.all((idx[seg] >= row_off[r]) & (idx[seg] < row_off[r + 1]))
    Xb, lab = assemble(split_rows(X, row_off), row_off, idx, order, counts, None if C is None else nearest(C))
    np.testing.assert_array_equal(Xb.view(np.int32), X[idx].view(np.int32))
    if C is not None:
        np.testing.assert_array_equal(lab, nearest(C)(X[idx]))


@pytest.mark.parametrize("world", range(1, 9))
def test_random_blocks(world):
    rs = np.random.RandomState(100 + world)
    N, D = 3000, 7
    X = rs.standard_normal((N, D)).astype(np.float32)
    C = rs.standard_normal((13, D)).astype(np.float32)
    for n_empty in (0, 1, world // 2):
        row_off = _random_offsets(rs, N, world, n_empty)
        for m in (1, 17, 1000, 2049):
            _check(X, row_off, rs.randint(0, N, m).astype(np.int64), C)


@pytest.mark.parametrize("world", [2, 3, 5, 8])
def test_duplicates_boundaries_and_one_owner(world):
    rs = np.random.RandomState(world)
    N, D = 500, 5
    X = rs.standard_normal((N, D)).astype(np.float32)
    C = rs.standard_normal((4, D)).astype(np.float32)
    row_off = _random_offsets(rs, N, world, 1)
    # every block's first and last row, each several times
    edges = np.concatenate([row_off[:-1], row_off[1:] - 1])
    edges = edges[(edges >= 0) & (edges < N)]
    _check(X, row_off, np.repeat(edges, 3)[rs.permutation(3 * len(edges))].astype(np.int64), C)
    # one id, many times
    _check(X, row_off, np.full(64, 7, np.int64), C)
    # all ids owned by the last rank with rows
    r = int(np.nonzero(np.diff(row_off))[0][-1])
    _check(X, row_off, rs.randint(row_off[r], row_off[r + 1], 300).astype(np.int64), C)
    # a batch of one on each boundary
    for e in edges:
        _check(X, row_off, np.array([e], np.int64), C)


def test_the_rank_without_rows_of_the_issue_layout():
    rs = np.random.RandomState(9)
    row_off = np.array([0, 9000, 20000, 20000, 30011], np.int64)
    X = rs.standard_normal((30011, 3)).astype(np.float32)
    idx = np.concatenate([[8999, 9000, 19999, 20000, 30010], rs.randint(0, 30011, 2043)]).astype(np.int64)
    order, counts = _plan()(idx, row_off)
    assert counts[2] == 0 and counts.sum() == 2048
    _check(X, row_off, idx, rs.standard_normal((9, 3)).astype(np.float32))


def test_plan_rejects_ids_outside_the_rows():
    with pytest.raises(ValueError):
        _plan()(np.array([0, 10], np.int64), np.array([0, 5, 10], np.int64))
    with pytest.raises(ValueError):
        _plan()(np.array([-1], np.int64), np.array([0, 5, 10], np.int64))


def test_state_digest():
    from gdr import parallel as par
    a, b = np.random.RandomState(3), np.random.RandomState(3)
    assert par.random_state_digest(a) == par.random_state_digest(b)
    assert par.random_state_digest(a) != par.random_state_digest(np.random.RandomState(4))
    a.random_sample(1)
    assert par.random_state_digest(a) != par.random_state_digest(b)
    b.random_sample(1)
    assert par.random_state_digest(a) == par.random_state_digest(b)
    a.standard_normal()       # the cached Gaussian is part of the state
    b.standard_normal()
    assert par.random_state_digest(a) == par.random_state_digest(b)
    st = a.get_state()
    c = np.random.RandomState()
    c.set_state(st)
    assert par.random_state_digest(c) == par.random_state_digest(a)
