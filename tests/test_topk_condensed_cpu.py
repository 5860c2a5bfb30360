"""CPU checks of the condensed top-K: the numpy mirror of the cluster walk (topk_condensed_ref) against topk_ref on the
expanded tables, argument rejection of gdr_topk_condensed[_ws_bytes] before any device work, and the workspace bound
at the Amazon-book shape."""
import numpy as np
import pytest

import topk_condensed_ref
import topk_ref

FAKE = 256   # a non-null pointer that the argument checks must reject before it is ever dereferenced


def _exclusion(rs, n_users, n_items, density, heavy=()):
    rowptr, cols = [0], []
    for u in range(n_users):
        p = 0.9 if u in heavy else density
        row = np.flatnonzero(rs.random_sample(n_items) < p)
        cols.extend(row.tolist())
        rowptr.append(len(cols))
    return np.asarray(rowptr, np.int32), np.asarray(cols, np.int32)


def _case(seed, n_users=60, n_items=90, n_cu=7, n_ci=12, d=5, ties=False):
    rs = np.random.RandomState(seed)
    # integer embeddings: scores are exact and tie often
    Ucl = rs.randint(-2, 3, (n_cu, d)).astype(np.float32)
    Icl = rs.randint(-2, 3, (n_ci, d)).astype(np.float32)
    if ties:
        Ucl[0] = 0                   # a zero super-user: every cluster ties
        Ucl[1] = -0.0                # -0 scores, ordered and reported as +0
        Icl[3] = Icl[2]              # duplicated cluster vectors: ties across distinct clusters
        Icl[5] = Icl[2]
        Icl[4] = -Icl[6]
    u2cu = rs.randint(0, n_cu, n_users).astype(np.int64)
    i2ci = rs.randint(0, n_ci, n_items).astype(np.int64)
    if ties:
        u2cu[:3] = [0, 1, 0]
        i2ci[i2ci == n_ci - 1] = 0   # an empty cluster
        i2ci[0] = 7                  # cluster 7 of size 1
        i2ci[i2ci == 7] = 8
        i2ci[0] = 7
    return Ucl, Icl, u2cu, i2ci


def _check(Ucl, Icl, k, u2cu, i2ci, rp=None, ci=None, rows=None):
    s, it, fb = topk_condensed_ref.topk_condensed(Ucl, Icl, k, u2cu, i2ci, rp, ci, rows)
    rs_, ri = topk_ref.topk(Ucl[u2cu], Icl[i2ci], k, rp, ci, rows)
    np.testing.assert_array_equal(it, ri)
    assert np.array_equal(s.view(np.uint32), rs_.view(np.uint32))
    return fb


@pytest.mark.parametrize("seed", range(6))
def test_walk_matches_expanded_reference_random(seed):
    Ucl, Icl, u2cu, i2ci = _case(seed)
    rs = np.random.RandomState(100 + seed)
    rp, ci = _exclusion(rs, len(u2cu), len(i2ci), 0.1, heavy=(4, 9))
    for k in (1, 5, 20, len(i2ci)):
        _check(Ucl, Icl, k, u2cu, i2ci)
        _check(Ucl, Icl, k, u2cu, i2ci, rp, ci)
        _check(Ucl, Icl, k, u2cu, i2ci, rp, ci, rows=np.array([4, 4, 9, 0, 17, 59]))


@pytest.mark.parametrize("seed", range(4))
def test_walk_matches_expanded_reference_ties(seed):
    Ucl, Icl, u2cu, i2ci = _case(seed, n_ci=40, n_items=120, ties=True)
    Icl[39] = np.nan   # an empty cluster: never read
    rs = np.random.RandomState(200 + seed)
    rp, ci = _exclusion(rs, len(u2cu), len(i2ci), 0.05, heavy=(2,))
    for k in (1, 3, 20, 119, 120):
        fb = _check(Ucl, Icl, k, u2cu, i2ci, rp, ci)
        assert 0 in fb   # user 0's super-user is zero: one tie run of every non-empty cluster (> 32)
        _check(Ucl, Icl, k, u2cu, i2ci)


def test_walk_pads_short_rows():
    Ucl, Icl, u2cu, i2ci = _case(3)
    n_items = len(i2ci)
    rp = np.array([0, n_items - 4] + [n_items - 4] * (len(u2cu) - 1), np.int32)   # user 0 keeps 4 items
    ci = np.arange(n_items - 4, dtype=np.int32)
    s, it, _ = topk_condensed_ref.topk_condensed(Ucl, Icl, 10, u2cu, i2ci, rp, ci)
    assert (it[0, 4:] == -1).all() and np.isneginf(s[0, 4:]).all() and (it[0, :4] >= n_items - 4).all()
    _check(Ucl, Icl, 10, u2cu, i2ci, rp, ci)


def test_walk_identity_maps_equal_plain_topk():
    rs = np.random.RandomState(9)
    U = rs.standard_normal((30, 6)).astype(np.float32)
    I = rs.standard_normal((50, 6)).astype(np.float32)
    rp, ci = _exclusion(rs, 30, 50, 0.2)
    s, it, fb = topk_condensed_ref.topk_condensed(U, I, 7, np.arange(30), np.arange(50), rp, ci)
    rs_, ri = topk_ref.topk(U, I, 7, rp, ci)
    assert not fb
    np.testing.assert_array_equal(it, ri)
    assert np.array_equal(s.view(np.uint32), rs_.view(np.uint32))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from gdr import _lib
    return _lib


def _call(lib, n_rows=4, n_users=4, n_items=10, n_cu=2, n_ci=3, d=8, k=3, U=FAKE, I=FAKE, umap=FAKE, imap=FAKE,
          exr=0, exc=0, ws=FAKE, ws_bytes=1 << 40, ld=None, lds=None):
    ld = d if ld is None else ld
    lds = k if lds is None else lds
    return lib.call("gdr_topk_condensed", n_rows, n_users, n_items, n_cu, n_ci, d, k, U, ld, I, ld, umap, imap, 0, exr,
                    exc, FAKE, lds, FAKE, k, FAKE, ws, ws_bytes, 0)


@pytest.mark.parametrize("kw", [dict(k=0), dict(k=11), dict(n_cu=0), dict(n_ci=0), dict(d=0), dict(U=0), dict(I=0),
                                dict(umap=0), dict(imap=0), dict(ws=0), dict(ld=4), dict(lds=2), dict(n_rows=5),
                                dict(exr=FAKE), dict(exc=FAKE)])
def test_condensed_rejects_bad_arguments(lib, kw):
    with pytest.raises(lib.GdrError) as e:
        _call(lib, **kw)
    assert e.value.code == -1


def test_condensed_rejects_small_workspace(lib):
    need = lib.query("gdr_topk_condensed_ws_bytes", 4, 4, 10, 2, 3, 8, 3)
    with pytest.raises(lib.GdrError) as e:
        _call(lib, ws_bytes=need - 1)
    assert e.value.code == -2


def test_condensed_workspace_is_bounded_by_shapes(lib):
    # Amazon-book shape at a 10 % condensation rate; the expanded score matrix would be 19 GB
    for k in (20, 100, 91599):
        wsb = lib.query("gdr_topk_condensed_ws_bytes", 52643, 52643, 91599, 5265, 9160, 64, k)
        assert 0 < wsb < 512 << 20, (k, wsb)
    # identity maps (no condensation) stay bounded too
    assert lib.query("gdr_topk_condensed_ws_bytes", 52643, 52643, 91599, 52643, 91599, 64, 20) < 1 << 30
