"""CPU checks of the BPR step: the numpy Philox4x32-10 of tests/bpr_ref.py against the Random123 known answers, the
complement select against brute force, the reference sampler's invariants, and argument validation of
gdr_bpr_sample / gdr_bpr_loss before any device work."""
import numpy as np
import pytest
import scipy.sparse as sp

import bpr_ref

FAKE = 256   # a non-null, 16-byte aligned pointer that the argument checks must reject before it is ever dereferenced


@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, want):
    got = bpr_ref.philox4x32_10(ctr, key)
    assert tuple(int(x) for x in got) == want


def test_draw_below_is_umulhi():
    rs = np.random.RandomState(0)
    lo = rs.randint(0, 1 << 32, 1000, dtype=np.uint64)
    hi = rs.randint(0, 1 << 32, 1000, dtype=np.uint64)
    n = rs.randint(1, 1 << 31, 1000).astype(np.uint64)
    got = bpr_ref.draw_below(lo, hi, n)
    want = [((int(h) << 32 | int(l)) * int(k)) >> 64 for l, h, k in zip(lo, hi, n)]
    assert got.tolist() == want and (got < n.astype(np.int64)).all()


@pytest.mark.parametrize("row", [[], list(range(1, 10)), list(range(0, 9)), [0, 2, 3, 7], [4], [0], [9]])
def test_complement_select_small_rows(row):
    n_items = 10
    comp = [j for j in range(n_items) if j not in set(row)]
    assert [bpr_ref.complement_select(row, r) for r in range(len(comp))] == comp


def test_complement_select_random_rows():
    rs = np.random.RandomState(1)
    for n_items in (2, 17, 300):
        for _ in range(30):
            k = rs.randint(0, n_items)
            row = np.sort(rs.choice(n_items, k, replace=False))
            comp = np.setdiff1d(np.arange(n_items), row)
            assert [bpr_ref.complement_select(row, r) for r in range(len(comp))] == comp.tolist()


def _random_csr(n_users, n_items, seed, density=0.1):
    rs = np.random.RandomState(seed)
    m = sp.random(n_users, n_items, density=density, format="csr", random_state=rs)
    m.data[:] = 1.0
    lil = m.tolil()
    lil[0, :] = 0                 # empty row
    lil[1, :] = 1                 # full row (not eligible)
    lil[2, :] = 1
    lil[2, 0] = 0                 # missing only item 0
    lil[3, :] = 1
    lil[3, n_items - 1] = 0       # missing only the last item
    m = lil.tocsr()
    m.eliminate_zeros()
    m.sort_indices()
    return m


def test_reference_sampler_invariants():
    R = _random_csr(60, 40, seed=2)
    for step in (0, 1, 2**32 - 1):
        users, pos, neg = bpr_ref.sample(R.indptr, R.indices, 40, seed=2**63 + 5, step=step, batch=5000)
        deg = np.diff(R.indptr)
        assert ((deg[users] > 0) & (deg[users] < 40)).all()
        dense = R.toarray() > 0
        assert dense[users, pos].all()
        assert not dense[users, neg].any()
        assert ((neg >= 0) & (neg < 40)).all()
        assert set(users.tolist()) >= {2, 3} and not set(users.tolist()) & {0, 1}
    # rows missing only item 0 / only the last item draw exactly that negative
    u, _, n = bpr_ref.sample(R.indptr, R.indices, 40, seed=7, step=0, batch=20000)
    assert (n[u == 2] == 0).all() and (n[u == 3] == 39).all()


def test_reference_sampler_distribution():
    # one eligible user with items {1, 4}: pos uniform over the row, neg uniform over the other 4 items
    R = sp.csr_matrix((np.ones(2), ([0, 0], [1, 4])), shape=(1, 6))
    _, pos, neg = bpr_ref.sample(R.indptr, R.indices, 6, seed=11, step=3, batch=60000)
    assert set(pos.tolist()) == {1, 4} and abs((pos == 1).mean() - 0.5) < 0.01
    assert set(neg.tolist()) == {0, 2, 3, 5}
    assert np.abs(np.bincount(neg, minlength=6)[[0, 2, 3, 5]] / 60000 - 0.25).max() < 0.01


def test_reference_sampler_no_eligible_user():
    R = sp.csr_matrix((np.ones(3), ([0, 1, 2], [0, 0, 0])), shape=(3, 1))
    with pytest.raises(ValueError):
        bpr_ref.sample(R.indptr, R.indices, 1, seed=0, step=0, batch=4)


# ---------------------------------------------------------------------------------------- C ABI argument checks
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from gdr import _lib
    return _lib


def _sample(lib, n_users=4, n_items=5, rowptr=FAKE, colidx=FAKE, n_elig=2, elig=FAKE, seed=1, step=0, batch=8,
            users=FAKE, pos=FAKE, neg=FAKE):
    return lib.call("gdr_bpr_sample", n_users, n_items, rowptr, colidx, n_elig, elig, seed, step, batch, users, pos,
                    neg, 0)


@pytest.mark.parametrize("kw", [dict(n_users=-1), dict(n_items=-1), dict(n_elig=-1), dict(batch=-1), dict(batch=0),
                                dict(batch=(1 << 31) // 3 + 1), dict(step=-1), dict(step=1 << 32), dict(n_elig=0),
                                dict(n_elig=5), dict(n_items=1)]
                         + [{k: 0} for k in ("rowptr", "colidx", "elig", "users", "pos", "neg")])
def test_sample_rejects_bad_arguments(lib, kw):
    with pytest.raises(lib.GdrError) as e:
        _sample(lib, **kw)
    assert e.value.code == -1


def _loss(lib, B=8, n_u=4, n_i=5, d=8, U=FAKE, ldu=8, I=FAKE, ldi=8, users=FAKE, pos=FAKE, neg=FAKE, loss=FAKE,
          gU=FAKE, ldgu=8, gI=FAKE, ldgi=8, status=FAKE, ws=FAKE, ws_bytes=1 << 40):
    return lib.call("gdr_bpr_loss", B, n_u, n_i, d, U, ldu, I, ldi, users, pos, neg, loss, gU, ldgu, gI, ldgi, status,
                    ws, ws_bytes, 0)


@pytest.mark.parametrize("kw", [dict(B=-1), dict(B=0), dict(B=(1 << 31) // 3 + 1), dict(n_u=-1), dict(n_i=-1),
                                dict(d=-1), dict(d=0), dict(n_u=0), dict(ldu=6), dict(ldu=4), dict(ldi=10),
                                dict(ldgu=6), dict(ldgi=4), dict(U=FAKE + 4), dict(I=FAKE + 8), dict(gU=FAKE + 4),
                                dict(gI=FAKE + 12)]
                         + [{k: 0} for k in ("U", "I", "users", "pos", "neg", "loss", "status", "ws")])
def test_loss_rejects_bad_arguments(lib, kw):
    with pytest.raises(lib.GdrError) as e:
        _loss(lib, **kw)
    assert e.value.code == -1


def test_loss_rejects_small_workspace(lib):
    need = lib.query("gdr_bpr_loss_ws_bytes", 8, 4, 5)
    assert need >= 8 * 4 + 24 * 8 + 24 * 4 + lib.query("gdr_sort_pairs_ws_bytes", 24)
    with pytest.raises(lib.GdrError) as e:
        _loss(lib, ws_bytes=need - 1)
    assert e.value.code == -2
