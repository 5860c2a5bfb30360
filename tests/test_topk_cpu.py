"""CPU checks of the top-K evaluation entry points: argument validation before any device work, workspace size at
the Amazon-book shape (no score matrix), and the CPU references against hand-worked values."""
import math

import numpy as np
import pytest

import topk_ref

FAKE = 256   # a non-null pointer that the argument checks must reject before it is ever dereferenced


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from gdr import _lib
    return _lib


def _topk(lib, n_rows=4, n_users=4, n_items=10, d=8, k=3, U=FAKE, I=FAKE, ws=FAKE, ws_bytes=1 << 40, ld=None):
    ld = d if ld is None else ld
    return lib.call("gdr_topk_scores", n_rows, n_users, n_items, d, k, U, ld, 0, I, ld, 0, 0, FAKE, k, FAKE, k, FAKE,
                    ws, ws_bytes, 0)


@pytest.mark.parametrize("kw", [dict(k=0), dict(k=11), dict(U=0), dict(I=0), dict(ws=0), dict(ld=4), dict(n_rows=5)])
def test_topk_rejects_bad_arguments(lib, kw):
    with pytest.raises(lib.GdrError) as e:
        _topk(lib, **kw)
    assert e.value.code == -1


def test_topk_rejects_small_workspace(lib):
    need = lib.query("gdr_topk_scores_ws_bytes", 4, 10, 8, 3)
    with pytest.raises(lib.GdrError) as e:
        _topk(lib, ws_bytes=need - 1)
    assert e.value.code == -2


def test_topk_exclusion_needs_both_arrays(lib):
    with pytest.raises(lib.GdrError) as e:
        lib.call("gdr_topk_scores", 4, 4, 10, 8, 3, FAKE, 8, 0, FAKE, 8, FAKE, 0, FAKE, 3, FAKE, 3, FAKE, FAKE, 1 << 40, 0)
    assert e.value.code == -1


def test_metrics_rejects_bad_arguments(lib):
    ks = np.array([5], dtype=np.int32)
    args = lambda k, ks_, n_ks, wsb: (4, 4, k, FAKE, k, 0, FAKE, FAKE, n_ks, ks_.ctypes.data, FAKE, FAKE, 0, FAKE, wsb, 0)
    with pytest.raises(lib.GdrError) as e:   # K > k
        lib.call("gdr_ranking_metrics", *args(3, ks, 1, 1 << 40))
    assert e.value.code == -1
    with pytest.raises(lib.GdrError) as e:   # no K
        lib.call("gdr_ranking_metrics", *args(5, ks, 0, 1 << 40))
    assert e.value.code == -1
    with pytest.raises(lib.GdrError) as e:
        lib.call("gdr_ranking_metrics", *args(5, ks, 1, 8))
    assert e.value.code == -2


def test_workspace_has_no_score_matrix(lib):
    # Amazon-book shape: the full score matrix would be 52 643 x 91 599 x 4 B = 19 GB
    for k in (20, 100, 91599):
        wsb = lib.query("gdr_topk_scores_ws_bytes", 52643, 91599, 64, k)
        assert 0 < wsb < 1 << 30, (k, wsb)


def test_reference_topk_orders_ties_and_pads():
    # integer embeddings: every product and sum is exact, so numpy's order-free scores equal the fmaf chain
    rs = np.random.RandomState(0)
    U = rs.randint(-2, 3, (6, 5)).astype(np.float32)
    U[1] = 0   # a zero user: every score ties
    I = rs.randint(-2, 3, (40, 5)).astype(np.float32)
    rowptr = np.array([0, 2, 2, 41, 41, 41, 41], dtype=np.int32)   # user 2 keeps only item 39
    colidx = np.concatenate([[3, 7], np.arange(39)]).astype(np.int32)
    s, it = topk_ref.topk(U, I, 4, rowptr, colidx)
    S = U.astype(np.float64) @ I.T.astype(np.float64)
    for u in range(6):
        ex = set(colidx[rowptr[u]:rowptr[u + 1]].tolist())
        keep = [j for j in range(40) if j not in ex]
        order = sorted(keep, key=lambda j: (-S[u, j], j))[:4]
        order += [-1] * (4 - len(order))
        assert it[u].tolist() == order, u
        for i, j in enumerate(order):
            assert s[u, i] == (S[u, j] if j >= 0 else -np.inf)
    assert it[1].tolist() == [0, 1, 2, 3] and it[2].tolist() == [39, -1, -1, -1]


def test_reference_metrics_hand_worked():
    items = np.array([[5, 2, 7], [0, 1, 2], [4, 1, 0]])
    # user 0: test {2, 9}; user 1: no test items (skipped); user 2: test {4} (|test| < K)
    rowptr = np.array([0, 2, 2, 3])
    colidx = np.array([2, 9, 4])
    m = topk_ref.metrics(items, rowptr, colidx, (1, 3))
    L = 1.0 / math.log2(3)
    want = {"recall@1": 0.5, "precision@1": 0.5, "ndcg@1": 0.5,
            "recall@3": (0.5 + 1.0) / 2, "precision@3": 1.0 / 3, "ndcg@3": (L / (1 + L) + 1.0) / 2}
    for key, v in want.items():
        assert m[key] == pytest.approx(v, rel=1e-15), key
    assert m["n_eval"] == 2 and m["n_skipped"] == 1
