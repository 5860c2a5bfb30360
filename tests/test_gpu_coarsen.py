"""Stage 4 without a sort: one CTA per coarse row, cells accumulated in shared memory (integer counts, fixed-point weight
sums) against the sort-based path and an fp64 scipy P^T A P (clustgdd_agent_transduct.py:234-250)."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import coarsen_ref

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None


@pytest.fixture(scope="module")
def gdr():
    import gdr
    return gdr


def _graph(n, avg_deg, hubs, seed):
    rng = np.random.RandomState(seed)
    m = n * avg_deg // 2
    u, v = rng.randint(0, n, m), rng.randint(0, n, m)
    for h in range(hubs):                    # a few very long rows (walked by the whole CTA)
        u = np.concatenate([u, np.full(6000, h)])
        v = np.concatenate([v, rng.randint(0, n, 6000)])
    return u.astype(np.int64), v.astype(np.int64)


def _coarsen(gdr, A, labels, k, dense, weights=True, drop_diag=True):
    from gdr import _lib
    _lib.call("gdr_debug_set", b"coarsen_dense", int(dense))
    try:
        out = gdr.coarsen_edges(labels, labels, k, k, csr=A, weights=A.vals if weights else None, drop_diag=drop_diag)
        torch.cuda.synchronize()
    finally:
        _lib.call("gdr_debug_set", b"coarsen_dense", 1)
    return out


@pytest.mark.parametrize("n,k,avg_deg,hubs,drop", [(5000, 50, 20, 0, True), (30000, 700, 30, 3, True), (30000, 700, 30, 3, False),
                                                   (2000, 1500, 16, 1, True), (60000, 9000, 24, 2, True)])
def test_dense_coarsen_equals_sort_path_and_fp64(gdr, n, k, avg_deg, hubs, drop):
    u, v = _graph(n, avg_deg, hubs, seed=n + k)
    A = gdr.sym_normalize(gdr.coo_to_csr(torch.from_numpy(u).to(DEV), torch.from_numpy(v).to(DEV), None, (n, n), symmetrize=True,
                                         binarize=True), 2)
    rng = np.random.RandomState(7)
    lab = rng.randint(0, k, n).astype(np.int32)
    lab[lab == 3] = 4                        # an empty cluster
    labels = torch.from_numpy(lab).to(DEV)
    rp_s, ci_s, cnt_s, ws_s = _coarsen(gdr, A, labels, k, dense=False, drop_diag=drop)
    rp_d, ci_d, cnt_d, ws_d = _coarsen(gdr, A, labels, k, dense=True, drop_diag=drop)
    assert torch.equal(rp_s, rp_d) and torch.equal(ci_s, ci_d) and torch.equal(cnt_s, cnt_d)
    torch.testing.assert_close(ws_d, ws_s, rtol=2e-6, atol=0)
    # fp64 reference: the fixed-point sums are within n*q_a/2 plus one fp32 rounding of the exact sums
    As = sp.csr_matrix((A.vals.cpu().numpy().astype(np.float64), A.colidx.cpu().numpy(), A.rowptr.cpu().numpy()), shape=(n, n))
    P = sp.csr_matrix((np.ones(n), (np.arange(n), lab)), shape=(n, k))
    S = (P.T @ As @ P).tocsr()
    if drop:
        S.setdiag(0)
        S.eliminate_zeros()
    S.sort_indices()
    assert np.array_equal(S.indptr, rp_d.cpu().numpy()) and np.array_equal(S.indices, ci_d.cpu().numpy())
    got = ws_d.cpu().numpy()
    r = coarsen_ref.csr_cells(A.rowptr.cpu().numpy(), A.colidx.cpu().numpy(), A.vals.cpu().numpy(), lab, lab, drop)
    q = coarsen_ref.steps(A.rowptr.cpu().numpy(), A.vals.cpu().numpy(), lab, k)[r["a"]]
    assert np.array_equal(r["count"], cnt_d.cpu().numpy())
    err = np.abs(got.astype(np.float64) - r["sum"])
    assert np.all(err <= coarsen_ref.dense_bound(r["sum"], r["count"], q))
    one = coarsen_ref.one_ulp_regime(r["sum"], r["count"], q)      # where n*q_a/2 <= ulp/4: within one ulp of fl32(exact)
    assert np.all(np.abs(got[one] - r["sum"][one].astype(np.float32)) <= coarsen_ref.ulp32(r["sum"][one]))
    # bit-reproducible although the shared-memory atomics land in any order
    _, _, _, ws_d2 = _coarsen(gdr, A, labels, k, dense=True, drop_diag=drop)
    assert torch.equal(ws_d, ws_d2)
    # counts only
    rp_c, ci_c, cnt_c, none = _coarsen(gdr, A, labels, k, dense=True, weights=False, drop_diag=drop)
    assert none is None and torch.equal(rp_c, rp_d) and torch.equal(ci_c, ci_d) and torch.equal(cnt_c, cnt_d)


def test_wide_coarse_rows_fall_back_to_the_sort(gdr):
    n, k = 40000, 30000                      # 30000 x 12 B does not fit in shared memory
    u, v = _graph(n, 12, 0, seed=5)
    A = gdr.sym_normalize(gdr.coo_to_csr(torch.from_numpy(u).to(DEV), torch.from_numpy(v).to(DEV), None, (n, n), symmetrize=True,
                                         binarize=True), 2)
    labels = torch.from_numpy(np.random.RandomState(1).randint(0, k, n).astype(np.int32)).to(DEV)
    a = _coarsen(gdr, A, labels, k, dense=True)
    b = _coarsen(gdr, A, labels, k, dense=False)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("n,k,world", [(60000, 9000, 2), (30000, 700, 3), (20000, 100, 2)])
def test_owner_side_merge_in_shared_memory(gdr, n, k, world):
    """The multi-GPU stage 4 at the owner of a key range, replayed on one GPU: the pairs gdr_coarsen_route addresses to
    each owner, merged by the sort and in shared memory (gdr_coarse_merge_edges_dense with the global per-cluster
    fixed-point step) — structure and counts equal, sums bit-identical to the single-GPU gdr_coarsen rows."""
    from gdr import parallel as par
    u, v = _graph(n, 24, 2, seed=n + k)
    A = gdr.sym_normalize(gdr.coo_to_csr(torch.from_numpy(u).to(DEV), torch.from_numpy(v).to(DEV), None, (n, n), symmetrize=True,
                                         binarize=True), 2)
    lab = np.random.RandomState(3).randint(0, k, n).astype(np.int32)
    labels = torch.from_numpy(lab).to(DEV)
    ops = par.CudaOps()
    rp1, ci1, cnt1, ws1 = _coarsen(gdr, A, labels, k, dense=True)
    keys, w, counts = ops.coarsen_route(A, labels, labels, k, world)
    stats = ops.cluster_stats(A, labels, k)
    cr = (k + world - 1) // world
    off = 0
    for r in range(world):
        a_lo = min(k, r * cr)
        n_rows = min(k, a_lo + cr) - a_lo
        seg_k, seg_w = keys[off: off + counts[r]], w[off: off + counts[r]]
        off += counts[r]
        d = ops.coarse_merge_edges(seg_k, seg_w, a_lo, n_rows, k, stats=stats)
        from gdr import _lib
        _lib.call("gdr_debug_set", b"coarsen_dense", 0)
        try:
            s = ops.coarse_merge_edges(seg_k, seg_w, a_lo, n_rows, k, stats=stats)
        finally:
            _lib.call("gdr_debug_set", b"coarsen_dense", 1)
        assert torch.equal(d[0], s[0]) and torch.equal(d[1], s[1]) and torch.equal(d[2], s[2])
        torch.testing.assert_close(d[3], s[3], rtol=2e-6, atol=0)
        b, e = int(rp1[a_lo]), int(rp1[a_lo + n_rows])
        assert torch.equal(d[0] + b, rp1[a_lo: a_lo + n_rows + 1]) and torch.equal(d[1], ci1[b:e]) and torch.equal(d[2], cnt1[b:e])
        assert torch.equal(d[3], ws1[b:e])                                  # the same fixed-point step: bit-identical sums
        c = ops.coarse_merge_edges(seg_k, None, a_lo, n_rows, k)             # counts only
        assert c[3] is None and torch.equal(c[0], d[0]) and torch.equal(c[1], d[1]) and torch.equal(c[2], d[2])
