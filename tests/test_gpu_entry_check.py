"""The collective entry check of the row-partitioned entry points (gdr_kmeans_plusplus_dist, gdr_sparsify_classes_dist,
gdr_dense_gram_dist).  One rank: every local rejection returns its own code, and a good call afterwards returns the
bytes it returned before.  Two and four ranks over NCCL (each skips when fewer GPUs are present): a rank rejecting its
own arguments gets its code and every other rank GDR_EINVAL; a value that differs on one rank or a shifted row block is
GDR_EINVAL everywhere; after each case a good call on the same communicator still matches the one-GPU result."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

EINVAL, EWORKSPACE, ERANGE, EUNSUPPORTED = -1, -2, -4, -5


def _code(fn):
    from gdr import _lib
    try:
        fn()
    except _lib.GdrError as e:
        return e.code
    return 0


def _padded(X, dev):
    from gdr._dev import new_padded
    t = new_padded(X.shape[0], X.shape[1], dev)
    t.copy_(torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)))
    return t


def _bits(t):
    return t.contiguous().view(torch.int32 if t.element_size() == 4 else torch.int64)


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert torch.equal(_bits(x), _bits(y))


# ---------------------------------------------------------------------------------------------------- k-means++
def _kpp_inputs(dev):
    from gdr import synth
    X = synth.clustered_features(30011, 100, 60, seed=12)
    K, L = 257, 7
    return X, _padded(X, dev), K, np.random.RandomState(5).uniform(size=(K, L))


def _kpp(h, world, X, K, rand, first=0, ws_delta=0, null_ws=False):
    """gdr_kmeans_plusplus_dist on this rank's rows X (padded fp32); rand holds at least K - 1 rows of draws."""
    from gdr import _lib
    from gdr._dev import ptr, stream, workspace
    N, D = X.shape
    L = rand.shape[1]
    rand = np.ascontiguousarray(rand[: K - 1])
    need = _lib.query("gdr_kmeans_plusplus_dist_ws_bytes", N, K, D, L, world)
    ws = workspace(need, X.device)
    C = torch.zeros((K, D), dtype=torch.float32, device=X.device)
    idx = torch.empty(K, dtype=torch.int64, device=X.device)
    _lib.call("gdr_kmeans_plusplus_dist", h, N, K, D, ptr(X) if N else 0, X.stride(0), first, rand.ctypes.data, L,
              ptr(C), D, ptr(idx), 0 if null_ws else ptr(ws), need + ws_delta, stream())
    return C, idx


def _kpp_one(X, K, rand, first=0):
    from gdr import _lib
    from gdr._dev import ptr, stream, workspace
    N, D = X.shape
    L = rand.shape[1]
    rand = np.ascontiguousarray(rand[: K - 1])
    ws = workspace(_lib.query("gdr_kmeans_plusplus_ws_bytes", N, K, D, L), X.device)
    C = torch.zeros((K, D), dtype=torch.float32, device=X.device)
    idx = torch.empty(K, dtype=torch.int64, device=X.device)
    _lib.call("gdr_kmeans_plusplus", N, K, D, ptr(X), X.stride(0), first, rand.ctypes.data, L, ptr(C), D, ptr(idx),
              ptr(ws), ws.numel(), stream())
    return C, idx


# ---------------------------------------------------------------------------------------------------- sparsify
def _graph(dev):
    """A seeded CSR of 3000 rows (sorted, distinct columns per row) and edge weights with many ties."""
    rs = np.random.RandomState(21)
    n = 3000
    deg = rs.randint(1, 13, size=n)
    cols = [np.unique(rs.randint(0, n, size=d)) for d in deg]
    rowptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int32)
    colidx = np.concatenate(cols).astype(np.int32)
    nnz = len(colidx)
    vals = rs.rand(nnz).astype(np.float32)
    er = (np.round(rs.rand(nnz) * 50) / 50).astype(np.float32)
    t = lambda a: torch.from_numpy(a).to(dev)
    return n, t(rowptr), t(colidx), t(vals), t(er), nnz // 3


def _sparsify(h, world, G, lo, hi, k, row_lo=None, nnz=None, ws_delta=0, null_ws=False):
    """gdr_sparsify_classes_dist without prob (one graph, weights er) on rows [lo, hi) of G."""
    from gdr import _lib
    from gdr._dev import ptr, stream, workspace
    n, rowptr, colidx, vals, er, _ = G
    s, e = int(rowptr[lo]), int(rowptr[hi])
    rp = (rowptr[lo:hi + 1] - s).contiguous()
    n_local, nnz_local = hi - lo, e - s
    cap = max(min(k, nnz_local), 1)
    out_rp = torch.empty(n_local + 1, dtype=torch.int32, device=rowptr.device)
    out_ci = torch.empty(cap, dtype=torch.int32, device=rowptr.device)
    out_v = torch.empty(cap, dtype=torch.float32, device=rowptr.device)
    cnt = torch.zeros(1, dtype=torch.int64, device=rowptr.device)
    need = _lib.query("gdr_sparsify_classes_dist_ws_bytes", n_local, nnz_local, 1, world)
    ws = workspace(need, rowptr.device)
    _lib.call("gdr_sparsify_classes_dist", h, n_local, nnz_local if nnz is None else nnz,
              lo if row_lo is None else row_lo, n, 1, ptr(rp), ptr(colidx[s:e]), ptr(vals[s:e]), ptr(er[s:e]), 0, 0, k, ptr(out_rp), ptr(out_ci),
              ptr(out_v), ptr(cnt), 0 if null_ws else ptr(ws), need + ws_delta, stream())
    m = int(cnt[0])
    return out_rp, out_ci[:m], out_v[:m]


def _sparsify_one(G, lo, hi):
    """Rows [lo, hi) of the one-GPU top-k (gdr_topk_filter_csr on the whole graph), as a local CSR."""
    from gdr import _lib
    from gdr._dev import ptr, stream, workspace
    n, rowptr, colidx, vals, er, k = G
    nnz = colidx.numel()
    out_rp = torch.empty(n + 1, dtype=torch.int32, device=rowptr.device)
    out_ci = torch.empty(k, dtype=torch.int32, device=rowptr.device)
    out_v = torch.empty(k, dtype=torch.float32, device=rowptr.device)
    cnt = torch.zeros(1, dtype=torch.int64, device=rowptr.device)
    ws = workspace(_lib.query("gdr_topk_filter_ws_bytes", n, nnz), rowptr.device)
    _lib.call("gdr_topk_filter_csr", n, nnz, ptr(rowptr), ptr(colidx), ptr(vals), ptr(er), k, ptr(out_rp), ptr(out_ci),
              ptr(out_v), ptr(cnt), ptr(ws), ws.numel(), stream())
    s, e = int(out_rp[lo]), int(out_rp[hi])
    return out_rp[lo:hi + 1] - s, out_ci[s:e], out_v[s:e]


# ---------------------------------------------------------------------------------------------------- Gram
def _gram_inputs(dev):
    rs = np.random.RandomState(7)
    W = torch.from_numpy(rs.standard_normal((5000, 40)) * np.exp(rs.uniform(-4, 4, (5000, 1)))).to(dev)
    return W[:, :24], W[:, 24:]


def _gram(h, world, n_global, row_lo, A, B, ws_delta=0, null_ws=False):
    from gdr import _lib
    from gdr._dev import ptr, stream, workspace
    n, p = A.shape
    r = B.shape[1]
    need = _lib.query("gdr_dense_gram_dist_ws_bytes", n_global, p, r, world)
    ws = workspace(need, A.device)
    C = torch.empty((p, r), dtype=torch.float64, device=A.device)
    _lib.call("gdr_dense_gram_dist", h, n_global, row_lo, n, p, r, ptr(A) if n else 0, A.stride(0), ptr(B) if n else 0,
              B.stride(0), ptr(C), r, 0 if null_ws else ptr(ws), need + ws_delta, stream())
    return (C,)


# ---------------------------------------------------------------------------------------------------- one rank
@pytest.fixture(scope="module")
def comm():
    from gdr import parallel as par
    c = par.Comm()
    yield c
    c.close()


def test_kmeans_plusplus_one_rank(comm):
    dev = torch.device("cuda", torch.cuda.current_device())
    h = comm.lib_handle()
    _, X, K, rand = _kpp_inputs(dev)
    before = _kpp(h, 1, X, K, rand)
    _same(before, _kpp_one(X, K, rand))
    assert _code(lambda: _kpp(h, 1, X, K, np.zeros((K, 17)))) == EINVAL            # n_trials > 16
    assert _code(lambda: _kpp(h, 1, X, K, rand, null_ws=True)) == EINVAL
    assert _code(lambda: _kpp(h, 1, X, K, rand, ws_delta=-1)) == EWORKSPACE
    wide = torch.zeros((100, 3300), dtype=torch.float32, device=dev)                 # 16 x 3300 floats of candidates
    assert _code(lambda: _kpp(h, 1, wide, 10, np.zeros((10, 16)))) == EUNSUPPORTED
    assert _code(lambda: _kpp(h, 1, X[:100], 101, rand)) == EINVAL                  # K > N_total
    assert _code(lambda: _kpp(h, 1, X[:100], 10, rand, first=100)) == EINVAL        # first centre out of range
    _same(_kpp(h, 1, X, K, rand), before)


def test_sparsify_one_rank(comm):
    dev = torch.device("cuda", torch.cuda.current_device())
    h = comm.lib_handle()
    G = _graph(dev)
    n, k = G[0], G[5]
    before = _sparsify(h, 1, G, 0, n, k)
    _same(before, _sparsify_one(G, 0, n))
    assert _code(lambda: _sparsify(h, 1, G, 0, n, -1)) == EINVAL
    assert _code(lambda: _sparsify(h, 1, G, 0, n, k, null_ws=True)) == EINVAL
    assert _code(lambda: _sparsify(h, 1, G, 0, n, k, nnz=1 << 31)) == ERANGE
    assert _code(lambda: _sparsify(h, 1, G, 0, n, k, ws_delta=-1)) == EWORKSPACE
    assert _code(lambda: _sparsify(h, 1, G, 0, n, G[2].numel() + 1)) == EINVAL     # k > nnz
    assert _code(lambda: _sparsify(h, 1, G, 0, n, k, row_lo=1)) == EINVAL           # the block must start at row 0
    _same(_sparsify(h, 1, G, 0, n, k), before)


def test_gram_one_rank(comm):
    from gdr import svd as gsvd
    dev = torch.device("cuda", torch.cuda.current_device())
    h = comm.lib_handle()
    A, B = _gram_inputs(dev)
    N = A.shape[0]
    before = _gram(h, 1, N, 0, A, B)
    _same(before, (gsvd._gram(A, B),))
    assert _code(lambda: _gram(h, 1, N, 0, A, B[:, :0])) == EINVAL                  # r = 0
    assert _code(lambda: _gram(h, 1, N, 0, A, B, null_ws=True)) == EINVAL
    assert _code(lambda: _gram(h, 1, N, 0, A, B, ws_delta=-1)) == EWORKSPACE
    assert _code(lambda: _gram(h, 1, N + 1, 0, A, B)) == EINVAL                     # the block does not cover N_global
    assert _code(lambda: _gram(h, 1, N + 1, 1, A, B)) == EINVAL                     # nor start at row 0
    _same(_gram(h, 1, N, 0, A, B), before)


# ---------------------------------------------------------------------------------------------------- 2 and 4 ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from gdr import _lib
        from gdr import parallel as par
        from gdr import svd as gsvd
        comm = par.Comm(dist)
        h = comm.lib_handle()
        last = rank == world - 1

        def expect(fn, mine, others=EINVAL):
            assert _code(fn) == (mine if last else others)

        def everywhere(fn):
            assert _code(fn) == EINVAL

        # k-means++: a different K on the last rank
        Xh, Xf, K, rand = _kpp_inputs(dev)
        p = par.RowPartition(Xh.shape[0], world, rank)
        X = _padded(Xh[p.lo:p.hi], dev)
        one = _kpp_one(Xf, K, rand)
        good = lambda: _same(_kpp(h, world, X, K, rand), one)
        good()
        expect(lambda: _kpp(h, world, X, K, rand, ws_delta=-1 if last else 0), EWORKSPACE)
        good()
        everywhere(lambda: _kpp(h, world, X, K + 1 if last else K, rand))
        good()

        # sparsification: a different k, a different batch cap, a shifted row block
        G = _graph(dev)
        n, k = G[0], G[5]
        p = par.RowPartition(n, world, rank)
        one = _sparsify_one(G, p.lo, p.hi)
        good = lambda: _same(_sparsify(h, world, G, p.lo, p.hi, k), one)
        good()
        expect(lambda: _sparsify(h, world, G, p.lo, p.hi, k, ws_delta=-1 if last else 0), EWORKSPACE)
        good()
        everywhere(lambda: _sparsify(h, world, G, p.lo, p.hi, k + 1 if last else k))
        good()
        _lib.call("gdr_debug_set", b"sparsify_batch", 3 if last else 0)
        everywhere(lambda: _sparsify(h, world, G, p.lo, p.hi, k))
        _lib.call("gdr_debug_set", b"sparsify_batch", 0)
        good()
        everywhere(lambda: _sparsify(h, world, G, p.lo, p.hi, k, row_lo=1 if rank == 0 else p.lo))
        good()

        # Gram: a different N_global, a different r, a shifted row block
        A, B = _gram_inputs(dev)
        N = A.shape[0]
        p = par.RowPartition(N, world, rank)
        Al, Bl = A[p.lo:p.hi], B[p.lo:p.hi]
        one = (gsvd._gram(A, B),)
        good = lambda: _same(_gram(h, world, N, p.lo, Al, Bl), one)
        good()
        expect(lambda: _gram(h, world, N, p.lo, Al, Bl, ws_delta=-1 if last else 0), EWORKSPACE)
        good()
        everywhere(lambda: _gram(h, world, N + 1 if last else N, p.lo, Al, Bl))
        good()
        everywhere(lambda: _gram(h, world, N, p.lo, Al, Bl[:, :-1] if last else Bl))
        good()
        everywhere(lambda: _gram(h, world, N, 1 if rank == 0 else p.lo, Al, Bl))
        good()
        torch.cuda.synchronize()
        comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_rejections_across_ranks(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    mp.spawn(_worker, args=(world, _free_port()), nprocs=world, join=True)
