"""MiniBatchKMeans on a row partition in an NCCL group of one rank: gdr_minibatch_batch_dist against Xp[idx] and
gdr_kmeans_assign(precision_mode=0) byte for byte, DistMiniBatchKMeans byte-equal to MiniBatchKMeans, the argument
rejections, and dist_kmeans_cluster on both sides of the 20 000-row switch."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def comm():
    import torch.distributed as dist
    from gdr import parallel as par
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    c = par.Comm(dist)
    yield c
    c.close()
    dist.destroy_process_group()


def _bits(t):
    return t.contiguous().view(torch.int32)


def _one_gpu_batch(Xp, idx, C):
    """What MiniBatchKMeans does for one batch: Xp[idx] padded, then gdr_kmeans_assign with precision_mode 0."""
    from gdr import kmeans
    from gdr._dev import padded_rows
    Xb = padded_rows(Xp[torch.from_numpy(idx).cuda()].contiguous())
    lab = torch.empty(idx.shape[0], dtype=torch.int32, device=Xp.device)
    kmeans.assign_labels(Xb, C, lab, precision_mode=0)
    return Xb, lab


@pytest.mark.parametrize("D", [7, 40, 47, 64, 100, 1433])
def test_batch_assembly_matches_one_gpu(comm, D):
    from gdr import parallel as par
    from gdr._dev import new_padded, padded_rows
    rs = np.random.RandomState(D)
    N = 12000
    Xp = padded_rows(torch.from_numpy(rs.standard_normal((N, D)).astype(np.float32)).cuda())
    ops = par.CudaOps()
    row_off = np.array([0, N], np.int64)
    for K in (1, 100, 9160):
        C = new_padded(K, D, Xp.device, zero=True)
        C.copy_(Xp[torch.from_numpy(rs.randint(0, N, K)).cuda()] + 0.01)
        for m in (1, 1000, 2048, 2049):
            idx = rs.randint(0, N, m).astype(np.int64)
            idx[m // 2:] = idx[: m - m // 2]                       # duplicates
            Xb_ref, lab_ref = _one_gpu_batch(Xp, idx, C)
            Xb = new_padded(m, D, Xp.device, zero=True)
            Xb.fill_(float("nan"))                                 # every element, padding included, is written
            lab = torch.full((m,), -7, dtype=torch.int32, device=Xp.device)
            ops.minibatch_batch(comm, idx, row_off, Xp, C, Xb, lab)
            wide = Xb.as_strided((m, Xb.stride(0)), (Xb.stride(0), 1))
            assert torch.equal(_bits(wide[:, D:]), torch.zeros_like(_bits(wide[:, D:])))
            assert torch.equal(_bits(Xb), _bits(Xb_ref)), (D, K, m)
            assert torch.equal(lab, lab_ref), (D, K, m)
            # rows only: labels untouched
            Xr = new_padded(m, D, Xp.device, zero=True)
            lab.fill_(-7)
            ops.minibatch_batch(comm, idx, row_off, Xp, None, Xr, lab)
            assert torch.equal(_bits(Xr), _bits(Xb_ref)) and bool((lab == -7).all())


def test_owner_labels_do_not_depend_on_the_launch(comm):
    """k_assign_simt tiles rows and scans all K per tile: a row's label is the same whichever rows share the launch."""
    from gdr import kmeans
    from gdr._dev import new_padded, padded_rows
    rs = np.random.RandomState(5)
    N, D, K = 5000, 47, 300
    Xp = padded_rows(torch.from_numpy(rs.standard_normal((N, D)).astype(np.float32)).cuda())
    C = new_padded(K, D, Xp.device, zero=True)
    C.copy_(Xp[:K])
    full = torch.empty(N, dtype=torch.int32, device=Xp.device)
    kmeans.assign_labels(Xp, C, full, precision_mode=0)
    for lo, hi in ((0, 1), (1, 130), (127, 1000), (4999, 5000), (2500, 5000)):
        part = torch.empty(hi - lo, dtype=torch.int32, device=Xp.device)
        kmeans.assign_labels(padded_rows(Xp[lo:hi].contiguous()), C, part, precision_mode=0)
        assert torch.equal(part, full[lo:hi])


def _fit_pair(comm, X, **kw):
    import gdr
    from gdr import parallel as par
    ref = gdr.MiniBatchKMeans(**kw).fit(X)
    got = par.DistMiniBatchKMeans(comm=comm, **kw).fit(X)
    assert torch.equal(_bits(got.cluster_centers_), _bits(ref.cluster_centers_)), kw
    assert got.n_steps_ == ref.n_steps_ and got.n_iter_ == ref.n_iter_, kw
    assert got.inertia_ == ref.inertia_, kw
    if kw.get("compute_labels", True):
        assert got.labels_.dtype == torch.int32 and got.labels_.is_cuda
        assert torch.equal(got.labels_, ref.labels_), kw
    return got, ref


def test_dist_minibatch_equals_one_gpu(comm):
    from gdr import synth
    X = torch.from_numpy(synth.clustered_features(30000, 40, 50, seed=2)).cuda()
    # the three configurations of test_minibatch_kmeans_follows_sklearn
    _fit_pair(comm, X, n_clusters=100, random_state=0, batch_size=1000)
    _fit_pair(comm, X, n_clusters=50, random_state=3, batch_size=2048, init="random", n_init=1)
    _fit_pair(comm, X, n_clusters=64, random_state=1, batch_size=512, max_iter=5, max_no_improvement=None)
    # three random inits, an array init, no labels
    _fit_pair(comm, X, n_clusters=30, random_state=4, batch_size=1024, init="random", n_init=3)
    C0 = synth.kmeans_init(X[:5000].cpu().numpy(), 40, 6)
    _fit_pair(comm, X, n_clusters=40, random_state=6, batch_size=1024, init=C0)
    _fit_pair(comm, X, n_clusters=40, random_state=7, batch_size=1024, compute_labels=False)
    # reassignment-heavy: many centres for the batch, a high ratio
    got, _ = _fit_pair(comm, X, n_clusters=600, random_state=8, batch_size=256, reassignment_ratio=0.3, max_iter=3)
    assert got.n_steps_ > 10
    # tol > 0: one rank sums the columns exactly as the ranks do
    _fit_pair(comm, X, n_clusters=20, random_state=9, batch_size=1024, tol=1e-3, max_iter=3)


@pytest.mark.parametrize("D", [47, 64])
def test_dist_minibatch_widths(comm, D):
    from gdr import synth
    X = torch.from_numpy(synth.clustered_features(21000, D, 80, seed=D)).cuda()
    _fit_pair(comm, X, n_clusters=2100, random_state=42, batch_size=2048)


def test_rejections(comm):
    from gdr import _lib
    from gdr import parallel as par
    from gdr._dev import new_padded
    X = torch.randn(500, 8, device="cuda")
    with pytest.raises(ValueError):       # a string init needs random_state
        par.DistMiniBatchKMeans(n_clusters=5, comm=comm).fit(X)
    with pytest.raises(ValueError):
        par.DistMiniBatchKMeans(n_clusters=5, init="kmeans++", random_state=0, comm=comm).fit(X)
    with pytest.raises(ValueError):
        par.DistMiniBatchKMeans(n_clusters=5, init=np.zeros((4, 8), np.float32), random_state=0, comm=comm).fit(X)
    with pytest.raises(ValueError):
        par.DistMiniBatchKMeans(n_clusters=501, random_state=0, comm=comm).fit(X)
    with pytest.raises(ValueError):
        par.DistMiniBatchKMeans(n_clusters=5, random_state=0, reassignment_ratio=-1.0, comm=comm).fit(X)
    with pytest.raises(ValueError):
        par.DistMiniBatchKMeans(n_clusters=5, random_state=0, precision="fp16", comm=comm).fit(X)
    with pytest.raises(NotImplementedError):
        par.DistMiniBatchKMeans(n_clusters=5, random_state=0, comm=comm, ops=object()).fit(X)

    # the C ABI: local checks only
    Xp = new_padded(100, 8, X.device)
    Xp.copy_(X[:100])
    m, K, D = 16, 4, 8
    idx = torch.arange(m, dtype=torch.int64, device=X.device)
    order = torch.arange(m, dtype=torch.int32, device=X.device)
    C = new_padded(K, D, X.device, zero=True)
    Xb = new_padded(m, D, X.device, zero=True)
    lab = torch.empty(m, dtype=torch.int32, device=X.device)
    need = _lib.query("gdr_minibatch_batch_dist_ws_bytes", m, K, D, 1)
    ws = torch.empty(need, dtype=torch.uint8, device=X.device)
    st = torch.cuda.current_stream().cuda_stream

    def call(counts=(m,), C_=C, lab_=lab, ldb=Xb.stride(0), ws_bytes=need, D_=D, comm_=None):
        cnt = (ctypes.c_int64 * 1)(*counts)
        h = comm.lib_handle() if comm_ is None else comm_
        _lib.call("gdr_minibatch_batch_dist", h, m, idx.data_ptr(), order.data_ptr(), ctypes.addressof(cnt), 0, 100, K, D_,
                  Xp.data_ptr(), Xp.stride(0), 0 if C_ is None else C_.data_ptr(), C.stride(0), Xb.data_ptr(), ldb,
                  0 if lab_ is None else lab_.data_ptr(), ws.data_ptr(), ws_bytes, st)

    for kw, code in ((dict(counts=(m - 1,)), -1), (dict(counts=(-1,)), -1), (dict(lab_=None), -1), (dict(ldb=7), -1),
                     (dict(D_=0), -1), (dict(ws_bytes=need - 256), -2), (dict(comm_=0), -1)):
        with pytest.raises(_lib.GdrError) as e:
            call(**kw)
        assert e.value.code == code, kw
    call(C_=None, lab_=None)              # rows only: labels_b may be null
    call()
    torch.cuda.synchronize()
    ref = torch.empty(m, dtype=torch.int32, device=X.device)
    from gdr import kmeans
    kmeans.assign_labels(Xb, C, ref, precision_mode=0)
    assert torch.equal(lab, ref) and torch.equal(Xb, Xp[:m])


def test_dist_kmeans_cluster(comm):
    from gdr import parallel as par
    from gdr import synth
    import gdr
    # above 20 000 rows: mini-batches, equal to MiniBatchKMeans on the dist-scaled rows
    X = torch.from_numpy(synth.clustered_features(20001, 64, 40, seed=3)).cuda()
    part = par.RowPartition(20001, 1, 0)
    lab, cen = par.dist_kmeans_cluster(comm, part, X, 2001, seed=42)
    Xs = par.dist_standard_scale(comm, X)
    ref = gdr.MiniBatchKMeans(n_clusters=2001, random_state=42, batch_size=2048, n_init="auto").fit(Xs)
    assert lab.dtype == torch.int64 and lab.is_cuda and torch.equal(lab, ref.labels_.to(torch.int64))
    assert torch.equal(_bits(cen), _bits(ref.cluster_centers_))
    # 20 000 rows: Lloyd (DistKMeans) with the same seed
    X2, part2 = X[:20000].contiguous(), par.RowPartition(20000, 1, 0)
    lab2, cen2 = par.dist_kmeans_cluster(comm, part2, X2, 200, seed=7)
    ref2 = par.DistKMeans(200, "k-means++", random_state=7, comm=comm).fit(par.dist_standard_scale(comm, X2))
    assert torch.equal(lab2, ref2.labels_.to(torch.int64)) and torch.equal(cen2, ref2.cluster_centers_)
    # minibatch=False: Lloyd above 20 000 rows too
    lab3, _ = par.dist_kmeans_cluster(comm, part, X, 50, seed=1, minibatch=False)
    ref3 = par.DistKMeans(50, "k-means++", random_state=1, comm=comm).fit(Xs)
    assert torch.equal(lab3, ref3.labels_.to(torch.int64))
    # K capped to N; K <= 0 rejected
    Xc = X[:300].contiguous()
    lab4, cen4 = par.dist_kmeans_cluster(comm, par.RowPartition(300, 1, 0), Xc, 1000, seed=0)
    assert tuple(cen4.shape) == (300, 64) and lab4.shape == (300,)
    with pytest.raises(ValueError):
        par.dist_kmeans_cluster(comm, part, X, 0, seed=0)
