"""gdr_kmeans_plusplus_dist with one rank: byte-identical to the one-GPU k-means++ (gdr_kmeans_plusplus) on the same
rows and draws, sklearn's golden picks, and the argument checks."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import golden

pytestmark = pytest.mark.gpu


def _dist(Xc, K, seed, comm):
    from gdr import parallel as par
    part = par.RowPartition(Xc.shape[0], 1, 0)
    return par.dist_kmeans_plusplus(comm, part, Xc, K, np.random.RandomState(seed), return_indices=True)


def _one(Xc, K, seed):
    from gdr.kmeans_init import kmeans_plusplus_device
    return kmeans_plusplus_device(Xc, K, np.random.RandomState(seed), return_indices=True)


def _padded(X):
    from gdr._dev import new_padded
    t = new_padded(X.shape[0], X.shape[1], torch.device("cuda"))
    t.copy_(torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)))
    return t


@pytest.fixture(scope="module")
def comm():
    from gdr import parallel as par
    c = par.Comm()
    yield c
    c.close()


def _same(a, b):
    assert torch.equal(a[1], b[1])
    assert torch.equal(a[0].contiguous().view(torch.int32), b[0].contiguous().view(torch.int32))


@pytest.mark.parametrize("k", [25, 60, 200])
def test_golden(k, comm):
    g = golden("kmeans_plusplus.npz")
    X = _padded(g["x"])
    got = _dist(X, k, int(g[f"k{k}_seed"]), comm)
    _same(got, _one(X, k, int(g[f"k{k}_seed"])))
    np.testing.assert_array_equal(got[1].cpu().numpy(), g[f"k{k}_indices"])


@pytest.mark.parametrize("n,d,k", [(30011, 100, 257), (30011, 47, 257), (5000, 1433, 1100), (3000, 100, 1)])
def test_clustered_features(n, d, k, comm):
    from gdr import synth
    X = _padded(synth.clustered_features(n, d, 60, seed=12))
    for seed in (0, 7):
        _same(_dist(X, k, seed, comm), _one(X, k, seed))


def test_duplicated_rows(comm):
    rng = np.random.RandomState(4)
    base = rng.randn(50, 20).astype(np.float32)
    X = _padded(base[rng.randint(0, 50, size=4000)])
    for k in (30, 50):      # K = 50: every distinct row becomes a centre and the potential reaches 0
        _same(_dist(X, k, 3, comm), _one(X, k, 3))


def test_crafted_draws_and_clip(comm):
    """Draws handed in directly: thresholds at 0 and above the potential (np.clip to the last row)."""
    from gdr import synth
    X = _padded(synth.clustered_features(3000, 16, 8, seed=2))
    K, L = 12, 4
    rand = np.random.RandomState(1).uniform(size=(K - 1, L))
    rand[2, :] = 0.0
    rand[5, 1] = 1.0 + 2.0 ** -30
    rand[7, :] = 1.0 + 2.0 ** -30
    one, dist = _both(X, K, 5, rand, comm)
    _same(one, dist)
    assert int(dist[1][8]) == X.shape[0] - 1


def _both(X, K, first, rand, comm):
    from gdr import _lib
    from gdr._dev import ptr, stream, workspace
    N, D = X.shape
    L = rand.shape[1]
    outs = []
    for name in ("one", "dist"):
        C = torch.zeros((K, D), dtype=torch.float32, device="cuda")
        idx = torch.empty(K, dtype=torch.int64, device="cuda")
        if name == "one":
            ws = workspace(_lib.query("gdr_kmeans_plusplus_ws_bytes", N, K, D, L), X.device)
            _lib.call("gdr_kmeans_plusplus", N, K, D, ptr(X), X.stride(0), first, rand.ctypes.data, L, ptr(C), D,
                      ptr(idx), ptr(ws), ws.numel(), stream())
        else:
            ws = workspace(_lib.query("gdr_kmeans_plusplus_dist_ws_bytes", N, K, D, L, 1), X.device)
            _lib.call("gdr_kmeans_plusplus_dist", comm.lib_handle(), N, K, D, ptr(X), X.stride(0), first,
                      rand.ctypes.data, L, ptr(C), D, ptr(idx), ptr(ws), ws.numel(), stream())
        outs.append((C, idx))
    return outs


def test_clip_inside_the_owner_block(comm):
    """A draw whose block prefix reaches the threshold while the row-level running sum inside that block rounds
    below it: np.clip takes the LAST row (here -0.0, whose bits differ from the first centre's +0.0).  Distances to
    row 0: [0, 1 x 24, 2^54, 0 x 38]; the block sum (warp-strided order) keeps 2 more than the 32-row warp scan, and
    u = 1 - 2^-53 puts the threshold between the two."""
    X = np.zeros((64, 1), dtype=np.float32)
    X[1:25] = 1.0
    X[25] = 2.0 ** 27
    X[63] = -0.0
    Xd = _padded(X)
    rand = np.full((1, 2), 1.0 - 2.0 ** -53)
    one, dist = _both(Xd, 2, 0, rand, comm)
    _same(one, dist)
    assert dist[1].tolist() == [0, 63]
    assert dist[0][1].view(torch.int32).item() == np.float32(-0.0).view(np.int32)


def test_rejections(comm):
    from gdr import _lib
    from gdr._dev import ptr, stream, workspace
    X = _padded(np.random.RandomState(0).randn(100, 8))
    C = torch.zeros((200, 8), dtype=torch.float32, device="cuda")
    rand = np.zeros((199, 17))

    def call(K, L, ws_bytes=None):
        need = _lib.query("gdr_kmeans_plusplus_dist_ws_bytes", 100, K, 8, L, 1)
        ws = workspace(need, X.device)
        _lib.call("gdr_kmeans_plusplus_dist", comm.lib_handle(), 100, K, 8, ptr(X), X.stride(0), 0, rand.ctypes.data, L,
                  ptr(C), 8, 0, ptr(ws), need if ws_bytes is None else ws_bytes(need), stream())

    with pytest.raises(_lib.GdrError) as e:
        call(10, 17)
    assert e.value.code == -1
    with pytest.raises(_lib.GdrError) as e:
        call(101, 6)
    assert e.value.code == -1
    with pytest.raises(_lib.GdrError) as e:
        call(10, 4, ws_bytes=lambda need: need - 256)
    assert e.value.code == -2
    call(10, 4)   # the communicator is still usable after the rejections


def test_dist_kmeans_string_inits_one_rank(comm):
    import gdr
    from gdr import parallel as par
    from gdr import synth
    t = torch.from_numpy(synth.clustered_features(30011, 100, 60, seed=12)).cuda()
    km = par.DistKMeans(257, "k-means++", random_state=3, max_iter=15, tol=0, comm=comm).fit(t)
    ref = gdr.KMeans(n_clusters=257, init="k-means++", random_state=3, n_init=1, max_iter=15, tol=0).fit(t)
    assert km.n_iter_ == ref.n_iter_
    assert (km.labels_ == ref.labels_).float().mean().item() > 0.99
    assert abs(km.inertia_ - ref.inertia_) <= 1e-4 * ref.inertia_
    km0 = par.DistKMeans(257, "random", random_state=4, max_iter=0, tol=0, comm=comm).fit(t)
    seeds = torch.from_numpy(np.random.RandomState(4).permutation(t.shape[0])[:257]).cuda()
    Xc = par.CudaOps().center(t, km0._mean)
    assert torch.equal(km0._centers_centered.contiguous(), Xc[seeds].contiguous())
