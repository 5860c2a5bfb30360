"""k-means++ on a row partition over NCCL (gdr_kmeans_plusplus_dist, DistKMeans string inits) against the one-GPU
seeding.  Needs >= 2 GPUs; the 4-rank case needs 4."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


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
        import gdr
        from gdr import _lib
        from gdr import parallel as par
        from gdr import synth
        from gdr._dev import new_padded
        from gdr.kmeans_init import kmeans_plusplus_device
        comm = par.Comm(dist)

        def padded(X):
            t = new_padded(X.shape[0], X.shape[1], dev)
            t.copy_(torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)))
            return t

        def check(X, K, seed, lo, hi):
            Xf = padded(X)
            c1, i1 = kmeans_plusplus_device(Xf, K, np.random.RandomState(seed), return_indices=True)
            part = par.RowPartition(X.shape[0], world, rank)
            cd, idd = par.dist_kmeans_plusplus(comm, part, padded(X[lo:hi]), K, np.random.RandomState(seed),
                                               return_indices=True)
            assert torch.equal(idd, i1), (K, seed)
            assert torch.equal(cd.contiguous().view(torch.int32), c1.contiguous().view(torch.int32))
            mx = cd.contiguous().clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            assert torch.equal(mx, cd.contiguous())
            return idd

        g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kmeans_plusplus.npz"))
        part = par.RowPartition(g["x"].shape[0], world, rank)
        for k in (25, 60, 200):
            idx = check(g["x"], k, int(g[f"k{k}_seed"]), part.lo, part.hi)
            np.testing.assert_array_equal(idx.cpu().numpy(), g[f"k{k}_indices"])
        X = synth.clustered_features(30011, 100, 60, seed=12)
        part = par.RowPartition(X.shape[0], world, rank)
        check(X, 257, 0, part.lo, part.hi)       # uneven last block
        if world == 4:                           # rank 2 owns no rows
            bounds = [0, 9000, 20000, 20000, 30011]
            check(X, 257, 1, bounds[rank], bounds[rank + 1])
        # mismatched seeds: every rank raises, none hangs
        with pytest.raises(_lib.GdrError):
            par.dist_kmeans_plusplus(comm, part, padded(X[part.lo:part.hi]), 50, np.random.RandomState(rank))
        # DistKMeans with the reference's default init against the one-GPU KMeans
        t = torch.from_numpy(X).to(dev)
        km = par.DistKMeans(257, "k-means++", random_state=3, max_iter=15, tol=0, comm=comm).fit(t[part.lo:part.hi])
        ref = gdr.KMeans(n_clusters=257, init="k-means++", random_state=3, n_init=1, max_iter=15, tol=0).fit(t)
        assert km.n_iter_ == ref.n_iter_
        same = (km.labels_ == ref.labels_[part.lo:part.hi]).float().mean().item()
        assert same > 0.99, same
        assert abs(km.inertia_ - ref.inertia_) <= 1e-4 * ref.inertia_
        # "random": exactly the centred rows of the permutation
        km0 = par.DistKMeans(257, "random", random_state=4, max_iter=0, tol=0, comm=comm).fit(t[part.lo:part.hi])
        seeds = torch.from_numpy(np.random.RandomState(4).permutation(X.shape[0])[:257]).to(dev)
        Xc = par.CudaOps().center(t, km0._mean)
        C0 = km0._centers_centered
        assert torch.equal(C0.contiguous(), Xc[seeds].contiguous())
        torch.cuda.synchronize()
        comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_row_partitioned_kmeans_plusplus(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    mp.spawn(_worker, args=(world, _free_port()), nprocs=world, join=True)
