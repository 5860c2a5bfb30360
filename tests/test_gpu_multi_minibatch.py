"""MiniBatchKMeans on a row partition over NCCL (DistMiniBatchKMeans, dist_kmeans_cluster) against the one-GPU
MiniBatchKMeans of the full rows: centres bit-identical and the same on every rank, each rank's labels its slice of the
one-GPU labels, the same n_steps_ / n_iter_, inertia within fp64 rounding of the rank grouping; even, uneven and empty
row blocks; a mismatched argument raises on every rank; the recsys chain interaction -> SVD embeddings -> clusters ->
condensed bipartite graph.  Needs >= 2 GPUs; the 4- and 8-rank cases need 4 and 8."""
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


def _layouts(N, world):
    """Row offsets [world + 1]: equal blocks, uneven blocks, and one with a rank without rows."""
    eq = [min(N, r * ((N + world - 1) // world)) for r in range(world)] + [N]
    w = np.arange(1, world + 1, dtype=np.float64) ** 2
    uneven = [0] + [int(v) for v in np.floor(np.cumsum(w)[:-1] / w.sum() * N)] + [N]
    if world == 4 and N == 30011:
        empty = [0, 9000, 20000, 20000, 30011]
    else:
        empty = list(eq)
        empty[world // 2] = empty[world // 2 - 1]      # rank world//2 - 1 gets no rows
    return [eq, uneven, empty]


def _worker(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import gdr
        from gdr import parallel as par
        from gdr import synth
        comm = par.Comm(dist)
        bits = lambda t: t.contiguous().view(torch.int32)      # noqa: E731

        def same_everywhere(t):
            hi, lo = bits(t).clone(), bits(t).clone()
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            return torch.equal(hi, bits(t)) and torch.equal(lo, bits(t))

        def check(X, row_off, **kw):
            ref = gdr.MiniBatchKMeans(**kw).fit(X)
            lo, hi = int(row_off[rank]), int(row_off[rank + 1])
            got = par.DistMiniBatchKMeans(comm=comm, **kw).fit(X[lo:hi].contiguous())
            assert torch.equal(bits(got.cluster_centers_), bits(ref.cluster_centers_)), (kw, row_off)
            assert same_everywhere(got.cluster_centers_)
            assert got.n_steps_ == ref.n_steps_ and got.n_iter_ == ref.n_iter_
            assert abs(got.inertia_ - ref.inertia_) <= 1e-12 * abs(ref.inertia_), (got.inertia_, ref.inertia_)
            if kw.get("compute_labels", True):
                assert got.labels_.shape == (hi - lo,) and torch.equal(got.labels_, ref.labels_[lo:hi])

        X = torch.from_numpy(synth.clustered_features(30011, 40, 50, seed=2)).to(dev)
        for row_off in _layouts(30011, world):
            check(X, row_off, n_clusters=100, random_state=0, batch_size=1000)
        row_off = _layouts(30011, world)[1]
        check(X, row_off, n_clusters=50, random_state=3, batch_size=2048, init="random", n_init=3)
        check(X, row_off, n_clusters=64, random_state=1, batch_size=512, max_iter=5, max_no_improvement=None)
        check(X, row_off, n_clusters=600, random_state=8, batch_size=256, reassignment_ratio=0.3, max_iter=3,
              compute_labels=False)
        X47 = torch.from_numpy(synth.clustered_features(21000, 47, 80, seed=47)).to(dev)
        check(X47, _layouts(21000, world)[2], n_clusters=2100, random_state=42, batch_size=2048)

        # a mismatched seed or batch_size on one rank: ValueError everywhere, the communicator stays usable
        part = par.RowPartition(30011, world, rank)
        Xl = X[part.lo:part.hi].contiguous()
        with pytest.raises(ValueError):
            par.DistMiniBatchKMeans(n_clusters=10, random_state=1 + (rank == world - 1), comm=comm).fit(Xl)
        with pytest.raises(ValueError):
            par.DistMiniBatchKMeans(n_clusters=10, random_state=1, batch_size=512 + (rank == 0), comm=comm).fit(Xl)
        with pytest.raises(ValueError):
            par.DistMiniBatchKMeans(n_clusters=10, comm=comm, random_state=None if rank == 1 else 1).fit(Xl)
        check(X, [part.bounds(r)[0] for r in range(world)] + [30011], n_clusters=10, random_state=1, batch_size=512,
              max_iter=2)

        # the recsys chain on a config-C-shaped interaction set
        cfg = synth.BIPARTITE["C"]
        nu, ni = cfg["users"], cfg["items"]
        u, i = synth.bipartite_interactions(nu, ni, cfg["inter"], seed=1236)
        pu, pi = par.RowPartition(nu, world, rank), par.RowPartition(ni, world, rank)
        u_sl = torch.from_numpy(np.ascontiguousarray(u[rank::world])).to(dev)
        i_sl = torch.from_numpy(np.ascontiguousarray(i[rank::world])).to(dev)
        R_l, RT_l = par.dist_build_interaction(comm, pu, pi, u_sl, i_sl)
        ue, ie = par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, cfg["d"], seed=42)
        ncu, nci = int(np.ceil(0.1 * nu)), int(np.ceil(0.1 * ni))
        u2cu, _ = par.dist_kmeans_cluster(comm, pu, ue, ncu, seed=42)
        i2ci, _ = par.dist_kmeans_cluster(comm, pi, ie, nci, seed=42)

        def gather_rows(x_local, p):
            x2 = x_local if x_local.dim() == 2 else x_local.reshape(-1, 1)
            blk = torch.zeros((p.rows_per, x2.shape[1]), dtype=x2.dtype, device=dev)
            blk[: x2.shape[0]] = x2
            full = torch.empty((p.rows_per * world, x2.shape[1]), dtype=x2.dtype, device=dev)
            dist.all_gather_into_tensor(full, blk)
            full = full[: p.n]
            return full if x_local.dim() == 2 else full.reshape(-1)

        labels = {}
        for name, emb, p, K, lab in (("u", ue, pu, ncu, u2cu), ("i", ie, pi, nci, i2ci)):
            xs = gather_rows(par.dist_standard_scale(comm, emb), p)
            ref = gdr.MiniBatchKMeans(n_clusters=K, random_state=42, batch_size=2048, n_init="auto").fit(xs)
            assert torch.equal(gather_rows(lab, p), ref.labels_.to(torch.int64)), name
            labels[name] = ref.labels_
        rpc, cic, vc = par.dist_build_condensed_bipartite(comm, pu, pi, u_sl, i_sl, u2cu.to(torch.int32),
                                                          i2ci.to(torch.int32), ncu, nci)
        C1 = gdr.build_condensed_bipartite(u, i, labels["u"], labels["i"], ncu, nci, device=dev, return_device=True)
        assert torch.equal(rpc, C1.rowptr) and torch.equal(cic, C1.colidx) and torch.equal(bits(vc), bits(C1.vals))
        assert int(vc.sum().item()) == len(u)
        torch.cuda.synchronize()
        comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_row_partitioned_minibatch_kmeans(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    mp.spawn(_worker, args=(world, _free_port()), nprocs=world, join=True)
