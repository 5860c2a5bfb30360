"""Cluster means and mean pooling on a row partition over NCCL (dist_segment_sum, dist_cluster_means,
dist_segment_mean_pool) against the one-GPU calls on the rows gathered in rank order: byte-equal on every rank, for
equal and uneven blocks and ranks without rows, and composed with the drivers that produce their inputs
(dist_propagate -> DistKMeans -> dist_cluster_means; dist_kmeans_cluster -> dist_segment_mean_pool).  Needs >= 2 GPUs;
the 4- and 8-rank cases need 4 and 8."""
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
    empty = list(eq)
    empty[world // 2] = empty[world // 2 - 1]          # rank world//2 - 1 gets no rows
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
        from gdr._dev import padded_rows
        comm = par.Comm(dist)
        ops = par.CudaOps()
        bits = lambda t: t.contiguous().view(torch.int32)      # noqa: E731

        def same_everywhere(t):
            hi, lo = bits(t).clone(), bits(t).clone()
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            return torch.equal(hi, bits(t)) and torch.equal(lo, bits(t))

        def gather_rows(x_local, p):
            x2 = x_local if x_local.dim() == 2 else x_local.reshape(-1, 1)
            blk = torch.zeros((p.rows_per, x2.shape[1]), dtype=x2.dtype, device=dev)
            blk[: x2.shape[0]] = x2
            full = torch.empty((p.rows_per * world, x2.shape[1]), dtype=x2.dtype, device=dev)
            dist.all_gather_into_tensor(full, blk)
            full = full[: p.n]
            return full if x_local.dim() == 2 else full.reshape(-1)

        def data(N, F, K, seed):
            rs = np.random.RandomState(seed)
            X = (rs.standard_normal((N, F)) * np.exp(rs.uniform(-6, 6, (N, 1)))).astype(np.float32)
            return torch.from_numpy(X).to(dev), torch.from_numpy(rs.randint(0, K, N).astype(np.int32)).to(dev)

        def check_sums(X, lab, K, row_off):
            # the ops layer takes any contiguous blocks; the drivers take a RowPartition's equal ones
            lo, hi = int(row_off[rank]), int(row_off[rank + 1])
            s1, c1 = gdr.segment_sum(padded_rows(X), lab, K)
            s2, c2 = ops.segment_sum_dist(comm, lo, padded_rows(X[lo:hi].contiguous()), lab[lo:hi].contiguous(), K)
            assert torch.equal(bits(s2), bits(s1)) and torch.equal(c2, c1), (K, row_off)
            assert same_everywhere(s2)

        def check_means(X, lab, K):
            part = par.RowPartition(X.shape[0], world, rank)
            Xl, ll = X[part.lo:part.hi].contiguous(), lab[part.lo:part.hi].contiguous()
            for one, multi in ((gdr.cluster_means, par.dist_cluster_means),
                               (gdr.segment_mean_pool, par.dist_segment_mean_pool)):
                ref, got = one(X, lab, K), multi(comm, part, Xl, ll, K)
                assert got.shape == ref.shape and torch.equal(bits(got), bits(ref)), (one.__name__, X.shape, K)
                assert same_everywhere(got)

        for N, F, K in ((30011, 100, 257), (4001, 47, 5000), (2708, 1433, 140), (5, 3, 4)):
            X, lab = data(N, F, K, seed=N + F)
            for row_off in _layouts(N, world):
                check_sums(X, lab, K, row_off)
            check_means(X, lab, K)
        # a cluster whose members lie on every rank, all other rows in one cluster; and empty clusters (NaN rows)
        X, lab = data(20000, 47, 2, seed=3)
        lab = (torch.arange(20000, device=dev, dtype=torch.int32) % 997 == 0).to(torch.int32)
        check_means(X, lab, 2)
        check_means(X, 4 * lab, 6)
        # N = 5 at world 4: blocks of 2, 2, 1, 0 rows
        X, lab = data(5, 7, 3, seed=4)
        check_means(X, lab, 3)

        # the transductive chain: dist_propagate -> DistKMeans on 47-wide rows -> dist_cluster_means of the F-wide rows
        n, f, k = 30011, 100, 47
        u, v = synth.skewed_graph(n, 200000, seed=11)
        feats = synth.clustered_features(n, f, 60, seed=12)
        part = par.RowPartition(n, world, rank)
        A_local, _ = par.build_local_adjacency(torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev), n, part, dev)
        prop, target = par.dist_propagate(comm, part, A_local, torch.from_numpy(feats[part.lo:part.hi].copy()).to(dev), 3,
                                          0.8, ops=ops)
        logits = target[:, :47].contiguous()
        C0 = synth.kmeans_init(gather_rows(logits, part).cpu().numpy(), 300, seed=13)
        km = par.DistKMeans(300, C0, max_iter=10, tol=0, ops=ops, comm=comm).fit(logits)
        assert km.labels_.dtype == torch.int32 and km.labels_.shape == (part.n_local,)
        feat_syn = par.dist_cluster_means(comm, part, prop, km.labels_, 300)
        ref = gdr.cluster_means(gather_rows(prop, part), gather_rows(km.labels_, part), 300)
        assert torch.equal(bits(feat_syn), bits(ref)) and same_everywhere(feat_syn)

        # the recsys chain: dist_kmeans_cluster -> dist_segment_mean_pool of the teacher rows
        nu, d = 24000, 64
        emb = torch.from_numpy(synth.clustered_features(nu, d, 40, seed=21)).to(dev)
        pu = par.RowPartition(nu, world, rank)
        u2cu, _ = par.dist_kmeans_cluster(comm, pu, emb[pu.lo:pu.hi].contiguous(), 2400, seed=42)
        teacher = emb[pu.lo:pu.hi] * 0.5 + 1.0
        pooled = par.dist_segment_mean_pool(comm, pu, teacher, u2cu, 2400)
        ref = gdr.segment_mean_pool(gather_rows(teacher, pu), gather_rows(u2cu, pu), 2400)
        assert torch.equal(bits(pooled), bits(ref)) and same_everywhere(pooled)

        # a label out of range on one rank, or K that differs on one rank: ValueError everywhere, then a valid call
        X, lab = data(4000, 47, 30, seed=5)
        part = par.RowPartition(4000, world, rank)
        Xl, ll = X[part.lo:part.hi].contiguous(), lab[part.lo:part.hi].clone()
        if rank == world - 1:
            ll[-1] = 30
        with pytest.raises(ValueError):
            par.dist_cluster_means(comm, part, Xl, ll, 30)
        with pytest.raises(ValueError):
            par.dist_cluster_means(comm, part, Xl, lab[part.lo:part.hi].contiguous(), 30 + (rank == 0))
        with pytest.raises(ValueError):
            par.dist_cluster_means(comm, part, Xl, lab[part.lo:part.hi].contiguous(), 0 if rank == 1 else 30)
        with pytest.raises(ValueError):
            par.dist_cluster_means(comm, part, Xl[:, : 46 + (rank == 0)], lab[part.lo:part.hi].contiguous(), 30)
        check_means(X, lab, 30)
        torch.cuda.synchronize()
        comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_row_partitioned_cluster_means(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    mp.spawn(_worker, args=(world, _free_port()), nprocs=world, join=True)
