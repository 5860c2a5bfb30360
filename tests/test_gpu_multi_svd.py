"""The truncated SVD embeddings on a row partition over NCCL (dist_compute_svd_embeddings) against the one-GPU
compute_svd_embeddings: the row blocks gathered in rank order are byte-equal, S is byte-equal on every rank.  Needs >= 2
GPUs; the 4- and 8-rank cases need 4 and 8."""
import os
import socket

import numpy as np
import pytest
import scipy.sparse as sp
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
        from gdr import parallel as par
        from gdr import synth
        comm = par.Comm(dist)

        def gather_rows(x_local, part):
            blk = torch.zeros((part.rows_per, x_local.shape[1]), dtype=x_local.dtype, device=dev)
            blk[: x_local.shape[0]] = x_local
            full = torch.empty((part.rows_per * world, x_local.shape[1]), dtype=x_local.dtype, device=dev)
            dist.all_gather_into_tensor(full, blk)
            return full[: part.n]

        def lines_of_rank(u, i):
            # every rank holds a strided slice of the interaction lines; dist_build_interaction routes them to the owners
            return (torch.from_numpy(np.ascontiguousarray(u[rank::world])).to(dev),
                    torch.from_numpy(np.ascontiguousarray(i[rank::world])).to(dev))

        def check(nu, ni, u, i, dim, seed):
            R = sp.csr_matrix((np.ones(len(u), np.float32), (u, i)), shape=(nu, ni))
            ue, ie = gdr.compute_svd_embeddings(R, dim, seed=seed)
            pu, pi = par.RowPartition(nu, world, rank), par.RowPartition(ni, world, rank)
            R_l, RT_l = par.dist_build_interaction(comm, pu, pi, *lines_of_rank(u, i))
            ud, idd = par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, dim, seed=seed)
            assert tuple(ud.shape) == (pu.n_local, ue.shape[1]) and tuple(idd.shape) == (pi.n_local, ie.shape[1])
            for got, ref, part in ((ud, ue, pu), (idd, ie, pi)):
                full = gather_rows(got, part).cpu().numpy()
                np.testing.assert_array_equal(full.view(np.int32), np.ascontiguousarray(ref).view(np.int32))
            _, S, _ = par.dist_truncated_svd(comm, pu, pi, R_l, RT_l, min(dim, min(nu, ni) - 1), seed=seed)
            S_max = S.clone()
            dist.all_reduce(S_max, op=dist.ReduceOp.MAX)
            S_min = S.clone()
            dist.all_reduce(S_min, op=dist.ReduceOp.MIN)
            assert torch.equal(S_max.view(torch.int32), S.view(torch.int32))
            assert torch.equal(S_min.view(torch.int32), S.view(torch.int32))

        def coo(M):
            M = M.tocoo()
            return M.row.astype(np.int64), M.col.astype(np.int64)

        # Yelp2018-shaped: the users are the small side
        cfg = synth.BIPARTITE["C"]
        u, i = synth.bipartite_interactions(cfg["users"], cfg["items"], cfg["inter"], seed=1236)
        check(cfg["users"], cfg["items"], u, i, cfg["d"], 42)
        # items are the small side
        rs = np.random.RandomState(3)
        P, Qm = rs.rand(3000, 24) < 0.08, rs.rand(24, 2000) < 0.08
        check(3000, 2000, *coo(sp.coo_matrix((P.astype(np.float32) @ Qm.astype(np.float32)) > 0)), 16, 1)
        # the exact path (small side <= 768)
        check(300, 100, *coo(sp.random(300, 100, density=0.15, random_state=np.random.RandomState(5))), 16, 3)
        # a Krylov side of 1500 rows: one Gram slab through every rank
        check(5000, 1500, *coo(sp.random(5000, 1500, density=0.01, random_state=np.random.RandomState(6))), 32, 7)
        # mismatched dim or seed on one rank: every rank raises, none hangs
        pu, pi = par.RowPartition(300, world, rank), par.RowPartition(100, world, rank)
        ur, ir = coo(sp.random(300, 100, density=0.15, random_state=np.random.RandomState(5)))
        R_l, RT_l = par.dist_build_interaction(comm, pu, pi, *lines_of_rank(ur, ir))
        with pytest.raises(ValueError):
            par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, 16 + (rank == 1), seed=3)
        with pytest.raises(ValueError):
            par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, 16, seed=3 + rank)
        torch.cuda.synchronize()
        comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_row_partitioned_svd_embeddings(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    mp.spawn(_worker, args=(world, _free_port()), nprocs=world, join=True)
