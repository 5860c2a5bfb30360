"""Edge sparsification on a row partition over NCCL (dist_graph_sparse, gdr_sparsify_classes_dist) and the coarsening
of the sparsified blocks (dist_graph_compress_list) against the one-GPU graph_sparse / graph_compress.  Each world
size skips when fewer GPUs are present."""
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
        from gdr.graph import CSR

        class Blocks(par.RowPartition):
            """A row partition with given block bounds (so that a rank can own no rows)."""
            def __init__(self, cuts, rank):
                super().__init__(cuts[-1], len(cuts) - 1, rank)
                self.cuts = cuts

            def bounds(self, rank=None):
                r = self.rank if rank is None else rank
                return self.cuts[r], self.cuts[r + 1]

        comm = par.Comm(dist)
        ops = par.CudaOps()
        cfg = synth.CONFIGS["B"]
        n, C, ratio = cfg["n"], cfg["d_logit"], 0.1
        assert n % world or world == 1
        u, v = synth.uniform_graph(n, cfg["pairs"], seed=31)
        part = par.RowPartition(n, world, rank)
        _, A_full = par.build_local_adjacency(torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev), n, part, dev)
        logits = torch.from_numpy((np.random.RandomState(32).randn(n, C) * 2).astype(np.float32)).to(dev)

        def bits(t):
            return t.contiguous().view(torch.int32)

        def check(A, ebd, sp_type, p):
            one = gdr.graph_sparse(A, ratio, ebd=ebd, sp_type=sp_type)
            lo, hi = p.bounds()
            A_loc = par.slice_rows(A, lo, hi) if hi > lo else None
            blocks = par.dist_graph_sparse(comm, p, A_loc, ratio, ebd[lo:hi], sp_type=sp_type, ops=ops)
            assert len(blocks) == len(one) == (C if sp_type == "attaw" else 1)
            kept = torch.zeros(len(one), dtype=torch.int64, device=dev)
            for c, (b, t) in enumerate(zip(blocks, one)):
                R = t._gdr_csr
                if b is None:
                    assert hi == lo
                    continue
                s, e = int(R.rowptr[lo]), int(R.rowptr[hi])
                assert torch.equal(b.rowptr, R.rowptr[lo:hi + 1] - s), (sp_type, c)
                assert torch.equal(b.colidx, R.colidx[s:e]), (sp_type, c)
                assert torch.equal(bits(b.vals), bits(R.vals[s:e])), (sp_type, c)
                kept[c] = b.nnz
            comm.all_reduce(kept)     # the blocks cover the one-GPU graph: nothing kept twice or lost
            assert kept.tolist() == [t._gdr_csr.nnz for t in one]
            return blocks, one, A_loc

        for sp_type in ("vanilla", "single", "attaw"):
            check(A_full, logits, sp_type, part)
        # class batches of 3: several rounds of collectives per call
        _lib.call("gdr_debug_set", b"sparsify_batch", 3)
        check(A_full, logits, "attaw", part)
        _lib.call("gdr_debug_set", b"sparsify_batch", 0)
        # ties everywhere: binary graph, constant logits
        A_bin = CSR(A_full.rowptr, A_full.colidx, torch.ones_like(A_full.vals), A_full.shape)
        flat = torch.ones_like(logits)
        for sp_type in ("vanilla", "single", "attaw"):
            check(A_bin, flat, sp_type, part)
        if world >= 2:     # rank 1 owns no rows
            cuts = [0, 60000, 60000] + [60000 + (n - 60000) * r // (world - 2) for r in range(1, world - 1)] \
                if world > 2 else [0, n, n]
            for sp_type in ("vanilla", "attaw"):
                check(A_full, logits, sp_type, Blocks(cuts, rank))
        # a k that differs on one rank (one rank: k above the edge count): every rank raises, none hangs
        A_loc = par.slice_rows(A_full, part.lo, part.hi)
        er = torch.ones(A_loc.nnz, dtype=torch.float32, device=dev)
        bad_k = 1000 + (rank == world - 1) if world > 1 else A_loc.nnz + 1
        with pytest.raises(_lib.GdrError):
            ops.sparsify_classes_dist(comm, A_loc, part.lo, n, er, None, bad_k)
        check(A_full, logits, "vanilla", part)      # the communicator still pairs up after the rejected call
        # stage 4 on the sparsified blocks: graph_compress(labels, A, sparsed_list) with the reference's shape
        labels = torch.from_numpy(np.random.RandomState(33).randint(0, 1000, n).astype(np.int64)).to(dev)
        blocks, one, A_loc = check(A_full, logits, "attaw", part)
        lab_l = labels[part.lo:part.hi].contiguous()
        comp1, syn1 = gdr.graph_compress(labels, A_full, one)
        compd, synd = par.dist_graph_compress_list(comm, part, lab_l, A_loc, blocks, ops=ops)
        assert len(compd) == len(comp1)
        for (sd, cnt), s1 in zip(compd + [synd], comp1 + [syn1]):
            assert torch.equal(sd._indices(), s1._indices())
            assert torch.equal(bits(sd._values()), bits(s1._values()))
        syn_alone, cnt_alone = par.dist_graph_compress(comm, part, lab_l, A_loc, ops=ops)
        assert torch.equal(syn_alone._indices(), synd[0]._indices())
        assert torch.equal(bits(syn_alone._values()), bits(synd[0]._values())) and torch.equal(cnt_alone, synd[1])
        torch.cuda.synchronize()
        comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_row_partitioned_graph_sparse(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    mp.spawn(_worker, args=(world, _free_port()), nprocs=world, join=True)
