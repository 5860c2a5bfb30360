"""2-rank NCCL run of the row-partitioned drivers with the real CUDA kernels; results must
match the single-GPU path (integers bit-exact, floats within the §8c tolerances).
Needs >= 2 GPUs (gpurun --gpus 2)."""
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
        from gdr import parallel as par
        from gdr import synth
        n, f, k = 30011, 100, 257
        u, v = synth.skewed_graph(n, 200000, seed=11)
        X = synth.clustered_features(n, f, 60, seed=12)
        part = par.RowPartition(n, world, rank)
        comm = par.Comm(dist)
        ops = par.CudaOps()
        u_d, v_d = torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev)
        A_local, A_full = par.build_local_adjacency(u_d, v_d, n, part, dev)
        # stage 1, exchange-based: each rank starts from a slice of the pair list; block == rows of the global build
        per = (u.shape[0] + world - 1) // world
        sl = slice(rank * per, min(u.shape[0], (rank + 1) * per))
        A_x = par.dist_build_adjacency(comm, part, u_d[sl].contiguous(), v_d[sl].contiguous(), n, ops=ops)
        assert torch.equal(A_x.rowptr, A_local.rowptr) and torch.equal(A_x.colidx, A_local.colidx)
        assert torch.equal(A_x.vals, A_local.vals)
        # pipelined hop (3 column slabs, async all-gathers) == one-pass hop
        x_l = torch.from_numpy(X[part.lo:part.hi].copy()).to(dev)
        # ONE hop: rows on the sequential path (<= 1024 non-zeros) are the same fp32 chain whatever the slab width;
        # hub rows are summed as fixed-order partials whose grouping follows the lane-group width (1e-5 contract)
        pa, ta = par.dist_propagate(comm, part, A_local, x_l, 2, 0.8, ops=ops, slabs=1)
        pb, tb = par.dist_propagate(comm, part, A_x, x_l, 2, 0.8, ops=ops, slabs=3)
        light = (A_local.rowptr[1:] - A_local.rowptr[:-1]) <= 1024
        assert torch.equal(pa[light], pb[light]) and torch.equal(ta[light], tb[light])
        # several hops: the hub rows' last-bit differences reach their neighbours
        pa, ta = par.dist_propagate(comm, part, A_local, x_l, 4, 0.8, ops=ops, slabs=1)
        pb, tb = par.dist_propagate(comm, part, A_x, x_l, 4, 0.8, ops=ops, slabs=3)
        torch.testing.assert_close(pa, pb, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(ta, tb, rtol=1e-5, atol=1e-6)
        # stage 2: the fused hop (SpMM epilogue stores into the peers' gathered operand over NVLink; default), the same
        # with the first distribution prefetched on a side stream, and the NCCL all-gather hop — all bit-identical to
        # the single-GPU propagation
        x_local = torch.from_numpy(X[part.lo:part.hi].copy()).to(dev)
        p1, t1 = gdr.propagate(A_full, torch.from_numpy(X).to(dev), 4, 0.8)
        for hop in ("p2p", "nccl", "auto"):
            prop, target = par.dist_propagate(comm, part, A_local, x_local, 4, 0.8, ops=ops, hop=hop)
            assert torch.equal(prop, p1[part.lo:part.hi]) and torch.equal(target, t1[part.lo:part.hi]), hop
        for rep in range(3):
            pre = par.prefetch_rows(comm, part, x_local, ops=ops)
            assert pre is not None
            prop, target = par.dist_propagate(comm, part, A_local, x_local, 4, 0.8, ops=ops, prefetched=pre)
            assert torch.equal(prop, p1[part.lo:part.hi]) and torch.equal(target, t1[part.lo:part.hi])
        prop2, target2 = par.dist_propagate(comm, part, A_local, x_local, 2, 0.8, ops=ops, hop="p2p")     # one hop only
        p2_, t2_ = gdr.propagate(A_full, torch.from_numpy(X).to(dev), 2, 0.8)
        assert torch.equal(prop2, p2_[part.lo:part.hi]) and torch.equal(target2, t2_[part.lo:part.hi])
        # stage 3
        tn = t1.cpu().numpy()
        C0 = synth.kmeans_init(tn, k, seed=13)
        # single step from shared centres (SURVEY §8c protocol 1): labels equal, centres to 1e-5
        # (rows of `target` are bit-identical to t1's, asserted above, so the labels must be EQUAL, not nearly equal)
        # max_iter = 0 is the E-step from the shared centres alone; after one update the centres differ in their last bits
        # (all-reduce order), so the labels of the E-step that follows may differ on near-tie rows
        km0 = par.DistKMeans(k, C0, max_iter=0, tol=0, ops=ops, comm=comm).fit(target)
        ref0 = gdr.KMeans(n_clusters=k, init=C0, n_init=1, max_iter=0, tol=0).fit(t1)
        assert km0.n_iter_ == 0 and torch.equal(km0.labels_, ref0.labels_[part.lo:part.hi])
        km1 = par.DistKMeans(k, C0, max_iter=1, tol=0, ops=ops, comm=comm).fit(target)
        ref1 = gdr.KMeans(n_clusters=k, init=C0, n_init=1, max_iter=1, tol=0).fit(t1)
        assert (km1.labels_ != ref1.labels_[part.lo:part.hi]).sum().item() <= 3
        torch.testing.assert_close(km1.cluster_centers_, ref1.cluster_centers_.contiguous(), rtol=1e-5, atol=1e-5)
        # the host-driven loop (torch.distributed collectives) and the in-library loop (NCCL inside libgdr_b200,
        # graph-replayed) are the same algorithm: identical fits
        kmp = par.DistKMeans(k, C0, max_iter=8, tol=0, ops=ops, comm=comm, python_loop=True).fit(target)
        kml = par.DistKMeans(k, C0, max_iter=8, tol=0, ops=ops, comm=comm).fit(target)
        assert kmp.n_iter_ == kml.n_iter_ and torch.equal(kmp.labels_, kml.labels_)
        assert torch.equal(kmp.cluster_centers_, kml.cluster_centers_)
        # replicated centres bit-identical on every rank
        cc = kml.cluster_centers_.clone()
        mx = cc.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        assert torch.equal(cc, mx)
        # empty clusters: duplicated initial centres -> distributed relocation == single-GPU relocation
        C0e = C0.copy()
        C0e[3] = C0e[2]
        C0e[4] = C0e[2]
        kme = par.DistKMeans(k, C0e, max_iter=1, tol=0, ops=ops, comm=comm).fit(target)
        refe = gdr.KMeans(n_clusters=k, init=C0e, n_init=1, max_iter=1, tol=0).fit(t1)
        torch.testing.assert_close(kme.cluster_centers_, refe.cluster_centers_.contiguous(), rtol=1e-5, atol=1e-5)
        assert (kme.labels_ != refe.labels_[part.lo:part.hi]).sum().item() <= 3
        # end to end (protocol 2): same iteration count, WCSS within 1e-4, labels nearly all equal
        km = par.DistKMeans(k, C0, max_iter=15, tol=0, ops=ops, comm=comm).fit(target)
        ref = gdr.KMeans(n_clusters=k, init=C0, n_init=1, max_iter=15, tol=0).fit(t1)
        assert km.n_iter_ == ref.n_iter_
        same = (km.labels_ == ref.labels_[part.lo:part.hi]).float().mean().item()
        # centres differ in the last bits across rank counts (all-reduce order), a flipped in-band row then
        # perturbs the trajectory: SURVEY §8c end-to-end protocol = WCSS within 1e-4, labels nearly all equal
        assert same > 0.99, same
        assert abs(km.inertia_ - ref.inertia_) <= 1e-4 * ref.inertia_
        # stage 4 (use the single-GPU labels so that the integer result is comparable bit for bit)
        labels = ref.labels_
        _, syn1 = gdr.graph_compress(labels, A_full, [])
        kk = int(labels.max()) + 1
        _, _, cnt1, _ = gdr.coarsen_edges(labels, labels, kk, kk, csr=A_full, drop_diag=True)
        # transports: NCCL send/recv (symm False) and posted stores through the symmetric buffer (gdr_symm_scatterv);
        # forms: cells accumulated in shared memory (dense 1: fixed-point sums with the GLOBAL per-cluster fixed-point
        # step) and the sort (dense 0: fp32 sums in global CSR order) — the routed result equals one GPU's bit for bit in both
        from gdr import _lib as _lib_dbg
        for dense in (1, 0):
            _lib_dbg.call("gdr_debug_set", b"coarsen_dense", dense)
            _, syn_d = gdr.graph_compress(labels, A_full, [])
            for merge, symm in (("records", True), ("route", False), ("route", True)):
                comm.use_symm_exchange = symm
                adj_syn, counts = par.dist_graph_compress(comm, part, labels[part.lo:part.hi].contiguous(), A_local, ops=ops,
                                                          merge=merge)
                assert torch.equal(adj_syn._indices(), syn1._indices())
                assert torch.equal(counts, cnt1)
                torch.testing.assert_close(adj_syn._values(), syn1._values(), rtol=1e-5, atol=1e-9)
                if merge == "route":
                    assert torch.equal(adj_syn._values(), syn_d._values())
        _lib_dbg.call("gdr_debug_set", b"coarsen_dense", 1)
        # not replicated: this rank's key range of the coarse rows
        a_lo, rp_p, ci_p, v_p, c_p = par.dist_graph_compress(comm, part, labels[part.lo:part.hi].contiguous(), A_local, ops=ops,
                                                             replicate=False)
        rp1, ci1, cnt1b, _ = gdr.coarsen_edges(labels, labels, kk, kk, csr=A_full, drop_diag=True)
        nr = rp_p.shape[0] - 1
        b, e = int(rp1[a_lo]), int(rp1[a_lo + nr])
        assert torch.equal(rp_p + b, rp1[a_lo:a_lo + nr + 1]) and torch.equal(ci_p, ci1[b:e]) and torch.equal(c_p, cnt1b[b:e])
        # feature widths that are not a multiple of 4 (row-padded, non-contiguous views in the collectives)
        for f2 in (7, 47):
            X2 = synth.clustered_features(n, f2, 20, seed=21 + f2)
            x2 = torch.from_numpy(X2[part.lo:part.hi].copy()).to(dev)
            for rc in (1, 3):
                p2, t2 = par.dist_propagate(comm, part, A_local, x2, 3, 0.8, ops=ops, row_chunks=rc)
                p2r, t2r = gdr.propagate(A_full, torch.from_numpy(X2).to(dev), 3, 0.8)
                assert torch.equal(p2, p2r[part.lo:part.hi]) and torch.equal(t2, t2r[part.lo:part.hi])
            C2 = synth.kmeans_init(X2, 50, seed=3)
            for py in (False, True):
                k0 = par.DistKMeans(50, C2, max_iter=0, tol=0, ops=ops, comm=comm, python_loop=py).fit(x2)
                r0 = gdr.KMeans(n_clusters=50, init=C2, n_init=1, max_iter=0, tol=0).fit(torch.from_numpy(X2).to(dev))
                assert torch.equal(k0.labels_, r0.labels_[part.lo:part.hi])
                k2 = par.DistKMeans(50, C2, max_iter=1, tol=0, ops=ops, comm=comm, python_loop=py).fit(x2)
                r2 = gdr.KMeans(n_clusters=50, init=C2, n_init=1, max_iter=1, tol=0).fit(torch.from_numpy(X2).to(dev))
                assert (k2.labels_ != r2.labels_[part.lo:part.hi]).sum().item() <= 3
                torch.testing.assert_close(k2.cluster_centers_, r2.cluster_centers_.contiguous(), rtol=1e-5, atol=1e-5)
        # distill_recsys on a row partition (users and items each split over the ranks) == the single-GPU path
        nu, ni, d, L = 6011, 4099, 64, 2
        uu, ii = synth.bipartite_interactions(nu, ni, 90000, seed=31)
        rs = np.random.RandomState(32)
        u0 = (0.1 * rs.standard_normal((nu, d))).astype(np.float32)
        i0 = (0.1 * rs.standard_normal((ni, d))).astype(np.float32)
        pu, pi = par.RowPartition(nu, world, rank), par.RowPartition(ni, world, rank)
        per = (uu.shape[0] + world - 1) // world
        sl = slice(rank * per, min(uu.shape[0], (rank + 1) * per))
        u_sl, i_sl = torch.from_numpy(uu[sl].copy()).to(dev), torch.from_numpy(ii[sl].copy()).to(dev)
        R_l, RT_l = par.dist_build_interaction(comm, pu, pi, u_sl, i_sl, ops=ops)
        A_l, AT_l, du_l, di_l = par.dist_bipartite_normalize(comm, pu, pi, R_l, RT_l, ops=ops)
        R = gdr.coo_to_csr(torch.from_numpy(uu).to(dev), torch.from_numpy(ii).to(dev), None, (nu, ni))
        graph = gdr.BipartiteGraph(R.coo_indices(), R.vals, nu, ni)
        Ar = par.slice_rows(graph.A, pu.lo, pu.hi)
        ATr = par.slice_rows(graph.AT, pi.lo, pi.hi)
        assert torch.equal(A_l.rowptr, Ar.rowptr) and torch.equal(A_l.colidx, Ar.colidx) and torch.equal(A_l.vals, Ar.vals)
        assert torch.equal(AT_l.rowptr, ATr.rowptr) and torch.equal(AT_l.colidx, ATr.colidx) and torch.equal(AT_l.vals, ATr.vals)
        assert torch.equal(du_l, graph.deg_u[pu.lo:pu.hi]) and torch.equal(di_l, graph.deg_i[pi.lo:pi.hi])
        u0d, i0d = torch.from_numpy(u0).to(dev), torch.from_numpy(i0).to(dev)
        uo, io = par.dist_lightgcn_propagate(comm, pu, pi, A_l, AT_l, u0d[pu.lo:pu.hi].contiguous(), i0d[pi.lo:pi.hi].contiguous(), L, ops=ops)
        uo1, io1 = gdr.lightgcn_propagate(graph, u0d, i0d, L)
        assert torch.equal(uo, uo1[pu.lo:pu.hi]) and torch.equal(io, io1[pi.lo:pi.hi])
        xs = par.dist_standard_scale(comm, u0d[pu.lo:pu.hi].contiguous(), ops=ops)
        xs1 = gdr.standard_scale(u0d)
        torch.testing.assert_close(xs, xs1[pu.lo:pu.hi], rtol=1e-6, atol=1e-6)
        ncu, nci = 601, 410
        u2cu = torch.from_numpy(rs.randint(0, ncu, nu).astype(np.int32)).to(dev)
        i2ci = torch.from_numpy(rs.randint(0, nci, ni).astype(np.int32)).to(dev)
        rpc, cic, vc = par.dist_build_condensed_bipartite(comm, pu, pi, u_sl, i_sl, u2cu[pu.lo:pu.hi].contiguous(),
                                                          i2ci[pi.lo:pi.hi].contiguous(), ncu, nci, ops=ops)
        C1 = gdr.build_condensed_bipartite(uu, ii, u2cu, i2ci, ncu, nci, device=dev, return_device=True)
        assert torch.equal(rpc, C1.rowptr) and torch.equal(cic, C1.colidx) and torch.equal(vc, C1.vals)
        assert int(vc.sum().item()) == uu.shape[0]
        torch.cuda.synchronize()
        comm.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_matches_single_gpu():
    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)
