"""Time the edge sparsification and the coarsening of the sparsified graphs on a row partition at config E
(ogbn-products shape: N = 2 449 029, 126 M stored entries of A_hat, C = 47 classes, ratio 0.1).

    python tools/sparsify_dist_bench.py [--steps 3] [--out FILE]
    python -m torch.distributed.run --nproc_per_node 8 tools/sparsify_dist_bench.py ...    (NCCL, one GPU per rank)

A_hat comes from dist_build_adjacency (each rank builds its rows from a slice of the synthetic pair list), the logits
are seeded normal draws.  Arms: "one" = the one-GPU graph_sparse('attaw') on the whole graph (rank 0, the other ranks
wait), "sparse" = dist_graph_sparse('attaw'), "compress" = dist_graph_compress_list on its blocks.  Each step is timed
with CUDA events after a 512 MB write that flushes the L2; the reported time is the largest over the ranks.  The parity
flag says whether every rank's blocks equal its rows of the one-GPU result byte for byte (and the coarsened graphs the
one-GPU graph_compress).  Prints one JSON line per arm on rank 0 with the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, PAIRS, C, RATIO, CLUSTERS = 2449029, 61859140, 47, 0.1, 10000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def bytes_per_class(nnz, kept):
    """Device-memory bytes of one class's select over nnz edges keeping `kept`, from shapes: weights (colidx, er,
    prob[dst] read, w written: 16 B), 4 histogram passes (16), tie flags (8) and their scan (8), selection flags (12)
    and their scan (8), compaction (positions 4 per edge; colidx and vals read and written for the kept ones: 16)."""
    return 72 * nnz + 16 * kept


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sparsify_dist_bench needs a CUDA device")
    import gdr
    from gdr import parallel as par
    from gdr import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        rank = int(os.environ["RANK"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    comm = par.Comm(dist)
    rank = comm.rank
    dev = torch.device("cuda", torch.cuda.current_device())
    gpu = card()
    part = par.RowPartition(N, world, rank)
    ops = par.CudaOps()

    u, v = synth.uniform_graph(N, PAIRS, seed=41)
    per = (u.shape[0] + world - 1) // world
    sl = slice(rank * per, min(u.shape[0], (rank + 1) * per))
    u_d, v_d = torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev)
    A_local = par.dist_build_adjacency(comm, part, u_d[sl].contiguous(), v_d[sl].contiguous(), N, ops=ops)
    _, A_full = par.build_local_adjacency(u_d, v_d, N, part, dev)     # the one-GPU operand (parity)
    del u_d, v_d
    logits = torch.from_numpy((np.random.RandomState(42).randn(N, C) * 2).astype(np.float32)).to(dev)
    labels = torch.from_numpy(np.random.RandomState(43).randint(0, CLUSTERS, N).astype(np.int64)).to(dev)
    e_l, lab_l = logits[part.lo:part.hi].contiguous(), labels[part.lo:part.hi].contiguous()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def timed(fn):
        flush.fill_(1)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        return comm.all_reduce(t, "max").item(), out

    one = gdr.graph_sparse(A_full, RATIO, ebd=logits, sp_type="attaw")    # warm-up and the parity reference
    blocks = par.dist_graph_sparse(comm, part, A_local, RATIO, e_l, sp_type="attaw", ops=ops)
    par.dist_graph_compress_list(comm, part, lab_l, A_local, blocks, ops=ops)
    times = {"one": [], "sparse": [], "compress": []}
    for _ in range(args.steps):
        if rank == 0:
            times["one"].append(timed(lambda: gdr.graph_sparse(A_full, RATIO, ebd=logits, sp_type="attaw"))[0])
        elif world > 1:
            timed(lambda: None)
        t, blocks = timed(lambda: par.dist_graph_sparse(comm, part, A_local, RATIO, e_l, sp_type="attaw", ops=ops))
        times["sparse"].append(t)
        t, (compd, synd) = timed(lambda: par.dist_graph_compress_list(comm, part, lab_l, A_local, blocks, ops=ops))
        times["compress"].append(t)

    # parity: this rank's rows of the one-GPU graphs, then the coarsened graphs against the one-GPU graph_compress
    ok = True
    for b, t in zip(blocks, one):
        R = t._gdr_csr
        s, e = int(R.rowptr[part.lo]), int(R.rowptr[part.hi])
        ok &= torch.equal(b.rowptr, R.rowptr[part.lo:part.hi + 1] - s) and torch.equal(b.colidx, R.colidx[s:e]) \
            and torch.equal(b.vals.view(torch.int32), R.vals[s:e].view(torch.int32))
    comp1, syn1 = gdr.graph_compress(labels, A_full, one)
    ok_c = True
    for (sd, _), s1 in zip(compd + [synd], comp1 + [syn1]):
        ok_c &= torch.equal(sd._indices(), s1._indices()) and \
            torch.equal(sd._values().view(torch.int32), s1._values().view(torch.int32))
    flags = torch.tensor([int(ok), int(ok_c)], dtype=torch.int64, device=dev)
    comm.all_reduce(flags, "min")
    nnz, k = A_full.nnz, int(A_full.nnz * RATIO)
    if rank == 0:
        lines = []
        for arm, ts in times.items():
            if not ts:
                continue
            ms = float(np.median(ts))
            w = 1 if arm == "one" else world
            rec = dict(config="E", N=N, nnz=nnz, C=C, ratio=RATIO, k=k, world=w, arm=arm, ms_median=ms,
                       ms_min=float(min(ts)), ms_max=float(max(ts)), steps=args.steps, gpu=gpu, l2_flushed=True)
            if arm != "compress":
                per_rank = bytes_per_class((nnz + w - 1) // w, (k + w - 1) // w)
                rec.update(bytes_per_class_pass=per_rank, TBps_per_gpu=C * per_rank / (ms * 1e-3) / 1e12)
            if arm != "one":
                rec["parity"] = "ok" if int(flags[0 if arm == "sparse" else 1]) else "MISMATCH"
            lines.append(rec)
        for r in lines:
            print(json.dumps(r))
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write("\n".join(json.dumps(r) for r in lines) + "\n")
    comm.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
