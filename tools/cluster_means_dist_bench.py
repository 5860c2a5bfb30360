"""Time the cluster means on a row partition (parallel.dist_cluster_means) against the one-GPU cluster_means and
against the only partitioned option without it (all-gather the rows and labels, then cluster_means), in the same job.

    python tools/cluster_means_dist_bench.py [--shapes E,B] [--reps 7] [--out FILE]
    python -m torch.distributed.run --nproc_per_node 4 tools/cluster_means_dist_bench.py ...    (NCCL, one GPU per rank)

Shapes: E = 2 449 029 x 100 rows, K = 10 000 (config E: the propagated features of ogbn-products' size);
B = 169 343 x 128, K = 1 000 (config B).  The rows are fp32 normal draws scaled over 12 binades, in the padded layout
dist_propagate returns, split into RowPartition's equal blocks; the labels are uniform int32.  Arms, alternated within
every repetition (the order is reversed every other repetition):
    one     cluster_means on all rows, on rank 0 while the other ranks wait;
    gather  every rank all-gathers the rows and the labels, then calls cluster_means;
    dist    dist_cluster_means (gdr_segment_sum_dist: the chain handed from rank to rank, nothing gathered).
Each call is timed with device events around a synchronised call (median over the repetitions).  peak_mb is the
largest rise of torch.cuda.max_memory_allocated over the memory held before the call, on any rank.  byte_parity
compares the gather and dist results with the one-GPU bytes (NaN rows included) and checks that every rank holds the
same bytes.  Prints one JSON line per (shape, arm) on rank 0, with the card name and power limit read in the same run.
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

SHAPES = {"E": (2449029, 100, 10000), "B": (169343, 128, 1000)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="E,B")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cluster_means_dist_bench needs a CUDA device")
    import gdr
    from gdr import parallel as par
    from gdr._dev import new_padded
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        rank = int(os.environ["RANK"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    else:
        # an NCCL group of one rank: the partitioned arms run the same code as at any world size
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29519")
        dist.init_process_group("nccl", rank=0, world_size=1,
                                device_id=torch.device("cuda", torch.cuda.current_device()))
    comm = par.Comm(dist)
    rank = comm.rank
    dev = torch.device("cuda", torch.cuda.current_device())
    gpu = card()
    lines = []
    for shape in args.shapes.split(","):
        N, F, K = SHAPES[shape]
        part = par.RowPartition(N, world, rank)
        g = torch.Generator(device=dev).manual_seed(1234)
        X = torch.randn((N, F), generator=g, device=dev)
        X *= torch.exp(torch.empty((N, 1), device=dev).uniform_(-4, 4, generator=g))
        lab = torch.randint(0, K, (N,), generator=g, device=dev, dtype=torch.int32)
        X_l = new_padded(part.n_local, F, dev)
        X_l.copy_(X[part.lo:part.hi])
        lab_l = lab[part.lo:part.hi].clone()
        if rank == 0:
            X_all = new_padded(N, F, dev)
            X_all.copy_(X)
        else:
            X_all = lab = None
        del X
        torch.cuda.empty_cache()

        def gather_then_means():
            blk = new_padded(part.rows_per, F, dev, zero=True)
            blk[: part.n_local].copy_(X_l)
            full = new_padded(part.rows_per * world, F, dev)
            comm.all_gather_rows(blk, full)
            lblk = torch.zeros(part.rows_per, dtype=torch.int32, device=dev)
            lblk[: part.n_local].copy_(lab_l)
            lfull = torch.empty(part.rows_per * world, dtype=torch.int32, device=dev)
            comm.all_gather_rows(lblk, lfull)
            return gdr.cluster_means(full[:N], lfull[:N], K)

        def run(arm):
            torch.cuda.synchronize()
            dist.barrier()
            if arm == "one" and rank != 0:
                return None, 0.0, 0
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            if arm == "one":
                out = gdr.cluster_means(X_all, lab, K)
            elif arm == "gather":
                out = gather_then_means()
            else:
                out = par.dist_cluster_means(comm, part, X_l, lab_l, K)
            ev1.record()
            ev1.synchronize()
            return out, ev0.elapsed_time(ev1) / 1e3, torch.cuda.max_memory_allocated() - base

        def same_everywhere(t):
            b = t.contiguous().view(torch.int32)
            hi, lo = b.clone(), b.clone()
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            return bool(torch.equal(hi, b) and torch.equal(lo, b))

        arms = ["one", "gather", "dist"]
        for a in arms:                           # warm-up: module loads, NCCL channels, function attributes
            run(a)
        times = {a: [] for a in arms}
        peaks = {a: 0 for a in arms}
        parity = {a: [] for a in arms[1:]}
        for rep in range(args.reps):
            outs = {}
            for a in (arms if rep % 2 == 0 else arms[::-1]):
                outs[a], t, peak = run(a)
                times[a].append(t)
                peaks[a] = max(peaks[a], peak)
            for a in arms[1:]:
                ok = same_everywhere(outs[a])
                if rank == 0:
                    ok = ok and torch.equal(outs[a].contiguous().view(torch.int32),
                                            outs["one"].contiguous().view(torch.int32))
                parity[a].append(ok)
            del outs
        pk = torch.tensor([peaks[a] for a in arms], dtype=torch.int64, device=dev)
        dist.all_reduce(pk, op=dist.ReduceOp.MAX)
        if rank == 0:
            for j, a in enumerate(arms):
                ts = np.array(times[a])
                row = dict(shape=shape, n=N, f=F, k=K, arm=a, world=1 if a == "one" else world,
                           ms_median=float(np.median(ts) * 1e3), ms_min=float(ts.min() * 1e3),
                           ms_max=float(ts.max() * 1e3), peak_mb=round(int(pk[j]) / 2**20, 1),
                           byte_parity=all(parity[a]) if a != "one" else None, reps=args.reps, gpu=gpu)
                if a != "one":
                    row["ratio_to_one_gpu"] = row["ms_median"] / float(np.median(times["one"]) * 1e3)
                lines.append(row)
                print(json.dumps(row), flush=True)
        del X_l, lab_l, X_all, lab
        torch.cuda.empty_cache()
    if rank == 0 and args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in lines) + "\n")
    comm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
