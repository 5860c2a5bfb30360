"""Time the SVD embeddings on a row partition (parallel.dist_compute_svd_embeddings) against the one-GPU
compute_svd_embeddings in the same job.

    python tools/svd_dist_bench.py [--shapes C,D,X] [--reps 5] [--out FILE]
    python -m torch.distributed.run --nproc_per_node 4 tools/svd_dist_bench.py ...    (NCCL, one GPU per rank)

Shapes: C = Yelp2018 (31 668 x 38 048, 1.56 M lines), D = Amazon-book (52 643 x 91 599, 2.98 M lines), X = a synthetic
shape with ten times Amazon-book's users, items and lines (29.8 M); dim 64, seed 42.  The one-GPU arm runs on rank 0
while the other ranks wait; the arms alternate within every repetition.  Each call is timed with device events
around a synchronised call (median over the repetitions) and counted in library launches.  One more run of each arm
with a synchronise around every library call splits the time into sections: the Krylov SpMMs (gdr_spmm_*), the
operand all-gathers and argument checks (exchange), the Gram matrices (gdr_dense_gram[_dist], on the partition the
rank-to-rank hand-off included), the replicated Ritz step (Jacobi + column gather) and the other dense steps (Cholesky,
triangular solve, tall x small products).  byte_parity compares the gathered row blocks with the one-GPU embeddings.
Prints one JSON line per (shape, arm) on rank 0, with the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"C": (31668, 38048, 1561406), "D": (52643, 91599, 2984108), "X": (526430, 915990, 29841080)}
SECTIONS = {"gdr_spmm_prop_planned": "spmm", "gdr_spmm_plan": "spmm", "gdr_dense_gram": "gram",
            "gdr_dense_gram_dist": "gram", "gdr_sym_eig_jacobi": "ritz", "gdr_dense_gather_cols": "ritz",
            "gdr_dense_chol": "dense_other", "gdr_dense_trsm_rows": "dense_other", "gdr_dense_gemm_small": "dense_other"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


class SectionTimer:
    """Stands in for the ctypes module in svd / propagation / CudaOps: every library call in SECTIONS is timed between
    two synchronises."""

    def __init__(self, lib):
        self.lib, self.t = lib, {}

    def __getattr__(self, name):
        return getattr(self.lib, name)

    def add(self, section, t):
        self.t[section] = self.t.get(section, 0.0) + t

    def call(self, name, *args):
        sec = SECTIONS.get(name)
        if sec is None:
            return self.lib.call(name, *args)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc = self.lib.call(name, *args)
        torch.cuda.synchronize()
        self.add(sec, time.perf_counter() - t0)
        return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="C,D,X")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--dim", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("svd_dist_bench needs a CUDA device")
    import gdr
    from gdr import _lib, parallel as par, propagation, svd, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        rank = int(os.environ["RANK"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    else:
        # an NCCL group of one rank: the partitioned arm runs the same code as at any world size
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29517")
        dist.init_process_group("nccl", rank=0, world_size=1,
                                device_id=torch.device("cuda", torch.cuda.current_device()))
    comm = par.Comm(dist)
    rank = comm.rank
    dev = torch.device("cuda", torch.cuda.current_device())
    gpu = card()
    lines = []
    for shape in args.shapes.split(","):
        nu, ni, inter = SHAPES[shape]
        u, i = synth.bipartite_interactions(nu, ni, inter, seed=1236)
        pu, pi = par.RowPartition(nu, world, rank), par.RowPartition(ni, world, rank)
        A = None
        if rank == 0:
            R = sp.csr_matrix((np.ones(inter, np.float32), (u, i)), shape=(nu, ni))
            A = gdr.CSR.from_scipy(R, device=dev)
            del R
        R_l, RT_l = par.dist_build_interaction(comm, pu, pi, torch.from_numpy(u[rank::world]).to(dev),
                                               torch.from_numpy(i[rank::world]).to(dev))
        del u, i

        def run(arm):
            torch.cuda.synchronize()
            dist.barrier()
            if arm == "one" and A is None:
                return None, 0.0, 0
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = gdr.launch_count()
            ev0.record()
            if arm == "one":
                out = gdr.compute_svd_embeddings(A, args.dim, seed=42)
            else:
                out = par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, args.dim, seed=42)
            ev1.record()
            ev1.synchronize()
            return out, ev0.elapsed_time(ev1) / 1e3, gdr.launch_count() - l0

        def gathered(x, part):
            blk = torch.zeros((part.rows_per, x.shape[1]), dtype=x.dtype, device=dev)
            blk[: x.shape[0]] = x
            full = torch.empty((part.rows_per * world, x.shape[1]), dtype=x.dtype, device=dev)
            comm.all_gather_rows(blk, full)
            return full[: part.n]

        run("one"), run("dist")                  # warm-up: module loads, NCCL channels, function attributes
        arms = ["one", "dist"]
        times = {a: [] for a in arms}
        launches, parity = {}, []
        for rep in range(args.reps):
            outs = {}
            for a in (arms if rep % 2 == 0 else arms[::-1]):
                outs[a], t, n = run(a)
                times[a].append(t)
                launches[a] = n
            full = [gathered(x, p) for x, p in zip(outs["dist"], (pu, pi))]
            if rank == 0:
                parity.append(all(np.array_equal(f.cpu().numpy().view(np.int32), o.view(np.int32))
                                  for f, o in zip(full, outs["one"])))
            del outs, full
        # the sectioned runs
        sections = {}
        for a in arms:
            timer = SectionTimer(_lib)
            ag = comm.all_gather_rows

            def timed_gather(*xs, **kw):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = ag(*xs, **kw)
                torch.cuda.synchronize()
                timer.add("exchange", time.perf_counter() - t0)
                return r
            svd._lib = propagation._lib = timer
            comm.all_gather_rows = timed_gather
            ops = par.CudaOps()
            ops._lib = timer
            try:
                torch.cuda.synchronize()
                dist.barrier()
                t0 = time.perf_counter()
                if a == "one":
                    if A is not None:
                        gdr.compute_svd_embeddings(A, args.dim, seed=42)
                else:
                    par.dist_compute_svd_embeddings(comm, pu, pi, R_l, RT_l, args.dim, seed=42, ops=ops)
                torch.cuda.synchronize()
                total = time.perf_counter() - t0
            finally:
                svd._lib = propagation._lib = _lib
                del comm.all_gather_rows
            sections[a] = dict({k: round(v * 1e3, 3) for k, v in sorted(timer.t.items())}, total_ms=round(total * 1e3, 3))
        if rank == 0:
            for a in arms:
                ts = np.array(times[a])
                lines.append(dict(shape=shape, users=nu, items=ni, lines=inter, dim=args.dim, arm=a,
                                  world=1 if a == "one" else world, ms_median=float(np.median(ts) * 1e3),
                                  ms_min=float(ts.min() * 1e3), ms_max=float(ts.max() * 1e3), launches=launches[a],
                                  sections_ms=sections[a], byte_parity=all(parity) if a == "dist" else None,
                                  reps=args.reps, gpu=gpu))
            one = lines[-2]["ms_median"]
            lines[-1]["speedup_vs_one_gpu"] = one / lines[-1]["ms_median"]
            print(json.dumps(lines[-2]), flush=True)
            print(json.dumps(lines[-1]), flush=True)
        del A, R_l, RT_l
        torch.cuda.empty_cache()
    if rank == 0 and args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in lines) + "\n")
    comm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
