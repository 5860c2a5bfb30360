"""Time k-means++ seeding at the stage-3 shapes: the one-GPU kmeans_plusplus_device, the row-partitioned
dist_kmeans_plusplus, and the latter with the score pass skipped ("no_score": the launches, the single-CTA pick /
reduce / choose kernels and the two all-gathers; with one rank the all-gathers are no-ops, so there it measures no
exchange at all).

    python tools/kpp_bench.py [--shapes E,Du,Di] [--reps 3] [--out FILE]
    python -m torch.distributed.run --nproc_per_node 8 tools/kpp_bench.py ...    (NCCL, one GPU per rank)

Shapes: E = config E (N = 2 449 029, D = 100, z-scored synthetic features, K = 10 000); Du / Di = the two sides of
config D (52 643 users / 91 599 items, d = 64, K = 10 %).  The arms alternate within every repetition; the indices of
every arm are compared with the one-GPU seeding at every size.  Prints one JSON line per (shape, arm) on rank 0, with
the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"E": (2449029, 100, 10000), "Du": (52643, 64, 5265), "Di": (91599, 64, 9160)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def features(n, d, seed):
    from gdr import synth
    if d == 100:
        return synth.features(n, d, seed, kind="zscore")
    return (0.1 * np.random.RandomState(seed).standard_normal((n, d))).astype(np.float32)


def bytes_per_round(n_rows, d, L, arm):
    """Device-memory bytes one round moves, from shapes (the rows this GPU holds)."""
    x = n_rows * d * 4
    if arm == "one":   # k_pp_update + k_pp_score each read X; closest read 3x, written once
        return 2 * x + 4 * n_rows * 4
    if arm == "dist":  # one pass: X, the last winner's column, L new columns
        return x + n_rows * 4 + L * n_rows * 4
    return 0           # no pass over X


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="E,Du,Di")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("kpp_bench needs a CUDA device")
    import gdr  # noqa: F401
    from gdr import _lib
    from gdr import parallel as par
    from gdr._dev import new_padded
    from gdr.kmeans_init import kmeans_plusplus_device

    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        rank = int(os.environ["RANK"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    comm = par.Comm(dist)
    dev = torch.device("cuda", torch.cuda.current_device())
    gpu = card()
    lines = []

    def padded(X):
        t = new_padded(X.shape[0], X.shape[1], dev)
        t.copy_(torch.from_numpy(X))
        return t

    for shape in args.shapes.split(","):
        N, D, K = SHAPES[shape]
        L = 2 + int(np.log(K))
        X = features(N, D, 1234)
        part = par.RowPartition(N, world, comm.rank)
        Xf = padded(X) if world == 1 or comm.rank == 0 else None
        Xl = padded(X[part.lo:part.hi])

        def run(arm, seed):
            # every rank enters the barrier of every arm (the same collective sequence on all ranks); the one-GPU
            # arm runs on rank 0 only while the others wait in the next barrier
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            if arm == "one":
                if Xf is None:
                    return 0.0, None
                out = kmeans_plusplus_device(Xf, K, np.random.RandomState(seed), return_indices=True)
            else:
                _lib.call("gdr_debug_set", b"kpp_dist_skip_score", int(arm == "no_score"))
                out = par.dist_kmeans_plusplus(comm, part, Xl, K, np.random.RandomState(seed), return_indices=True)
                _lib.call("gdr_debug_set", b"kpp_dist_skip_score", 0)
            torch.cuda.synchronize()
            return time.perf_counter() - t0, out[1]

        arms = ["one", "dist", "no_score"]
        # warm-up at a small K (module loads, NCCL channels, the attribute opt-in)
        if Xf is not None:
            kmeans_plusplus_device(Xf, 20, np.random.RandomState(0))
        par.dist_kmeans_plusplus(comm, part, Xl, 20, np.random.RandomState(0))
        times = {a: [] for a in arms}
        same = []
        for rep in range(args.reps):
            order = arms if rep % 2 == 0 else arms[::-1]
            idx = {}
            for a in order:
                t, i = run(a, rep)
                times[a].append(t)
                idx[a] = i
            if idx["one"] is not None:
                same.append(bool(torch.equal(idx["one"], idx["dist"])))
        if comm.rank == 0:    # rank 0 holds the one-GPU arm
            for a in arms:
                ts = np.array(times[a])
                rows = N if a == "one" else part.n_local
                rec = dict(shape=shape, N=N, D=D, K=K, n_trials=L, world=1 if a == "one" else world, arm=a,
                           seconds_median=float(np.median(ts)), seconds_min=float(ts.min()), seconds_max=float(ts.max()),
                           us_per_round=float(np.median(ts)) / (K - 1) * 1e6,
                           bytes_per_round=bytes_per_round(rows, D, L, a),
                           no_score_share=None, indices_equal_one_gpu=same if a == "dist" else None, gpu=gpu,
                           reps=args.reps)
                lines.append(rec)
            d_med = next(r for r in lines if r["shape"] == shape and r["arm"] == "dist")["seconds_median"]
            for r in lines:
                if r["shape"] == shape and r["arm"] == "no_score":
                    r["no_score_share"] = r["seconds_median"] / d_med
        del Xf, Xl
        torch.cuda.empty_cache()
    if comm.rank == 0:
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
