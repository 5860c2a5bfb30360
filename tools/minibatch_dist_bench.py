"""Time MiniBatchKMeans on a row partition (parallel.DistMiniBatchKMeans) against the one-GPU MiniBatchKMeans in the
same job.

    python tools/minibatch_dist_bench.py [--configs Cu,Ci,Du,Di,B] [--reps 3] [--out FILE]
    python -m torch.distributed.run --nproc_per_node 4 tools/minibatch_dist_bench.py ...    (NCCL, one GPU per rank)

Configurations (synthetic clustered rows, synth.clustered_features, seed 42):
  Cu / Ci  config C (Yelp2018) users / items: 31 668 / 38 048 x 64, K = ceil(0.1 N), batch 2048
  Du / Di  config D (Amazon-book) users / items: 52 643 / 91 599 x 64, K = ceil(0.1 N), batch 2048
  B        config B (ogbn-arxiv) logit space: 169 343 x 40, K = 1 000, batch 1 000
random_state 0, every other argument sklearn's default (tol 0, max_no_improvement 10).  The one-GPU arm runs on rank 0
(the other ranks wait); the arms alternate within every repetition.  Per fit: the wall time of the fit between two
synchronises (median over the repetitions) split at synchronises into subsets + init (validation subset, init subset,
k-means++), steps (from the validation E-step of the last init candidate on) and the final E-step; us per step; launches (library launch counter,
rank 0).  One more run of each arm synchronises around every library call of a step to split a step into
  exchange   the partitioned arm's batch assembly without labels (a second, rows-only gdr_minibatch_batch_dist of the
             same batch, run only in this sectioned run);
  estep      gdr_kmeans_assign (one GPU), or the labelled assembly minus the rows-only one (partition);
  update     gdr_inertia + gdr_minibatch_update;
the rest of a step (the draws, H2D of the plan, reassignment, the read-back) is "other".  byte_parity: centres, labels,
n_steps_ and n_iter_ of the partitioned fit equal the one-GPU fit's.  Prints one JSON line per (configuration, arm) on
rank 0 with the card name and power limit read in the same run.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {"Cu": (31668, 64, None, 2048), "Ci": (38048, 64, None, 2048), "Du": (52643, 64, None, 2048),
           "Di": (91599, 64, None, 2048), "B": (169343, 40, 1000, 1000)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


class Phases:
    """Synchronised time stamps at the end of the init (last _mb_init + validation E-step) and of the step loop."""

    def __init__(self):
        self.t = {}

    def mark(self, name):
        torch.cuda.synchronize()
        self.t[name] = time.perf_counter()


class StepSections:
    """Stands in for the ctypes module of kmeans / CudaOps during the step loop: times the step's library calls between
    synchronises; a labelled gdr_minibatch_batch_dist is timed again without labels to isolate the exchange."""
    SECTIONS = {"gdr_kmeans_assign": "estep", "gdr_inertia": "update", "gdr_minibatch_update": "update"}

    def __init__(self, lib):
        self.lib, self.t, self.active = lib, {}, False

    def __getattr__(self, name):
        return getattr(self.lib, name)

    def _timed(self, name, *args):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        self.lib.call(name, *args)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def call(self, name, *args):
        if not self.active:
            return self.lib.call(name, *args)
        if name == "gdr_minibatch_batch_dist" and args[11]:
            full = self._timed(name, *args)
            a = list(args)
            a[11], a[12], a[15] = 0, 0, 0            # C, ldc, labels_b: rows only, the same bytes into Xb
            rows = self._timed(name, *a)
            self.t["exchange"] = self.t.get("exchange", 0.0) + rows
            self.t["estep"] = self.t.get("estep", 0.0) + max(full - rows, 0.0)
            return 0
        sec = self.SECTIONS.get(name)
        if sec is None:
            return self.lib.call(name, *args)
        self.t[sec] = self.t.get(sec, 0.0) + self._timed(name, *args)
        return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="Cu,Ci,Du,Di,B")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("minibatch_dist_bench needs a CUDA device")
    import gdr
    import torch.distributed as dist
    from gdr import _lib, kmeans, parallel as par, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        rank = int(os.environ["RANK"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    else:
        # an NCCL group of one rank: the partitioned arm runs the same code as at any world size
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29519")
        dist.init_process_group("nccl", rank=0, world_size=1,
                                device_id=torch.device("cuda", torch.cuda.current_device()))
    comm = par.Comm(dist)
    rank = comm.rank
    dev = torch.device("cuda", torch.cuda.current_device())
    gpu = card()
    ops = par.CudaOps()
    lines = []
    orig_init, orig_loop = kmeans.MiniBatchKMeans._mb_init, kmeans.minibatch_loop

    for name in args.configs.split(","):
        N, D, K, batch = CONFIGS[name]
        K = K or math.ceil(0.1 * N)
        X = torch.from_numpy(synth.clustered_features(N, D, max(K // 10, 8), seed=42)).to(dev)
        part = par.RowPartition(N, world, rank)
        X_local = X[part.lo:part.hi].contiguous()
        kw = dict(n_clusters=K, random_state=0, batch_size=batch)

        def fit(arm, ph):
            """One fit with phase marks; returns the estimator (None on ranks that only wait)."""
            def mb_init(self, *a, **k):
                out = orig_init(self, *a, **k)
                ph.mark("init_call")
                return out

            def loop(est, *a, **k):
                out = orig_loop(est, *a, **k)
                ph.mark("loop_end")
                return out

            kmeans.MiniBatchKMeans._mb_init, kmeans.minibatch_loop = mb_init, loop
            try:
                ph.mark("start")
                if arm == "one":
                    est = gdr.MiniBatchKMeans(**kw).fit(X)
                else:
                    est = par.DistMiniBatchKMeans(comm=comm, ops=ops, **kw).fit(X_local)
                ph.mark("end")
            finally:
                kmeans.MiniBatchKMeans._mb_init, kmeans.minibatch_loop = orig_init, orig_loop
            return est

        res = {"one": [], "dist": []}
        ests = {}
        for rep in range(args.reps + 1):               # repetition 0 warms up
            for arm in ("one", "dist"):
                torch.cuda.synchronize()
                dist.barrier()
                if arm == "one" and rank != 0:
                    continue
                ph = Phases()
                l0 = gdr.launch_count()
                est = fit(arm, ph)
                launches = gdr.launch_count() - l0
                ests[arm] = est
                if rep == 0:
                    continue
                t = ph.t
                # the validation E-step of the last init candidate (one E-step of init_size rows) lands in "steps"
                res[arm].append(dict(total=t["end"] - t["start"], init=t["init_call"] - t["start"],
                                     steps=t["loop_end"] - t["init_call"], final=t["end"] - t["loop_end"],
                                     launches=launches))
        # byte parity of the partitioned fit against the one-GPU fit
        d, one = ests["dist"], ests.get("one")
        lab = d.labels_.to(torch.int32)
        blk = torch.full((part.rows_per,), -1, dtype=torch.int32, device=dev)
        blk[: lab.shape[0]] = lab
        full = torch.empty(part.rows_per * world, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(full, blk)
        parity = None
        if rank == 0:
            parity = bool(torch.equal(d.cluster_centers_.contiguous().view(torch.int32),
                                      one.cluster_centers_.contiguous().view(torch.int32))
                          and torch.equal(full[:N], one.labels_) and d.n_steps_ == one.n_steps_
                          and d.n_iter_ == one.n_iter_)
        # per-step sections, one more fit of each arm
        sect = {}
        for arm in ("one", "dist"):
            torch.cuda.synchronize()
            dist.barrier()
            if arm == "one" and rank != 0:
                continue
            timer = StepSections(_lib)
            kmeans._lib, ops._lib = timer, timer
            orig_first = orig_init

            def mb_init(self, *a, **k):
                out = orig_first(self, *a, **k)
                timer.active = True                  # everything after the (last) init is the loop
                return out

            kmeans.MiniBatchKMeans._mb_init = mb_init
            try:
                est = (gdr.MiniBatchKMeans(compute_labels=False, **kw).fit(X) if arm == "one" else
                       par.DistMiniBatchKMeans(comm=comm, ops=ops, compute_labels=False, **kw).fit(X_local))
            finally:
                kmeans._lib, ops._lib = _lib, _lib
                kmeans.MiniBatchKMeans._mb_init = orig_init
            sect[arm] = {k: v / est.n_steps_ * 1e6 for k, v in timer.t.items()}
        if rank == 0:
            for arm in ("one", "dist"):
                r = res[arm]
                med = {k: float(np.median([x[k] for x in r])) for k in ("total", "init", "steps", "final")}
                e = ests[arm]
                line = dict(bench="minibatch_dist", config=name, arm=arm, world=1 if arm == "one" else world, N=N, D=D,
                            K=K, batch=batch, reps=len(r), fit_s=round(med["total"], 4),
                            init_s=round(med["init"], 4), steps_s=round(med["steps"], 4),
                            final_estep_s=round(med["final"], 4), n_steps=e.n_steps_, n_iter=e.n_iter_,
                            us_per_step=round(med["steps"] / e.n_steps_ * 1e6, 1),
                            step_split_us={k: round(v, 1) for k, v in sect.get(arm, {}).items()},
                            launches=int(np.median([x["launches"] for x in r])),
                            byte_parity=("ok" if parity else "DIFFERS") if arm == "dist" else None,
                            inertia=e.inertia_, gpu=gpu)
                print(json.dumps(line), flush=True)
                lines.append(line)
    if rank == 0 and args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")
    comm.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
