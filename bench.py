#!/usr/bin/env python
"""bench.py — one "step" = one pass of the distillation core over a synthetic graph of a BASELINE.json shape:
stage 1 (CSR build + D^-1/2 A D^-1/2)  ->  stage 2 (K hops)  ->  stage 3 (20 Lloyd iterations from a fixed
init, tol = 0)  ->  stage 4 (P^T A P).  Bipartite workloads (C, D) run the distill_recsys form of the same four
stages: interaction CSR + LightGCN normalisation -> L propagation layers -> per-side k-means -> condensed counts.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload E|B|A|C|D] [--precision fp32|tc]
    python bench.py --impl reference ...        # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR      # also write the last timed step's outputs as DIR/<name>.npy

The default workload is config E (BASELINE.json configs[4], ogbn-products-shaped: the shape the target is quoted
on; it fits one GPU) for EVERY N, so the N = 1, 2, 4, 8 lines are one strong-scaling experiment.

Prints ONE JSON line (rank 0).  `value` = k-means iterations / s (whole job), the quantity BASELINE.json's
speed-up target is quoted on; `prop` carries the A^K.X GB/s figure of the same metric string with its own HBM
roofline.  See DESIGN.md §Measurement.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LLOYD_ITERS = 20
ALPHA = 0.8
HOMOGENEOUS = {"A": 0, "B": 1, "E": 4}
BIPARTITE = {"C": 2, "D": 3}
CPU_SAMPLE_ROWS = 200_000   # bounded k-means sample of the large workload (all K centres, first rows of X)


# ----------------------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d["bf16_tflops"]),
                    bf16_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


def load_synth():
    """The workload generators, loaded BY PATH: `import gdr` would map libgdr_b200.so into the process, and the
    reference arm must stay a pure CPU process (no product code anywhere near it)."""
    spec = importlib.util.spec_from_file_location(
        "_bench_synth", os.path.join(ROOT, "graph-distillation-for-recommendation_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def product_so_mapped() -> bool:
    try:
        return "libgdr_b200" in open("/proc/self/maps").read()
    except OSError:
        return False


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_ev = index, [], threading.Event()
        self.nvml = None
        try:  # in-process NVML: no fork, negligible GIL time (a forked nvidia-smi stalls the launch thread)
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip() != ""]
            if index < len(ids) and ids[index].strip().isdigit():
                return int(ids[index])
        return index

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flag = lambda bit: "Active" if (r & bit) else "Not Active"
        return [str(sm), str(mx), str(pw), flag(0x8), flag(0x40), flag(0x20), flag(0x4)]

    def sample_now(self):
        """One sample from the CALLING thread (used between timed steps: an NVML query running
        concurrently with the launch thread contends on the driver lock and was measured to
        double the step time)."""
        try:
            if self.nvml is not None:
                self.rows.append(self._sample_nvml())
        except Exception:
            pass

    def run(self):
        if self.nvml is not None:
            return   # NVML available: samples are taken by sample_now() from the main thread
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop_ev.wait(0.5)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    samples=len(sm), reasons=reasons)


def make_workload(name, synth, graph="uniform"):
    """Host arrays of one BASELINE.json config (seed = 1234 + config index, SURVEY §8d); the same arrays go to
    the GPU path and to the CPU reference."""
    if name in BIPARTITE:
        cfg = dict(synth.BIPARTITE[name])
        seed = 1234 + BIPARTITE[name]
        u, i = synth.bipartite_interactions(cfg["users"], cfg["items"], cfg["inter"], seed)
        rs = np.random.RandomState(seed + 100)
        u0 = (0.1 * rs.standard_normal((cfg["users"], cfg["d"]))).astype(np.float32)   # nn.init.normal_(std=0.1)
        i0 = (0.1 * rs.standard_normal((cfg["items"], cfg["d"]))).astype(np.float32)
        cfg.update(u=u, i=i, u0=u0, i0=i0, seed=seed, ku=int(np.ceil(0.1 * cfg["users"])), ki=int(np.ceil(0.1 * cfg["items"])),
                   bipartite=True)
        return cfg
    cfg = dict(synth.CONFIGS[name])
    seed = 1234 + HOMOGENEOUS[name]
    gen = synth.uniform_graph if graph == "uniform" else synth.skewed_graph
    u, v = gen(cfg["n"], cfg["pairs"], seed)
    X = synth.features(cfg["n"], cfg["f"], seed + 100, kind="l1" if name == "A" else "zscore")
    cfg.update(u=u, v=v, X=X, seed=seed, bipartite=False)
    return cfg


def workload_string(name, w, kmeans_d=None):
    """ONE string for both arms (the driver compares the two lines' config.workload)."""
    if w.get("bipartite"):
        return (f"config {name}: {w['name']}-shaped user-item bipartite graph, users={w['users']}, items={w['items']}, "
                f"interaction lines={w['inter']} (~4% duplicates), d={w['d']}, LightGCN layers={w['layers']}, "
                f"K_users={w['ku']}, K_items={w['ki']}, {LLOYD_ITERS} Lloyd iterations per side tol=0")
    d = w["f"] if kmeans_d is None else kmeans_d
    return (f"config {name}: {w['name']}-shaped uniform graph, N={w['n']}, undirected input pairs={w['u'].shape[0]}, "
            f"F={w['f']}, hops={w['hops']}, K={w['k']}, k-means D={d}, {LLOYD_ITERS} Lloyd iterations tol=0")


def spmm_bytes(nnz, rows, xrows, F, fused=True, model="min"):
    """SURVEY §8(d): compulsory (B_min) or gather (B_gather) bytes of one hop."""
    if model == "min":
        b = nnz * 8 + (rows + 1) * 4 + xrows * F * 4 + rows * F * 4
    else:
        b = nnz * (8 + 4 * F) + (rows + 1) * 4 + rows * F * 4
    return b + (2 * rows * F * 4 if fused else 0)


# ----------------------------------------------------------------------------------------
# --dump-outputs DIR: what the last timed step computed, so that two builds can be compared output for output.
# Outputs larger than the budget are written as a fixed sample of their rows (seed 0: the same rows every run).
DUMP_ROWS = 16384          # rows written of a per-node feature matrix
DUMP_GRAPH_ROWS = 128      # rows of a coarsened graph written as dense rows
DUMP_MAX_BYTES = 64 << 20


def dump_rows(n, cap):
    """Sorted indices of the rows written of an n-row output: all of them, or a seeded sample of cap rows."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.RandomState(0).choice(n, cap, replace=False))


def csr_rows_dense(A, rows):
    """Rows `rows` of a device CSR as a dense float32 host array."""
    import torch
    rp = A.rowptr.cpu().numpy().astype(np.int64)
    lo, hi = rp[rows], rp[rows + 1]
    pos = torch.from_numpy(np.concatenate([np.arange(a, b) for a, b in zip(lo, hi)] + [np.zeros(0, np.int64)])).to(A.device)
    out = np.zeros((len(rows), A.shape[1]), np.float32)
    out[np.repeat(np.arange(len(rows)), hi - lo), A.colidx[pos].cpu().numpy()] = A.vals[pos].cpu().numpy()
    return out


def graph_outputs(name, A):
    """A coarsened graph as <name> (DUMP_GRAPH_ROWS dense rows), <name>_rows (their indices) and <name>_row_nnz
    (the non-zero count of every row)."""
    rows = dump_rows(A.shape[0], DUMP_GRAPH_ROWS)
    return {name: csr_rows_dense(A, rows), name + "_rows": rows, name + "_row_nnz": np.diff(A.rowptr.cpu().numpy())}


def write_outputs(out_dir, arrays):
    """<out_dir>/<name>.npy for every entry: float32 stays float32, everything else (labels, indices, scalars)
    is written as float64."""
    host = {}
    for name, a in arrays.items():
        a = np.asarray(a.cpu().numpy() if hasattr(a, "cpu") else a)
        host[name] = a if a.dtype == np.float32 else a.astype(np.float64)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_THREAD_LIMIT = None


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the reference's CPU path has to run on ALL the host cores
    (the other ranks of the reference arm exit at once), so the BLAS / OpenMP / torch pools are raised at run time."""
    global _THREAD_LIMIT
    n = len(os.sched_getaffinity(0))
    try:
        import torch
        torch.set_num_threads(n)
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_limits
        _THREAD_LIMIT = threadpool_limits(limits=n)   # kept alive for the rest of the process
    except Exception:
        pass
    return n


# ========================================================================================
# reference arm: the reference's own CPU path (oracle/ref_port.py restates its call sites on scipy /
# torch-CPU sparse / scikit-learn, the libraries that own its arithmetic).  Pure CPU process.
# ========================================================================================
def run_reference(args, rank, world):
    if rank != 0:
        return
    import torch
    from oracle import ref_port as rp
    synth = load_synth()
    assert not product_so_mapped(), "the reference arm must not load the product library"
    use_all_host_threads()
    w = make_workload(args.workload, synth)
    info = rp.host_info()
    if w["bipartite"]:
        return run_reference_bipartite(args, w, info, rp, synth)
    n, F, K, hops = w["n"], w["f"], w["k"], w["hops"]
    if n * K > 1e9:
        return run_reference_bounded(args, w, info, rp, synth)
    t_s1, t_s2, t_s3, t_s4, per_step = [], [], [], [], []
    it_lo, it_hi = 3, 3 + args.ref_kmeans_iters
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        A = rp.build_adjacency(w["u"], w["v"], n)
        adj = rp.to_tensor_sparse(A)
        adj_norm = rp.normalize_adj_tensor_sparse(adj)
        t1 = time.perf_counter()
        _, target = rp.propagate(adj_norm, torch.from_numpy(w["X"]), hops + 1, ALPHA)
        t2 = time.perf_counter()
        tn = target.numpy()
        C0 = synth.kmeans_init(tn, K, w["seed"])
        rp.kmeans_fit(tn, C0, 1)  # first call pays thread-pool start-up; keep it out of the difference
        t3 = time.perf_counter()
        rp.kmeans_fit(tn, C0, it_lo)
        t3a = time.perf_counter()
        km = rp.kmeans_fit(tn, C0, it_hi)
        t3b = time.perf_counter()
        rp.graph_compress_sparse(km.labels_.astype(np.int64), adj_norm)
        t4 = time.perf_counter()
        if s >= args.warmup:
            t_s1.append(t1 - t0)
            t_s2.append(t2 - t1)
            # differenced: (fit with it_hi) - (fit with it_lo) cancels validation / centring / final E-step
            d_it = ((t3b - t3a) - (t3a - t3)) / (it_hi - it_lo)
            if d_it <= 0:   # tiny problems converge before it_lo: fall back to the undifferenced fit
                d_it = (t3b - t3a) / max(1, int(km.n_iter_))
            t_s3.append(d_it)
            t_s4.append(t4 - t3b)
            per_step.append(t4 - t0)
    nnz = adj_norm._nnz()
    s_iter = float(np.mean(t_s3))
    iters_per_s = 1.0 / s_iter
    prop_gbs = hops * spmm_bytes(nnz, n, n, F) / np.mean(t_s2) / 1e9
    line = {
        "impl": "reference", "metric": "kmeans_iters_per_s", "value": iters_per_s, "unit": "iters/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(per_step)) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, w), "nnz_a_hat": int(nnz),
                   "lloyd_iters_timed": f"sklearn fit(max_iter={it_hi}) - fit(max_iter={it_lo})", "full_size": True},
        "prop": {"metric": "A^K.X", "value": prop_gbs, "unit": "GB/s", "bytes_model": "B_min",
                 "s_per_hop": float(np.mean(t_s2)) / hops},
        "stages_ms": {"s1_build_normalize": np.mean(t_s1) * 1e3, "s2_propagate": np.mean(t_s2) * 1e3,
                      "s3_kmeans_per_iter": s_iter * 1e3, "s4_coarsen": np.mean(t_s4) * 1e3},
        "cpu_baseline": {"value": iters_per_s, "unit": "iters/s", "cores": info["affinity"], "kind": "port",
                         "sample": f"full config {args.workload}; sklearn/scipy/torch-CPU with all host threads", "host": info},
        "e2e": {"value": iters_per_s, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "product_so_mapped": product_so_mapped(),
    }
    print(json.dumps(line))


def reference_full_size_legs(w, rp, synth, budget_s):
    """Config E at FULL size on the host, once per run (not per step): every stage of the reference's CPU path
    as BASELINE.md §4 prescribes, each leg skipped (null + reason) when the remaining budget cannot hold it.
      s1  utils_graphsaint.py:18-22 build + deep_robust_utils.to_tensor + normalize_adj_tensor(sparse=True).  The
          reference's normalize_adj goes through scipy `tolil()` (Python-object lists: 126 M entries, hours and
          > 60 GB) — timed here on a 1/32 row block and reported as infeasible at full size; the downstream legs use
          the same arithmetic without the LIL detour (csr + diags products).
      s2  ONE hop of clustgdd_agent_transduct.py:59-65 on torch-CPU sparse COO ((alpha*adj_norm) @ X), reported per hop
      s3  sklearn KMeans(init=C0, n_init=1, tol=0): fit(max_iter=3) - fit(max_iter=1) on all 2.45 M rows
      s4  graph_compress with a sparse one-hot (the dense N x n one-hot is 196 GB): scipy P^T A_hat P"""
    import scipy.sparse as sp
    import torch
    n, F, K, hops = w["n"], w["f"], w["k"], w["hops"]
    t_start = time.perf_counter()
    left = lambda: budget_s - (time.perf_counter() - t_start)
    out = {"budget_s": budget_s, "notes": []}
    adj_norm = None
    if left() > 0:
        t0 = time.perf_counter()
        A = rp.build_adjacency(w["u"], w["v"], n)
        t1 = time.perf_counter()
        adj = rp.to_tensor_sparse(A)
        t2 = time.perf_counter()
        # normalize_adj (deep_robust_utils.py:180-207) without tolil(): identical arithmetic (fp64 rowsum, power -1/2,
        # two diagonal products), then back to a torch COO as normalize_adj_tensor does
        mx = sp.csr_matrix((adj._values().numpy(), adj._indices().numpy()), shape=(n, n))
        if mx[0, 0] == 0:
            mx = mx + sp.eye(n, format="csr")
        rowsum = np.asarray(mx.sum(1)).ravel()
        with np.errstate(divide="ignore"):
            r_inv = np.power(rowsum, -0.5)
        r_inv[np.isinf(r_inv)] = 0.0
        mx = sp.diags(r_inv).dot(mx).dot(sp.diags(r_inv))
        adj_norm = rp.to_tensor_sparse(mx.tocsr())
        t3 = time.perf_counter()
        out["s1_build_adjacency_s"] = t1 - t0
        out["s1_to_tensor_s"] = t2 - t1
        out["s1_normalize_without_tolil_s"] = t3 - t2
        out["s1_build_normalize_s"] = t3 - t0
        out["nnz_a_hat"] = int(adj_norm._nnz())
        # the reference's own normalize_adj_tensor (with tolil) on a 1/32 row block, to document why it is not run whole
        m = n // 32
        blk = A[:m, :m].tocsr()
        t4 = time.perf_counter()
        rp.normalize_adj_tensor_sparse(rp.to_tensor_sparse(blk))
        out["s1_reference_tolil_path_on_1_32_block_s"] = time.perf_counter() - t4
        out["notes"].append("normalize_adj's tolil() detour is not run at full size (Python-object lists for 126 M entries); "
                            "s1 uses the same fp64 arithmetic on CSR")
        del A, adj, mx, blk
    if adj_norm is not None and left() > 60:
        X = torch.from_numpy(w["X"])
        t0 = time.perf_counter()
        prop = ALPHA * adj_norm @ X
        _ = (1 - ALPHA) * X + (1 - ALPHA) * prop
        out["s2_one_hop_s"] = time.perf_counter() - t0
        out["s2_propagate_s"] = out["s2_one_hop_s"] * hops
        out["s2_b_gather_gbs"] = spmm_bytes(out["nnz_a_hat"], n, n, F, model="gather") / out["s2_one_hop_s"] / 1e9
        out["notes"].append(f"s2: one hop timed, s2_propagate_s = {hops} x that")
        del prop
    else:
        out["notes"].append("s2 skipped: budget")
    if left() > 45:
        Xh = w["X"]
        C0 = synth.kmeans_init(Xh, K, w["seed"])
        rp.kmeans_fit(Xh[:20000], C0[:100], 2)
        t0 = time.perf_counter()
        rp.kmeans_fit(Xh, C0, 1)
        t1 = time.perf_counter()
        km = rp.kmeans_fit(Xh, C0, 3)
        t2 = time.perf_counter()
        s_iter = ((t2 - t1) - (t1 - t0)) / 2.0
        out["s3_fit1_s"], out["s3_fit3_s"] = t1 - t0, t2 - t1
        out["s3_kmeans_per_iter_s"] = s_iter
        out["s3_kmeans_iters_per_s"] = 1.0 / s_iter if s_iter > 0 else None
        labels = km.labels_.astype(np.int64)
    else:
        out["notes"].append("s3 skipped: budget")
        labels = np.random.RandomState(0).randint(0, K, n).astype(np.int64)
    if adj_norm is not None and left() > 45:
        t0 = time.perf_counter()
        S = rp.graph_compress_sparse(labels, adj_norm)
        out["s4_coarsen_s"] = time.perf_counter() - t0
        out["s4_syn_nnz"] = int(S.nnz)
    else:
        out["notes"].append("s4 skipped: budget")
    out["wall_s"] = time.perf_counter() - t_start
    return out


def run_reference_bounded(args, w, info, rp, synth):
    """Large workload (config E).  Per STEP: a bounded sample of the same workload — sklearn Lloyd on the first
    CPU_SAMPLE_ROWS rows of the feature matrix against all K centres, differenced between max_iter 1 and 3, rate
    scaled by rows/N (an iteration costs the same flops whatever the rows hold).  Once per RUN: every stage at full
    size (reference_full_size_legs), printed beside the sampled rate."""
    n, F, K, hops = w["n"], w["f"], w["k"], w["hops"]
    full = reference_full_size_legs(w, rp, synth, args.ref_full_budget) if args.ref_full_budget > 0 else None
    rates, what, per_step = [], "", []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        rate, what = cpu_kmeans_rate(w, 1, 3, CPU_SAMPLE_ROWS, synth=synth)
        if s >= args.warmup:
            rates.append(rate)
            per_step.append(time.perf_counter() - t0)
    iters_per_s = float(np.mean(rates))
    g = (lambda k, sc=1e3: (None if (full is None or full.get(k) is None) else full[k] * sc))
    line = {
        "impl": "reference", "metric": "kmeans_iters_per_s", "value": iters_per_s, "unit": "iters/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(per_step)) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, w), "per_step_sample": what,
                   "full_size": "every stage once per run, see full_size"},
        "stages_ms": {"s1_build_normalize": g("s1_build_normalize_s"), "s2_propagate": g("s2_propagate_s"),
                      "s3_kmeans_per_iter": 1e3 / iters_per_s, "s3_kmeans_per_iter_full_size": g("s3_kmeans_per_iter_s"),
                      "s4_coarsen": g("s4_coarsen_s")},
        "full_size": full,
        "prop": None if g("s2_one_hop_s") is None else {
            "metric": "A^K.X", "value": full["s2_b_gather_gbs"], "unit": "GB/s", "bytes_model": "B_gather",
            "s_per_hop": full["s2_one_hop_s"]},
        "cpu_baseline": {"value": iters_per_s, "unit": "iters/s", "cores": info["affinity"], "kind": "port",
                         "sample": what, "full_size_iters_per_s": None if full is None else full.get("s3_kmeans_iters_per_s"),
                         "host": info},
        "e2e": {"value": iters_per_s, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "product_so_mapped": product_so_mapped(),
    }
    print(json.dumps(line))


def run_reference_bipartite(args, w, info, rp, synth):
    """distill_recsys on the host (configs C / D), full size every step: build_interaction_matrix, LightGCN
    propagate (torch index_add_), StandardScaler + sklearn KMeans per side (init pinned), build_condensed_bipartite."""
    import torch
    nu, ni = w["users"], w["items"]
    it_lo, it_hi = 2, 2 + max(2, args.ref_kmeans_iters // 2)
    t_s1, t_s2, t_s3, t_s4, per_step = [], [], [], [], []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        R = rp.build_interaction_matrix(nu, ni, w["u"], w["i"])
        coo = R.tocoo()
        cu, ci = torch.from_numpy(coo.row.astype(np.int64)), torch.from_numpy(coo.col.astype(np.int64))
        wgt = torch.from_numpy(coo.data.astype(np.float32))
        t1 = time.perf_counter()
        rp.lightgcn_propagate(cu, ci, wgt, torch.from_numpy(w["u0"]), torch.from_numpy(w["i0"]), w["layers"])
        t2 = time.perf_counter()
        d_it, maps = 0.0, []
        for emb, K in ((w["u0"], w["ku"]), (w["i0"], w["ki"])):
            Xs = rp.standard_scale(emb).astype(np.float32)
            C0 = synth.kmeans_init(Xs, K, w["seed"])
            ta = time.perf_counter()
            rp.kmeans_fit(Xs, C0, it_lo)
            tb = time.perf_counter()
            km = rp.kmeans_fit(Xs, C0, it_hi)
            tc = time.perf_counter()
            d = ((tc - tb) - (tb - ta)) / (it_hi - it_lo)
            d_it += d if d > 0 else (tc - tb) / max(1, int(km.n_iter_))
            maps.append(km.labels_.astype(np.int64))
        t3 = time.perf_counter()
        rp.build_condensed_bipartite(w["u"], w["i"], maps[0], maps[1], w["ku"], w["ki"])
        t4 = time.perf_counter()
        if s >= args.warmup:
            t_s1.append(t1 - t0)
            t_s2.append(t2 - t1)
            t_s3.append(d_it)
            t_s4.append(t4 - t3)
            per_step.append(t4 - t0)
    s_iter = float(np.mean(t_s3))
    line = {
        "impl": "reference", "metric": "kmeans_iters_per_s", "value": 1.0 / s_iter, "unit": "iters/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(per_step)) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, w), "full_size": True,
                   "iteration": "one Lloyd iteration over BOTH sides (users + items)",
                   "lloyd_iters_timed": f"sklearn fit(max_iter={it_hi}) - fit(max_iter={it_lo}) per side"},
        "stages_ms": {"s1_build_normalize": np.mean(t_s1) * 1e3, "s2_propagate": np.mean(t_s2) * 1e3,
                      "s3_kmeans_per_iter": s_iter * 1e3, "s4_coarsen": np.mean(t_s4) * 1e3},
        "cpu_baseline": {"value": 1.0 / s_iter, "unit": "iters/s", "cores": info["affinity"], "kind": "port",
                         "sample": f"full config {args.workload}; scipy / torch-CPU index_add_ / sklearn with all host threads",
                         "host": info},
        "e2e": {"value": 1.0 / s_iter, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "product_so_mapped": product_so_mapped(),
    }
    print(json.dumps(line))


def cpu_kmeans_rate(w, it_lo, it_hi, rows_cap=None, synth=None, X=None, K=None):
    """k-means iterations/s of the reference's CPU path (sklearn Lloyd, all host threads) on workload w,
    differenced between two max_iter values so that validation / centring / the final E-step cancel.
    With rows_cap the fit runs on the first rows_cap rows against all K centres and the rate is scaled by
    rows_cap / N (the E-step is linear in the rows and dominates: 2*N*K*D flops per iteration)."""
    from oracle import ref_port as rp
    synth = synth or load_synth()
    X = w["X"] if X is None else X
    K = w["k"] if K is None else K
    n = X.shape[0]
    m = n if rows_cap is None else min(n, int(rows_cap))
    Xs = np.ascontiguousarray(X[:m])
    C0 = synth.kmeans_init(Xs, K, w["seed"])       # the init rows lie inside the sample
    rp.kmeans_fit(Xs[:20000], C0[: min(K, 100)], 2)  # warm the thread pools
    t0 = time.perf_counter()
    rp.kmeans_fit(Xs, C0, it_lo)
    t1 = time.perf_counter()
    km = rp.kmeans_fit(Xs, C0, it_hi)
    t2 = time.perf_counter()
    s_iter = ((t2 - t1) - (t1 - t0)) / float(it_hi - it_lo)
    if s_iter <= 0:   # noisy or converged before it_lo: undifferenced fit
        s_iter = (t2 - t1) / max(1, int(km.n_iter_))
    rate = (1.0 / s_iter) * (m / n)
    what = (f"sklearn KMeans(init=C0,n_init=1,tol=0) on "
            + (f"the full {n}x{X.shape[1]} matrix" if m == n else f"the first {m} of {n} rows (x{X.shape[1]}), rate scaled by {m}/{n}")
            + f", K={K}: fit({it_hi} it) - fit({it_lo} it)")
    return rate, what


def cpu_baseline(w, args, synth):
    """Bounded CPU sample on this box's host cores (oracle-side port of the reference)."""
    from oracle import ref_port as rp
    info = rp.host_info()
    if w.get("bipartite"):
        s_iter, what = 0.0, []
        for emb, K in ((w["u0"], w["ku"]), (w["i0"], w["ki"])):
            Xs = rp.standard_scale(emb).astype(np.float32)
            r, wh = cpu_kmeans_rate(w, 2, 6, synth=synth, X=Xs, K=K)
            s_iter += 1.0 / r
            what.append(wh)
        return {"value": 1.0 / s_iter, "unit": "iters/s", "cores": info["affinity"], "kind": "port",
                "sample": " + ".join(what), "host": info}
    big = w["n"] * w["k"] > 1e9
    rate, what = cpu_kmeans_rate(w, 1, 3, CPU_SAMPLE_ROWS, synth=synth) if big else cpu_kmeans_rate(w, 2, 12, synth=synth)
    return {"value": rate, "unit": "iters/s", "cores": info["affinity"], "kind": "port", "sample": what, "host": info}


# ========================================================================================
# our arm, one GPU
# ========================================================================================
def _profile_kernel(_lib, kind, fn, reps, flush):
    """Average duration of the launches of one kernel kind inside fn(), by the CUDA-event pairs the library records
    on its own launch stream (gdr_profile_enable): (ms per launch, launches)."""
    import ctypes
    import torch
    tot_ms, n_l = ctypes.c_double(0), ctypes.c_int64(0)
    _lib.call("gdr_profile_enable", kind)
    for _ in range(reps):
        flush.fill_(1)
        fn()
    torch.cuda.synchronize()
    _lib.call("gdr_profile_collect", ctypes.addressof(tot_ms), ctypes.addressof(n_l))
    _lib.call("gdr_profile_enable", 0)
    return tot_ms.value / max(1, n_l.value), int(n_l.value)


def _ncu_traffic(workload):
    """DRAM bytes per launch from the committed `ncu --set full` capture of this same command
    (profiles/ncu_traffic.json: a constant of the profile, not a measurement of this run)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(workload, {})
    except Exception:
        return {}


def run_ours(args, rank, world):
    import torch
    import gdr
    from gdr import synth
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.tc_screen:
        from gdr import _lib as _l
        _l.call("gdr_debug_set", b"tc_screen", int(args.tc_screen))
    w = make_workload(args.workload, synth)
    if world > 1:
        if w["bipartite"]:
            return run_ours_multi_bipartite(args, rank, world, dev, w)
        return run_ours_multi(args, rank, world, dev, w)
    if w["bipartite"]:
        return run_ours_bipartite(args, dev, w)

    from gdr import _lib
    n, F, K, hops, seed = w["n"], w["f"], w["k"], w["hops"], w["seed"]
    pk = peaks()

    # inputs resident in HBM before the timed region
    u_d = torch.from_numpy(w["u"]).to(dev)
    v_d = torch.from_numpy(w["v"]).to(dev)
    X_d = torch.from_numpy(w["X"]).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def build():
        return gdr.sym_normalize(gdr.coo_to_csr(u_d, v_d, None, (n, n), symmetrize=True, binarize=True), 2)

    # k-means init: C0 = X_target[perm[:K]] needs the propagated features -> computed once, untimed
    A0 = build()
    _, tgt0 = gdr.propagate(A0, X_d, hops + 1, ALPHA)
    perm = torch.from_numpy(np.random.RandomState(seed).permutation(n)[:K].astype(np.int64)).to(dev)
    C0 = tgt0[perm].clone()
    nnz = A0.nnz
    del A0, tgt0

    def step(keep=False):
        e = [ev() for _ in range(5)]
        e[0].record()
        An = build()
        e[1].record()
        prop, target = gdr.propagate(An, X_d, hops + 1, ALPHA)
        e[2].record()
        km = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=LLOYD_ITERS, tol=0, precision=args.precision)
        km.fit(target)
        e[3].record()
        _, adj_syn = gdr.graph_compress(km.labels_, An, [])
        e[4].record()
        # keep only scalars: holding km / adj_syn of every step alive fragments the caching allocator
        # and forces cudaMalloc (a device-wide sync) inside later timed steps; `keep` (the last timed step
        # under --dump-outputs) also returns the outputs themselves
        out = dict(prop=prop, target=target, labels=km.labels_, centers=km.cluster_centers_, inertia=km.inertia_,
                   n_iter=km.n_iter_, adj_syn=gdr.CSR.from_torch_coo(adj_syn)) if keep else None
        return e, types.SimpleNamespace(n_iter_=km.n_iter_, inertia_=km.inertia_), int(adj_syn._nnz()), out

    # W warm-up steps, continued until the GPU has been busy for >= 2 s: a fresh process starts
    # with the GPU in its idle power state and the first ~0.5 s of work runs at about half speed
    t_warm = time.perf_counter()
    n_warm = 0
    while n_warm < args.warmup or (not args.profile and time.perf_counter() - t_warm < 2.0):
        step()
        flush.fill_(1)
        n_warm += 1
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = gdr.launch_count()
    recs = []
    t_wall0 = time.perf_counter()
    for s in range(args.steps):
        flush.fill_(1)          # L2 flush between timed iterations (untimed)
        torch.cuda.synchronize()
        recs.append(step(keep=args.dump_outputs is not None and s == args.steps - 1))
        sampler.sample_now()    # clocks / throttle reasons while the GPU is still under load
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    launches = gdr.launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs is not None:
        o = recs[-1][3]
        rows = dump_rows(n, DUMP_ROWS)
        rows_d = torch.from_numpy(rows).to(dev)
        o.update(prop=o["prop"][rows_d], target=o["target"][rows_d], feature_rows=rows)
        o.update(graph_outputs("adj_syn", o.pop("adj_syn")))
        write_outputs(args.dump_outputs, o)
        del o, rows_d
        recs[-1] = recs[-1][:3]

    st = np.array([[r[0][i].elapsed_time(r[0][i + 1]) for i in range(4)] for r in recs])  # ms per stage
    step_ms = st.sum(axis=1)
    n_iter = [r[1].n_iter_ for r in recs]
    km_ms, prop_ms = st[:, 2], st[:, 1]
    iters_per_s = float(np.sum(n_iter) / (km_ms.sum() / 1e3))

    # roofline legs: the E-step screen and the SpMM kernel alone, timed by CUDA-event pairs recorded inside the
    # library on its launch stream (separate passes: event pairs cannot live inside the replayed graph)
    assign_ms, _ = _profile_kernel(_lib, 1, step, 3, flush)
    assign_total_ms = assign_ms * (LLOYD_ITERS + 1) * args.steps   # launches per step: 20 iterations + final E-step
    A_t = build()
    spmm_ms, _ = _profile_kernel(_lib, 2, lambda: gdr.propagate(A_t, X_d, hops + 1, ALPHA), 5, flush)
    # SURVEY §8(d) headline rule: B_gather when X does not fit L2 (N*F*4 > 96 MB), else B_min
    prop_model = "gather" if n * F * 4 > 96e6 else "min"
    b_hop = spmm_bytes(nnz, n, n, F, model=prop_model)
    b_prop = hops * b_hop + 2 * n * F * 4  # + the t = 0 scale pass
    prop_gbs = float(b_prop / (prop_ms.mean() / 1e3) / 1e9)

    traffic = _ncu_traffic(args.workload)
    flops = 2.0 * n * K * F
    a_tf = float(flops / (assign_ms / 1e3) / 1e12)
    tc = args.precision in ("tc", "auto") and F <= 128
    two_level = tc and (args.tc_screen >= 2 or (args.tc_screen == 0 and -(-n // 128) >= 4 * 148))
    roofline = {"kernel": ("k_assign_tc two-level screen (tcgen05 1xTF32 all rows -> select -> compact -> 3xTF32 undecided rows)" if two_level
                           else "k_assign_tc (tcgen05 3xTF32)") if tc else "k_assign_simt (exact fp32 FFMA)",
                "bound": "tensor", "achieved": a_tf, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                "frac": a_tf / pk["bf16_sustained"], "traffic": traffic.get("k_assign_tc") if tc else None,
                "traffic_source": "profiles/ncu_traffic.json (ncu --set full capture of this command; not measured in this run)",
                "peak_source": pk["src"] + " bf16 sustained",
                "note": "useful flops 2NKD per E-step over the time of the whole tensor-core screen; fp32 inputs run as TF32 "
                        "(1/2 the bf16 rate), so 0.5 is the ceiling of this fraction",
                "launch_ms": float(assign_ms), "share_of_step": float(assign_total_ms / step_ms.sum())}
    b_head = spmm_bytes(nnz, n, n, F, model=prop_model)
    roofline_spmm = {"kernel": "k_spmm", "bound": "hbm", "achieved": float(b_head / (spmm_ms / 1e3) / 1e9), "peak": pk["hbm"],
                     "unit": "GB/s", "frac": float(b_head / (spmm_ms / 1e3) / 1e9 / pk["hbm"]),
                     "traffic": traffic.get("k_spmm"), "launch_ms": float(spmm_ms),
                     "bytes_model": "B_gather (X exceeds L2)" if prop_model == "gather" else "B_min (X fits L2; the gathers run out of L2)",
                     "b_min_gbs": float(spmm_bytes(nnz, n, n, F) / (spmm_ms / 1e3) / 1e9),
                     "b_gather_gbs": float(spmm_bytes(nnz, n, n, F, model='gather') / (spmm_ms / 1e3) / 1e9),
                     "peak_source": pk["src"]}
    del A_t

    # ---- §8(d) secondary legs: the reference-faithful logit-space k-means width and the skewed (hub-heavy) graph ----
    legs = {}
    if not args.profile and not args.no_extra_legs:
        legs["kmeans_logit"] = logit_leg(args, gdr, _lib, synth, w, dev, flush, pk)
        legs["prop_skewed"] = skewed_leg(args, gdr, _lib, synth, w, dev, flush, pk, X_d)

    # ---- e2e through the public API with HOST buffers ----
    e2e = e2e_homogeneous(args, gdr, w, dev, flush, C0, build, X_d)

    cpu = cpu_baseline(w, args, synth) if not (args.no_cpu_baseline or args.profile) else None
    line = {
        "metric": "kmeans_iters_per_s", "value": iters_per_s, "unit": "iters/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(step_ms.mean()), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, w), "nnz_a_hat": int(nnz),
                   "precision": args.precision, "tc_screen": args.tc_screen, "l2": "flushed between timed steps (256 MB write)"},
        "prop": {"metric": "A^K.X", "value": prop_gbs, "unit": "GB/s", "frac_hbm_measured": prop_gbs / pk["hbm"],
                 "frac_hbm_8TBs": prop_gbs / 8000.0, "bytes_model": "B_gather" if prop_model == "gather" else "B_min",
                 "ms": float(prop_ms.mean())},
        "stages_ms": {"s1_build_normalize": float(st[:, 0].mean()), "s2_propagate": float(prop_ms.mean()),
                      "s3_kmeans": float(km_ms.mean()), "s3_kmeans_per_iter": float(km_ms.sum() / np.sum(n_iter)),
                      "s4_coarsen": float(st[:, 3].mean())},
        "stage_rooflines": {
            "s1": {"bytes_model": "E_in*16 + nnz*8", "gbs": float((w["u"].shape[0] * 16 + nnz * 8) / (st[:, 0].mean() / 1e3) / 1e9),
                   "edges_per_s": float(w["u"].shape[0] / (st[:, 0].mean() / 1e3))},
            "s4": {"bytes_model": "nnz*24", "gbs": float(nnz * 24 / (st[:, 3].mean() / 1e3) / 1e9),
                   "edges_per_s": float(nnz / (st[:, 3].mean() / 1e3))}},
        "roofline": roofline, "roofline_spmm": roofline_spmm, **legs, "cpu_baseline": cpu,
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "wall_s": t_wall,
        "result": {"inertia": recs[-1][1].inertia_, "n_iter": int(n_iter[-1]), "syn_nnz": int(recs[-1][2])},
    }
    print(json.dumps(line))


def logit_leg(args, gdr, _lib, synth, w, dev, flush, pk):
    """k-means on the width ClustGDD actually clusters: the MLP probe's logits, N x nclass
    (clustgdd_agent_transduct.py:88-105; 47 classes at ogbn-products, 40 at arxiv, 7 at Cora)."""
    import torch
    n, K, D = w["n"], w["k"], w["d_logit"]
    Xl = torch.from_numpy(synth.clustered_features(n, D, D, seed=w["seed"] + 200)).to(dev)
    perm = torch.from_numpy(np.random.RandomState(w["seed"]).permutation(n)[:K].astype(np.int64)).to(dev)
    C0 = Xl[perm].clone()

    def fit():
        return gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=LLOYD_ITERS, tol=0, precision=args.precision).fit(Xl)

    fit()
    ts, its = [], []
    for _ in range(3):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        km = fit()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
        its.append(km.n_iter_)
    screen_ms, _ = _profile_kernel(_lib, 1, fit, 2, flush)
    tf = 2.0 * n * K * D / (screen_ms / 1e3) / 1e12
    return {"D": D, "value": float(sum(its) / (sum(ts) / 1e3)), "unit": "iters/s", "ms_per_iter": float(sum(ts) / sum(its)),
            "screen_ms": float(screen_ms), "tflops": float(tf), "frac": float(tf / pk["bf16_sustained"]),
            "note": "synthetic logits: mixture of nclass Gaussians; same K, init rule and iteration count as the headline"}


def skewed_leg(args, gdr, _lib, synth, w, dev, flush, pk, X_d):
    """SURVEY §8(d) secondary graph: hub-biased destinations (v = floor(N r^3) for half of the pairs) — exercises the
    load balancing of the SpMM; hub rows hit L2, so DRAM bytes < B_gather here."""
    import torch
    n, F, hops = w["n"], w["f"], w["hops"]
    u, v = synth.skewed_graph(n, w["pairs"], w["seed"] + 7)
    A = gdr.sym_normalize(gdr.coo_to_csr(torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev), None, (n, n),
                                         symmetrize=True, binarize=True), 2)
    deg = (A.rowptr[1:] - A.rowptr[:-1])
    gdr.propagate(A, X_d, hops + 1, ALPHA)
    ms, _ = _profile_kernel(_lib, 2, lambda: gdr.propagate(A, X_d, hops + 1, ALPHA), 5, flush)
    model = "gather" if n * F * 4 > 96e6 else "min"
    b = spmm_bytes(A.nnz, n, n, F, model=model)
    return {"graph": "skewed (50% of destinations floor(N r^3))", "nnz": int(A.nnz), "max_degree": int(deg.max()),
            "mean_degree": float(A.nnz / n), "ms_per_hop": float(ms), "gbs": float(b / (ms / 1e3) / 1e9),
            "frac": float(b / (ms / 1e3) / 1e9 / pk["hbm"]), "bytes_model": "B_gather" if model == "gather" else "B_min"}


def e2e_homogeneous(args, gdr, w, dev, flush, C0, build, X_d):
    """The same metric through the public API from pinned HOST buffers.  `value`: KMeans.fit with the H2D copy of the
    propagated rows and the D2H read of labels + centres inside the timed region.  `pipeline`: the WHOLE step from
    host buffers — H2D of the pair list and the features, stages 1-4, D2H of labels, centres and the coarsened graph."""
    import torch
    n, F, K, hops = w["n"], w["f"], w["k"], w["hops"]
    C0_host = C0.cpu().numpy()
    target_host = torch.empty((n, F), dtype=torch.float32).pin_memory()
    target_host.copy_(gdr.propagate(build(), X_d, hops + 1, ALPHA)[1])
    e2e_t = []
    for i in range(2 if args.profile else max(3, min(args.steps, 6))):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x_dev = target_host.to(dev, non_blocking=True)
        km = gdr.KMeans(n_clusters=K, init=C0_host, n_init=1, max_iter=LLOYD_ITERS, tol=0, precision=args.precision).fit(x_dev)
        km.labels_.cpu()
        km.cluster_centers_.cpu()
        torch.cuda.synchronize()
        e2e_t.append((time.perf_counter() - t0, km.n_iter_))
    e2e_t = e2e_t[1:]
    out = {"value": float(sum(k for _, k in e2e_t) / sum(t for t, _ in e2e_t)), "unit": "iters/s",
           "h2d_bytes_per_step": n * F * 4 + K * F * 4, "d2h_bytes_per_step": n * 4 + K * F * 4}
    if args.profile:
        return out
    del target_host
    u_pin, v_pin = torch.from_numpy(w["u"]).pin_memory(), torch.from_numpy(w["v"]).pin_memory()
    X_pin = torch.from_numpy(w["X"]).pin_memory()
    ts = []
    out_pin = {}

    def d2h(name, t):
        """device -> pinned host buffer (allocated on the first, untimed repetition)"""
        if name not in out_pin or out_pin[name].shape != t.shape:
            out_pin[name] = torch.empty(tuple(t.shape), dtype=t.dtype).pin_memory()
        out_pin[name].copy_(t, non_blocking=True)
        return out_pin[name]

    for i in range(3):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        u_e, v_e, X_e = u_pin.to(dev, non_blocking=True), v_pin.to(dev, non_blocking=True), X_pin.to(dev, non_blocking=True)
        An = gdr.sym_normalize(gdr.coo_to_csr(u_e, v_e, None, (n, n), symmetrize=True, binarize=True), 2)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        _, target = gdr.propagate(An, X_e, hops + 1, ALPHA)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        km = gdr.KMeans(n_clusters=K, init=C0_host, n_init=1, max_iter=LLOYD_ITERS, tol=0, precision=args.precision).fit(target)
        d2h("labels", km.labels_)
        d2h("centres", km.cluster_centers_)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        _, adj_syn = gdr.graph_compress(km.labels_, An, [])
        d2h("syn_idx", adj_syn._indices())
        val_h = d2h("syn_val", adj_syn._values())
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        ts.append((t1 - t0, t2 - t1, t3 - t2, t4 - t3, int(val_h.numel())))
    ts = np.array(ts[1:], dtype=np.float64)
    m = ts.mean(axis=0)
    out["pipeline"] = {
        "ms": float(m[:4].sum() * 1e3),
        "stages_ms": {"s1_h2d_pairs_features_build_normalize": float(m[0] * 1e3), "s2_propagate": float(m[1] * 1e3),
                      "s3_kmeans_d2h_labels_centres": float(m[2] * 1e3), "s4_coarsen_d2h_graph": float(m[3] * 1e3)},
        "h2d_bytes": int(w["u"].shape[0] * 16 + n * F * 4 + K * F * 4),
        "d2h_bytes": int(n * 4 + K * F * 4 + m[4] * 20),
        "note": "wall clock with a synchronize per stage; pinned host buffers; whole step incl. all copies"}
    return out


# ========================================================================================
# our arm, one GPU, bipartite (configs C / D)
# ========================================================================================
def run_ours_bipartite(args, dev, w):
    import torch
    import gdr
    from gdr import _lib, synth
    pk = peaks()
    nu, ni, d, L, ku, ki, seed = w["users"], w["items"], w["d"], w["layers"], w["ku"], w["ki"], w["seed"]
    u_d, i_d = torch.from_numpy(w["u"]).to(dev), torch.from_numpy(w["i"]).to(dev)
    u0, i0 = torch.from_numpy(w["u0"]).to(dev), torch.from_numpy(w["i0"]).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # fixed init per side: rows perm[:K] of the z-scored embeddings (distill_recsys.py:172)
    C0 = []
    for emb, K in ((u0, ku), (i0, ki)):
        Xs = gdr.standard_scale(emb)
        perm = torch.from_numpy(np.random.RandomState(seed).permutation(emb.shape[0])[:K].astype(np.int64)).to(dev)
        C0.append(Xs[perm].clone())

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def step(keep=False):
        e = [ev() for _ in range(5)]
        e[0].record()
        R = gdr.coo_to_csr(u_d, i_d, None, (nu, ni))                 # build_interaction_matrix: duplicates summed
        graph = gdr.BipartiteGraph(R.coo_indices(), R.vals, nu, ni)  # degrees + LightGCN edge norm, R and R^T
        e[1].record()
        emb_out = gdr.lightgcn_propagate(graph, u0, i0, L)
        e[2].record()
        its, maps, inertia = 0, [], 0.0
        out = dict(u_emb=emb_out[0], i_emb=emb_out[1]) if keep else None   # keep: the last timed step under --dump-outputs
        del emb_out
        for side, emb, K, c0 in (("u", u0, ku, C0[0]), ("i", i0, ki, C0[1])):
            km = gdr.KMeans(n_clusters=K, init=c0, n_init=1, max_iter=LLOYD_ITERS, tol=0, precision=args.precision)
            km.fit(gdr.standard_scale(emb))
            its += km.n_iter_
            inertia += km.inertia_
            maps.append(km.labels_)
            if keep:
                out.update({f"labels_{side}": km.labels_, f"centers_{side}": km.cluster_centers_,
                            f"inertia_{side}": km.inertia_, f"n_iter_{side}": km.n_iter_})
        e[3].record()
        C = gdr.build_condensed_bipartite(u_d, i_d, maps[0], maps[1], ku, ki, device=dev, return_device=True)
        e[4].record()
        if keep:
            out["condensed"] = C
        return e, types.SimpleNamespace(n_iter_=its / 2.0, inertia_=inertia), int(C.nnz), out

    t_warm, n_warm = time.perf_counter(), 0
    while n_warm < args.warmup or (not args.profile and time.perf_counter() - t_warm < 2.0):
        step()
        flush.fill_(1)
        n_warm += 1
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index)
    sampler.start()
    launches0 = gdr.launch_count()
    recs = []
    t_wall0 = time.perf_counter()
    for s in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        recs.append(step(keep=args.dump_outputs is not None and s == args.steps - 1))
        sampler.sample_now()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    launches = gdr.launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs is not None:
        o = recs[-1][3]
        for side, n_side in (("u", nu), ("i", ni)):
            rows = dump_rows(n_side, DUMP_ROWS)
            o[f"{side}_emb"] = o[f"{side}_emb"][torch.from_numpy(rows).to(dev)]
            o[f"{side}_emb_rows"] = rows
        o.update(graph_outputs("condensed", o.pop("condensed")))
        write_outputs(args.dump_outputs, o)
        del o
        recs[-1] = recs[-1][:3]
    st = np.array([[r[0][i].elapsed_time(r[0][i + 1]) for i in range(4)] for r in recs])
    n_iter = [r[1].n_iter_ for r in recs]
    iters_per_s = float(np.sum(n_iter) / (st[:, 2].sum() / 1e3))
    assign_ms, n_l = _profile_kernel(_lib, 1, step, 3, flush)
    flops = 2.0 * (nu * ku + ni * ki) * d / 2.0     # mean over the two sides' E-steps (launches alternate)
    a_tf = float(flops / (assign_ms / 1e3) / 1e12)
    R = gdr.coo_to_csr(u_d, i_d, None, (nu, ni))
    graph = gdr.BipartiteGraph(R.coo_indices(), R.vals, nu, ni)
    spmm_ms, _ = _profile_kernel(_lib, 2, lambda: gdr.lightgcn_propagate(graph, u0, i0, L), 5, flush)
    nnz = R.nnz
    b_layer = 2 * nnz * 8 + (nu + ni + 2) * 4 + 2 * (nu + ni) * d * 4 + 2 * (nu + ni) * d * 4   # both directions of one layer (B_min, fused accumulate)
    prop_gbs = float(L * b_layer / (st[:, 1].mean() / 1e3) / 1e9)

    # e2e: kmeans_cluster-style call from HOST arrays (H2D of the embeddings, D2H of labels + centres), both sides
    e2e_t = []
    u0_pin, i0_pin = torch.from_numpy(w["u0"]).pin_memory(), torch.from_numpy(w["i0"]).pin_memory()
    c0_host = [c.cpu().numpy() for c in C0]
    for _ in range(max(3, min(args.steps, 6))):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        its = 0
        for pin, K, c0 in ((u0_pin, ku, c0_host[0]), (i0_pin, ki, c0_host[1])):
            km = gdr.KMeans(n_clusters=K, init=c0, n_init=1, max_iter=LLOYD_ITERS, tol=0, precision=args.precision)
            km.fit(gdr.standard_scale(pin.to(dev, non_blocking=True)))
            km.labels_.cpu()
            km.cluster_centers_.cpu()
            its += km.n_iter_
        torch.cuda.synchronize()
        e2e_t.append((time.perf_counter() - t0, its / 2.0))
    e2e_t = e2e_t[1:]
    cpu = cpu_baseline(w, args, synth) if not (args.no_cpu_baseline or args.profile) else None
    line = {
        "metric": "kmeans_iters_per_s", "value": iters_per_s, "unit": "iters/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(st.sum(axis=1).mean()), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, w), "nnz_r": int(nnz),
                   "iteration": "one Lloyd iteration over BOTH sides (users + items)", "precision": args.precision,
                   "l2": "flushed between timed steps (256 MB write)"},
        "prop": {"metric": "LightGCN layers on R / R^T", "value": prop_gbs, "unit": "GB/s", "frac_hbm_measured": prop_gbs / pk["hbm"],
                 "bytes_model": "B_min (embeddings fit L2)", "ms": float(st[:, 1].mean())},
        "stages_ms": {"s1_build_normalize": float(st[:, 0].mean()), "s2_propagate": float(st[:, 1].mean()),
                      "s3_kmeans": float(st[:, 2].mean()), "s3_kmeans_per_iter": float(st[:, 2].sum() / np.sum(n_iter)),
                      "s4_coarsen": float(st[:, 3].mean())},
        "roofline": {"kernel": "k_assign_tc (tcgen05), mean over the users' and items' E-steps", "bound": "tensor", "achieved": a_tf,
                     "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": a_tf / pk["bf16_sustained"], "traffic": None,
                     "launch_ms": float(assign_ms), "peak_source": pk["src"] + " bf16 sustained"},
        "roofline_spmm": {"kernel": "k_spmm", "bound": "hbm", "launch_ms": float(spmm_ms), "peak": pk["hbm"], "unit": "GB/s",
                          "achieved": float(b_layer / 2 / (spmm_ms / 1e3) / 1e9), "frac": float(b_layer / 2 / (spmm_ms / 1e3) / 1e9 / pk["hbm"]),
                          "bytes_model": "B_min per direction", "traffic": None},
        "cpu_baseline": cpu,
        "e2e": {"value": float(sum(k for _, k in e2e_t) / sum(t for t, _ in e2e_t)), "unit": "iters/s",
                "h2d_bytes_per_step": (nu + ni) * d * 4 + (ku + ki) * d * 4, "d2h_bytes_per_step": (nu + ni) * 4 + (ku + ki) * d * 4},
        "gpu_launches": int(launches), "clocks": clocks, "wall_s": t_wall,
        "result": {"inertia": recs[-1][1].inertia_, "n_iter": float(n_iter[-1]), "condensed_nnz": int(recs[-1][2])},
    }
    print(json.dumps(line))


# ========================================================================================
# our arm, N > 1
# ========================================================================================
def one_gpu_reference(workload):
    """The committed single-GPU measurement of the same workload (for the strong-scaling ratio)."""
    name = {"E": "r2_bench_configE_1gpu.json", "B": "r2_bench_configB_1gpu.json"}.get(workload)
    try:
        d = json.loads(open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1])
        return {"value": d["value"], "unit": d["unit"], "ms_per_step": d["ms_per_step"], "source": "profiles/" + name}
    except Exception:
        return None


def multi_parity(gdr, par, comm, part, ops, dev, w, A_ref, tgt_ref, C0, u_sl, v_sl):
    """N > 1 parity record, computed OUTSIDE the timed region on every rank and reduced with MIN: this rank's
    block of each stage against the same rows of the single-GPU path run on this very GPU.
      adj_block_equal   rows of A_hat built by the all-to-all exchange == rows of the one-GPU build (rowptr/colidx/vals)
      prop_rows_equal   distributed hops == one-GPU hops on this rank's rows (bit-exact: same fp32 chains)
      labels_equal      the E-step from shared centres on bit-identical rows: labels torch.equal to the one-GPU labels
      centres_close     centres after ONE Lloyd step within 1e-5 (the all-reduce order changes the last bits; the labels
                        of the E-step that follows may then differ on a few near-tie rows: labels_differ_after_update)
      counts_equal      integer cell counts of the coarsened graph == one-GPU counts (same labels in)"""
    import torch
    import torch.distributed as dist
    n, K, hops = w["n"], w["k"], w["hops"]
    lo, hi = part.lo, part.hi
    out = {}
    A_blk = par.dist_build_adjacency(comm, part, u_sl, v_sl, n, ops=ops)
    A_rows = par.slice_rows(A_ref, lo, hi)
    out["adj_block_equal"] = bool(torch.equal(A_blk.rowptr, A_rows.rowptr) and torch.equal(A_blk.colidx, A_rows.colidx)
                                  and torch.equal(A_blk.vals, A_rows.vals))
    x_local = torch.from_numpy(w["X"][lo:hi].copy()).to(dev)
    _, t_l = par.dist_propagate(comm, part, A_blk, x_local, hops + 1, ALPHA, ops=ops)
    out["prop_rows_equal"] = bool(torch.equal(t_l, tgt_ref[lo:hi]))
    out["prop_rows_max_rel_err"] = float(((t_l - tgt_ref[lo:hi]).abs().max() / tgt_ref.abs().max()).item())
    # the E-step from the SHARED centres (max_iter = 0: no update, labels of C0) must agree bit for bit; after one update
    # the centres differ in their last bits (all-reduce order), so only their closeness is part of the contract
    x_blk = tgt_ref[lo:hi].contiguous()
    km0 = par.DistKMeans(K, C0, max_iter=0, tol=0, ops=ops, comm=comm).fit(x_blk)
    ref0 = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=0, tol=0).fit(tgt_ref)
    out["labels_equal"] = bool(torch.equal(km0.labels_, ref0.labels_[lo:hi]))
    out["labels_differ"] = int((km0.labels_ != ref0.labels_[lo:hi]).sum().item())
    km1 = par.DistKMeans(K, C0, max_iter=1, tol=0, ops=ops, comm=comm).fit(x_blk)
    ref1 = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=1, tol=0).fit(tgt_ref)
    cdiff = (km1.cluster_centers_ - ref1.cluster_centers_).abs().max() / ref1.cluster_centers_.abs().max()
    out["centres_close"] = bool(cdiff.item() <= 1e-5)
    out["labels_differ_after_update"] = int((km1.labels_ != ref1.labels_[lo:hi]).sum().item())
    labels = ref1.labels_
    adj_syn, counts = par.dist_graph_compress(comm, part, labels[lo:hi].contiguous(), A_blk, ops=ops)
    kk = int(labels.max()) + 1
    rp1, ci1, cnt1, _ = gdr.coarsen_edges(labels, labels, kk, kk, csr=A_ref, drop_diag=True)
    _, syn1 = gdr.graph_compress(labels, A_ref, [])
    out["counts_equal"] = bool(counts.shape == cnt1.shape and torch.equal(counts, cnt1)
                               and torch.equal(adj_syn._indices(), syn1._indices()))
    vdiff = (adj_syn._values() - syn1._values()).abs().max() / syn1._values().abs().max() if out["counts_equal"] else torch.tensor(1.0)
    out["coarse_values_close"] = bool(vdiff.item() <= 1e-5)
    # informative, not part of `status`: the owner-side shared-memory merge uses the single-GPU fixed-point step
    out["coarse_values_bit_equal"] = bool(out["counts_equal"] and torch.equal(adj_syn._values(), syn1._values()))
    flags = [k for k, v in out.items() if isinstance(v, bool)]
    t = torch.tensor([1 if out[k] else 0 for k in flags], dtype=torch.int32, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    d = torch.tensor([out["labels_differ"], out["labels_differ_after_update"]], dtype=torch.int64, device=dev)
    dist.all_reduce(d)
    e = torch.tensor([out["prop_rows_max_rel_err"]], dtype=torch.float64, device=dev)
    dist.all_reduce(e, op=dist.ReduceOp.MAX)
    res = {k: bool(v) for k, v in zip(flags, t.tolist())}
    res["labels_differ"], res["labels_differ_after_update"] = int(d[0].item()), int(d[1].item())
    res["prop_rows_max_rel_err"] = float(e.item())
    must = ["adj_block_equal", "labels_equal", "centres_close", "counts_equal", "coarse_values_close"]
    res["status"] = "ok" if all(res[k] for k in must) and res["prop_rows_max_rel_err"] <= 1e-5 else "MISMATCH"
    res["what"] = "each rank's block vs the same rows of the single-GPU path (MIN over ranks); single Lloyd step from shared centres"
    return res


def run_ours_multi(args, rank, world, dev, w):
    """N > 1: the same step on the same graph, nodes row-partitioned over the ranks (strong
    scaling).  NCCL all-gather of the propagated rows per hop, all-reduce of the centroid
    partial sums / counts per Lloyd iteration, key-range exchange merge of the coarsened graph."""
    import torch
    import torch.distributed as dist
    import gdr
    from gdr import _lib
    from gdr import parallel as par
    dist.init_process_group("nccl", device_id=dev)
    n, F, K, hops, seed = w["n"], w["f"], w["k"], w["hops"], w["seed"]
    pk = peaks()
    part = par.RowPartition(n, world, rank)
    comm = par.Comm(dist)
    ops = par.CudaOps(precision=args.precision)
    u_d = torch.from_numpy(w["u"]).to(dev)
    v_d = torch.from_numpy(w["v"]).to(dev)
    x_local = torch.from_numpy(w["X"][part.lo:part.hi].copy()).to(dev)
    per = (u_d.shape[0] + world - 1) // world
    u_sl = u_d[rank * per: (rank + 1) * per].contiguous()      # this rank's slice of the undirected pair list
    v_sl = v_d[rank * per: (rank + 1) * per].contiguous()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # fixed init: rows perm[:K] of the propagated features (computed once on every rank, untimed)
    A0 = gdr.sym_normalize(gdr.coo_to_csr(u_d, v_d, None, (n, n), symmetrize=True, binarize=True), 2)
    _, tgt0 = gdr.propagate(A0, torch.from_numpy(w["X"]).to(dev), hops + 1, ALPHA)
    perm = torch.from_numpy(np.random.RandomState(seed).permutation(n)[:K].astype(np.int64)).to(dev)
    C0 = tgt0[perm].clone()
    nnz = A0.nnz
    parity = None
    if not args.no_parity:
        parity = multi_parity(gdr, par, comm, part, ops, dev, w, A0, tgt0, C0, u_sl, v_sl)
    del A0, tgt0, u_d, v_d
    torch.cuda.empty_cache()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def step():
        e = [ev() for _ in range(5)]
        e[0].record()
        # the feature rows start travelling to the peers' gathered operand (side stream, NVLink) under stage 1
        # (started right after stage 1's own all-to-all so that the two do not share the links)
        box = []
        hook = (lambda: box.append(par.prefetch_rows(comm, part, x_local, ops=ops))) \
            if args.hop in ("auto", "p2p") and not args.no_prefetch else None
        A_local = par.dist_build_adjacency(comm, part, u_sl, v_sl, n, ops=ops, after_exchange=hook)   # 1/world of the pairs per rank
        pre = box[0] if box else None
        e[1].record()
        prop, target = par.dist_propagate(comm, part, A_local, x_local, hops + 1, ALPHA, ops=ops, slabs=args.slabs,
                                          row_chunks=args.row_chunks, hop=args.hop, prefetched=pre)
        e[2].record()
        km = par.DistKMeans(K, C0, max_iter=LLOYD_ITERS, tol=0, ops=ops, comm=comm).fit(target)
        e[3].record()
        adj_syn, _ = par.dist_graph_compress(comm, part, km.labels_, A_local, ops=ops)
        e[4].record()
        return e, types.SimpleNamespace(n_iter_=km.n_iter_, inertia_=km.inertia_), int(adj_syn._nnz())

    t_warm = time.perf_counter()
    n_warm = 0
    while True:   # W warm-up steps, and at least 2 s of work on every rank (same count everywhere)
        go = torch.tensor([1 if (n_warm < args.warmup or time.perf_counter() - t_warm < 2.0) else 0], device=dev)
        dist.all_reduce(go, op=dist.ReduceOp.MAX)
        if int(go.item()) == 0:
            break
        step()
        flush.fill_(1)
        n_warm += 1
    torch.cuda.synchronize()
    dist.barrier()
    sampler = ClockSampler(dev.index)
    sampler.start()
    launches0 = gdr.launch_count()
    recs = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        dist.barrier()
        recs.append(step())
        sampler.sample_now()
    torch.cuda.synchronize()
    dist.barrier()
    t_wall = time.perf_counter() - t0
    launches = gdr.launch_count() - launches0
    clocks = sampler.stop()
    st = torch.tensor([[r[0][i].elapsed_time(r[0][i + 1]) for i in range(4)] for r in recs], dtype=torch.float64, device=dev)
    dist.all_reduce(st, op=dist.ReduceOp.MAX)     # device time, max over ranks, per step and stage
    st = st.cpu().numpy()
    lt = torch.tensor([launches], dtype=torch.int64, device=dev)
    dist.all_reduce(lt)
    n_iter = [r[1].n_iter_ for r in recs]

    # ---- roofline leg (per GPU): the E-step tensor-core screen of this rank's row block, timed by the
    #      library's own CUDA-event pairs on its launch stream ----
    A_local = par.dist_build_adjacency(comm, part, u_sl, v_sl, n, ops=ops)
    _, target_l = par.dist_propagate(comm, part, A_local, x_local, hops + 1, ALPHA, ops=ops, hop=args.hop)
    assign_ms, _ = _profile_kernel(
        _lib, 1, lambda: par.DistKMeans(K, C0, max_iter=LLOYD_ITERS, tol=0, ops=ops, comm=comm).fit(target_l), 1, flush)
    am = torch.tensor([assign_ms], dtype=torch.float64, device=dev)
    dist.all_reduce(am, op=dist.ReduceOp.MAX)
    assign_ms = float(am.item())
    # per-hop split: the SpMM of this rank's rows alone (library event pairs) beside the whole hop
    spmm_ms, n_sp = _profile_kernel(
        _lib, 2, lambda: par.dist_propagate(comm, part, A_local, x_local, hops + 1, ALPHA, ops=ops, slabs=args.slabs,
                                            row_chunks=args.row_chunks, hop=args.hop), 3, flush)
    sm = torch.tensor([spmm_ms * n_sp / 3.0 / hops], dtype=torch.float64, device=dev)   # SpMM kernel time per hop
    dist.all_reduce(sm, op=dist.ReduceOp.MAX)
    spmm_per_hop = float(sm.item())

    # ---- e2e: DistKMeans.fit through the public API from pinned HOST rows (H2D of this rank's block of the
    #      propagated features, D2H of its labels + the centres), max over ranks ----
    target_host = torch.empty(tuple(target_l.shape), dtype=torch.float32).pin_memory()
    target_host.copy_(target_l)
    del target_l, A_local
    C0_host = C0.cpu()
    e2e_t = []
    for i in range(max(4, min(args.steps, 8))):
        flush.fill_(1)
        torch.cuda.synchronize()
        dist.barrier()
        t0e = time.perf_counter()
        x_dev = target_host.to(dev, non_blocking=True)
        km = par.DistKMeans(K, C0_host, max_iter=LLOYD_ITERS, tol=0, ops=ops, comm=comm).fit(x_dev)
        km.labels_.cpu()
        km.cluster_centers_.cpu()
        torch.cuda.synchronize()
        tt = torch.tensor([time.perf_counter() - t0e], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_t.append((float(tt.item()), km.n_iter_))
    e2e_reps_ms = [round(t * 1e3, 3) for t, _ in e2e_t]
    e2e_t = e2e_t[1:]
    e2e_val = float(sum(k for _, k in e2e_t) / sum(t for t, _ in e2e_t))

    if rank == 0:
        step_ms = st.sum(axis=1)
        km_ms, prop_ms = st[:, 2], st[:, 1]
        flops_rank = 2.0 * part.rows_per * K * F
        a_tf = flops_rank / (assign_ms / 1e3) / 1e12
        roofline = {"kernel": "k_assign_tc two-level screen (per GPU, this rank's row block)", "bound": "tensor",
                    "achieved": a_tf, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": a_tf / pk["bf16_sustained"],
                    "traffic": None, "peak_source": pk["src"] + " bf16 sustained", "launch_ms": assign_ms,
                    "note": "useful flops 2*(N/world)*K*D per E-step over the slowest rank's screen time; fp32 inputs run as TF32"}
        e2e = {"value": e2e_val, "unit": "iters/s", "h2d_bytes_per_step": n * F * 4 + world * K * F * 4,
               "d2h_bytes_per_step": n * 4 + world * K * F * 4, "reps_ms": e2e_reps_ms}
        prop_model = "gather" if n * F * 4 > 96e6 else "min"   # SURVEY §8(d) headline rule
        b_prop = hops * spmm_bytes(nnz, n, n, F, model=prop_model) + 2 * n * F * 4
        prop_gbs = float(b_prop / (prop_ms.mean() / 1e3) / 1e9)
        iters_per_s = float(np.sum(n_iter) / (km_ms.sum() / 1e3))
        line = {
            "metric": "kmeans_iters_per_s", "value": iters_per_s, "unit": "iters/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(step_ms.mean()), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.workload, w), "nnz_a_hat": int(nnz),
                       "parallelism": f"row-partition x{world}: " + par.describe(world, args.row_chunks, args.hop),
                       "precision": args.precision, "l2": "flushed between timed steps (256 MB write)"},
            "prop": {"metric": "A^K.X", "value": prop_gbs, "unit": "GB/s", "frac_hbm_measured": prop_gbs / (pk["hbm"] * world),
                     "bytes_model": ("B_gather" if prop_model == "gather" else "B_min") + " (whole job, incl. the all-gather time)",
                     "ms": float(prop_ms.mean()), "ms_per_hop": float(prop_ms.mean() / hops),
                     "spmm_kernel_ms_per_hop": spmm_per_hop,
                     "exposed_gather_ms_per_hop": float(max(0.0, prop_ms.mean() / hops - spmm_per_hop))},
            "stages_ms": {"s1_build_normalize": float(st[:, 0].mean()), "s2_propagate": float(prop_ms.mean()),
                          "s3_kmeans": float(km_ms.mean()), "s3_kmeans_per_iter": float(km_ms.sum() / np.sum(n_iter)),
                          "s4_coarsen": float(st[:, 3].mean())},
            "roofline": roofline, "parity": parity, "cpu_baseline": None, "same_workload_1gpu": one_gpu_reference(args.workload),
            "e2e": e2e, "gpu_launches": int(lt.item()), "clocks": clocks, "wall_s": t_wall,
            "result": {"inertia": recs[-1][1].inertia_, "n_iter": int(n_iter[-1]), "syn_nnz": int(recs[-1][2])},
        }
        print(json.dumps(line))
    dist.barrier()
    comm.close()
    dist.destroy_process_group()


def run_ours_multi_bipartite(args, rank, world, dev, w):
    """Configs C / D on N GPUs: users and items each split N ways (SURVEY §8e).  Stage 1: two all-to-alls of the
    interaction lines (by owner of u / of i) + all-gather of the degree vectors; stage 2: all-gather of the user and item
    rows per LightGCN layer; stage 3: DistKMeans per side on the z-scored rows (column statistics all-reduced); stage 4:
    all-gather of the cluster maps, local line counting, key-range exchange merge."""
    import torch
    import torch.distributed as dist
    import gdr
    from gdr import parallel as par
    dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    nu, ni, d, L, ku, ki, seed = w["users"], w["items"], w["d"], w["layers"], w["ku"], w["ki"], w["seed"]
    pu, pi = par.RowPartition(nu, world, rank), par.RowPartition(ni, world, rank)
    comm = par.Comm(dist)
    ops = par.CudaOps(precision=args.precision)
    per = (w["u"].shape[0] + world - 1) // world
    u_sl = torch.from_numpy(w["u"][rank * per:(rank + 1) * per].copy()).to(dev)
    i_sl = torch.from_numpy(w["i"][rank * per:(rank + 1) * per].copy()).to(dev)
    u0_l = torch.from_numpy(w["u0"][pu.lo:pu.hi].copy()).to(dev)
    i0_l = torch.from_numpy(w["i0"][pi.lo:pi.hi].copy()).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    # fixed init per side (replicated): rows perm[:K] of the z-scored embeddings, computed on every rank
    C0 = []
    u_d, i_d = torch.from_numpy(w["u"]).to(dev), torch.from_numpy(w["i"]).to(dev)
    u0, i0 = torch.from_numpy(w["u0"]).to(dev), torch.from_numpy(w["i0"]).to(dev)
    Xs_full = []
    for emb, K in ((u0, ku), (i0, ki)):
        Xs = gdr.standard_scale(emb)
        perm = torch.from_numpy(np.random.RandomState(seed).permutation(emb.shape[0])[:K].astype(np.int64)).to(dev)
        C0.append(Xs[perm].clone())
        Xs_full.append(Xs)

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def step(keep=False):
        e = [ev() for _ in range(5)]
        e[0].record()
        R_l, RT_l = par.dist_build_interaction(comm, pu, pi, u_sl, i_sl, ops=ops)
        A_l, AT_l, _, _ = par.dist_bipartite_normalize(comm, pu, pi, R_l, RT_l, ops=ops)
        e[1].record()
        uo, io = par.dist_lightgcn_propagate(comm, pu, pi, A_l, AT_l, u0_l, i0_l, L, ops=ops)
        e[2].record()
        its, maps, inertia = 0, [], 0.0
        for emb_l, K, c0 in ((u0_l, ku, C0[0]), (i0_l, ki, C0[1])):
            km = par.DistKMeans(K, c0, max_iter=LLOYD_ITERS, tol=0, ops=ops, comm=comm).fit(par.dist_standard_scale(comm, emb_l, ops=ops))
            its += km.n_iter_
            inertia += km.inertia_
            maps.append(km.labels_)
        e[3].record()
        rpc, cic, vc = par.dist_build_condensed_bipartite(comm, pu, pi, u_sl, i_sl, maps[0], maps[1], ku, ki, ops=ops)
        e[4].record()
        out = (e, types.SimpleNamespace(n_iter_=its / 2.0, inertia_=inertia), int(cic.shape[0]))
        return out + ((A_l, uo, io, maps, rpc, cic, vc),) if keep else out

    # ---- parity (outside the timed region): this rank's blocks against the single-GPU path on this GPU ----
    parity = None
    if not args.no_parity:
        R = gdr.coo_to_csr(u_d, i_d, None, (nu, ni))
        graph = gdr.BipartiteGraph(R.coo_indices(), R.vals, nu, ni)
        uo1, io1 = gdr.lightgcn_propagate(graph, u0, i0, L)
        rec = step(keep=True)[3]
        A_l, uo, io, maps, rpc, cic, vc = rec
        A_rows = par.slice_rows(graph.A, pu.lo, pu.hi)
        flags = {
            "interaction_block_equal": bool(torch.equal(A_l.rowptr, A_rows.rowptr) and torch.equal(A_l.colidx, A_rows.colidx)
                                            and torch.equal(A_l.vals, A_rows.vals)),
            "lightgcn_rows_equal": bool(torch.equal(uo, uo1[pu.lo:pu.hi]) and torch.equal(io, io1[pi.lo:pi.hi])),
        }
        lab_ok, cen_ok, maps1 = True, True, []
        for Xs, part, K, c0 in ((Xs_full[0], pu, ku, C0[0]), (Xs_full[1], pi, ki, C0[1])):
            km0 = par.DistKMeans(K, c0, max_iter=0, tol=0, ops=ops, comm=comm).fit(Xs[part.lo:part.hi].contiguous())
            ref0 = gdr.KMeans(n_clusters=K, init=c0, n_init=1, max_iter=0, tol=0).fit(Xs)
            lab_ok &= bool(torch.equal(km0.labels_, ref0.labels_[part.lo:part.hi]))
            km1 = par.DistKMeans(K, c0, max_iter=1, tol=0, ops=ops, comm=comm).fit(Xs[part.lo:part.hi].contiguous())
            ref1 = gdr.KMeans(n_clusters=K, init=c0, n_init=1, max_iter=1, tol=0).fit(Xs)
            cen_ok &= bool(((km1.cluster_centers_ - ref1.cluster_centers_).abs().max() / ref1.cluster_centers_.abs().max()).item() <= 1e-5)
            maps1.append(ref1.labels_)
        flags["labels_equal"], flags["centres_close"] = lab_ok, cen_ok
        C1 = gdr.build_condensed_bipartite(u_d, i_d, maps1[0], maps1[1], ku, ki, device=dev, return_device=True)
        rp2, ci2, v2 = par.dist_build_condensed_bipartite(comm, pu, pi, u_sl, i_sl, maps1[0][pu.lo:pu.hi].contiguous(),
                                                          maps1[1][pi.lo:pi.hi].contiguous(), ku, ki, ops=ops)
        flags["counts_equal"] = bool(torch.equal(rp2, C1.rowptr) and torch.equal(ci2, C1.colidx) and torch.equal(v2, C1.vals)
                                     and int(v2.sum().item()) == w["u"].shape[0])
        t = torch.tensor([1 if v else 0 for v in flags.values()], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        parity = {k: bool(v) for k, v in zip(flags, t.tolist())}
        parity["status"] = "ok" if all(parity.values()) else "MISMATCH"
        parity["what"] = "each rank's blocks vs the single-GPU path (MIN over ranks); single Lloyd step per side from shared centres"
        del R, graph, uo1, io1, rec
    del u_d, i_d

    t_warm, n_warm = time.perf_counter(), 0
    while True:
        go = torch.tensor([1 if (n_warm < args.warmup or time.perf_counter() - t_warm < 2.0) else 0], device=dev)
        dist.all_reduce(go, op=dist.ReduceOp.MAX)
        if int(go.item()) == 0:
            break
        step()
        flush.fill_(1)
        n_warm += 1
    torch.cuda.synchronize()
    dist.barrier()
    sampler = ClockSampler(dev.index)
    sampler.start()
    launches0 = gdr.launch_count()
    recs = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        dist.barrier()
        recs.append(step())
        sampler.sample_now()
    torch.cuda.synchronize()
    dist.barrier()
    t_wall = time.perf_counter() - t0
    launches = gdr.launch_count() - launches0
    clocks = sampler.stop()
    st = torch.tensor([[r[0][i].elapsed_time(r[0][i + 1]) for i in range(4)] for r in recs], dtype=torch.float64, device=dev)
    dist.all_reduce(st, op=dist.ReduceOp.MAX)
    st = st.cpu().numpy()
    lt = torch.tensor([launches], dtype=torch.int64, device=dev)
    dist.all_reduce(lt)
    n_iter = [r[1].n_iter_ for r in recs]
    # e2e: both sides' DistKMeans from pinned HOST rows of this rank's blocks
    u0_pin, i0_pin = torch.from_numpy(w["u0"][pu.lo:pu.hi].copy()).pin_memory(), torch.from_numpy(w["i0"][pi.lo:pi.hi].copy()).pin_memory()
    c0_host = [c.cpu() for c in C0]
    e2e_t = []
    for _ in range(max(3, min(args.steps, 5))):
        flush.fill_(1)
        torch.cuda.synchronize()
        dist.barrier()
        t0e = time.perf_counter()
        its = 0
        for pin, K, c0 in ((u0_pin, ku, c0_host[0]), (i0_pin, ki, c0_host[1])):
            km = par.DistKMeans(K, c0, max_iter=LLOYD_ITERS, tol=0, ops=ops, comm=comm).fit(
                par.dist_standard_scale(comm, pin.to(dev, non_blocking=True), ops=ops))
            km.labels_.cpu()
            km.cluster_centers_.cpu()
            its += km.n_iter_
        torch.cuda.synchronize()
        tt = torch.tensor([time.perf_counter() - t0e], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_t.append((float(tt.item()), its / 2.0))
    e2e_t = e2e_t[1:]
    if rank == 0:
        line = {
            "metric": "kmeans_iters_per_s", "value": float(np.sum(n_iter) / (st[:, 2].sum() / 1e3)), "unit": "iters/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(st.sum(axis=1).mean()),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.workload, w),
                       "iteration": "one Lloyd iteration over BOTH sides (users + items)",
                       "parallelism": f"users and items each row-partitioned x{world}: all-to-all of the interaction lines by owner, "
                                      "all-gather of degrees / embedding rows / cluster maps, packed all-reduce per Lloyd iteration, "
                                      "key-range exchange of the condensed counts",
                       "precision": args.precision, "l2": "flushed between timed steps (256 MB write)"},
            "stages_ms": {"s1_build_normalize": float(st[:, 0].mean()), "s2_propagate": float(st[:, 1].mean()),
                          "s3_kmeans": float(st[:, 2].mean()), "s3_kmeans_per_iter": float(st[:, 2].sum() / np.sum(n_iter)),
                          "s4_coarsen": float(st[:, 3].mean())},
            "roofline": None, "parity": parity, "cpu_baseline": None,
            "e2e": {"value": float(sum(k for _, k in e2e_t) / sum(t for t, _ in e2e_t)), "unit": "iters/s",
                    "h2d_bytes_per_step": (nu + ni) * d * 4 + world * (ku + ki) * d * 4,
                    "d2h_bytes_per_step": (nu + ni) * 4 + world * (ku + ki) * d * 4},
            "gpu_launches": int(lt.item()), "clocks": clocks, "wall_s": t_wall,
            "result": {"inertia": recs[-1][1].inertia_, "n_iter": float(n_iter[-1]), "condensed_nnz": int(recs[-1][2])},
        }
        print(json.dumps(line))
    dist.barrier()
    comm.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=["A", "B", "C", "D", "E"])
    ap.add_argument("--precision", default="tc", choices=["fp32", "tc", "auto"])
    ap.add_argument("--slabs", type=int, default=None, help="N > 1: column slabs of the pipelined hop (default: automatic)")
    ap.add_argument("--row-chunks", type=int, default=None, help="N > 1: row chunks of the pipelined hop (default: automatic)")
    ap.add_argument("--hop", default="auto", choices=["auto", "p2p", "nccl"],
                    help="N > 1: fused NVLink hop (SpMM epilogue stores into the peers' gathered operand) or NCCL all-gather hop")
    ap.add_argument("--no-prefetch", action="store_true", help="N > 1: do not start the first row distribution under stage 1")
    ap.add_argument("--tc-screen", type=int, default=0, help="debug: 0 auto, 1 direct 3xTF32, 2/3 two-level screen (BN 128/256)")
    ap.add_argument("--ref-kmeans-iters", type=int, default=10)
    ap.add_argument("--ref-full-budget", type=float, default=420.0,
                    help="reference arm, config E: seconds the once-per-run full-size legs may take (0 = skip them)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-legs", action="store_true", help="skip the logit-space and skewed-graph legs")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the parity record")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: no CPU baseline, minimal e2e leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU: write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, "
                         "large outputs as a fixed sample of rows, at most 64 MB in all)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs writes the outputs of the one-GPU path (--impl ours, one process)")
    if args.workload is None:
        # ONE workload for every N, so that the per-N lines are one strong-scaling experiment: config E
        # (configs[4], ogbn-products-shaped), the shape BASELINE.json's target is quoted on; it fits one GPU
        # (~6 GB resident).  `--workload B` is configs[1] (ogbn-arxiv-shaped), the shape of most parity tests.
        args.workload = "E"
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
