#!/usr/bin/env python
"""E-step of the two-level tensor-core screen with the second level on candidate centres (tc_cand 1) or over all
centres (tc_cand 0), at a BASELINE shape: whole E-step by CUDA events (L2 flushed before each), per-kernel times from
torch.profiler (a separate pass), and the row counts of each level.  Run on the GPU box:
    python tools/cand_probe.py [E|B] [reps]"""
import ctypes, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gdr  # noqa: F401
from gdr import synth, _lib
from gdr._dev import padded_rows
from gdr.kmeans import TcOperand, assign_labels, segment_sum

dev = torch.device("cuda:0")
name = sys.argv[1] if len(sys.argv) > 1 else "E"
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
cfg = synth.CONFIGS[name]
n, f, K = cfg["n"], cfg["f"], cfg["k"]
# the data of tests/test_gpu_tc.py::test_tc_full_size_labels_equal_exact_kernel: unclustered z-scored rows, centres
# after one Lloyd update from random rows
X = torch.from_numpy(synth.features(n, f, seed=17)).to(dev)
X = padded_rows((X - X.mean(0)).contiguous())
C = padded_rows(X[torch.from_numpy(np.random.RandomState(3).permutation(n)[:K].astype(np.int64)).to(dev)].clone())
op = TcOperand(X)
lab0 = torch.empty(n, dtype=torch.int32, device=dev)
assign_labels(X, C, lab0, tc_operand=op)
sums, counts = segment_sum(X, lab0, K)
C = padded_rows((sums / counts.clamp_min(1).unsqueeze(1)).contiguous())
ws = torch.empty(_lib.query("gdr_kmeans_assign_tc_ws_bytes", n, K, f), dtype=torch.uint8, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
print(f"{torch.cuda.get_device_name(0)}  config {name}: N={n} D={f} K={K}", flush=True)


def get(key):
    v = ctypes.c_int64(-1)
    _lib.call("gdr_debug_get", key.encode(), ctypes.addressof(v))
    return int(v.value)


def run(lab, nref, nch):
    nref.zero_(); nch.zero_()
    assign_labels(X, C, lab, labels_prev=lab0, n_changed=nch, tc_operand=op, n_refined=nref, ws=ws)


res = {}
for it in range(2):            # two alternations of the arms
    for cand in (0, 1):
        _lib.call("gdr_debug_set", b"tc_cand", cand)
        lab = torch.empty(n, dtype=torch.int32, device=dev)
        nref = torch.zeros(1, dtype=torch.int32, device=dev)
        nch = torch.zeros(1, dtype=torch.int32, device=dev)
        ts = []
        for r in range(reps + 1):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); run(lab, nref, nch); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts = sorted(ts[1:])
        res.setdefault(cand, []).extend(ts)
        cnt = dict(level2=get("tc_level2_rows"), n_refined=int(nref.item()), n_changed=int(nch.item()))
        if cand:
            cnt.update(cand_rows=get("tc_cand_rows"), overflow=get("tc_cand_overflow_rows"), entries=get("tc_cand_entries"))
        print(f"pass {it} tc_cand {cand}: E-step median {ts[len(ts)//2]*1e3:.0f} us (min {ts[0]*1e3:.0f}, max {ts[-1]*1e3:.0f})  {cnt}",
              flush=True)
        res.setdefault(f"lab{cand}", lab.clone())
print("labels equal:", torch.equal(res["lab0"], res["lab1"]), flush=True)

# per-kernel times (separate pass: the profiler slows the host)
from torch.profiler import profile, ProfilerActivity
for cand in (0, 1):
    _lib.call("gdr_debug_set", b"tc_cand", cand)
    lab = torch.empty(n, dtype=torch.int32, device=dev)
    nref = torch.zeros(1, dtype=torch.int32, device=dev)
    nch = torch.zeros(1, dtype=torch.int32, device=dev)
    run(lab, nref, nch); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for r in range(reps):
            flush.fill_(1)
            run(lab, nref, nch)
        torch.cuda.synchronize()
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        if t > 0 and "fill" not in e.key and "elementwise" not in e.key.lower():
            rows.append((t / reps, e.count / reps, e.key))
    print(f"tc_cand {cand}: per-kernel time per E-step (us, torch.profiler)  total {sum(r[0] for r in rows):.0f}")
    for t, c, k_ in sorted(rows, reverse=True):
        print(f"  {t:9.1f}  x{c:.0f}  {k_[:110]}")
_lib.call("gdr_debug_set", b"tc_cand", 1)
