#!/usr/bin/env python
"""E-step alone at a BASELINE shape: direct 3xTF32 (tc_screen 1) vs the two-level screen (tc_screen 3).
Run on the GPU box:  python tools/estep_probe.py [B|E]"""
import ctypes, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gdr
from gdr import synth, _lib
from gdr._dev import padded_rows
from gdr.kmeans import TcOperand, assign_labels, segment_sum

dev = torch.device("cuda:0")
name = sys.argv[1] if len(sys.argv) > 1 else "B"
cfg = synth.CONFIGS[name]
n, f, K = cfg["n"], cfg["f"], cfg["k"]
if name == "E":   # the E-step does not care where X came from: skip the graph at this size
    Xc = torch.from_numpy(synth.features(n, f, 1338)).to(dev)
else:
    u, v = synth.uniform_graph(n, cfg["pairs"], 1235)
    A = gdr.sym_normalize(gdr.coo_to_csr(torch.from_numpy(u).to(dev), torch.from_numpy(v).to(dev), None, (n, n), symmetrize=True, binarize=True), 2)
    X = torch.from_numpy(synth.features(n, f, 1335)).to(dev)
    _, Xc = gdr.propagate(A, X, cfg["hops"] + 1, 0.8)
Xc = padded_rows((Xc - Xc.mean(0)).contiguous())
perm = torch.from_numpy(np.random.RandomState(1235).permutation(n)[:K].astype(np.int64)).to(dev)
C = padded_rows(Xc[perm].clone())
op = TcOperand(Xc)
ws = torch.empty(_lib.query("gdr_kmeans_assign_tc_ws_bytes", n, K, f), dtype=torch.uint8, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
MODES = (1, 3)
for it in range(int(os.environ.get("PROBE_ITERS", "4"))):
    res = {}
    for mode in MODES:
        _lib.call("gdr_debug_set", b"tc_screen", mode)
        lab = torch.empty(n, dtype=torch.int32, device=dev)
        nref = torch.zeros(1, dtype=torch.int32, device=dev)
        ts = []
        for rep in range(4):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            assign_labels(Xc, C, lab, tc_operand=op, n_refined=nref, ws=ws)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        lvl2 = ctypes.c_int64(-1)
        if mode > 1:
            _lib.call("gdr_debug_get", b"tc_level2_rows", ctypes.addressof(lvl2))
        res[mode] = (min(ts[1:]), lvl2.value, int(nref.item()), lab.clone())
    same = all(torch.equal(res[MODES[0]][3], res[m][3]) for m in MODES)
    print(f"iter {it}: " + "  ".join(f"mode{m}: {res[m][0]*1e3:.0f} us (level2 {res[m][1]}, exact {res[m][2]})" for m in MODES) + f"  labels equal: {same}", flush=True)
    sums, counts = segment_sum(Xc, res[MODES[0]][3], K)
    C = padded_rows((sums / counts.clamp_min(1).unsqueeze(1)).contiguous())
_lib.call("gdr_debug_set", b"tc_screen", 0)
