"""Time full-ranking top-K of a condensed model from its cluster tables (gdr.recommend_topk_condensed) against
gdr.recommend_topk on the expanded tables user_emb[u2cu], item_emb[i2ci] (the only way to rank it before).

Workloads: the condensed models at the Yelp2018 (C) and Amazon-book (D) shapes of tests/test_gpu_topk_condensed.py
(bench.py's seeds and synthetic interactions, gdr.kmeans_cluster maps at a 10 % rate, tables from a seeded
LightGCNPropagate forward, d = 64), k = 20, the training CSR excluded.  Arms, in one process, alternated
until each has >= 1 s of calls, median per arm, whole calls (the status read included):
  condensed        recommend_topk_condensed(U, I, 20, u2cu, i2ci, exclude=R)
  expanded_auto    recommend_topk(U[u2cu], I[i2ci], 20, exclude=R), automatic path (tables expanded outside the timing)
  expanded_exact   the same with gdr_debug_set("topk_path", 1)
  expanded_screen  the same with gdr_debug_set("topk_path", 2)
  entry_point      gdr_topk_condensed alone on preallocated outputs and workspace, CUDA events around it
Also printed: the screen's overflow rows on the expanded inputs, the condensed call's fallback rows, flops and score
bytes from shapes, and the card's name and power limit read in the same run.  Outputs of every arm are compared.

Usage: python tools/topk_condensed_bench.py [C] [D]
"""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gdr  # noqa: E402
from gdr import _lib  # noqa: E402
from gdr._dev import ptr, stream  # noqa: E402
from test_gpu_topk_condensed import condensed_workload  # noqa: E402

K = 20


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = out.stdout.strip().splitlines()[torch.cuda.current_device()] if out.returncode == 0 else ""
    vals = [v.strip() for v in line.split(",")] if line else []
    return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"nvidia_smi": "unavailable"}


def debug_get(key):
    v = ctypes.c_int64(0)
    _lib.call("gdr_debug_get", key, ctypes.addressof(v))
    return v.value


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), out


def main():
    assert torch.cuda.is_available(), "topk_condensed_bench needs a GPU"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = card()
    for name in sys.argv[1:] or ["C", "D"]:
        Ucl, Icl, u2cu, i2ci, R = condensed_workload(gdr, name, dev)
        Ucl, Icl = Ucl.contiguous(), Icl.contiguous()
        um, im = torch.from_numpy(u2cu).to(dev), torch.from_numpy(i2ci).to(dev)
        Ue, Ie = Ucl[um].contiguous(), Icl[im].contiguous()
        n_users, n_items, n_cu, n_ci, d = len(u2cu), len(i2ci), Ucl.shape[0], Icl.shape[0], Ucl.shape[1]

        def expanded(path):
            def run():
                _lib.call("gdr_debug_set", b"topk_path", path)
                try:
                    return gdr.recommend_topk(Ue, Ie, K, exclude=R)
                finally:
                    _lib.call("gdr_debug_set", b"topk_path", 0)
            return run

        # the entry point alone
        scores = torch.empty((n_users, K), dtype=torch.float32, device=dev)
        items = torch.empty((n_users, K), dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        wsb = _lib.query("gdr_topk_condensed_ws_bytes", n_users, n_users, n_items, n_cu, n_ci, d, K)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        args = (n_users, n_users, n_items, n_cu, n_ci, d, K, ptr(Ucl), Ucl.stride(0), ptr(Icl), Icl.stride(0), ptr(um),
                ptr(im), 0, ptr(R.rowptr), ptr(R.colidx), ptr(scores), K, ptr(items), K, ptr(status), ptr(ws), wsb,
                stream())

        arms = {
            "condensed": lambda: gdr.recommend_topk_condensed(Ucl, Icl, K, um, im, exclude=R),
            "expanded_auto": expanded(0),
            "expanded_exact": expanded(1),
            "expanded_screen": expanded(2),
            "entry_point": lambda: _lib.call("gdr_topk_condensed", *args),
        }
        outs = {a: fn() for a, fn in arms.items()}   # warm-up, and the outputs compared below
        counts = {"condensed_fallback_rows": None, "screen_overflow_rows": None}
        arms["condensed"]()
        counts["condensed_fallback_rows"] = debug_get(b"topk_condensed_fallback_rows")
        arms["expanded_screen"]()
        counts["screen_overflow_rows"] = debug_get(b"topk_overflow_rows")
        ref = outs["condensed"]
        same = {a: bool(torch.equal(o[1], ref[1]) and torch.equal(o[0].view(torch.int32), ref[0].view(torch.int32)))
                for a, o in outs.items() if a.startswith("expanded")}
        same["entry_point"] = bool(torch.equal(items.long(), ref[1]) and torch.equal(scores.view(torch.int32),
                                                                                     ref[0].view(torch.int32)))
        assert int(status.item()) == 0
        times = {a: [] for a in arms}
        while min(sum(t) for t in times.values()) < 1000.0:
            for a, fn in arms.items():   # alternated; an arm stops once it has 1 s of calls
                if sum(times[a]) < 1000.0:
                    times[a].append(timed(fn)[0])
        med = {a: round(float(np.median(t)), 3) for a, t in times.items()}
        n_g = int(np.unique(u2cu).shape[0])
        print(json.dumps({
            "workload": {"C": "yelp2018 condensed", "D": "amazon-book condensed"}[name],
            "n_users": n_users, "n_items": n_items, "n_cu": n_cu, "n_ci": n_ci, "used_super_users": n_g, "d": d, "k": K,
            "excluded": int(R.nnz), "ms": med, "speedup_vs_expanded_auto": round(med["expanded_auto"] / med["condensed"], 2),
            "calls": {a: len(t) for a, t in times.items()}, "identical_to_condensed": same, **counts,
            "multiply_adds": {"condensed": n_g * n_ci * d, "expanded": n_users * n_items * d},
            "score_table_bytes": {"condensed": n_g * n_ci * 4, "expanded_if_held": n_users * n_items * 4},
            "workspace_bytes": wsb, "card": info}), flush=True)


if __name__ == "__main__":
    main()
