"""Time gdr.recommend_topk against the torch full-ranking baseline at the Yelp2018 (C) and Amazon-book (D) shapes.

Inputs as bench.py builds them (bench seeds, d = 64, training interactions excluded), embeddings N(0, 0.1^2)
z-scored per column; k = 20.  Arms, alternated, each timed with CUDA events after one warm-up call, over >= 1 s:
  gdr_tc     gdr.recommend_topk forced onto the 3xTF32 tensor-core screen (exact finish of its candidates)
  gdr_exact  gdr.recommend_topk forced onto the exact SIMT path (score slabs + radix top-k per row)
  torch      user blocks of 4096: fp32 mm (TF32 off) + masked_fill of the training items + torch.topk
Each time is one whole call as a user makes it: the gdr arms include the workspace allocation (from torch's caching
allocator), the status read-back and, on the tensor-core path, its one read of the overflow count; the torch arm
includes the per-block index slicing (the COO indices and row pointers are prepared once, outside the timing).
"ms" is the total time of all timed calls of an arm over their number.
The embeddings (37 MB at D) fit the 126 MB L2; the score slabs of either arm (hundreds of MB) do not.
Prints one JSON line per (shape, arm): ms per call, useful TFLOP/s (2 n_users n_items d over the time) and its share of
the data-sheet dense TF32 rate of one B200 (1125 TFLOP/s), with the card name, power limit and SM clock read in the
same run.  Also checks that every gdr call returned identical bytes and that the two arms pick the same top-k sets
for the users whose k-th and (k+1)-th exact scores are apart by more than 2^-15 |u| max|i|.
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

import gdr  # noqa: E402
from gdr import synth  # noqa: E402

DATASHEET_TF32 = 1125.0   # TFLOP/s, dense TF32, one B200 (NVIDIA HGX B200 data sheet / 8)
K = 20
BLOCK = 4096


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = out.stdout.strip().splitlines()[torch.cuda.current_device()] if out.returncode == 0 else ""
    vals = [v.strip() for v in line.split(",")] if line else []
    return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"nvidia_smi": "unavailable"}


def inputs(name, dev):
    cfg = synth.BIPARTITE[name]
    seed = 1234 + {"C": 2, "D": 3}[name]
    u, i = synth.bipartite_interactions(cfg["users"], cfg["items"], cfg["inter"], seed)
    rs = np.random.RandomState(seed + 100)
    z = lambda x: ((x - x.mean(0)) / x.std(0)).astype(np.float32)
    U = torch.from_numpy(z(0.1 * rs.standard_normal((cfg["users"], 64)))).to(dev)
    I = torch.from_numpy(z(0.1 * rs.standard_normal((cfg["items"], 64)))).to(dev)
    R = gdr.coo_to_csr(u, i, None, (cfg["users"], cfg["items"]), device=dev)
    return U, I, R


def torch_topk(U, I, rows, cols, rp, k):
    out_s, out_i = [], []
    for b0 in range(0, U.shape[0], BLOCK):
        b1 = min(b0 + BLOCK, U.shape[0])
        S = U[b0:b1] @ I.T
        e0, e1 = int(rp[b0]), int(rp[b1])
        S[rows[e0:e1] - b0, cols[e0:e1]] = -float("inf")
        s, i = torch.topk(S, k, dim=1)
        out_s.append(s)
        out_i.append(i)
    return torch.cat(out_s), torch.cat(out_i)


def timed(fn, min_s=1.0):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    out = fn()
    ev1.record()
    ev1.synchronize()
    return out, ev0.elapsed_time(ev1)


def main():
    assert torch.cuda.is_available(), "topk_bench needs a GPU"
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    info = card()
    for name in ("C", "D"):
        U, I, R = inputs(name, dev)
        flops = 2.0 * U.shape[0] * I.shape[0] * U.shape[1]
        rows, cols = R.coo_indices()
        rp = R.rowptr.long().cpu()

        def forced(path):
            def run():
                gdr._lib.call("gdr_debug_set", b"topk_path", path)
                try:
                    return gdr.recommend_topk(U, I, K, exclude=R)
                finally:
                    gdr._lib.call("gdr_debug_set", b"topk_path", 0)
            return run

        arms = {"gdr_tc": forced(2), "gdr_exact": forced(1), "torch": lambda: torch_topk(U, I, rows, cols, rp, K)}
        ref = {}
        overflow = {}
        for a, fn in arms.items():   # warm-up (module load, cuBLAS algorithm choice)
            ref[a] = fn()
            if a == "gdr_tc":
                v = ctypes.c_int64(0)
                gdr._lib.call("gdr_debug_get", b"topk_overflow_rows", ctypes.addressof(v))
                overflow[a] = v.value
        assert torch.equal(ref["gdr_tc"][0], ref["gdr_exact"][0]) and torch.equal(ref["gdr_tc"][1], ref["gdr_exact"][1]), \
            "tensor-core and exact paths differ"
        times = {a: [] for a in arms}
        while min(sum(t) for t in times.values()) < 1000.0:
            for a, fn in arms.items():
                out, ms = timed(fn)
                times[a].append(ms)
                if a != "torch":
                    assert torch.equal(out[0], ref[a][0]) and torch.equal(out[1], ref[a][1]), f"{a} run differs"
        # set agreement outside the rounding band
        s1, i1 = gdr.recommend_topk(U, I, K + 1, exclude=R)
        band = 2.0 ** -15 * U.norm(dim=1) * I.norm(dim=1).max()
        clear = (s1[:, K - 1] - s1[:, K]) > band
        same = torch.equal(torch.sort(i1[:, :K], 1).values[clear], torch.sort(ref["torch"][1], 1).values[clear])
        for a, t in times.items():
            ms = float(sum(t) / len(t))
            print(json.dumps({"shape": name, "arm": a, "users": U.shape[0], "items": I.shape[0], "d": U.shape[1],
                              "k": K, "ms": round(ms, 3), "calls": len(t), "useful_tflops": round(flops / ms / 1e9, 2),
                              "share_of_datasheet_tf32_1125": round(flops / ms / 1e9 / DATASHEET_TF32, 4),
                              "overflow_rows": overflow.get(a), "sets_agree_outside_band": bool(same),
                              "rows_outside_band": int(clear.sum()),
                              "card": info}), flush=True)


if __name__ == "__main__":
    main()
