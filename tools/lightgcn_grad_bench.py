"""Time one refinement step of the condensed LightGCN through gdr.LightGCNPropagate against the reference expression
under torch autograd, both on the GPU.

Step = propagate (L = 2, d = 64) + BPR loss over 2 048 fixed triplets + backward to the user / item embeddings and the
edge weights (w = softplus(raw), the gradient flows to raw); no optimiser.  Arms, alternated, each timed with CUDA
events per step after 3 warm-up steps, until each has >= 1 s of steps:
  gdr    graph built once (outside the timing); LightGCNPropagate.apply(u, i, w, graph, L) per step
  torch  oracle/ref_port.lightgcn_propagate (index_add_ degrees, edge norm, index_add_ layers) under autograd
Workloads: the condensed graphs at the Yelp2018 (C) and Amazon-book (D) shapes (bench seeds, synth interactions,
N(0, 0.1^2) embeddings, gdr.kmeans_cluster at 10 %, build_condensed_bipartite), and the full Yelp2018-shaped
interaction graph for callers that train a full LightGCN.  "grad_err" = max |gdr - fp64| / max |fp64| of d u0, d i0 and
d w on one backward, against torch fp64 autograd of the same expression.  The kernel leg times gdr_lightgcn_edge_grad
alone with CUDA events (100 launches) against its gathered bytes E * 2L * d * 4; these operands fit the 126 MB L2,
which is also the regime of a real refinement loop, so the figure is an L2 rate, not an HBM one.
Prints one JSON line per workload with the card name and power limit read in the same run.
"""
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
from gdr import _lib, synth  # noqa: E402
from gdr._dev import pad4, ptr, stream  # noqa: E402
from oracle import ref_port as rp  # noqa: E402
from test_lightgcn_grad_cpu import ref_autograd_f64  # noqa: E402

D, L, N_TRIPLETS = 64, 2, 2048


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = out.stdout.strip().splitlines()[torch.cuda.current_device()] if out.returncode == 0 else ""
    vals = [v.strip() for v in line.split(",")] if line else []
    return dict(zip(q.split(","), vals)) if len(vals) == 4 else {"nvidia_smi": "unavailable"}


def workload(name, dev):
    cfg = synth.BIPARTITE["C" if name in ("C", "C_full") else "D"]
    seed = 1234 + (3 if name == "D" else 2)
    U, I = cfg["users"], cfg["items"]
    u, i = synth.bipartite_interactions(U, I, cfg["inter"], seed)
    if name == "C_full":
        R = gdr.coo_to_csr(u, i, None, (U, I), device=dev)
        ei, ew = gdr.condensed_csr_to_edge_index(R, dev)
        return ei, ew, U, I
    rs = np.random.RandomState(seed + 100)
    emb_u = (rs.standard_normal((U, D)) * 0.1).astype(np.float32)
    emb_i = (rs.standard_normal((I, D)) * 0.1).astype(np.float32)
    ncu, nci = int(np.ceil(U * 0.1)), int(np.ceil(I * 0.1))
    u2cu, _ = gdr.kmeans_cluster(emb_u, ncu, seed=42, init="random", device=dev)
    i2ci, _ = gdr.kmeans_cluster(emb_i, nci, seed=42, init="random", device=dev)
    C = gdr.build_condensed_bipartite(u, i, u2cu, i2ci, ncu, nci, device=dev, return_device=True)
    ei, ew = gdr.condensed_csr_to_edge_index(C, dev)
    return ei, ew, ncu, nci


def main():
    assert torch.cuda.is_available(), "lightgcn_grad_bench needs a GPU"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = card()
    for name in ("C", "D", "C_full"):
        ei, ew, nu, ni = workload(name, dev)
        E = int(ei.shape[1])
        rs = np.random.RandomState(7)
        u0 = torch.from_numpy((rs.standard_normal((nu, D)) * 0.1).astype(np.float32)).to(dev).requires_grad_(True)
        i0 = torch.from_numpy((rs.standard_normal((ni, D)) * 0.1).astype(np.float32)).to(dev).requires_grad_(True)
        raw = torch.log(torch.expm1(ew.clamp_min(0.05))).requires_grad_(True)
        tu = torch.from_numpy(rs.randint(0, nu, N_TRIPLETS)).to(dev)
        tp = torch.from_numpy(rs.randint(0, ni, N_TRIPLETS)).to(dev)
        tn = torch.from_numpy(rs.randint(0, ni, N_TRIPLETS)).to(dev)
        cu, ci = ei[0].contiguous(), ei[1].contiguous()
        graph = gdr.BipartiteGraph(ei, ew, nu, ni)

        def step(arm):
            u0.grad = i0.grad = raw.grad = None
            w = torch.nn.functional.softplus(raw)
            if arm == "gdr":
                uo, io = gdr.LightGCNPropagate.apply(u0, i0, w, graph, L)
            else:
                with torch.device(dev):
                    uo, io = rp.lightgcn_propagate(cu, ci, w, u0, i0, L)
            x = (uo[tu] * io[tp]).sum(1) - (uo[tu] * io[tn]).sum(1)
            (-torch.nn.functional.logsigmoid(x).mean()).backward()

        arms = ("gdr", "torch")
        for a in arms:
            for _ in range(3):
                step(a)
        times = {a: [] for a in arms}
        while min(sum(t) for t in times.values()) < 1000.0:
            for a in arms:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                step(a)
                e1.record()
                e1.synchronize()
                times[a].append(e0.elapsed_time(e1))
        med = {a: float(np.median(t)) for a, t in times.items()}

        # gradient error of one gdr backward against fp64 autograd, with a random upstream gradient
        g_u = torch.randn(nu, D, device=dev, generator=torch.Generator(dev).manual_seed(1))
        g_i = torch.randn(ni, D, device=dev, generator=torch.Generator(dev).manual_seed(2))
        w = ew.clone().requires_grad_(True)
        U, I = u0.detach().clone().requires_grad_(True), i0.detach().clone().requires_grad_(True)
        uo, io = gdr.LightGCNPropagate.apply(U, I, w, graph, L)
        ((uo * g_u).sum() + (io * g_i).sum()).backward()
        ref = ref_autograd_f64(cu, ci, ew, u0.detach(), i0.detach(), g_u, g_i, L)
        err = {k: float((got.double() - r).abs().max() / r.abs().max())
               for k, got, r in zip(("du0", "di0", "dw"), (U.grad, I.grad, w.grad), ref)}

        # kernel leg: gdr_lightgcn_edge_grad alone on stacked layers of the right shape
        A = graph.A
        ld = pad4(D)
        Xu, Yu = (torch.randn(L, nu, ld, device=dev) for _ in range(2))
        Xi, Yi = (torch.randn(L, ni, ld, device=dev) for _ in range(2))
        G = torch.empty(A.nnz, device=dev)
        S_u = torch.empty(nu, dtype=torch.float64, device=dev)
        args = (nu, ni, A.nnz, ptr(A.rowptr), ptr(A.colidx), ptr(A.vals), L, D, ptr(Xu), ptr(Xi), ptr(Yu), ptr(Yi), ld,
                1.0 / (L + 1), ptr(G), ptr(S_u), stream())
        for _ in range(5):
            _lib.call("gdr_lightgcn_edge_grad", *args)
        n_k = 100
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(n_k):
            _lib.call("gdr_lightgcn_edge_grad", *args)
        k1.record()
        k1.synchronize()
        k_ms = k0.elapsed_time(k1) / n_k
        gathered = E * 2 * L * D * 4
        print(json.dumps({"workload": {"C": "yelp2018 condensed", "D": "amazon-book condensed",
                                       "C_full": "yelp2018 full interaction graph"}[name],
                          "n_u": nu, "n_i": ni, "E": E, "d": D, "L": L, "triplets": N_TRIPLETS,
                          "gdr_ms_per_step": round(med["gdr"], 3), "torch_ms_per_step": round(med["torch"], 3),
                          "speedup": round(med["torch"] / med["gdr"], 2), "steps": {a: len(t) for a, t in times.items()},
                          "max_grad_err_vs_fp64": {k: float(f"{v:.3e}") for k, v in err.items()},
                          "edge_grad_kernel_ms": round(k_ms, 4), "edge_grad_gathered_bytes": gathered,
                          "edge_grad_gathered_GBps_L2_resident": round(gathered / k_ms / 1e6, 1),
                          "card": info}), flush=True)


if __name__ == "__main__":
    main()
