"""Time one BPR refinement step of LightGCN three ways on the GPU, and the two BPR entry points alone.

Step = sample B triplets + LightGCNPropagate (L = 2, d = 64; gradients to u0, i0 and the raw edge weights through
softplus) + BPR loss + backward + torch.optim.Adam (fused).  Arms, alternated, each timed with CUDA events around a
synchronised step after 3 warm-up steps, until each has >= 1 s of steps; the median is reported:
  library  gdr.BPRSampler.sample + gdr.bpr_loss
  host     a LightGCN-style host sampler (one Python iteration per triplet: uniform user, uniform positive, negatives
           by rejection against the user's item array), an H2D copy of the triplets, and the torch BPR expression.
           It stands in for the reference's own sampler (distill_recsys.py:234-270), which is not in this checkout.
  torch    a vectorised on-device rejection sampler in torch (membership by searchsorted over the row-major
           (user, item) keys; rejected negatives redrawn until none is left) and the torch BPR expression.
Kernel leg: gdr_bpr_sample and gdr_bpr_loss (with both gradients) alone, CUDA events over 100 launches each.
Bytes: sample = B * 40 (eligible id, row bounds, positive column, 3 int64 ids out; the binary search adds
log2(deg) colidx reads); loss = B * (24 + 3 * 4d) for the scores plus B * 4 * 4d for the gradient gathers
(2 item rows per user slot, 1 user row per item slot) plus the sort of the 3B (8 + 4)-byte slots.  These operands
fit the 126 MB L2, the regime of a real refinement loop, so the rates are L2 rates.
Workloads: the condensed Yelp2018 and Amazon-book graphs (bench seeds, as tools/lightgcn_grad_bench.py) and the full
Yelp2018-shaped interaction graph; B in {2048, 65536}.  One JSON line per (workload, B), with the card name and power
limit read in the same run.
"""
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import gdr  # noqa: E402
from gdr import _lib  # noqa: E402
from gdr._dev import ptr, stream, workspace  # noqa: E402
from lightgcn_grad_bench import card, workload  # noqa: E402

D, L = 64, 2


def _inv_softplus(w):
    """softplus^-1(w) = w + log(1 - exp(-w)), finite for the large counts of a condensed graph."""
    return w + torch.log(-torch.expm1(-w))


def torch_bpr(uo, io, u, p, n):
    x = (uo[u] * io[p]).sum(1) - (uo[u] * io[n]).sum(1)
    return -F.logsigmoid(x).mean()


class HostSampler:
    """LightGCN's UniformSample_original_python: a Python loop over triplets with rejection for the negatives."""

    def __init__(self, rowptr, colidx, n_items, seed):
        self.pos_for_user = [colidx[rowptr[u]:rowptr[u + 1]] for u in range(len(rowptr) - 1)]
        deg = np.diff(rowptr)
        self.users = np.nonzero((deg > 0) & (deg < n_items))[0]
        self.n_items = n_items
        self.rng = np.random.RandomState(seed)

    def sample(self, B, dev):
        out = np.empty((3, B), dtype=np.int64)
        rng = self.rng
        for b in range(B):
            user = self.users[rng.randint(0, len(self.users))]
            pos_items = self.pos_for_user[user]
            pos = pos_items[rng.randint(0, len(pos_items))]
            while True:
                neg = rng.randint(0, self.n_items)
                if neg in pos_items:
                    continue
                break
            out[0, b], out[1, b], out[2, b] = user, pos, neg
        t = torch.from_numpy(out).to(dev)
        return t[0], t[1], t[2]


class TorchSampler:
    """Vectorised rejection sampler on the device."""

    def __init__(self, R, seed):
        n_u, self.n_i = R.shape
        deg = (R.rowptr[1:] - R.rowptr[:-1]).long()
        self.deg, self.start = deg, R.rowptr[:-1].long()
        self.elig = torch.nonzero((deg > 0) & (deg < self.n_i)).reshape(-1)
        rows = torch.repeat_interleave(torch.arange(n_u, device=deg.device), deg)
        self.keys = rows * self.n_i + R.colidx.long()   # ascending: rows in order, columns sorted
        self.colidx = R.colidx.long()
        self.gen = torch.Generator(deg.device).manual_seed(seed)

    def _member(self, u, j):
        k = u * self.n_i + j
        at = torch.searchsorted(self.keys, k).clamp_max(self.keys.numel() - 1)
        return self.keys[at] == k

    def sample(self, B, dev):
        g = self.gen
        u = self.elig[torch.randint(0, self.elig.numel(), (B,), device=dev, generator=g)]
        r = torch.rand(B, device=dev, generator=g)
        p = self.colidx[self.start[u] + (r * self.deg[u]).long().clamp_max(self.deg[u] - 1)]
        n = torch.randint(0, self.n_i, (B,), device=dev, generator=g)
        bad = self._member(u, n)
        while bool(bad.any()):
            idx = torch.nonzero(bad).reshape(-1)
            n[idx] = torch.randint(0, self.n_i, (idx.numel(),), device=dev, generator=g)
            bad[idx] = self._member(u[idx], n[idx])
        return u, p, n


def event_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    assert torch.cuda.is_available(), "bpr_bench needs a GPU"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = card()
    for name in ("C", "D", "C_full"):
        ei, ew, nu, ni = workload(name, dev)
        R = gdr.BipartiteGraph(ei, ew, nu, ni).W
        graph = gdr.BipartiteGraph(ei, ew, nu, ni)
        rowptr, colidx = R.rowptr.cpu().numpy().astype(np.int64), R.colidx.cpu().numpy().astype(np.int64)
        raw0 = _inv_softplus(ew.clamp_min(0.05))
        rs = np.random.RandomState(7)
        u_init = torch.from_numpy((rs.standard_normal((nu, D)) * 0.1).astype(np.float32)).to(dev)
        i_init = torch.from_numpy((rs.standard_normal((ni, D)) * 0.1).astype(np.float32)).to(dev)
        for B in (2048, 65536):
            samplers = {"library": gdr.BPRSampler(R, 1), "host": HostSampler(rowptr, colidx, ni, 1),
                        "torch": TorchSampler(R, 1)}
            state = {}
            for arm in samplers:
                u0, i0, raw = (x.clone().requires_grad_(True) for x in (u_init, i_init, raw0))
                state[arm] = [u0, i0, raw, torch.optim.Adam([u0, i0, raw], lr=1e-3, fused=True), 0]

            def step(arm):
                u0, i0, raw, opt, k = state[arm]
                if arm == "library":
                    u, p, n = samplers[arm].sample(B, k)
                else:
                    u, p, n = samplers[arm].sample(B, dev)
                uo, io = gdr.LightGCNPropagate.apply(u0, i0, F.softplus(raw), graph, L)
                loss = gdr.bpr_loss(uo, io, u, p, n) if arm == "library" else torch_bpr(uo, io, u, p, n)
                opt.zero_grad(set_to_none=True)
                loss.backward()
                opt.step()
                state[arm][4] = k + 1

            for a in samplers:
                for _ in range(3):
                    step(a)
            times = {a: [] for a in samplers}
            while min(sum(t) for t in times.values()) < 1000.0:
                for a in samplers:   # alternated; an arm that has its second of steps sits out the later rounds
                    if sum(times[a]) < 1000.0:
                        times[a].append(event_ms(lambda: step(a), 1))
            med = {a: float(np.median(t)) for a, t in times.items()}

            # kernel leg: the two entry points alone
            s = samplers["library"]
            out = torch.empty((3, B), dtype=torch.int64, device=dev)
            sample_args = (nu, ni, ptr(R.rowptr), ptr(R.colidx), s.n_eligible, ptr(s.eligible), s.seed, 5, B,
                           ptr(out[0]), ptr(out[1]), ptr(out[2]), stream())
            _lib.call("gdr_bpr_sample", *sample_args)
            Ue, Ie = u_init.clone(), i_init.clone()
            gU, gI = torch.empty_like(Ue), torch.empty_like(Ie)
            loss = torch.empty((), device=dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            ws = workspace(_lib.query("gdr_bpr_loss_ws_bytes", B, nu, ni), dev)
            loss_args = (B, nu, ni, D, ptr(Ue), D, ptr(Ie), D, ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(loss),
                         ptr(gU), D, ptr(gI), D, ptr(status), ptr(ws), ws.numel(), stream())
            for _ in range(5):
                _lib.call("gdr_bpr_sample", *sample_args)
                _lib.call("gdr_bpr_loss", *loss_args)
            ks = event_ms(lambda: _lib.call("gdr_bpr_sample", *sample_args), 100)
            kl = event_ms(lambda: _lib.call("gdr_bpr_loss", *loss_args), 100)
            assert int(status.item()) == 0
            sample_bytes = B * 40
            loss_bytes = B * (24 + 3 * 4 * D) + B * 4 * 4 * D + 3 * B * 12 * 2
            print(json.dumps({
                "workload": {"C": "yelp2018 condensed", "D": "amazon-book condensed",
                             "C_full": "yelp2018 full interaction graph"}[name],
                "n_u": nu, "n_i": ni, "E": int(ei.shape[1]), "d": D, "L": L, "B": B,
                "ms_per_step": {a: round(v, 3) for a, v in med.items()},
                "speedup_vs_host": round(med["host"] / med["library"], 2),
                "speedup_vs_torch": round(med["torch"] / med["library"], 2),
                "steps": {a: len(t) for a, t in times.items()},
                "bpr_sample_kernel_ms": round(ks, 4), "bpr_sample_bytes": sample_bytes,
                "bpr_loss_call_ms": round(kl, 4), "bpr_loss_bytes": loss_bytes,
                "card": info}), flush=True)
    hub_leg(dev, info)


def hub_leg(dev, info):
    """gdr_bpr_loss alone at B = 2^20 on the condensed Yelp2018 sizes, with uniform triplets and with every triplet on
    user 0 and positive item 0 (two rows of 2^20 slots, each summed by one CTA): the cost of the hub path."""
    nu, ni, B = 3167, 3805, 1 << 20
    g = torch.Generator(dev).manual_seed(3)
    U = torch.randn(nu, D, device=dev, generator=g) * 0.1
    I = torch.randn(ni, D, device=dev, generator=g) * 0.1
    gU, gI = torch.empty_like(U), torch.empty_like(I)
    loss = torch.empty((), device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = workspace(_lib.query("gdr_bpr_loss_ws_bytes", B, nu, ni), dev)
    uni = [torch.randint(0, n, (B,), device=dev, generator=g) for n in (nu, ni, ni)]
    hub = [torch.zeros(B, dtype=torch.int64, device=dev), torch.zeros(B, dtype=torch.int64, device=dev), uni[2]]
    res = {}
    for name, (u, p, n) in (("uniform", uni), ("hub", hub)):
        args = (B, nu, ni, D, ptr(U), D, ptr(I), D, ptr(u), ptr(p), ptr(n), ptr(loss), ptr(gU), D, ptr(gI), D,
                ptr(status), ptr(ws), ws.numel(), stream())
        for _ in range(3):
            _lib.call("gdr_bpr_loss", *args)
        res[name] = round(event_ms(lambda: _lib.call("gdr_bpr_loss", *args), 20), 4)
    assert int(status.item()) == 0
    print(json.dumps({"workload": "bpr_loss hub rows", "n_u": nu, "n_i": ni, "d": D, "B": B,
                      "bpr_loss_call_ms": res, "card": info}), flush=True)


if __name__ == "__main__":
    main()
