"""LightGCNPropagate on the B200: gradients w.r.t. the embeddings and the edge weights against torch fp64 autograd of
the reference expression, bit-identity with the forward-only path and with BipartitePropagate, in-place reweighting,
the full condensed shapes, and a short training run against the fp32 torch reference."""
import numpy as np
import pytest
import torch

from conftest import golden
from test_lightgcn_grad_cpu import random_graph, ref_autograd_f64

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
BOUND = 1e-4   # max |gdr - fp64| <= BOUND * max |fp64|, per gradient


@pytest.fixture(scope="module")
def gdr():
    import gdr as g
    assert torch.cuda.is_available()
    torch.cuda.set_device(DEV)
    return g


def _dev(a, dt=None):
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
    return t.to(DEV, dt) if dt is not None else t.to(DEV)


def run_gdr(gdr, cu, ci, w, u0, i0, gu, gi, L, nu, ni, graph=None):
    """(du0, di0, dw, graph) of <gu, u_out> + <gi, i_out> through gdr.LightGCNPropagate."""
    if graph is None:
        graph = gdr.BipartiteGraph(torch.stack([_dev(cu, torch.int64), _dev(ci, torch.int64)]), _dev(w, torch.float32),
                                   nu, ni)
    W = _dev(w, torch.float32).clone().requires_grad_(True)
    U = _dev(u0, torch.float32).clone().requires_grad_(True)
    I = _dev(i0, torch.float32).clone().requires_grad_(True)
    uo, io = gdr.LightGCNPropagate.apply(U, I, W, graph, L)
    ((uo * _dev(gu, torch.float32)).sum() + (io * _dev(gi, torch.float32)).sum()).backward()
    return U.grad, I.grad, W.grad, graph


def check_vs_fp64(gdr, cu, ci, w, u0, i0, gu, gi, L, nu, ni):
    du, di, dw, _ = run_gdr(gdr, cu, ci, w, u0, i0, gu, gi, L, nu, ni)
    ru, ri, rw = ref_autograd_f64(_dev(cu), _dev(ci), _dev(w), _dev(u0), _dev(i0), _dev(gu), _dev(gi), L)
    errs = {}
    for name, got, ref in (("du0", du, ru), ("di0", di, ri), ("dw", dw, rw)):
        assert got.shape == ref.shape, name
        assert torch.isfinite(got).all(), name
        err = float((got.double() - ref).abs().max()) if ref.numel() else 0.0
        scale = float(ref.abs().max()) if ref.numel() else 0.0
        assert err <= BOUND * scale, f"{name}: max|err| {err:.3e} > {BOUND} * max|ref| {scale:.3e}"
        errs[name] = err / scale if scale else 0.0
    if L == 0:
        assert not dw.any()
    return errs


def _inputs(nu, ni, d, seed):
    rs = np.random.RandomState(seed)
    return [rs.standard_normal(s).astype(np.float32) * 0.1 for s in ((nu, d), (ni, d), (nu, d), (ni, d))]


# ------------------------------------------------------------------------------------- gradients vs fp64 autograd
@pytest.mark.parametrize("L", [0, 1, 2, 3])
@pytest.mark.parametrize("d", [1, 7, 16, 64, 100])
def test_random_graph_with_hubs(gdr, L, d):
    nu, ni = 400, 6000
    cu, ci, w = random_graph(nu, ni, 20000, seed=d + 10 * L, hub_row=5500, hub_col=300)
    assert np.bincount(cu).max() >= 5000
    check_vs_fp64(gdr, cu, ci, w, *_inputs(nu, ni, d, seed=L), L, nu, ni)


@pytest.mark.parametrize("L", [0, 1, 2, 3])
def test_golden_graph(gdr, L):
    g = golden("lightgcn.npz")
    ei = g["edge_index"]
    nu, ni = g["u0"].shape[0], g["i0"].shape[0]
    rs = np.random.RandomState(7)
    gu = rs.standard_normal(g["u0"].shape).astype(np.float32)
    gi = rs.standard_normal(g["i0"].shape).astype(np.float32)
    check_vs_fp64(gdr, ei[0], ei[1], g["w"], g["u0"], g["i0"], gu, gi, L, nu, ni)


@pytest.mark.parametrize("d", [5, 300])
def test_deep_and_wide(gdr, d):
    # L > 4 and d > 256 run as several passes (layer chunks / column windows) adding into G
    nu, ni = 120, 90
    cu, ci, w = random_graph(nu, ni, 1500, seed=d, hub_row=60)
    check_vs_fp64(gdr, cu, ci, w, *_inputs(nu, ni, d, seed=d), 6, nu, ni)


def test_no_edges(gdr):
    nu, ni, d = 5, 4, 8
    cu = ci = np.zeros(0, dtype=np.int64)
    w = np.zeros(0, dtype=np.float32)
    check_vs_fp64(gdr, cu, ci, w, *_inputs(nu, ni, d, seed=1), 2, nu, ni)


# ------------------------------------------------------------------------------------------------- bit identity
def _small(seed=0, nu=300, ni=200, d=24):
    cu, ci, w = random_graph(nu, ni, 6000, seed=seed, hub_row=150)
    return cu, ci, w, nu, ni, _inputs(nu, ni, d, seed)


def test_forward_matches_lightgcn_propagate(gdr):
    cu, ci, w, nu, ni, (u0, i0, _, _) = _small()
    ei = torch.stack([_dev(cu), _dev(ci)])
    g1 = gdr.BipartiteGraph(ei, _dev(np.ones_like(w)), nu, ni)   # built with other weights, reweighted by the forward
    uo, io = gdr.LightGCNPropagate.apply(_dev(u0), _dev(i0), _dev(w).requires_grad_(True), g1, 3)
    g2 = gdr.BipartiteGraph(ei, _dev(w), nu, ni)
    ur, ir = gdr.lightgcn_propagate(g2, _dev(u0), _dev(i0), 3)
    assert torch.equal(uo, ur) and torch.equal(io, ir)


def test_set_edge_weight_matches_fresh_build(gdr):
    cu, ci, w, nu, ni, _ = _small(1)
    ei = torch.stack([_dev(cu), _dev(ci)])
    g = gdr.BipartiteGraph(ei, _dev(w), nu, ni)
    w2 = np.random.RandomState(5).uniform(0.0, 2.0, w.shape).astype(np.float32)
    w2[:50] = 0.0
    g.set_edge_weight(_dev(w2))
    f = gdr.BipartiteGraph(ei, _dev(w2), nu, ni)
    for a, b in ((g.A.vals, f.A.vals), (g.AT.vals, f.AT.vals), (g.deg_u, f.deg_u), (g.deg_i, f.deg_i),
                 (g.W.vals, f.W.vals)):
        assert torch.equal(a, b)


def test_embedding_grads_match_bipartite_propagate(gdr):
    cu, ci, w, nu, ni, (u0, i0, gu, gi) = _small(2)
    du, di, _, _ = run_gdr(gdr, cu, ci, w, u0, i0, gu, gi, 2, nu, ni)
    g = gdr.BipartiteGraph(torch.stack([_dev(cu), _dev(ci)]), _dev(w), nu, ni)
    U = _dev(u0).requires_grad_(True)
    I = _dev(i0).requires_grad_(True)
    uo, io = gdr.BipartitePropagate.apply(U, I, g, 2)
    ((uo * _dev(gu)).sum() + (io * _dev(gi)).sum()).backward()
    assert torch.equal(du, U.grad) and torch.equal(di, I.grad)


def test_edge_grad_is_deterministic(gdr):
    cu, ci, w, nu, ni, (u0, i0, gu, gi) = _small(3, d=64)
    _, _, dw1, g = run_gdr(gdr, cu, ci, w, u0, i0, gu, gi, 3, nu, ni)
    _, _, dw2, _ = run_gdr(gdr, cu, ci, w, u0, i0, gu, gi, 3, nu, ni, graph=g)
    assert torch.equal(dw1, dw2)


def test_two_forwards_one_backward(gdr):
    # the second forward reweights the shared graph; the first call's backward must use its own weights
    cu, ci, w, nu, ni, (u0, i0, gu, gi) = _small(4)
    w2 = (w * 0.5 + 0.25).astype(np.float32)
    g = gdr.BipartiteGraph(torch.stack([_dev(cu), _dev(ci)]), _dev(w), nu, ni)
    single = [run_gdr(gdr, cu, ci, ww, u0, i0, gu, gi, 2, nu, ni, graph=g)[:3] for ww in (w, w2)]
    U = _dev(u0).requires_grad_(True)
    I = _dev(i0).requires_grad_(True)
    W1 = _dev(w).requires_grad_(True)
    W2 = _dev(w2).requires_grad_(True)
    u1, i1 = gdr.LightGCNPropagate.apply(U, I, W1, g, 2)
    u2, i2 = gdr.LightGCNPropagate.apply(U, I, W2, g, 2)
    ((u1 * _dev(gu)).sum() + (i1 * _dev(gi)).sum() + (u2 * _dev(gu)).sum() + (i2 * _dev(gi)).sum()).backward()
    assert torch.equal(W1.grad, single[0][2]) and torch.equal(W2.grad, single[1][2])
    assert torch.equal(U.grad, single[0][0] + single[1][0]) and torch.equal(I.grad, single[0][1] + single[1][1])


def test_duplicate_pair_raises(gdr):
    ei = _dev(np.array([[0, 1, 1, 2], [0, 2, 2, 1]], dtype=np.int64))
    g = gdr.BipartiteGraph(ei, _dev(np.ones(4, dtype=np.float32)), 3, 3)
    assert g.W.nnz == 3
    u0 = _dev(np.ones((3, 4), dtype=np.float32))
    gdr.lightgcn_propagate(g, u0, u0, 2)   # the forward-only path keeps accepting duplicates
    with pytest.raises(ValueError):
        g.set_edge_weight(_dev(np.ones(4, dtype=np.float32)))
    with pytest.raises(ValueError):
        gdr.LightGCNPropagate.apply(u0, u0, _dev(np.ones(4, dtype=np.float32)).requires_grad_(True), g, 2)


# --------------------------------------------------------------------------------------- full condensed shapes
@pytest.mark.parametrize("cfg_id", ["C", "D"])
def test_full_condensed_shapes(gdr, cfg_id):
    from gdr import synth
    cfg = synth.BIPARTITE[cfg_id]
    U, I, E, d, L = cfg["users"], cfg["items"], cfg["inter"], cfg["d"], cfg["layers"]
    u, i = synth.bipartite_interactions(U, I, E, seed=1236)
    rs = np.random.RandomState(3)
    emb_u = (rs.standard_normal((U, d)) * 0.1).astype(np.float32)
    emb_i = (rs.standard_normal((I, d)) * 0.1).astype(np.float32)
    ncu, nci = int(np.ceil(U * 0.1)), int(np.ceil(I * 0.1))
    u2cu, _ = gdr.kmeans_cluster(emb_u, ncu, seed=42, init="random")
    i2ci, _ = gdr.kmeans_cluster(emb_i, nci, seed=42, init="random")
    C = gdr.build_condensed_bipartite(u, i, u2cu, i2ci, ncu, nci, device=DEV, return_device=True)
    ei, ew = gdr.condensed_csr_to_edge_index(C, DEV)
    u0, i0, gu, gi = _inputs(ncu, nci, d, seed=11)
    errs = check_vs_fp64(gdr, ei[0], ei[1], ew, u0, i0, gu, gi, L, ncu, nci)
    print(f"\n{cfg['name']} condensed: {ncu} x {nci}, E = {ei.shape[1]}, d = {d}, L = {L}, "
          f"max|err|/max|ref|: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))


# -------------------------------------------------------------------------------------------- training smoke test
def test_training_matches_fp32_reference(gdr):
    from oracle import ref_port as rp
    nu, ni, d, L, steps, lr = 400, 300, 32, 2, 20, 50.0
    cu, ci, w0 = random_graph(nu, ni, 8000, seed=9, hub_row=200)
    rs = np.random.RandomState(10)
    base_u = _dev((rs.standard_normal((nu, d)) * 0.1).astype(np.float32))
    base_i = _dev((rs.standard_normal((ni, d)) * 0.1).astype(np.float32))
    n_t = 2048
    tu = _dev(rs.randint(0, nu, n_t).astype(np.int64))
    tp = _dev(rs.randint(0, ni, n_t).astype(np.int64))
    tn = _dev(rs.randint(0, ni, n_t).astype(np.int64))
    raw0 = _dev(np.log(np.expm1(np.maximum(w0, 0.05))).astype(np.float32))   # softplus^-1 of the initial weights
    cu_d, ci_d = _dev(cu), _dev(ci)
    graph = gdr.BipartiteGraph(torch.stack([cu_d, ci_d]), _dev(w0), nu, ni)

    def bpr(uo, io):
        x = (uo[tu] * io[tp]).sum(1) - (uo[tu] * io[tn]).sum(1)
        return -torch.nn.functional.logsigmoid(x).mean()

    def train(use_gdr):
        ud = torch.zeros(nu, d, device=DEV, requires_grad=True)
        idl = torch.zeros(ni, d, device=DEV, requires_grad=True)
        raw = raw0.clone().requires_grad_(True)
        losses = []
        for _ in range(steps):
            w = torch.nn.functional.softplus(raw)
            if use_gdr:
                uo, io = gdr.LightGCNPropagate.apply(base_u + ud, base_i + idl, w, graph, L)
            else:
                with torch.device(DEV):
                    uo, io = rp.lightgcn_propagate(cu_d, ci_d, w, base_u + ud, base_i + idl, L)
            loss = bpr(uo, io)
            ud.grad = idl.grad = raw.grad = None
            loss.backward()
            with torch.no_grad():
                for p in (ud, idl, raw):
                    p -= lr * p.grad
            losses.append(float(loss.detach()))
        return losses

    got, ref = train(True), train(False)
    for s, (a, b) in enumerate(zip(got, ref)):
        assert abs(a - b) <= 1e-4 * abs(b), f"step {s}: gdr {a} vs torch {b}"
    assert all(b < a for a, b in zip(got, got[1:])) and got[-1] < got[0] - 1e-3, got
