"""BPRSampler and bpr_loss on the B200: the sampler bit-identical to the numpy reference (tests/bpr_ref.py) on edge
case graphs and at the condensed / full dataset shapes; the fused loss and gradients against torch fp32 / fp64
autograd of -logsigmoid(x).mean(); run-to-run bit identity; and a seeded 20-step refinement (sampler ->
LightGCNPropagate -> bpr_loss -> Adam) that is bit-reproducible and follows the torch BPR expression."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.nn.functional as F

import bpr_ref
from test_lightgcn_grad_cpu import random_graph

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def gdr():
    import gdr as g
    assert torch.cuda.is_available()
    torch.cuda.set_device(DEV)
    return g


def _check_sampler(gdr, R, seed, steps, batch):
    s = gdr.BPRSampler(R, seed)
    rp, ci = s.R.rowptr.cpu().numpy(), s.R.colidx.cpu().numpy()
    for step in steps:
        got = [t.cpu().numpy() for t in s.sample(batch, step)]
        want = bpr_ref.sample(rp, ci, s.R.shape[1], seed, step, batch)
        for g, w in zip(got, want):
            assert g.dtype == np.int64 and np.array_equal(g, w)
    return s


# ------------------------------------------------------------------------------------------------------- sampler
def test_sampler_matches_reference_on_edge_cases(gdr):
    rs = np.random.RandomState(0)
    n_u, n_i = 500, 7000
    m = sp.random(n_u, n_i, density=0.002, format="lil", random_state=rs)
    m[0, :] = 0                                   # empty row
    m[1, :] = 1                                   # full row: not eligible
    m[2, :] = 1
    m[2, 0] = 0                                   # missing only item 0
    m[3, :] = 1
    m[3, n_i - 1] = 0                             # missing only the last item
    m[4, rs.choice(n_i, 6000, replace=False)] = 1   # hub row
    m = m.tocsr()
    m.eliminate_zeros()
    s = _check_sampler(gdr, m, seed=0x123456789ABCDEF, steps=(0, 1, 2**32 - 1), batch=100_000)
    u, _, n = (t.cpu().numpy() for t in s.sample(100_000, 5))
    assert not np.isin([0, 1], u).any()
    assert (n[u == 2] == 0).all() and (n[u == 3] == n_i - 1).all()
    # the torch sparse and gdr.CSR spellings give the same triplets
    idx = torch.from_numpy(np.stack(m.nonzero()).astype(np.int64))
    t = torch.sparse_coo_tensor(idx, torch.ones(m.nnz), m.shape).to(DEV)
    for R in (t, s.R):
        assert all(torch.equal(a, b) for a, b in zip(gdr.BPRSampler(R, 0x123456789ABCDEF).sample(777, 9),
                                                     s.sample(777, 9)))


def test_sampler_one_item_catalogue_raises(gdr):
    m = sp.csr_matrix((np.ones(3), ([0, 1, 2], [0, 0, 0])), shape=(4, 1))
    with pytest.raises(ValueError):
        gdr.BPRSampler(m, 1)


def test_sampler_rejects_unsorted_columns(gdr):
    R = gdr.CSR(torch.tensor([0, 2], dtype=torch.int32, device=DEV), torch.tensor([3, 1], dtype=torch.int32,
                device=DEV), torch.ones(2, device=DEV), (1, 5))
    with pytest.raises(ValueError):
        gdr.BPRSampler(R, 1)


def test_sampler_argument_ranges(gdr):
    s = gdr.BPRSampler(sp.csr_matrix(np.eye(3, 4)), 3)
    for B, step in ((0, 0), ((1 << 31) // 3 + 1, 0), (4, -1), (4, 1 << 32)):
        with pytest.raises(ValueError):
            s.sample(B, step)


def test_sampler_same_step_same_output(gdr):
    cu, ci, _ = random_graph(300, 200, 5000, seed=1, hub_row=150)
    s = gdr.BPRSampler(sp.csr_matrix((np.ones(len(cu)), (cu, ci)), shape=(300, 200)), 42)
    a, b, c = s.sample(4096, 17), s.sample(4096, 17), s.sample(4096, 18)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert not all(torch.equal(x, y) for x, y in zip(a, c))


@pytest.fixture(scope="module")
def shapes(gdr):
    """Interaction CSRs: the condensed Yelp2018 and Amazon-book shapes (as in test_full_condensed_shapes) and the
    full Yelp2018-shaped training graph."""
    from gdr import synth
    out = {}
    for cfg_id in ("C", "D"):
        cfg = synth.BIPARTITE[cfg_id]
        U, I, d = cfg["users"], cfg["items"], cfg["d"]
        u, i = synth.bipartite_interactions(U, I, cfg["inter"], seed=1236)
        rs = np.random.RandomState(3)
        emb_u = (rs.standard_normal((U, d)) * 0.1).astype(np.float32)
        emb_i = (rs.standard_normal((I, d)) * 0.1).astype(np.float32)
        ncu, nci = int(np.ceil(U * 0.1)), int(np.ceil(I * 0.1))
        u2cu, _ = gdr.kmeans_cluster(emb_u, ncu, seed=42, init="random")
        i2ci, _ = gdr.kmeans_cluster(emb_i, nci, seed=42, init="random")
        out[cfg["name"] + " condensed"] = gdr.build_condensed_bipartite(u, i, u2cu, i2ci, ncu, nci, device=DEV,
                                                                        return_device=True)
        if cfg_id == "C":
            out["yelp2018 full"] = gdr.coo_to_csr(u, i, None, (U, I), device=DEV)
    return out


@pytest.mark.parametrize("batch", [2048, 1 << 20])
@pytest.mark.parametrize("name", ["yelp2018 condensed", "amazon-book condensed", "yelp2018 full"])
def test_sampler_matches_reference_at_dataset_shapes(gdr, shapes, name, batch):
    _check_sampler(gdr, shapes[name], seed=2024, steps=(0, 733), batch=batch)


# ---------------------------------------------------------------------------------------------- loss and gradient
def _emb(n, d, seed, scale=0.1):
    g = torch.Generator(DEV).manual_seed(seed)
    return torch.randn(n, d, device=DEV, generator=g) * scale


def _triplets(n_u, n_i, B, seed):
    g = torch.Generator(DEV).manual_seed(seed)
    return tuple(torch.randint(0, n, (B,), device=DEV, generator=g) for n in (n_u, n_i, n_i))


def _inv_softplus(w):
    """softplus^-1(w) = w + log(1 - exp(-w)), finite for the large counts of a condensed graph."""
    return w + torch.log(-torch.expm1(-w))


def torch_bpr(U, I, u, p, n):
    x = (U[u] * I[p]).sum(1) - (U[u] * I[n]).sum(1)
    return -F.logsigmoid(x).mean()


def check_loss(gdr, U, I, u, p, n):
    """gdr loss vs torch fp32 (1e-6 relative); gdr gU / gI vs torch fp64 autograd (1e-5 max|ref|).  Inputs that
    already require grad are passed to bpr_loss as they are (strides and padding included)."""
    Ug = U if U.requires_grad else U.detach().clone().requires_grad_(True)
    Ig = I if I.requires_grad else I.detach().clone().requires_grad_(True)
    loss = gdr.bpr_loss(Ug, Ig, u, p, n)
    gU, gI = torch.autograd.grad(loss, (Ug, Ig))
    assert loss.dtype == torch.float32 and loss.dim() == 0
    ref32 = torch_bpr(U.detach(), I.detach(), u, p, n)
    assert abs(float(loss) - float(ref32)) <= 1e-6 * abs(float(ref32)), (float(loss), float(ref32))
    U64 = U.detach().double().requires_grad_(True)
    I64 = I.detach().double().requires_grad_(True)
    torch_bpr(U64, I64, u, p, n).backward()
    for name, got, ref in (("gU", gU, U64.grad), ("gI", gI, I64.grad)):
        assert got.shape == ref.shape and torch.isfinite(got).all(), name
        err, scale = float((got.double() - ref).abs().max()), float(ref.abs().max())
        assert err <= 1e-5 * scale, f"{name}: max|err| {err:.3e} > 1e-5 * max|ref| {scale:.3e}"
    return loss, gU, gI


@pytest.mark.parametrize("B", [1, 2048, 1 << 20])
@pytest.mark.parametrize("d", [1, 7, 16, 64, 100, 300])
def test_loss_and_gradients(gdr, d, B):
    n_u, n_i = 3000, 4000
    check_loss(gdr, _emb(n_u, d, 1), _emb(n_i, d, 2), *_triplets(n_u, n_i, B, seed=d + B))


@pytest.mark.parametrize("d", [7, 64, 300])
def test_all_triplets_on_one_user_and_one_item(gdr, d):
    # one user row and one item row take every slot: the rows split over the whole CTA
    B, n_u, n_i = 1 << 20, 50, 80
    _, _, n = _triplets(n_u, n_i, B, seed=5)
    z = torch.zeros(B, dtype=torch.int64, device=DEV)
    check_loss(gdr, _emb(n_u, d, 3), _emb(n_i, d, 4), z, z, n)
    check_loss(gdr, _emb(n_u, d, 3), _emb(n_i, d, 4), z, z, torch.full_like(z, 1))


@pytest.mark.parametrize("d", [7, 64])
def test_inputs_from_lightgcn_propagate(gdr, d, monkeypatch):
    # LightGCNPropagate's outputs go into bpr_loss as they are: padded rows are read in place, without a copy
    from gdr import recsys
    in_place = []
    orig = recsys.padded_rows

    def spy(x):
        y = orig(x)
        in_place.append(y.data_ptr() == x.data_ptr())
        return y

    cu, ci, w = random_graph(300, 200, 6000, seed=3, hub_row=150)
    ei = torch.stack([torch.from_numpy(cu), torch.from_numpy(ci)]).to(DEV)
    g = gdr.BipartiteGraph(ei, torch.from_numpy(w).to(DEV), 300, 200)
    u0, i0 = _emb(300, d, 5).requires_grad_(True), _emb(200, d, 6).requires_grad_(True)
    uo, io = gdr.LightGCNPropagate.apply(u0, i0, torch.from_numpy(w).to(DEV), g, 2)
    monkeypatch.setattr(recsys, "padded_rows", spy)   # from here on: bpr_loss's two operands only
    assert uo.stride(0) % 4 == 0 and (d % 4 == 0 or uo.stride(0) > d)
    check_loss(gdr, uo, io, *_triplets(300, 200, 4096, seed=7))
    assert in_place == [True, True]


def test_padding_columns_are_not_read(gdr):
    # rows with stride 8 and d = 7 whose padding column holds NaN: read in place, the NaN never reaches a score
    n_u, n_i, d = 40, 50, 7
    bu = torch.full((n_u, 8), float("nan"), device=DEV)
    bi = torch.full((n_i, 8), float("nan"), device=DEV)
    bu[:, :d] = _emb(n_u, d, 1)
    bi[:, :d] = _emb(n_i, d, 2)
    U, I = bu[:, :d].requires_grad_(True), bi[:, :d].requires_grad_(True)
    _, gU, gI = check_loss(gdr, U, I, *_triplets(n_u, n_i, 3000, seed=4))
    assert torch.isnan(bu[:, d]).all() and torch.isnan(bi[:, d]).all()


def test_gradients_are_bit_identical(gdr):
    U, I = _emb(500, 64, 8), _emb(700, 64, 9)
    t = _triplets(500, 700, 1 << 16, seed=10)
    a, b = check_loss(gdr, U, I, *t), check_loss(gdr, U, I, *t)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_backward_scales_by_upstream_gradient(gdr):
    U, I = _emb(50, 16, 1).requires_grad_(True), _emb(60, 16, 2).requires_grad_(True)
    t = _triplets(50, 60, 300, seed=3)
    gdr.bpr_loss(U, I, *t).backward()
    g1 = U.grad.clone(), I.grad.clone()
    U.grad = I.grad = None
    (2.5 * gdr.BPRLoss.apply(U, I, *t)).backward()
    assert torch.equal(U.grad, g1[0] * 2.5) and torch.equal(I.grad, g1[1] * 2.5)


def test_bad_inputs_raise(gdr):
    U, I = _emb(10, 8, 1), _emb(12, 8, 2)
    u, p, n = _triplets(10, 12, 64, seed=1)
    for bad in ((u.clone().fill_(10), p, n), (u, p.clone().fill_(-1), n), (u, p, n.clone().fill_(12))):
        with pytest.raises(ValueError):
            gdr.bpr_loss(U, I, *bad)
    Un = U.clone()
    Un[int(u[0]), 3] = float("nan")
    In = I.clone()
    In[int(n[5]), 0] = float("inf")
    for a, b in ((Un, I), (U, In)):
        with pytest.raises(ValueError):
            gdr.bpr_loss(a, b, u, p, n)
    e = torch.zeros(0, dtype=torch.int64, device=DEV)
    with pytest.raises(ValueError):
        gdr.bpr_loss(U, I, e, e, e)


# ---------------------------------------------------------------------------------------------------- end to end
def test_refinement_is_reproducible_and_matches_torch_bpr(gdr, shapes):
    C = shapes["yelp2018 condensed"]
    ei, ew = gdr.condensed_csr_to_edge_index(C, DEV)
    n_u, n_i = C.shape
    d, L, B, steps = 64, 2, 4096, 20
    graph = gdr.BipartiteGraph(ei, ew, n_u, n_i)
    sampler = gdr.BPRSampler(C, seed=99)
    raw0 = _inv_softplus(ew.clamp_min(0.05))

    def run(use_gdr_loss):
        u0 = _emb(n_u, d, 21).requires_grad_(True)
        i0 = _emb(n_i, d, 22).requires_grad_(True)
        raw = raw0.clone().requires_grad_(True)
        opt = torch.optim.Adam([u0, i0, raw], lr=1e-2)
        losses = []
        for s in range(steps):
            u, p, n = sampler.sample(B, s)
            uo, io = gdr.LightGCNPropagate.apply(u0, i0, F.softplus(raw), graph, L)
            loss = gdr.bpr_loss(uo, io, u, p, n) if use_gdr_loss else torch_bpr(uo, io, u, p, n)
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(float(loss))
        return losses, (u0.detach(), i0.detach(), raw.detach())

    l1, p1 = run(True)
    l2, p2 = run(True)
    assert l1 == l2 and all(torch.equal(a, b) for a, b in zip(p1, p2))
    lt, _ = run(False)
    for s, (a, b) in enumerate(zip(l1, lt)):
        assert abs(a - b) <= 1e-4 * abs(b), f"step {s}: gdr {a} vs torch {b}"
    assert l1[-1] < l1[0] and np.mean(l1[-5:]) < np.mean(l1[:5]) - 1e-3, l1
