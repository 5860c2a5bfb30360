"""CPU checks of the LightGCN edge-weight backward: the closed form the kernels implement (numpy fp64) against torch
fp64 autograd through the reference expression, and argument validation of the new entry points before any device
work.  The helpers here are shared with tests/test_gpu_lightgcn_grad.py."""
import numpy as np
import pytest
import torch

FAKE = 256   # a non-null pointer that the argument checks must reject before it is ever dereferenced
EPS = 1e-8


def random_graph(nu, ni, e, seed, hub_row=0, hub_col=0):
    """Unique (u, i) pairs with positive weights, plus: the last user row and the last item column empty, user 0 with
    all-zero weights, and optionally a hub row (user 1) / hub column (item 1) of the given lengths."""
    rs = np.random.RandomState(seed)
    keys = set()
    pairs = []

    def add(u, i):
        if (u, i) not in keys:
            keys.add((u, i))
            pairs.append((u, i))

    for u, i in zip(rs.randint(0, nu - 1, e), rs.randint(0, ni - 1, e)):
        add(int(u), int(i))
    for i in range(min(3, ni - 1)):
        add(0, i)
    for i in rs.permutation(ni - 1)[:hub_row]:
        add(1, int(i))
    for u in rs.permutation(nu - 1)[:hub_col]:
        add(int(u), 1)
    p = np.array(pairs, dtype=np.int64).reshape(-1, 2)[rs.permutation(len(pairs))]
    cu, ci = p[:, 0].copy(), p[:, 1].copy()
    w = rs.uniform(0.2, 3.0, len(cu)).astype(np.float32)
    w[cu == 0] = 0.0
    return cu, ci, w


def ref_autograd_f64(cu, ci, w, u0, i0, gu, gi, L):
    """dL/d(u0, i0, w) by torch fp64 autograd of oracle/ref_port.lightgcn_propagate, L = <gu, u_out> + <gi, i_out>.
    Runs on the device of the inputs (torch tensors or numpy arrays -> CPU)."""
    from oracle import ref_port as rp
    dev = cu.device if isinstance(cu, torch.Tensor) else torch.device("cpu")
    t = lambda a, dt: (a if isinstance(a, torch.Tensor) else torch.from_numpy(np.asarray(a))).to(dev, dt)
    old_dtype = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.device(dev):   # scoped: leaves no default-device mode behind
            W = t(w, torch.float64).requires_grad_(True)
            U = t(u0, torch.float64).requires_grad_(True)
            I = t(i0, torch.float64).requires_grad_(True)
            uo, io = rp.lightgcn_propagate(t(cu, torch.int64), t(ci, torch.int64), W, U, I, L)
            ((uo * t(gu, torch.float64)).sum() + (io * t(gi, torch.float64)).sum()).backward()
        return U.grad, I.grad, (W.grad if W.grad is not None else torch.zeros_like(W))   # L = 0: out ignores w
    finally:
        torch.set_default_dtype(old_dtype)


def closed_form_f64(cu, ci, w, u0, i0, gu, gi, L, nu, ni):
    """The math of csrc/lightgcn_grad.cu in numpy fp64: (du0, di0, dw, G)."""
    import scipy.sparse as sp
    w = w.astype(np.float64)
    du = np.bincount(cu, w, nu)
    di = np.bincount(ci, w, ni)
    ru, ri = 1.0 / np.sqrt(du + EPS), 1.0 / np.sqrt(di + EPS)
    norm = w * ru[cu] * ri[ci]
    A = sp.csr_matrix((norm, (cu, ci)), shape=(nu, ni))
    AT = A.T.tocsr()

    def layers(x_u, x_i):
        Xu, Xi = [x_u.astype(np.float64)], [x_i.astype(np.float64)]
        for _ in range(L):
            Xu.append(A @ Xi[-1])
            Xi.append(AT @ Xu[-2])
        return Xu, Xi

    Xu, Xi = layers(u0, i0)
    Yu, Yi = layers(gu, gi)
    c = 1.0 / (L + 1)
    G = np.zeros(len(cu))
    for j in range(L):
        PY = sum(Yu[: L - j])   # sum_{m <= L-1-j} Yu_m
        PX = sum(Xu[: L - j])
        G += (Xi[j][ci] * PY[cu]).sum(1) + (Yi[j][ci] * PX[cu]).sum(1)
    G *= c
    S_u = np.bincount(cu, G * norm, nu)
    S_i = np.bincount(ci, G * norm, ni)
    dw = G * ru[cu] * ri[ci] - 0.5 * S_u[cu] / (du[cu] + EPS) - 0.5 * S_i[ci] / (di[ci] + EPS)
    return c * sum(Yu), c * sum(Yi), dw, G


@pytest.mark.parametrize("L", [0, 1, 2, 3])
@pytest.mark.parametrize("seed", [0, 1])
def test_closed_form_matches_autograd(L, seed):
    nu, ni, d = 23, 17, 5
    cu, ci, w = random_graph(nu, ni, 90, seed, hub_row=12, hub_col=9)
    assert (np.bincount(cu, minlength=nu)[nu - 1] == 0) and (np.bincount(ci, minlength=ni)[ni - 1] == 0)
    rs = np.random.RandomState(100 + seed)
    u0, i0 = rs.standard_normal((nu, d)), rs.standard_normal((ni, d))
    gu, gi = rs.standard_normal((nu, d)), rs.standard_normal((ni, d))
    du0, di0, dw, _ = closed_form_f64(cu, ci, w, u0, i0, gu, gi, L, nu, ni)
    ru, ri, rw = (x.numpy() for x in ref_autograd_f64(cu, ci, w, u0, i0, gu, gi, L))
    np.testing.assert_allclose(du0, ru, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(di0, ri, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(dw, rw, rtol=1e-9, atol=1e-9 * np.abs(rw).max())
    if L == 0:
        assert not dw.any()
    else:
        assert np.abs(dw[w == 0]).max() > 0   # zero weights still get a gradient (the zero-weight row)


def test_closed_form_with_empty_graph_and_isolated_nodes():
    cu = ci = np.zeros(0, dtype=np.int64)
    w = np.zeros(0, dtype=np.float32)
    rs = np.random.RandomState(3)
    u0, i0, gu, gi = (rs.standard_normal((4, 3)) for _ in range(4))
    du0, di0, dw, _ = closed_form_f64(cu, ci, w, u0, i0, gu, gi, 2, 4, 4)
    ru, ri, _ = ref_autograd_f64(cu, ci, w, u0, i0, gu, gi, 2)
    np.testing.assert_allclose(du0, ru.numpy(), rtol=1e-12)
    np.testing.assert_allclose(di0, ri.numpy(), rtol=1e-12)
    assert dw.shape == (0,)


# ---------------------------------------------------------------------------------------- C ABI argument checks
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from gdr import _lib
    return _lib


def _locate(lib, n_rows=4, n_cols=5, nnz=6, rowptr=FAKE, colidx=FAKE, E=6, row=FAKE, col=FAKE, pos=FAKE, status=FAKE):
    return lib.call("gdr_csr_locate", n_rows, n_cols, nnz, rowptr, colidx, E, row, col, pos, status, 0)


@pytest.mark.parametrize("kw", [dict(n_rows=-1), dict(nnz=-1), dict(E=-1), dict(rowptr=0), dict(colidx=0),
                                dict(row=0), dict(col=0), dict(pos=0), dict(status=0)])
def test_locate_rejects_bad_arguments(lib, kw):
    with pytest.raises(lib.GdrError) as e:
        _locate(lib, **kw)
    assert e.value.code == -1


def _edge_grad(lib, n_u=4, n_i=5, nnz=6, rowptr=FAKE, colidx=FAKE, norm=FAKE, L=2, d=8, Xu=FAKE, Xi=FAKE, Yu=FAKE,
               Yi=FAKE, ld=8, G=FAKE, S_u=FAKE):
    return lib.call("gdr_lightgcn_edge_grad", n_u, n_i, nnz, rowptr, colidx, norm, L, d, Xu, Xi, Yu, Yi, ld, 1.0 / 3,
                    G, S_u, 0)


@pytest.mark.parametrize("kw", [dict(n_u=-1), dict(n_i=-1), dict(nnz=-1), dict(d=-1), dict(L=-1), dict(rowptr=0),
                                dict(colidx=0), dict(norm=0), dict(Xu=0), dict(Xi=0), dict(Yu=0), dict(Yi=0), dict(G=0),
                                dict(S_u=0), dict(ld=6), dict(ld=4), dict(Xu=FAKE + 4)])
def test_edge_grad_rejects_bad_arguments(lib, kw):
    with pytest.raises(lib.GdrError) as e:
        _edge_grad(lib, **kw)
    assert e.value.code == -1


def _norm_bwd(lib, n_u=4, n_i=5, nnz=6, E=6, ws_bytes=1 << 40, **ptrs):
    p = dict(rowptr=FAKE, colidx=FAKE, t_rowptr=FAKE, t_perm=FAKE, norm=FAKE, deg_u=FAKE, deg_i=FAKE, G=FAKE, S_u=FAKE,
             pos=FAKE, dw=FAKE, ws=FAKE)
    p.update(ptrs)
    return lib.call("gdr_bipartite_normalize_backward", n_u, n_i, nnz, p["rowptr"], p["colidx"], p["t_rowptr"],
                    p["t_perm"], p["norm"], p["deg_u"], p["deg_i"], EPS, p["G"], p["S_u"], E, p["pos"], p["dw"],
                    p["ws"], ws_bytes, 0)


@pytest.mark.parametrize("kw", [dict(n_u=-1), dict(n_i=-1), dict(nnz=-1), dict(E=-1), dict(nnz=0)]
                         + [{k: 0} for k in ("rowptr", "colidx", "t_rowptr", "t_perm", "norm", "deg_u", "deg_i", "G",
                                             "S_u", "pos", "dw", "ws")])
def test_normalize_backward_rejects_bad_arguments(lib, kw):
    with pytest.raises(lib.GdrError) as e:
        _norm_bwd(lib, **kw)
    assert e.value.code == -1


def test_normalize_backward_rejects_small_workspace(lib):
    need = lib.query("gdr_bipartite_normalize_backward_ws_bytes", 5, 6)
    assert need >= 5 * 8 + 6 * 4
    with pytest.raises(lib.GdrError) as e:
        _norm_bwd(lib, ws_bytes=need - 1)
    assert e.value.code == -2
