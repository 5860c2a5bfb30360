"""Stage 4's weight sums against exact cell sums (tests/coarsen_ref.py) on the inputs where fixed-point and fp32 sums go
wrong: cosine-reweighted graphs (signed, cancelling, down to exact zeros), weights over 60 binades, exact and near
cancellation, a cluster whose sum fills the 64-bit accumulator, all-zero clusters, more hub rows than hub slots and both
sides of every form switch.  Each form is held to its own bound: the shared-memory form to n*q_a/2 plus one fp32 rounding
(one ulp where the cell is large next to n*q_a), the sort form to gamma_{n-1} * sum |w|."""
import numpy as np
import pytest
import torch

import coarsen_ref as ref

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None


@pytest.fixture(scope="module")
def gdr():
    import gdr
    return gdr


# ---------------------------------------------------------------- graphs built on the host
class Case:
    """A CSR adjacency (host arrays) with a cluster label per row and per column."""

    def __init__(self, rowptr, colidx, w, labels_src, labels_dst, n_src, n_dst):
        self.rowptr, self.colidx = rowptr.astype(np.int32), colidx.astype(np.int32)
        self.w = w.astype(np.float32)
        self.ls, self.ld = labels_src.astype(np.int32), labels_dst.astype(np.int32)
        self.n_src, self.n_dst = int(n_src), int(n_dst)

    @property
    def E(self):
        return int(self.colidx.shape[0])

    def csr(self, gdr):
        t = lambda x: torch.from_numpy(x).to(DEV)  # noqa: E731
        return gdr.CSR(t(self.rowptr), t(self.colidx), t(self.w), (self.rowptr.shape[0] - 1, self.ld.shape[0]))


def _from_edges(u, v, w, n_rows):
    """CSR of the distinct (u, v) pairs (the first weight of a repeated pair), columns sorted in a row."""
    key = u.astype(np.int64) * (1 << 32) + v
    _, first = np.unique(key, return_index=True)
    u, v, w = u[first], v[first], w[first]
    o = np.lexsort((v, u))
    u, v, w = u[o], v[o], w[o]
    return np.searchsorted(u, np.arange(n_rows + 1)), v, w


def _wide(rng, n, lo=-60, hi=0):
    """+-m * 2^k, m uniform in [1, 2), k uniform in [lo, hi]: below 2 in magnitude."""
    m = (1.0 + rng.rand(n)).astype(np.float32)
    return (m * np.ldexp(1.0, rng.randint(lo, hi + 1, n)) * rng.choice([-1.0, 1.0], n)).astype(np.float32)


def _square(u, v, w, labels, k):
    rp, ci, ww = _from_edges(u, v, w, labels.shape[0])
    return Case(rp, ci, ww, labels, labels, k, k)


def case_wide(seed=2):
    """Each cluster: a weight-1 self-loop, signed weights +-m * 2^k with k in [-60, 0]; some cells hold tiny weights only."""
    rng = np.random.RandomState(seed)
    n, k, m = 6000, 60, 150000
    lab = rng.randint(0, k, n)
    lab[:k] = np.arange(k)
    u, v = rng.randint(0, n, m), rng.randint(0, n, m)
    w = _wide(rng, m)
    tiny = ((lab[u] * 7 + lab[v]) % 5) == 0                   # a fifth of the cells: only weights below 2^-40
    w[tiny] = _wide(rng, int(tiny.sum()), -60, -40)
    u, v, w = np.concatenate([np.arange(k), u]), np.concatenate([np.arange(k), v]), np.concatenate([np.ones(k), w])
    return _square(u, v, w, lab, k)


def case_cancel(seed=3):
    """Cells made only of pairs +-w of one magnitude (exact partial sums: must come out +0.0), cells of near-cancelling
    pairs w, -w(1 - 2^-23), and ordinary signed cells around them."""
    rng = np.random.RandomState(seed)
    k, per = 24, 120
    n = k * per
    lab = np.arange(n) % k
    members = [np.flatnonzero(lab == a) for a in range(k)]
    us, vs, ws, zero_cells = [], [], [], []
    for a in range(k):
        for b in range(k):
            kind = (a * 5 + b) % 3
            p = int(rng.randint(1, 30))
            pick = rng.choice(per * per, 2 * p, replace=False)
            u, v = members[a][pick // per], members[b][pick % per]
            if kind == 0:                                          # +-w, |w| with 16 significant bits
                mag = np.float32((1 + rng.randint(0, 1 << 15) / 2.0 ** 15) * 2.0 ** rng.randint(-30, 1))
                w = np.repeat(np.array([mag, -mag], dtype=np.float32), p)
                zero_cells.append((a, b))
            elif kind == 1:                                        # w, -w (1 - 2^-23)
                w = _wide(rng, p, -30, 0)
                w = np.stack([w, -(w * np.float32(1 - 2.0 ** -23))], 1).reshape(-1)
            else:
                w = _wide(rng, 2 * p, -30, 0)
            us.append(u), vs.append(v), ws.append(w)
    c = _square(np.concatenate(us), np.concatenate(vs), np.concatenate(ws).astype(np.float32), lab, k)
    c.zero_cells = zero_cells
    return c


SAT = [(0x3F7FFFFF, (1 << 14) - 1, 1), (0x3F7FFFFF, 1 << 14, 1), (0x3F7FFFFF, (1 << 14) - 1, -1), (0x3F7FFFFF, 1 << 14, -1),
       (0x497FFFFF, (1 << 14) - 1, 1), (0x497FFFFF, 1 << 14, 1), (0x497FFFFF, (1 << 14) - 1, -1), (0x497FFFFF, 1 << 14, -1)]


def case_saturate():
    """Every edge of cluster a goes to the one cell (a, a + 8), all of weight +-w: n*|w| fills the 64-bit fixed-point sum
    to within a factor 2 of its range, every term is an exact multiple of q, so the sum must be exactly fl32(n*w).  With
    -0x497fffff the cluster's largest |w| belongs to a negative weight above 1."""
    per = 128
    lab = np.repeat(np.arange(2 * len(SAT)), per)
    us, vs, ws = [], [], []
    for a, (bits, cnt, sign) in enumerate(SAT):
        w = sign * np.array([bits], dtype=np.uint32).view(np.float32)[0]
        src, dst = a * per, (a + len(SAT)) * per
        pick = np.arange(cnt)
        us.append(src + pick // per), vs.append(dst + pick % per), ws.append(np.full(cnt, w, dtype=np.float32))
    c = _square(np.concatenate(us), np.concatenate(vs), np.concatenate(ws), lab, 2 * len(SAT))
    c.expect = {(a, a + len(SAT)): np.float32(float(cnt) * float(sign * np.array([bits], np.uint32).view(np.float32)[0]))
                for a, (bits, cnt, sign) in enumerate(SAT)}
    return c


def case_zeros(seed=5):
    """Cluster 0: weights +0.0 only (max |w| = 0); cluster 1: -0.0 only; cluster 2: both; cluster 3: ordinary weights."""
    rng = np.random.RandomState(seed)
    k, n, m = 4, 800, 20000
    lab = np.arange(n) % k
    u, v = rng.randint(0, n, m), rng.randint(0, n, m)
    w = _wide(rng, m, -20, 0)
    w[lab[u] == 0] = 0.0
    w[lab[u] == 1] = -0.0
    w[lab[u] == 2] = np.where(rng.rand(int((lab[u] == 2).sum())) < 0.5, 0.0, -0.0)
    return _square(u, v, w, lab, k)


def case_hubs(seed=6):
    """Cluster 0 holds 70 rows of >= 4096 edges — more than the 64 hub slots of a CTA — and cluster 1 rows of exactly
    4095 and 4096 edges (CD_HUB); ordinary rows around them."""
    rng = np.random.RandomState(seed)
    k, n = 40, 6000
    lab = rng.randint(2, k, n)
    hub_rows, edge_rows = np.arange(70), np.array([70, 71, 72, 73])
    lab[hub_rows], lab[edge_rows] = 0, 1
    us, vs = [], []
    for r, d in [(r, 4096 + int(rng.randint(0, 200))) for r in hub_rows] + list(zip(edge_rows, [4095, 4096, 4095, 4096])):
        us.append(np.full(d, r)), vs.append(rng.choice(n, d, replace=False))
    m = 60000
    us.append(rng.randint(74, n, m)), vs.append(rng.randint(0, n, m))
    u, v = np.concatenate(us), np.concatenate(vs)
    return _square(u, v, _wide(rng, u.shape[0], -30, 0), lab, k)


def case_threshold(n_src, n_dst, E, seed=7):
    """n_src one-row clusters, column labels in [0, n_dst), E edges.  Row 0 carries two probe cells that tell the forms
    apart: cell (0, 0) = 1.0 then 63 x 2^-26 (a sequential fp32 sum drops all 63, 8 ulps; the fixed-point sum does not)
    and cell (0, 1) = one edge of 1e-13 (exact in fp32; the fixed-point step of cluster 0 is coarser)."""
    rng = np.random.RandomState(seed)
    M = n_dst + 63
    ld = np.concatenate([np.zeros(64, np.int64), [1], 2 + rng.permutation(M - 65) % (n_dst - 2)])
    probe_w = np.concatenate([[1.0], np.full(63, 2.0 ** -26), [1e-13]]).astype(np.float32)
    rest = E - 65
    u = np.concatenate([np.zeros(65, np.int64), 1 + np.arange(rest) % (n_src - 1)])
    v = np.concatenate([np.arange(65), 65 + rng.choice(M - 65, rest, replace=False)])
    w = np.concatenate([probe_w, _wide(rng, rest, -30, -1)])
    rp, ci, ww = _from_edges(u, v, w, n_src)
    assert ci.shape[0] == E
    return Case(rp, ci, ww, np.arange(n_src), ld, n_src, n_dst)


def case_cosine(gdr, seed=1):
    """A normalised skewed graph reweighted by the cosine of its end points' embeddings (cosine_reweight): integer
    orthogonal rows (cos exactly 0), nearly orthogonal ones (|cos| 1e-9 .. 1e-5), opposite ones (cos -1), random ones."""
    from gdr import synth
    n, k = 6000, 50
    u, v = synth.skewed_graph(n, 60000, seed=seed)
    A = gdr.sym_normalize(gdr.coo_to_csr(torch.from_numpy(u).to(DEV), torch.from_numpy(v).to(DEV), None, (n, n),
                                         symmetrize=True, binarize=True), 2)
    rng = np.random.RandomState(seed)
    e = rng.randn(n, 4).astype(np.float32)
    kind = np.arange(n) % 5
    e[kind == 0] = [2, 0, 0, 0]
    e[kind == 1] = [0, 3, 0, 0]
    eps = 10.0 ** rng.uniform(-9, -5, n) * rng.choice([-1.0, 1.0], n)
    e[kind == 2] = np.stack([eps, np.zeros(n), np.ones(n), np.zeros(n)], 1)[kind == 2]
    e[kind == 3] = [-1, 0, 0, 0]
    ebd = torch.from_numpy(e).to(DEV)
    labels = rng.randint(0, k, n).astype(np.int32)
    labels[:k] = np.arange(k)
    return A, ebd, labels, k


def _host(gdr, A, labels, k):
    return Case(A.rowptr.cpu().numpy(), A.colidx.cpu().numpy(), A.vals.cpu().numpy(), labels, labels, k, k)


# ---------------------------------------------------------------- checks
def _dense_selected(c, has_w, dense_flag):
    """cd_applicable: CSR input, the coarse row in shared memory, at least 4 edges per coarse row."""
    return bool(dense_flag) and c.n_dst * (12 if has_w else 4) <= ref.SMEM_BYTES and c.E >= 4 * c.n_src


def _coarsen(gdr, c, dense, drop, weights=True, coo=False):
    from gdr import _lib
    A = c.csr(gdr)
    ls, ld = torch.from_numpy(c.ls).to(DEV), torch.from_numpy(c.ld).to(DEV)
    _lib.call("gdr_debug_set", b"coarsen_dense", int(dense))
    try:
        if coo:
            src = torch.repeat_interleave(torch.arange(A.shape[0], device=DEV), (A.rowptr[1:] - A.rowptr[:-1]).long())
            out = gdr.coarsen_edges(ls, ld, c.n_src, c.n_dst, src=src, dst=A.colidx.long(), weights=A.vals, drop_diag=drop)
        else:
            out = gdr.coarsen_edges(ls, ld, c.n_src, c.n_dst, csr=A, weights=A.vals if weights else None, drop_diag=drop)
        torch.cuda.synchronize()
    finally:
        _lib.call("gdr_debug_set", b"coarsen_dense", 1)
    return [None if x is None else x.cpu().numpy() for x in out]


def _check_structure(got, r, n_src):
    rp, ci, cnt = got[0], got[1], got[2]
    assert np.array_equal(rp, np.searchsorted(r["a"], np.arange(n_src + 1))), "stored cells differ from the cells with edges"
    assert np.array_equal(ci, r["b"]) and np.array_equal(cnt, r["count"]), "cell columns or counts differ"


def _within(got, S, bound, what):
    err = np.abs(got.astype(np.float64) - S)
    bad = np.flatnonzero(err > bound)
    assert bad.size == 0, (f"{what}: {bad.size} cells outside the bound, e.g. cell {bad[0]}: got {got[bad[0]]!r}, "
                           f"exact {S[bad[0]]!r}, error {err[bad[0]]:.3e} > {bound[bad[0]]:.3e}")


def _check_dense_sums(got, r, q, what):
    S, n = r["sum"], r["count"]
    _within(got, S, ref.dense_bound(S, n, q), what + " (shared-memory bound)")
    one = ref.one_ulp_regime(S, n, q)
    _within(got[one], S[one].astype(np.float32).astype(np.float64), ref.ulp32(S[one]), what + " (one ulp where n*q/2 <= ulp/4)")


def check_case(gdr, c, drop_list=(True, False)):
    """Both forms, drop_diag on and off: structure and counts exact, sums within the bound of the form the dispatch
    selects, the shared-memory sums bit-reproducible.  Returns {(form, drop): (got sums, reference cells, q per cell)}."""
    out = {}
    for drop in drop_list:
        r = ref.csr_cells(c.rowptr, c.colidx, c.w, c.ls, c.ld, drop)
        q = ref.steps(c.rowptr, c.w, c.ls, c.n_src)[r["a"]]
        for dense in (1, 0):
            got = _coarsen(gdr, c, dense, drop)
            _check_structure(got, r, c.n_src)
            form = "dense" if _dense_selected(c, True, dense) else "sort"
            what = f"{form} form, drop_diag={drop}"
            if form == "dense":
                _check_dense_sums(got[3], r, q, what)
                again = _coarsen(gdr, c, dense, drop)
                assert np.array_equal(again[3].view(np.uint32), got[3].view(np.uint32)), "shared-memory sums not reproducible"
            else:
                _within(got[3], r["sum"], ref.sort_bound(r["count"], r["abs_sum"]), what + " (sort bound)")
            out[(form, drop)] = (got[3], r, q)
        counts_only = _coarsen(gdr, c, 1, drop, weights=False)
        assert counts_only[3] is None
        _check_structure(counts_only, r, c.n_src)
    return out


def _cell_value(res, a, b):
    got, r, _ = res
    i = np.flatnonzero((r["a"] == a) & (r["b"] == b))
    assert i.size == 1, f"cell ({a}, {b}) not stored"
    return got[i[0]]


# ---------------------------------------------------------------- 1. cosine-reweighted graphs
def test_cosine_reweighted_graphs(gdr, oracle):
    A, ebd, labels, k = case_cosine(gdr)
    R = gdr.cosine_reweight(A, ebd)
    w = R.vals.cpu().numpy()
    assert (w == 0).sum() > 1000 and (w < 0).sum() > 1000 and ((w != 0) & (np.abs(w) < 1e-6)).sum() > 1000
    graphs = [R] + [gdr.CSR.from_torch_coo(t) for t in gdr.graph_sparse(A, 0.5, ebd=ebd, sp_type="single")]
    graphs += [gdr.CSR.from_torch_coo(t) for t in gdr.graph_sparse(A, 0.5, ebd=ebd, sp_type="attaw")]
    for G in graphs:
        check_case(gdr, _host(gdr, G, labels, k))
    # graph_compress end to end, against the exact cells and against the fp64 dense reference
    lab_d = torch.from_numpy(labels).to(DEV)
    syn_list, syn = gdr.graph_compress(lab_d, A, graphs[1:])
    sizes = np.bincount(labels, minlength=k).astype(np.float64)
    for G, T in zip(graphs[1:] + [A], syn_list + [syn]):
        c = _host(gdr, G, labels, k)
        r = ref.csr_cells(c.rowptr, c.colidx, c.w, labels, labels, drop_diag=True)
        q = ref.steps(c.rowptr, c.w, labels, k)[r["a"]]
        cell_bound = ref.dense_bound(r["sum"], r["count"], q) if _dense_selected(c, True, 1) else \
            ref.sort_bound(r["count"], r["abs_sum"])
        na, nb = sizes[r["a"]], sizes[r["b"]]
        bound = ref.scale_bound(cell_bound, r["sum"], na, nb)
        idx, val = T._indices().cpu().numpy(), T._values().cpu().numpy()
        o = np.lexsort((idx[1], idx[0]))
        idx, val = idx[:, o], val[o]
        assert np.array_equal(idx[0], r["a"]) and np.array_equal(idx[1], r["b"]), "graph_compress stores other cells"
        _within(val, r["sum"] / (na * nb), bound, "graph_compress")
        dense = oracle.graph_compress_dense(labels.astype(np.int64), c.rowptr, c.colidx, c.w, k)
        slack = (r["count"] + 3) * 2.0 ** -53 * r["abs_sum"] / (na * nb)      # the fp64 reference's own rounding
        _within(val, dense[r["a"], r["b"]], bound + slack, "graph_compress against the fp64 dense reference")


# ---------------------------------------------------------------- 2. weights over 60 binades
def test_wide_range_weights(gdr):
    c = case_wide()
    res = check_case(gdr, c)
    got, r, q = res[("dense", True)]
    S = r["sum"]
    assert np.any(~ref.one_ulp_regime(S, r["count"], q))
    # the corrected bound is the one that applies: some cells are more than one ulp from the exact sum
    assert np.any(np.abs(got.astype(np.float64) - S.astype(np.float32).astype(np.float64)) > ref.ulp32(S))


# ---------------------------------------------------------------- 3. cancellation
def test_cancelling_pairs(gdr):
    c = case_cancel()
    res = check_case(gdr, c)
    for key, val in res.items():
        for a, b in c.zero_cells:
            if key[1] and a == b:
                continue
            v = _cell_value(val, a, b)
            assert v.view(np.uint32) == 0, f"{key}: cell ({a}, {b}) of pairs +-w is {v!r}, not +0.0"
    # graph_compress keeps such a cell as an explicit +0.0 (a dense reference's .to_sparse() would drop it)
    _, syn = gdr.graph_compress(torch.from_numpy(c.ls).to(DEV), c.csr(gdr), [])
    idx, val = syn._indices().cpu().numpy(), syn._values().cpu().numpy()
    stored = {(int(a), int(b)): v for a, b, v in zip(idx[0], idx[1], val)}
    for a, b in c.zero_cells:
        if a != b:
            assert (a, b) in stored and stored[(a, b)].view(np.uint32) == 0


# ---------------------------------------------------------------- 4. a full 64-bit accumulator
def test_saturated_fixed_point_sum(gdr):
    c = case_saturate()
    res = check_case(gdr, c)
    for drop in (True, False):
        got = res[("dense", drop)]
        for (a, b), want in c.expect.items():
            v = _cell_value(got, a, b)
            assert v == want, f"cell ({a}, {b}): {v!r}, want fl32(n*w) = {want!r}"


# ---------------------------------------------------------------- 5. zeros
def test_zero_and_negative_zero_weights(gdr):
    c = case_zeros()
    res = check_case(gdr, c)
    for (form, drop), (got, r, _) in res.items():
        z = r["a"] < 3
        assert z.any() and np.all(got[z].view(np.uint32) == 0), f"{form} form: a cell of +-0.0 weights is not +0.0"


# ---------------------------------------------------------------- 6. hub rows
def test_more_hub_rows_than_hub_slots(gdr):
    c = case_hubs()
    assert (np.diff(c.rowptr)[:70] >= 4096).all() and list(np.diff(c.rowptr)[70:74]) == [4095, 4096, 4095, 4096]
    check_case(gdr, c)


# ---------------------------------------------------------------- 7. form thresholds
def _form_of(res):
    """Which form produced these sums, from the probe cells of case_threshold."""
    got, r, q = res
    i0, i1 = [int(np.flatnonzero((r["a"] == 0) & (r["b"] == b))[0]) for b in (0, 1)]
    fits_dense = all(abs(float(got[i]) - r["sum"][i]) <= ref.dense_bound(r["sum"][i], r["count"][i], q[i]) for i in (i0, i1))
    fits_sort = all(abs(float(got[i]) - r["sum"][i]) <= ref.sort_bound(r["count"][i], r["abs_sum"][i]) for i in (i0, i1))
    assert fits_dense != fits_sort, "the probe cells do not tell the forms apart"
    return "dense" if fits_dense else "sort"


@pytest.mark.parametrize("n_src,n_dst,E", [(8, 17066, 4000), (8, 17067, 4000), (40, 100, 159), (40, 100, 160)])
def test_form_switch_with_weights(gdr, n_src, n_dst, E):
    c = case_threshold(n_src, n_dst, E)
    res = check_case(gdr, c, drop_list=(False,))
    want = "dense" if _dense_selected(c, True, 1) else "sort"
    assert want == ("dense" if (n_dst, E) in [(17066, 4000), (100, 160)] else "sort")
    assert (want, False) in res and _form_of(res[(want, False)]) == want


@pytest.mark.parametrize("n_dst", [51200, 51201])
def test_form_switch_counts_only(gdr, n_dst):
    c = case_threshold(8, n_dst, 4000)
    for drop in (True, False):
        r = ref.csr_cells(c.rowptr, c.colidx, None, c.ls, c.ld, drop)
        for dense in (1, 0):
            got = _coarsen(gdr, c, dense, drop, weights=False)
            assert got[3] is None
            _check_structure(got, r, c.n_src)


# ---------------------------------------------------------------- 8. COO input with weights (always the sort form)
@pytest.mark.parametrize("make", [case_wide, case_cancel])
def test_coo_input_with_weights(gdr, make):
    c = make()
    for drop in (True, False):
        r = ref.csr_cells(c.rowptr, c.colidx, c.w, c.ls, c.ld, drop)
        got = _coarsen(gdr, c, 1, drop, coo=True)
        _check_structure(got, r, c.n_src)
        _within(got[3], r["sum"], ref.sort_bound(r["count"], r["abs_sum"]), f"COO input, drop_diag={drop}")


# ---------------------------------------------------------------- 9. owner-side merge of the multi-GPU form
@pytest.mark.parametrize("which", ["cosine", "wide", "cancel", "saturate"])
def test_owner_side_merge(gdr, which):
    """The pairs gdr_coarsen_route addresses to each owner of a key range, merged in shared memory with the global
    per-cluster step (bit-identical to the single-GPU rows) and by the sort (within the sort bound), worlds 2, 3, 5."""
    from gdr import _lib
    from gdr import parallel as par
    if which == "cosine":
        A, ebd, labels, k = case_cosine(gdr)
        c = _host(gdr, gdr.cosine_reweight(A, ebd), labels, k)
    else:
        c = {"wide": case_wide, "cancel": case_cancel, "saturate": case_saturate}[which]()
    A = c.csr(gdr)
    k = c.n_src
    labels = torch.from_numpy(c.ls).to(DEV)
    single = _coarsen(gdr, c, 1, True)
    assert _dense_selected(c, True, 1)
    r = ref.csr_cells(c.rowptr, c.colidx, c.w, c.ls, c.ld, True)
    ops = par.CudaOps()
    stats = ops.cluster_stats(A, labels, k)
    for world in (2, 3, 5):
        keys, w, counts = ops.coarsen_route(A, labels, labels, k, world)
        cr = (k + world - 1) // world
        off = 0
        for rank in range(world):
            a_lo = min(k, rank * cr)
            n_rows = min(k, a_lo + cr) - a_lo
            seg_k, seg_w = keys[off: off + counts[rank]], w[off: off + counts[rank]]
            off += counts[rank]
            if n_rows == 0:
                continue
            d = [x.cpu().numpy() for x in ops.coarse_merge_edges(seg_k, seg_w, a_lo, n_rows, k, stats=stats)]
            _lib.call("gdr_debug_set", b"coarsen_dense", 0)
            try:
                s = [x.cpu().numpy() for x in ops.coarse_merge_edges(seg_k, seg_w, a_lo, n_rows, k, stats=stats)]
            finally:
                _lib.call("gdr_debug_set", b"coarsen_dense", 1)
            b, e = int(single[0][a_lo]), int(single[0][a_lo + n_rows])
            for x in (d, s):
                assert np.array_equal(x[0] + b, single[0][a_lo: a_lo + n_rows + 1])
                assert np.array_equal(x[1], single[1][b:e]) and np.array_equal(x[2], single[2][b:e])
            assert np.array_equal(d[3].view(np.uint32), single[3][b:e].view(np.uint32)), \
                f"world {world}, rank {rank}: shared-memory merge differs from one GPU"
            _within(s[3], r["sum"][b:e], ref.sort_bound(r["count"][b:e], r["abs_sum"][b:e]), f"sort merge, world {world}")
