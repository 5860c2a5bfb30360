"""The oracle (oracle/oracle.py + oracle.c) against the golden vectors produced by the
reference's own functions (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

from conftest import golden


def csr_from(o, g, prefix="in_", n=None):
    n = int(g["n"]) if n is None else n
    return o.coo_to_csr(g[prefix + "row"], g[prefix + "col"], g[prefix + "val"], (n, n))


def test_csr_build_duplicates_summed(oracle):
    g = golden("csr_build.npz")
    n = int(g["n"])
    rp, ci, v = oracle.coo_to_csr(g["row"], g["col"], None, (n, n))
    assert np.array_equal(rp, g["a_indptr"]) and np.array_equal(ci, g["a_indices"])
    assert np.array_equal(v, g["a_data"])
    assert v.max() > 1  # the fixture really has duplicates


def test_csr_build_symmetrize_binarize(oracle):
    g = golden("csr_build.npz")
    n = int(g["n"])
    rp, ci, v = oracle.coo_to_csr(g["row"], g["col"], None, (n, n), symmetrize=True, binarize=True)
    assert np.array_equal(rp, g["b_indptr"]) and np.array_equal(ci, g["b_indices"])
    assert np.array_equal(v, g["b_data"])


def test_recsys_builders_subset(oracle):
    g = golden("recsys_ali_subset.npz")
    nu, ni = int(g["nu"]), int(g["ni"])
    rp, ci, v = oracle.coo_to_csr(g["u"], g["i"], None, (nu, ni))
    assert np.array_equal(rp, g["r_indptr"]) and np.array_equal(ci, g["r_indices"]) and np.array_equal(v, g["r_data"])
    rp, ci, cnt, _ = oracle.coarsen_counts(g["u"], g["i"], g["u2cu"], g["i2ci"], 211, 97)
    assert np.array_equal(rp, g["c_indptr"]) and np.array_equal(ci, g["c_indices"])
    assert np.array_equal(cnt.astype(np.float32), g["c_data"])
    assert cnt.sum() == g["u"].shape[0]  # counts LINES, duplicates included (distill_recsys.py:184-201)


@pytest.mark.parametrize("case", ["plain", "loop0", "isolated", "loop0_isolated", "weighted"])
def test_sym_normalize(oracle, case):
    g = golden(f"normalize_{case}.npz")
    n = int(g["n"])
    rp, ci, v = csr_from(oracle, g)
    rpo, cio, vo, _ = oracle.sym_normalize(rp, ci, v, n, self_loop_mode=2)
    rows = np.repeat(np.arange(n), np.diff(rpo))
    assert np.array_equal(np.stack([rows, cio]), g["out_idx"])
    if case in ("plain", "isolated"):          # +I path: fp64 arithmetic, bit-exact
        assert np.array_equal(vo, g["out_val"])
    else:                                       # fp32 path / float weights: 1 ulp
        np.testing.assert_allclose(vo, g["out_val"], rtol=2e-7, atol=0)


def test_sym_normalize_dense(oracle):
    g = golden("normalize_dense.npz")
    np.testing.assert_allclose(oracle.sym_normalize_dense(g["a"]), g["out"], rtol=3e-7, atol=0)


def test_propagate(oracle):
    g = golden("propagate.npz")
    n = int(g["n"])
    rp, ci, v = csr_from(oracle, g)
    rpo, cio, vo, _ = oracle.sym_normalize(rp, ci, v, n)
    prop, target = oracle.propagate(rpo, cio, vo, g["x"], int(g["T"]), float(g["alpha"]))
    scale = np.abs(g["x"]).max()
    np.testing.assert_allclose(prop, g["prop"], rtol=1e-5, atol=1e-6 * scale)
    np.testing.assert_allclose(target, g["target"], rtol=1e-5, atol=1e-6 * scale)
    p64, t64 = oracle.propagate_f64(rpo, cio, vo, g["x"], int(g["T"]), float(g["alpha"]))
    np.testing.assert_allclose(target, t64, rtol=1e-5, atol=1e-6 * scale)


def test_kmeans_single_iteration(oracle):
    g = golden("kmeans.npz")
    res = oracle.kmeans_fit(g["x"], g["c0"], max_iter=1, tol=0)
    assert np.array_equal(res["labels"], g["it1_labels"])
    np.testing.assert_allclose(res["centers"], g["it1_centers"], rtol=1e-5, atol=1e-6)
    assert abs(res["inertia"] - float(g["it1_inertia"])) <= 1e-4 * float(g["it1_inertia"])


def test_kmeans_full_fit(oracle):
    g = golden("kmeans.npz")
    res = oracle.kmeans_fit(g["x"], g["c0"], max_iter=300, tol=1e-4)
    assert res["n_iter"] == int(g["fit_n_iter"])
    assert np.array_equal(res["labels"], g["fit_labels"])
    np.testing.assert_allclose(res["centers"], g["fit_centers"], rtol=1e-5, atol=1e-5)
    assert abs(res["inertia"] - float(g["fit_inertia"])) <= 1e-4 * float(g["fit_inertia"])
    res0 = oracle.kmeans_fit(g["x"], g["c0"], max_iter=12, tol=0)
    assert res0["n_iter"] == int(g["tol0_n_iter"])
    assert np.array_equal(res0["labels"], g["tol0_labels"])


def test_kmeans_margin_contract(oracle):
    g = golden("kmeans.npz")
    x = g["x"] - g["x"].mean(axis=0)
    c = g["c0"] - g["x"].mean(axis=0)
    labels, _ = oracle.kmeans_assign(x, c)
    ok, n_band, n_bad = oracle.labels_match(labels, x, c)
    assert ok and n_bad == 0


def test_kmeans_empty_cluster_relocation(oracle):
    g = golden("kmeans.npz")
    res = oracle.kmeans_fit(g["x"], g["c0_empty"], max_iter=1, tol=0)
    # relocation picks the farthest samples; sklearn's order inside the top set is unspecified
    # (argpartition), so compare the SET of centres and the inertia.
    a = np.sort(res["centers"].round(4), axis=0)
    b = np.sort(g["empty_centers"].round(4), axis=0)
    np.testing.assert_allclose(a, b, rtol=1e-4, atol=1e-4)
    assert abs(res["inertia"] - float(g["empty_inertia"])) <= 1e-4 * float(g["empty_inertia"])


def test_kmeans_empty_clusters_filled_in_place(oracle):
    """More clusters than distinct rows: relocation is skipped (all distances zero) and sklearn's in-place
    _average_centers gives an empty cluster BELOW the largest one that cluster's raw sum, one above it the mean."""
    g = golden("kmeans_edge.npz")
    for it in (1, 2, 5):
        res = oracle.kmeans_fit(g["x"], g["c0"], max_iter=it, tol=0)
        assert res["n_iter"] == int(g[f"it{it}_n_iter"])
        assert np.array_equal(res["labels"], g[f"it{it}_labels"])
        np.testing.assert_allclose(res["centers"], g[f"it{it}_centers"], rtol=1e-5, atol=2e-6)


def test_standard_scaler(oracle):
    g = golden("standard_scaler.npz")
    np.testing.assert_allclose(oracle.standard_scale(g["x"]), g["out"], rtol=1e-6, atol=1e-6)


def test_cluster_means_and_graph_compress(oracle):
    g = golden("graph_compress.npz")
    n = int(g["n"])
    rp, ci, v = csr_from(oracle, g)
    rpo, cio, vo, _ = oracle.sym_normalize(rp, ci, v, n)
    labels = g["labels"].astype(np.int64)
    means = oracle.cluster_means(g["feat"], labels, 20)
    assert np.isnan(means[13]).all() and np.isnan(g["means"][13]).all()  # empty cluster -> NaN row
    ok = ~np.isnan(g["means"])
    np.testing.assert_allclose(means[ok], g["means"][ok], rtol=1e-5, atol=1e-6)
    k = int(labels.max()) + 1
    S = oracle.graph_compress_dense(labels, rpo, cio, vo, k)
    ref = g["syn_dense"]
    fin = np.isfinite(ref)
    np.testing.assert_allclose(S[fin], ref[fin], rtol=1e-5, atol=1e-8)
    # the count/sum form used by the kernel gives the same matrix
    rows = np.repeat(np.arange(n), np.diff(rpo))
    rpc, cic, cnt, wsum = oracle.coarsen_counts(rows, cio, labels, labels, k, k, w=vo, drop_diag=True)
    sizes = np.bincount(labels, minlength=k).astype(np.float64)
    rr = np.repeat(np.arange(k), np.diff(rpc))
    S2 = np.zeros((k, k))
    S2[rr, cic] = wsum / sizes[rr] / sizes[cic]
    np.testing.assert_allclose(S2[fin], ref[fin], rtol=1e-5, atol=1e-8)


def test_lightgcn_propagate(oracle):
    g = golden("lightgcn.npz")
    ei = g["edge_index"]
    rp, ci, w = oracle.coo_to_csr(ei[0], ei[1], g["w"], (g["u0"].shape[0], g["i0"].shape[0]))
    u, i = oracle.lightgcn_propagate(rp, ci, w, g["u0"], g["i0"], int(g["layers"]))
    np.testing.assert_allclose(u, g["u_out"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(i, g["i_out"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("k", [25, 60, 200])
def test_kmeans_plusplus_matches_sklearn(oracle, k):
    g = golden("kmeans_plusplus.npz")
    seed = int(g[f"k{k}_seed"])
    for dt in (np.float32, np.float64):
        c, idx = oracle.kmeans_plusplus(g["x"], k, np.random.RandomState(seed), cumsum_dtype=dt)
        assert np.array_equal(idx, g[f"k{k}_indices"])
        assert np.array_equal(c, g[f"k{k}_centers"])


# ---------------------------------------------------------------- SURVEY §8f item 1: sparsification
def _sparsify_case():
    g = golden("sparsify.npz")
    n = int(g["n"])
    rp = np.zeros(n + 1, np.int64)
    np.add.at(rp, g["src"] + 1, 1)
    return g, n, np.cumsum(rp).astype(np.int32), g["dst"].astype(np.int32), g["val"]


def _edge_set(rp, ci):
    rows = np.repeat(np.arange(rp.shape[0] - 1), np.diff(rp))
    return set(zip(rows.tolist(), ci.tolist()))


def test_er_estimator_matches_reference(oracle):
    g, n, rp, ci, va = _sparsify_case()
    assert np.array_equal(oracle.er_lower(rp, ci, va), g["er"])                 # utils_clustgdd.ER_estimator, bit-exact
    er_att, rew = oracle.attaw_er_lower(rp, ci, va, g["ebd"])                   # attaw_ER_estimator
    np.testing.assert_allclose(rew, g["rew_val"], rtol=0, atol=2e-7 * np.abs(va).max())
    # degrees of the re-weighted graph are sums with cancellation: compare against their magnitude
    np.testing.assert_allclose(er_att, g["er_att"], rtol=1e-3, atol=1e-4 * np.abs(g["er_att"]).max())


def test_graph_sparse_matches_reference(oracle):
    g, n, rp, ci, va = _sparsify_case()
    ratio = float(g["ratio"])
    k = int(va.shape[0] * ratio)
    for tag, tp in (("van", "vanilla"), ("sin", "single")):
        rpo, cio, vo = oracle.graph_sparse(rp, ci, va, ratio, ebd=g["ebd"], sp_type=tp)[0]
        assert cio.shape[0] == k
        ref = set(zip(g[tag + "_row"].tolist(), g[tag + "_col"].tolist()))
        assert len(_edge_set(rpo, cio) ^ ref) <= 2        # only edges AT the threshold may differ (ties / last-bit weights)
    gl = oracle.graph_sparse(rp, ci, va, ratio, ebd=g["ebd"], sp_type="attaw")
    assert len(gl) == int(g["C"])
    for i, (rpo, cio, vo) in enumerate(gl):
        ref = set(zip(g[f"att{i}_row"].tolist(), g[f"att{i}_col"].tolist()))
        assert cio.shape[0] == k and len(_edge_set(rpo, cio) ^ ref) <= 4


def test_topk_edges_ties_take_first_in_index_order(oracle):
    w = np.array([1, 3, 3, 2, 3, 0, 3], np.float32)
    assert oracle.topk_edges(w, 3).tolist() == [1, 2, 4]
    assert oracle.topk_edges(w, 5).tolist() == [1, 2, 3, 4, 6]
    assert oracle.topk_edges(w, 0).tolist() == []
