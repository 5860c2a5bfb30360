"""Tensor-core (tcgen05 3xTF32 + exact re-score) E-step against the oracle.  GPU only."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gdr():
    import gdr as g
    assert torch.cuda.is_available()
    return g


DEV = "cuda:0"


def np_(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("N,K,D", [(128, 128, 32), (300, 7, 3), (5000, 140, 7), (4099, 129, 100), (20000, 1000, 40),
                                   (20000, 333, 128), (1, 1, 1)])
def test_tc_assign_vs_oracle(gdr, oracle, N, K, D):
    from gdr import synth
    from gdr._dev import padded_rows
    from gdr.kmeans import TcOperand
    X = synth.clustered_features(N, D, max(2, K // 3), seed=N + K)
    X -= X.mean(axis=0)
    C = synth.kmeans_init(X, K, seed=1)
    Xd, Cd = padded_rows(torch.from_numpy(X).to(DEV)), padded_rows(torch.from_numpy(C).to(DEV))
    op = TcOperand(Xd)
    labels = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    best = torch.full((N,), float("nan"), dtype=torch.float32, device=DEV)
    n_ref = torch.zeros(1, dtype=torch.int32, device=DEV)
    gdr.assign_labels(Xd, Cd, labels, best=best, tc_operand=op, n_refined=n_ref)
    torch.cuda.synchronize()
    lab = np_(labels)
    assert lab.min() >= 0 and lab.max() < K
    ok, n_band, n_bad = oracle.labels_match(lab, X, C, band=1e-6)
    assert ok, f"{n_bad} rows outside the 1e-6 margin band disagree with the exact argmin"
    l32, b32 = oracle.kmeans_assign(X, C)
    np.testing.assert_allclose(np_(best), b32, rtol=1e-4, atol=1e-4 * max(1.0, np.abs(b32).max()))
    # the screen must decide most rows on its own (refine set small on well-separated data)
    assert int(n_ref.item()) <= max(64, N // 5)
    # and the result equals the exact-fp32 kernel's labels
    lab32 = torch.empty(N, dtype=torch.int32, device=DEV)
    gdr.assign_labels(Xd, Cd, lab32)
    assert np.array_equal(np_(lab32), lab)


@pytest.fixture
def screen_mode():
    """Force a tensor-core screen variant (gdr_debug_set "tc_screen"); reset to auto afterwards."""
    from gdr import _lib
    yield lambda v: _lib.call("gdr_debug_set", b"tc_screen", int(v))
    _lib.call("gdr_debug_set", b"tc_screen", 0)


@pytest.mark.parametrize("mode", [3])   # the two-level screen whatever N
@pytest.mark.parametrize("N,K,D,kind", [(300, 7, 3, "clustered"), (4099, 129, 100, "clustered"), (20000, 1000, 40, "clustered"),
                                        (20000, 333, 128, "zscore"), (50000, 1000, 128, "zscore"), (30011, 700, 100, "zscore"),
                                        (1, 1, 1, "clustered")])
def test_tc_two_level_screen_equals_exact_kernel(gdr, oracle, screen_mode, mode, N, K, D, kind):
    """1xTF32 lower-bound screen -> 3xTF32 on the compacted undecided rows -> exact re-score: the labels
    are those of the exact fp32 kernel, also on unclustered data where many rows reach level 2."""
    from gdr import synth
    from gdr._dev import padded_rows
    from gdr.kmeans import TcOperand
    X = synth.clustered_features(N, D, max(2, K // 3), seed=N + K) if kind == "clustered" else synth.features(N, D, seed=N + K)
    X -= X.mean(axis=0)
    C = synth.kmeans_init(X, K, seed=1)
    Xd, Cd = padded_rows(torch.from_numpy(X).to(DEV)), padded_rows(torch.from_numpy(C).to(DEV))
    op = TcOperand(Xd)
    prev = torch.zeros(N, dtype=torch.int32, device=DEV)
    lab32 = torch.empty(N, dtype=torch.int32, device=DEV)
    nch32 = torch.zeros(1, dtype=torch.int32, device=DEV)
    gdr.assign_labels(Xd, Cd, lab32, labels_prev=prev, n_changed=nch32)
    screen_mode(mode)
    labels = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    nch = torch.zeros(1, dtype=torch.int32, device=DEV)
    n_ref = torch.zeros(1, dtype=torch.int32, device=DEV)
    gdr.assign_labels(Xd, Cd, labels, labels_prev=prev, n_changed=nch, tc_operand=op, n_refined=n_ref)
    torch.cuda.synchronize()
    assert np.array_equal(np_(lab32), np_(labels))
    assert int(nch.item()) == int(nch32.item())
    ok, n_band, n_bad = oracle.labels_match(np_(labels), X, C, band=1e-6)
    assert ok, f"{n_bad} rows outside the 1e-6 margin band disagree with the exact argmin"
    assert int(n_ref.item()) <= max(64, N // 5)


@pytest.mark.parametrize("mode", [1, 3])   # direct 3xTF32, two-level screen
def test_tc_full_fit_same_for_every_screen(gdr, screen_mode, mode):
    from gdr import synth
    N, K, D = 40000, 300, 100
    X = synth.features(N, D, seed=11)
    C0 = synth.kmeans_init(X, K, seed=3)
    a = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=6, tol=0, precision="fp32").fit(X)
    screen_mode(mode)
    b = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=6, tol=0, precision="tc").fit(X)
    assert np.array_equal(a.labels_, b.labels_)
    np.testing.assert_array_equal(a.cluster_centers_, b.cluster_centers_)
    assert a.inertia_ == b.inertia_


def test_tc_full_fit_matches_fp32_path(gdr):
    from gdr import synth
    N, K, D = 30000, 500, 64
    X = synth.clustered_features(N, D, 200, seed=5)
    C0 = synth.kmeans_init(X, K, seed=2)
    a = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=8, tol=0, precision="fp32").fit(X)
    b = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=8, tol=0, precision="tc").fit(X)
    assert a.n_iter_ == b.n_iter_
    assert np.array_equal(a.labels_, b.labels_)
    np.testing.assert_array_equal(a.cluster_centers_, b.cluster_centers_)
    assert a.inertia_ == b.inertia_


def test_tc_unsupported_width_fails_loudly(gdr):
    x = torch.randn(1000, 200, device=DEV)
    with pytest.raises(gdr.GdrError):
        gdr.KMeans(n_clusters=10, init="random", random_state=0, precision="tc", max_iter=2).fit(x)


@pytest.mark.parametrize("cfg_name", ["B", "E"])
def test_tc_full_size_labels_equal_exact_kernel(gdr, cfg_name):
    """BASELINE full sizes (config B: 169 343 x 128, K = 1 000; config E: 2 449 029 x 100, K = 10 000): one E-step of
    the production path (automatic two-level tensor-core screen) gives exactly the labels of the exact fp32 SIMT
    kernel, on unclustered z-scored data where thousands of rows reach the exact re-score."""
    from gdr import synth, _lib
    from gdr._dev import padded_rows
    from gdr.kmeans import TcOperand
    import ctypes
    cfg = synth.CONFIGS[cfg_name]
    n, d, k = cfg["n"], cfg["f"], cfg["k"]
    X = torch.from_numpy(synth.features(n, d, seed=17)).to(DEV)
    X = padded_rows((X - X.mean(0)).contiguous())
    C = padded_rows(X[torch.from_numpy(np.random.RandomState(3).permutation(n)[:k].astype(np.int64)).to(DEV)].clone())
    # one Lloyd update so that the centres are means (small norms, tight margins), not data points
    lab0 = torch.empty(n, dtype=torch.int32, device=DEV)
    op = TcOperand(X)
    gdr.assign_labels(X, C, lab0, tc_operand=op)
    sums, counts = gdr.segment_sum(X, lab0, k)
    C = padded_rows((sums / counts.clamp_min(1).unsqueeze(1)).contiguous())
    lab_tc = torch.empty(n, dtype=torch.int32, device=DEV)
    n_ref = torch.zeros(1, dtype=torch.int32, device=DEV)
    gdr.assign_labels(X, C, lab_tc, tc_operand=op, n_refined=n_ref)
    lvl2 = ctypes.c_int64(-1)
    _lib.call("gdr_debug_get", b"tc_level2_rows", ctypes.addressof(lvl2))
    lab_32 = torch.empty(n, dtype=torch.int32, device=DEV)
    gdr.assign_labels(X, C, lab_32)
    torch.cuda.synchronize()
    assert torch.equal(lab_tc, lab_32)
    assert 0 < int(n_ref.item()) < n // 100 and 0 < lvl2.value < n // 5     # both refinement levels were exercised


@pytest.fixture
def gate_mode():
    """First-level epilogue gate (gdr_debug_set "tc_gate": 0 off, 1 on the running best)."""
    from gdr import _lib
    yield lambda v: _lib.call("gdr_debug_set", b"tc_gate", int(v))
    _lib.call("gdr_debug_set", b"tc_gate", 1)


@pytest.mark.parametrize("N,K,D,kind", [(100000, 4096, 100, "zscore"), (80000, 5000, 47, "clustered"), (90001, 4100, 128, "zscore")])
def test_tc_gate_modes_take_identical_decisions(gdr, oracle, gate_mode, screen_mode, N, K, D, kind):
    """The gated first-level epilogue (chunks are looked at only when they hold a score within tolmax_i of a lower
    bound of the row's best) must hand EXACTLY the same rows to level 2 and produce the same labels as the ungated
    running top-2 — with good hints (the true labels), useless hints (all zero) and no hints."""
    import ctypes
    from gdr import synth, _lib
    from gdr._dev import padded_rows
    from gdr.kmeans import TcOperand
    X = synth.clustered_features(N, D, max(2, K // 3), seed=N + K) if kind == "clustered" else synth.features(N, D, seed=N + K)
    X -= X.mean(axis=0)
    C = synth.kmeans_init(X, K, seed=1)
    Xd, Cd = padded_rows(torch.from_numpy(X).to(DEV)), padded_rows(torch.from_numpy(C).to(DEV))
    op = TcOperand(Xd)
    screen_mode(3)          # two-level screen whatever N

    def run(gate, prev):
        gate_mode(gate)
        labels = torch.full((N,), -7, dtype=torch.int32, device=DEV)
        nch = torch.zeros(1, dtype=torch.int32, device=DEV)
        n_ref = torch.zeros(1, dtype=torch.int32, device=DEV)
        gdr.assign_labels(Xd, Cd, labels, labels_prev=prev, n_changed=None if prev is None else nch, tc_operand=op,
                          n_refined=n_ref)
        lvl2 = ctypes.c_int64(-1)
        _lib.call("gdr_debug_get", b"tc_level2_rows", ctypes.addressof(lvl2))
        return labels, int(lvl2.value), int(n_ref.item()), int(nch.item())

    lab0, l2_0, ref_0, _ = run(0, None)
    ok, _, n_bad = oracle.labels_match(np_(lab0), X, C, band=1e-6)
    assert ok, n_bad
    truth = lab0.clone()
    zeros = torch.zeros(N, dtype=torch.int32, device=DEV)
    shuffled = truth[torch.randperm(N, device=DEV)]
    for prev in (None, truth, zeros, shuffled):
        lab, l2, ref, nch = run(1, prev)
        assert torch.equal(lab, lab0), "labels differ"
        assert (l2, ref) == (l2_0, ref_0), (l2, l2_0, ref, ref_0)
        if prev is not None:
            assert nch == int((prev != lab0).sum().item())


def test_tc_gate_full_fit_equals_ungated(gdr, gate_mode):
    from gdr import synth
    N, K, D = 120000, 4500, 100
    X = synth.features(N, D, seed=21)
    C0 = synth.kmeans_init(X, K, seed=5)
    gate_mode(0)
    a = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=6, tol=0, precision="tc").fit(X)
    gate_mode(1)
    b = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=6, tol=0, precision="tc").fit(X)
    assert np.array_equal(a.labels_, b.labels_)
    np.testing.assert_array_equal(a.cluster_centers_, b.cluster_centers_)
    assert a.inertia_ == b.inertia_ and a.n_iter_ == b.n_iter_
