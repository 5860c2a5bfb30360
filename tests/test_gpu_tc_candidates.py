"""Second level of the two-level tensor-core screen on candidate centres (seeded 1xTF32 pass that records the centres
within tolmax of the row's best, exact fp32 re-score of the kept ones, 3xTF32 fallback for the rest).  GPU only."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def gdr():
    import gdr as g
    assert torch.cuda.is_available()
    return g


@pytest.fixture
def knob():
    """gdr_debug_set(key, value); every key touched is put back to its default afterwards."""
    from gdr import _lib
    defaults = {"tc_cand": 1, "tc_cand_cap": 0, "tc_screen": 0, "tc_gate": 1}
    touched = set()

    def set_(key, value):
        touched.add(key)
        _lib.call("gdr_debug_set", key.encode(), int(value))
    yield set_
    for key in touched:
        _lib.call("gdr_debug_set", key.encode(), defaults[key])


def debug_get(key):
    from gdr import _lib
    v = ctypes.c_int64(-7)
    _lib.call("gdr_debug_get", key.encode(), ctypes.addressof(v))
    return int(v.value)


def np_(t):
    return t.detach().cpu().numpy()


def make(N, K, D, kind, seed=None):
    from gdr import synth
    seed = N + K if seed is None else seed
    X = synth.clustered_features(N, D, max(2, K // 3), seed=seed) if kind == "clustered" else synth.features(N, D, seed=seed)
    X -= X.mean(axis=0)
    C = synth.kmeans_init(X, K, seed=1)
    return X, C


def assign(gdr, Xd, Cd, prev=None):
    from gdr.kmeans import TcOperand
    N = Xd.shape[0]
    labels = torch.full((N,), -7, dtype=torch.int32, device=DEV)
    nch = torch.zeros(1, dtype=torch.int32, device=DEV)
    n_ref = torch.zeros(1, dtype=torch.int32, device=DEV)
    gdr.assign_labels(Xd, Cd, labels, labels_prev=prev, n_changed=None if prev is None else nch,
                      tc_operand=TcOperand(Xd), n_refined=n_ref)
    torch.cuda.synchronize()
    return labels, int(nch.item()), int(n_ref.item())


def exact(gdr, Xd, Cd, prev=None):
    N = Xd.shape[0]
    lab = torch.empty(N, dtype=torch.int32, device=DEV)
    nch = torch.zeros(1, dtype=torch.int32, device=DEV)
    gdr.assign_labels(Xd, Cd, lab, labels_prev=prev, n_changed=None if prev is None else nch)
    torch.cuda.synchronize()
    return lab, int(nch.item())


@pytest.mark.parametrize("N,K,D,kind", [(300, 7, 3, "clustered"), (4099, 129, 100, "clustered"), (20000, 1000, 40, "clustered"),
                                        (20000, 333, 128, "zscore"), (50000, 1000, 128, "zscore"), (30011, 700, 100, "zscore"),
                                        (1, 1, 1, "clustered"), (60000, 4100, 47, "zscore"), (70001, 2000, 47, "clustered")])
def test_candidate_level_equals_exact_and_previous_level(gdr, knob, N, K, D, kind):
    from gdr._dev import padded_rows
    X, C = make(N, K, D, kind)
    Xd, Cd = padded_rows(torch.from_numpy(X).to(DEV)), padded_rows(torch.from_numpy(C).to(DEV))
    prev = torch.zeros(N, dtype=torch.int32, device=DEV)
    lab32, nch32 = exact(gdr, Xd, Cd, prev)
    knob("tc_screen", 3)    # two-level screen whatever N
    knob("tc_cand", 0)
    lab0, nch0, _ = assign(gdr, Xd, Cd, prev)
    knob("tc_cand", 1)
    lab1, nch1, ref1 = assign(gdr, Xd, Cd, prev)
    assert torch.equal(lab1, lab32) and torch.equal(lab0, lab32)
    assert nch1 == nch0 == nch32
    assert ref1 <= max(64, N // 5)


@pytest.mark.parametrize("cfg_name", ["B", "E"])
def test_candidate_level_full_size(gdr, knob, cfg_name):
    """BASELINE full sizes after one Lloyd update (as test_gpu_tc.py): candidate level, previous level and the exact
    kernel agree; most undecided rows are decided on their candidates."""
    from gdr import synth
    from gdr._dev import padded_rows
    from gdr.kmeans import TcOperand
    cfg = synth.CONFIGS[cfg_name]
    n, d, k = cfg["n"], cfg["f"], cfg["k"]
    X = torch.from_numpy(synth.features(n, d, seed=17)).to(DEV)
    X = padded_rows((X - X.mean(0)).contiguous())
    C = padded_rows(X[torch.from_numpy(np.random.RandomState(3).permutation(n)[:k].astype(np.int64)).to(DEV)].clone())
    lab0 = torch.empty(n, dtype=torch.int32, device=DEV)
    gdr.assign_labels(X, C, lab0, tc_operand=TcOperand(X))
    sums, counts = gdr.segment_sum(X, lab0, k)
    C = padded_rows((sums / counts.clamp_min(1).unsqueeze(1)).contiguous())
    lab_32, nch_32 = exact(gdr, X, C, lab0)
    knob("tc_cand", 0)
    lab_a, nch_a, _ = assign(gdr, X, C, lab0)
    knob("tc_cand", 1)
    lab_b, nch_b, ref_b = assign(gdr, X, C, lab0)
    lvl2, cand_rows = debug_get("tc_level2_rows"), debug_get("tc_cand_rows")
    assert torch.equal(lab_a, lab_32) and torch.equal(lab_b, lab_32)
    assert nch_b == nch_a == nch_32
    assert 0 < ref_b < n // 100
    assert 0 < lvl2 < n // 5 and lvl2 // 2 < cand_rows <= lvl2


def test_duplicated_centres_resolve_to_lowest_index(gdr, knob):
    from gdr._dev import padded_rows
    N, K, D = 40000, 4096, 64
    X, C = make(N, K // 2, D, "zscore", seed=5)
    # every centre twice (j and j + K/2), one pair mirrored in sign and zero rows: exact ties everywhere
    C[7] = -C[9]
    C = np.ascontiguousarray(np.concatenate([C, C], axis=0))
    X[:100] = 0.0
    Xd, Cd = padded_rows(torch.from_numpy(X).to(DEV)), padded_rows(torch.from_numpy(C).to(DEV))
    lab32, _ = exact(gdr, Xd, Cd)
    knob("tc_screen", 3)
    lab, _, _ = assign(gdr, Xd, Cd)
    assert torch.equal(lab, lab32)
    assert int(lab.max().item()) < K // 2     # the lower copy of each pair wins
    assert debug_get("tc_cand_rows") >= 0


def test_capacity_one_sends_rows_to_the_fallback(gdr, knob):
    from gdr._dev import padded_rows
    N, K, D = 50000, 4096, 100
    X, C = make(N, K, D, "zscore")
    Xd, Cd = padded_rows(torch.from_numpy(X).to(DEV)), padded_rows(torch.from_numpy(C).to(DEV))
    prev = torch.zeros(N, dtype=torch.int32, device=DEV)
    lab32, nch32 = exact(gdr, Xd, Cd, prev)
    knob("tc_screen", 3)
    lab_d, _, _ = assign(gdr, Xd, Cd, prev)
    entries_d, overflow_d = debug_get("tc_cand_entries"), debug_get("tc_cand_overflow_rows")
    knob("tc_cand_cap", 1)
    lab1, nch1, _ = assign(gdr, Xd, Cd, prev)
    lvl2, cand_rows, overflow = debug_get("tc_level2_rows"), debug_get("tc_cand_rows"), debug_get("tc_cand_overflow_rows")
    assert torch.equal(lab1, lab32) and torch.equal(lab_d, lab32) and nch1 == nch32
    assert lvl2 > 0 and overflow > overflow_d and cand_rows + overflow <= lvl2 and entries_d > 0


def test_candidate_counts_identical_across_gate_modes(gdr, knob):
    """Level-2 rows, n_refined and the candidate counters do not depend on the first-level gate or its hints."""
    from gdr._dev import padded_rows
    N, K, D = 100000, 4096, 100
    X, C = make(N, K, D, "zscore")
    Xd, Cd = padded_rows(torch.from_numpy(X).to(DEV)), padded_rows(torch.from_numpy(C).to(DEV))
    knob("tc_screen", 3)
    ref = None
    truth = None
    for gate in (0, 1, 2):
        knob("tc_gate", gate)
        for prev in ((None,) if truth is None else (None, truth, torch.zeros(N, dtype=torch.int32, device=DEV))):
            lab, _, n_ref = assign(gdr, Xd, Cd, prev)
            got = (np_(lab).tobytes(), n_ref, debug_get("tc_level2_rows"), debug_get("tc_cand_rows"),
                   debug_get("tc_cand_overflow_rows"), debug_get("tc_cand_entries"))
            if ref is None:
                ref, truth = got, lab.clone()
            assert got == ref, (gate, got[1:], ref[1:])


def test_full_fit_same_with_and_without_candidates(gdr, knob):
    from gdr import synth
    N, K, D = 120000, 4500, 100
    X = synth.features(N, D, seed=21)
    C0 = synth.kmeans_init(X, K, seed=5)
    knob("tc_cand", 0)
    a = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=6, tol=0, precision="tc").fit(X)
    knob("tc_cand", 1)
    b = gdr.KMeans(n_clusters=K, init=C0, n_init=1, max_iter=6, tol=0, precision="tc").fit(X)
    assert np.array_equal(a.labels_, b.labels_)
    np.testing.assert_array_equal(a.cluster_centers_, b.cluster_centers_)
    assert a.inertia_ == b.inertia_ and a.n_iter_ == b.n_iter_
