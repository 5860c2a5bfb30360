"""The arithmetic of the shared-memory coarsening (csrc/graph.cu k_cd_accumulate), restated in numpy and checked on the
CPU: per-cluster fixed-point step q = 2^(e_w + e_n - 62) from (max |w|, edge count), terms round(w / q) accumulated as a
64-bit integer kept in two 32-bit words with a carry, in ANY order -> bit-reproducible, no overflow, and within
n_cell * q / 2 plus one fp32 rounding of the exact sum: one ulp when the cell is at least about n_cell * q * 2^24, not for
a cell small next to the cluster's largest weight."""
from fractions import Fraction

import numpy as np
import pytest

from coarsen_ref import dense_bound, fixed_point_sum, one_ulp_regime, step as _step, ulp32


def _accumulate_two_words(terms: np.ndarray, order: np.ndarray) -> int:
    """lo / hi 32-bit words with the carry rule of the kernel: old = atomicAdd(lo, v_lo); hi += v_hi + (old + v_lo wrapped)"""
    lo = hi = 0
    for i in order:
        v = int(terms[i]) & 0xFFFFFFFFFFFFFFFF       # two's complement of the signed 64-bit term
        v_lo, v_hi = v & 0xFFFFFFFF, v >> 32
        old = lo
        lo = (lo + v_lo) & 0xFFFFFFFF
        hi = (hi + v_hi + (1 if lo < old else 0)) & 0xFFFFFFFF
    s = (hi << 32) | lo
    return s - (1 << 64) if s >> 63 else s           # back to signed


@pytest.mark.parametrize("seed,n,scale,signed", [(0, 50, 1.0, False), (1, 3000, 1e-4, False), (2, 500, 37.0, True),
                                                 (3, 1, 1e-20, False), (4, 2000, 1e12, True)])
def test_fixed_point_sum_is_the_exact_sum_rounded_once_in_any_order(seed, n, scale, signed):
    rng = np.random.RandomState(seed)
    w = (rng.rand(n) * scale).astype(np.float32)
    w[rng.randint(n)] = np.float32(scale)                      # the maximum
    if signed:
        w *= rng.choice([-1.0, 1.0], n).astype(np.float32)
    # hub-like spread: most weights far below the maximum
    w[: n // 2] *= np.float32(1e-5)
    wmax = np.abs(w).max()
    n_cluster_edges = n + rng.randint(0, 1000)                 # the cluster has more edges than this cell
    e = _step(wmax, n_cluster_edges)
    terms = np.array([int(np.rint(np.float64(x) * 2.0 ** (-e))) for x in w], dtype=object)
    assert all(abs(int(t)) < 2 ** (62 - int(np.frexp(float(n_cluster_edges))[1]) + 1) for t in terms)   # |w| / q < 2^(62 - ee)
    exact = sum(Fraction(float(x)) for x in w)
    results = set()
    for rep in range(4):
        order = rng.permutation(n)
        total = _accumulate_two_words(terms, order)
        assert abs(total) < 2 ** 62                            # no overflow, whatever the order
        results.add(total)
        got = np.float32(np.float64(total) * 2.0 ** e)
        assert got == fixed_point_sum(w, e)
        # the integer sum differs from the exact sum by at most n/2 steps of q ~ 2^-48 of the largest weight; this cell
        # holds that weight, so it is large next to n*q and its fp32 rounding is within one ulp of the exact sum's
        S = float(exact)
        assert abs(Fraction(float(got)) - exact) <= Fraction(float(dense_bound(S, n, 2.0 ** e)))
        assert one_ulp_regime(S, n, 2.0 ** e)
        assert abs(float(got) - float(np.float32(S))) <= float(ulp32(S))
    assert len(results) == 1                                   # associative: bit-reproducible


def test_step_is_a_function_of_the_global_cluster_stats_only():
    """Every rank of a partition derives q from the all-reduced (edges, max |w|): the same q as one GPU."""
    assert _step(np.float32(0.5), 12600) == _step(np.float32(0.5), 12600)
    assert _step(np.float32(0.5), 12600) == 0 + 14 - 62        # 0.5 = 0.5 * 2^0 -> ew 0; 12600 < 2^14 -> ee 14
    assert _step(np.float32(0.0), 0) == 0 + 1 - 62


@pytest.mark.parametrize("w_cell,ulps", [(1e-9, 31), (1e-12, 17204)])
def test_small_cell_next_to_a_large_weight_is_off_by_more_than_one_ulp(w_cell, ulps):
    """A cluster with a weight-1 self-loop and 12 600 edges: q = 2^-47 for every cell of it.  A one-edge cell of weight
    1e-9 is rounded to a multiple of q — dozens of ulps from the exact (and fp32-exact) value — so 'within one ulp' does
    not hold; the bound n*q/2 + one fp32 rounding does."""
    e = _step(np.float32(1.0), 12600)
    assert e == -47
    w = np.array([w_cell], dtype=np.float32)
    got = fixed_point_sum(w, e)
    S = float(w[0])                                            # a one-edge cell: the exact sum is the fp32 weight itself
    err = abs(float(got) - S)
    assert err <= dense_bound(S, 1, 2.0 ** e)
    assert not one_ulp_regime(S, 1, 2.0 ** e)
    assert err > ulp32(S)                                      # the old 'within one ulp of the exact sum' fails here
    assert round(err / ulp32(S)) == ulps
