"""CPU model of the candidate second level of the two-level tensor-core screen (tools/cand_estimate.py: the level-1
operands of k_split_tf32, the seeded limit of k_tc_cand and the final filter of k_tc_cand_resolve): the exact fp32
argmin is always among the kept candidates, also when every modelled score is moved by the full TMEM accumulation
allowance (D + 4) 2^-23 |x||c| against it."""
import importlib.util
import os
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def model():
    spec = importlib.util.spec_from_file_location("cand_estimate", os.path.join(ROOT, "tools", "cand_estimate.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def inputs(kind, rng):
    N, D, K = 600, 47, 700
    if kind == "random":
        X = rng.standard_normal((N, D)).astype(np.float32)
        C = rng.standard_normal((K, D)).astype(np.float32) * 0.3
    elif kind == "clustered":
        C = rng.standard_normal((K, D)).astype(np.float32) * 3
        X = C[rng.integers(0, K, N)] + 0.05 * rng.standard_normal((N, D)).astype(np.float32)
    elif kind == "duplicated":
        C = rng.standard_normal((K // 2, D)).astype(np.float32)
        C = np.concatenate([C, C])
        X = C[rng.integers(0, K, N)] * 0.5 + 0.01 * rng.standard_normal((N, D)).astype(np.float32)
    elif kind == "mirrored":
        C = rng.standard_normal((K // 2, D)).astype(np.float32)
        C = np.concatenate([C, -C])
        X = rng.standard_normal((N, D)).astype(np.float32) * 1e-3
        X[: N // 4] = 0.0
    elif kind == "large":
        X = rng.standard_normal((N, D)).astype(np.float32) * 1e6
        C = X[rng.permutation(N)[:K // 2]] + rng.standard_normal((K // 2, D)).astype(np.float32)
    else:
        raise ValueError(kind)
    return np.ascontiguousarray(X, dtype=np.float32), np.ascontiguousarray(C, dtype=np.float32)


@pytest.mark.parametrize("kind", ["random", "clustered", "duplicated", "mirrored", "large"])
@pytest.mark.parametrize("push", [None, "against", "random"])
def test_exact_argmin_is_a_kept_candidate(model, oracle, kind, push):
    rng = np.random.default_rng(zlib.crc32(f"{kind}/{push}".encode()))
    X, C = inputs(kind, rng)
    lab, _ = oracle.kmeans_assign(X, C)
    lab = lab.astype(np.int64)
    n = X.shape[0]

    def perturb(d, bound):
        if push == "against":        # the exact argmin's score as bad as allowed, every other one as good as allowed
            s = -np.ones_like(d)
            s[np.arange(n), lab] = 1.0
        else:
            s = rng.uniform(-1, 1, d.shape)
        return d + s * bound

    und, counts, kept, d = model.screen(X, C, None if push is None else perturb)
    assert kept[np.arange(n), lab].all(), np.flatnonzero(~kept[np.arange(n), lab])[:10]
    assert (counts.sum(1) >= kept.sum(1)).all() and (kept.sum(1) >= 1).all()
