"""CPU references of gdr.recommend_topk (topk_ref.c, the exact fmaf chain) and gdr.ranking_metrics (fp64 numpy,
ascending row order).  Test infrastructure only; the library never imports it."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _c():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="gdr_topk_ref_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libtopk_ref.so")
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC",
                               os.path.join(_HERE, "topk_ref.c"), "-o", out, "-lm"])
        _lib = C.CDLL(out)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def topk(U, I, k, ex_rowptr=None, ex_colidx=None, rows=None):
    """(scores [n_rows, k] f32, items [n_rows, k] int32) of the exact full-ranking top-k."""
    U = np.ascontiguousarray(U, dtype=np.float32)
    I = np.ascontiguousarray(I, dtype=np.float32)
    rows = None if rows is None else np.ascontiguousarray(rows, dtype=np.int64)
    n_rows = U.shape[0] if rows is None else rows.shape[0]
    rp = None if ex_rowptr is None else np.ascontiguousarray(ex_rowptr, dtype=np.int32)
    ci = None if ex_colidx is None else np.ascontiguousarray(ex_colidx, dtype=np.int32)
    scores = np.empty((n_rows, k), dtype=np.float32)
    items = np.empty((n_rows, k), dtype=np.int32)
    I64 = C.c_int64
    _c().ref_topk(I64(n_rows), I64(I.shape[0]), I64(U.shape[1]), I64(k), _p(U), I64(U.shape[1]), _p(rows), _p(I),
                  I64(I.shape[1]), _p(rp), _p(ci), _p(scores), _p(items))
    return scores, items


def metrics(items, test_rowptr, test_colidx, ks, rows=None):
    """Recall / Precision / NDCG@K means (fp64, evaluated rows summed in ascending row order), n_eval, n_skipped."""
    items = np.asarray(items)
    n_rows = items.shape[0]
    users = np.arange(n_rows) if rows is None else np.asarray(rows, dtype=np.int64)
    out = {}
    per = {K: ([], [], []) for K in ks}
    n_eval = 0
    for r in range(n_rows):
        u = users[r]
        test = set(np.asarray(test_colidx[test_rowptr[u]:test_rowptr[u + 1]]).tolist())
        if not test:
            continue
        n_eval += 1
        for K in ks:
            hit = [int(items[r, i]) in test for i in range(K)]
            h = float(sum(hit))
            dcg = sum(1.0 / np.log2(i + 2) for i in range(K) if hit[i])
            idcg = sum(1.0 / np.log2(i + 2) for i in range(min(K, len(test))))
            per[K][0].append(h / len(test))
            per[K][1].append(h / K)
            per[K][2].append(dcg / idcg)
    for K in ks:
        for name, vals in zip(("recall", "precision", "ndcg"), per[K]):
            acc = 0.0
            for v in vals:
                acc += v
            out[f"{name}@{K}"] = acc / n_eval if n_eval else float("nan")
    out.update(n_eval=n_eval, n_skipped=n_rows - n_eval)
    return out
