"""Truncated SVD embeddings of the interaction matrix (SURVEY §8f item 3).

``compute_svd_embeddings(R, dim, seed)`` of distill_recsys.py:124-155 — the step right before the k-means
stage of distill_recsys — returns ``(U sqrt(S), V sqrt(S))`` of the ``dim`` leading singular triplets.  The
reference calls scipy's ``svds`` (ARPACK, fp64, host).  Here the factorisation is a **block Krylov
Rayleigh-Ritz** on the device:

  * the sparse products R·Q and Rᵀ·Q run on the stage-2 CSR SpMM kernel (R and Rᵀ as device CSR) — the hot
    operation is the same HBM-bound gather kernel as the propagation;
  * every dense step is a hand-written fp64 kernel of csrc/svd.cu (no cuSOLVER / cuBLAS): CholeskyQR2 of the tall
    blocks (``gdr_dense_gram`` -> ``gdr_dense_chol`` -> ``gdr_dense_trsm_rows``), block Gram-Schmidt against the earlier
    blocks (``gdr_dense_gram`` + ``gdr_dense_gemm_small``), the (q·b)² Ritz problem by parallel cyclic Jacobi on the
    Gram matrix of R·Q (``gdr_sym_eig_jacobi``) and the Ritz vectors (``gdr_dense_gemm_small``).

The Krylov space lives on the SMALLER side of R and never exceeds it (blocks stop when the space is exhausted or a
block loses rank), so small matrices are factorised exactly instead of on noise.

Parity with the reference is defined on what it determines uniquely: the singular values (relative 1e-4) and
the singular vectors of well separated values up to sign; the tail of a slowly decaying spectrum is only
determined as a subspace (the reference itself depends on ARPACK's starting vector there).
"""
from __future__ import annotations

import ctypes
from typing import Tuple, Union

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib
from ._dev import device_of, ptr, stream, workspace
from .graph import CSR
from .propagation import spmm


EXACT_SIDE = 768     # smaller side up to which the factorisation is the exact Gram eigen-problem (no Krylov space)


def _gram(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """AᵀB for fp64 row-major (possibly column-sliced) tall matrices."""
    N, p, r = A.shape[0], A.shape[1], B.shape[1]
    C = torch.empty((p, r), dtype=torch.float64, device=A.device)
    ws = workspace(_lib.query("gdr_dense_gram_ws_bytes", N, p, r), A.device)
    _lib.call("gdr_dense_gram", N, p, r, ptr(A), A.stride(0), ptr(B), B.stride(0), ptr(C), r, ptr(ws), ws.numel(), stream())
    return C


def _cholqr2(Y: torch.Tensor, gram=_gram) -> bool:
    """In-place orthonormalisation of the columns of the fp64 block Y [N, b] (CholeskyQR, twice).  False when the block
    has lost rank (a pivot of the Gram matrix is below 1e-13 of its largest diagonal entry).  ``gram(X, Y)`` is XᵀY
    over all rows of the block (on a row partition: over every rank's rows, replicated)."""
    N, b = Y.shape
    info = torch.zeros(1, dtype=torch.int32, device=Y.device)
    L = torch.empty((b, b), dtype=torch.float64, device=Y.device)
    for _ in range(2):
        S = gram(Y, Y)
        _lib.call("gdr_dense_chol", b, ptr(S), b, ptr(L), b, ptr(info), 1e-13, stream())
        if int(info.item()):
            return False
        _lib.call("gdr_dense_trsm_rows", N, b, ptr(Y), Y.stride(0), ptr(L), b, stream())
    return True


def _project_out(Z: torch.Tensor, Q: torch.Tensor, gram=_gram):
    """Z <- Z - Q (Qᵀ Z), twice (block Gram-Schmidt with re-orthogonalisation), Q [N, m] orthonormal."""
    N, b = Z.shape
    m = Q.shape[1]
    for _ in range(2):
        P = gram(Q, Z)
        if N:
            _lib.call("gdr_dense_gemm_small", N, m, b, -1.0, ptr(Q), Q.stride(0), ptr(P), b, 1.0, ptr(Z), Z.stride(0), 0, 0,
                      0, stream())


def krylov_ritz(ns: int, rows: slice, k: int, seed: int, block, n_blocks, dev, gram_s, gram_o, mul_A, mul_At
                ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """The factorisation of truncated_svd, written for the rows ``rows`` of the small side (ns rows) that this process
    holds: all of them on one GPU, a row block on a partition (parallel.dist_truncated_svd).  ``gram_s(X, Y)`` / ``gram_o``
    = XᵀY over all rows of the small / other side; ``mul_A(X)`` = the held rows of the other side of A X for the held
    fp64 rows X of small-side vectors (fp32 result), ``mul_At(Y)`` = the held small-side rows of Aᵀ Y.  Every branch is
    decided on replicated data.  Returns (Uo [held other-side rows, k], S [k] fp32 descending, Vs [held small-side rows, k])."""
    k = int(min(k, ns))
    n_s = rows.stop - rows.start
    if ns <= EXACT_SIDE and block is None and n_blocks is None:
        # the whole space of the smaller side: Q = I, the Ritz problem below is the exact Gram eigen-problem of A
        # (a Krylov space clamped to a few dimensions short of ns interlaces the spectrum instead of matching it)
        m = ns
        Qm = torch.eye(ns, dtype=torch.float64, device=dev)[rows]
    else:
        b = int(min(block or (k + 8), ns, 128))
        q = int(n_blocks or max(6, min(14, 600 // b)))
        q = max(1, min(q, ns // b))                              # q b <= ns: the space cannot be larger than the side
        gen = torch.Generator(device="cpu").manual_seed(int(seed))
        G = torch.randn((ns, b), generator=gen, dtype=torch.float32)[rows].to(dev)
        Q = torch.zeros((n_s, q * b), dtype=torch.float64, device=dev)
        V = Q[:, :b]
        V.copy_(G)
        if not _cholqr2(V, gram_s):
            raise ValueError("truncated_svd: the random start block is rank deficient")
        m = b
        for j in range(1, q):
            Y = mul_A(Q[:, (j - 1) * b: j * b])                  # [n_other, b]  sparse x dense on the CSR kernel
            Z = mul_At(Y)                                        # [ns, b]
            Vn = Q[:, j * b: (j + 1) * b]
            Vn.copy_(Z)
            _project_out(Vn, Q[:, :m], gram_s)
            if not _cholqr2(Vn, gram_s):                         # Krylov space exhausted: keep the blocks so far
                break
            m += b
        Qm = Q[:, :m]
    B = mul_A(Qm).double()                                       # [n_other, m] = A Q
    # Rayleigh-Ritz on the Gram matrix of B (fp64; the leading Ritz values lose nothing to the squared condition number)
    T = gram_o(B, B).contiguous()
    W = torch.empty((m, m), dtype=torch.float64, device=dev)
    evals = torch.empty(m, dtype=torch.float64, device=dev)
    order = torch.empty(m, dtype=torch.int32, device=dev)
    sweeps = ctypes.c_int32(0)
    ws = workspace(_lib.query("gdr_sym_eig_jacobi_ws_bytes", m), dev)
    _lib.call("gdr_sym_eig_jacobi", m, ptr(T), ptr(W), ptr(evals), ptr(order), 30, 1e-14, ctypes.addressof(sweeps), ptr(ws),
              ws.numel(), stream())
    kk = min(k, m)
    Wk = torch.empty((m, kk), dtype=torch.float64, device=dev)
    _lib.call("gdr_dense_gather_cols", m, kk, ptr(W), ptr(order), ptr(Wk), stream())
    S = evals[:kk].clamp_min(0).sqrt()
    inv_s = torch.where(S > 0, 1.0 / S, torch.zeros_like(S)).contiguous()
    n_other = B.shape[0]
    Vs = torch.empty((n_s, kk), dtype=torch.float32, device=dev)         # small-side vectors  Q W
    Uo = torch.empty((n_other, kk), dtype=torch.float32, device=dev)     # other-side vectors  B W / sigma
    if n_s:
        _lib.call("gdr_dense_gemm_small", n_s, m, kk, 1.0, ptr(Qm), Qm.stride(0), ptr(Wk), kk, 0.0, 0, 0, ptr(Vs), kk, 0,
                  stream())
    if n_other:
        _lib.call("gdr_dense_gemm_small", n_other, m, kk, 1.0, ptr(B), B.stride(0), ptr(Wk), kk, 0.0, 0, 0, ptr(Uo), kk,
                  ptr(inv_s), stream())
    return Uo, S.to(torch.float32), Vs


def truncated_svd(R: CSR, k: int, seed: int = 42, block: int = None, n_blocks: int = None
                  ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(U [n_rows, k], S [k] descending, V [n_cols, k]) of the k largest singular triplets of the device CSR ``R``."""
    n_rows, n_cols = R.shape
    Rt, _ = R.transpose()
    # Krylov space on the smaller side: A maps it to the larger one
    A, At = (R, Rt) if n_cols <= n_rows else (Rt, R)
    ns = min(n_rows, n_cols)
    Uo, S, Vs = krylov_ritz(ns, slice(0, ns), k, seed, block, n_blocks, R.device, _gram, _gram,
                            lambda X: spmm(A, X.to(torch.float32).contiguous()), lambda Y: spmm(At, Y.contiguous()))
    return (Uo, S, Vs) if n_cols <= n_rows else (Vs, S, Uo)


def compute_svd_embeddings(R: Union[sp.spmatrix, CSR], dim: int, seed: int = 42, device=None
                           ) -> Tuple[np.ndarray, np.ndarray]:
    """distill_recsys.py:124-155: ``(user_emb, item_emb) = (U sqrt(S), V sqrt(S))`` as float32 numpy arrays, singular
    values in descending order; raises the reference's ValueError when no factorisation is possible."""
    shape = R.shape
    k = min(int(dim), min(shape) - 1)
    if k <= 0:
        raise ValueError(f"Cannot compute SVD with shape={tuple(shape)} and dim={dim}")
    A = R if isinstance(R, CSR) else CSR.from_scipy(sp.csr_matrix(R, dtype=np.float32), device=device_of(device))
    U, S, V = truncated_svd(A, k, seed=seed)
    sqrt_s = torch.sqrt(torch.clamp_min(S, 1e-12)).reshape(1, -1)
    return (U * sqrt_s).cpu().numpy().astype(np.float32), (V * sqrt_s).cpu().numpy().astype(np.float32)
