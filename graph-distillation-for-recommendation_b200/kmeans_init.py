"""k-means++ seeding on the device (sklearn/_kmeans.py:180-278).

The host draws the random numbers from numpy's RandomState in exactly the order sklearn's
``_kmeans_plusplus`` consumes them (one ``choice`` with uniform p, then ``uniform(size=
n_local_trials)`` per further centre); every distance, potential and cumulative-sum step runs
in libgdr_b200 (``gdr_kmeans_plusplus``).  With the same ``random_state`` the chosen seeds
equal sklearn's except when a draw lands within rounding of a cumulative-sum boundary (the
kernel accumulates in fp64, sklearn in fp32).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._dev import new_padded, ptr, stream, workspace


def draw_plusplus(random_state, n_samples: int, n_clusters: int):
    """The host draws of sklearn's ``_kmeans_plusplus``, in its order: (first centre, [K-1, n_trials] uniforms,
    n_trials)."""
    K = int(n_clusters)
    n_trials = 2 + int(np.log(K))
    if n_trials > 16:
        raise ValueError("n_clusters too large for the k-means++ kernel (n_local_trials > 16)")
    # random_state.choice(n_samples, p=sample_weight / sample_weight.sum())  (:232)
    first = int(random_state.choice(n_samples, p=np.full(n_samples, 1.0 / n_samples)))
    rand = np.empty((max(K - 1, 1), n_trials), dtype=np.float64)
    for c in range(K - 1):
        rand[c] = random_state.uniform(size=n_trials)   # (:251)
    return first, rand, n_trials


def kmeans_plusplus_device(Xc: torch.Tensor, n_clusters: int, random_state, return_indices: bool = False):
    """Xc: row-padded f32 [N, D] on the GPU.  Returns centres [K, D] (padded rows) on the GPU."""
    N, D = Xc.shape
    K = int(n_clusters)
    first, rand, n_trials = draw_plusplus(random_state, N, K)
    centers = new_padded(K, D, Xc.device, zero=True)
    indices = torch.empty(K, dtype=torch.int64, device=Xc.device)
    ws = workspace(_lib.query("gdr_kmeans_plusplus_ws_bytes", N, K, D, n_trials), Xc.device)
    _lib.call("gdr_kmeans_plusplus", N, K, D, ptr(Xc), Xc.stride(0), first, rand.ctypes.data, n_trials,
              ptr(centers), centers.stride(0), ptr(indices), ptr(ws), ws.numel(), stream())
    return (centers, indices) if return_indices else centers
