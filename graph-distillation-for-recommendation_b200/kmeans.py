"""Stage 3 — k-means / WCSS clustering on the GPU.

``KMeans`` mirrors the estimator surface the reference uses from scikit-learn
(constructor keywords, ``fit`` / ``fit_predict`` / ``predict``, ``cluster_centers_``,
``labels_``, ``inertia_``, ``n_iter_``) at these call sites:
    clustgdd_agent_transduct.py:102-107, clustgdd_agent_induct.py:131-136,
    distill_recsys.py:172-180 (``kmeans_cluster``).
The control flow follows ``sklearn/cluster/_kmeans.py`` (fit :1436-1560,
_kmeans_single_lloyd :630-758, _tolerance :285-293); the arithmetic of every step is a
libgdr_b200 kernel (see csrc/kmeans.cu for the .pyx lines each one follows).

Parity is defined for a *given initialisation* (``init=<array>``): the reference's own
call ``KMeans(n_clusters=n)`` has no random_state and is not reproducible with itself.
"""
from __future__ import annotations

import numbers
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._dev import device_of, new_padded, pad4, padded_rows, ptr, stream, workspace


def _check_random_state(seed):
    if seed is None or isinstance(seed, numbers.Integral):
        return np.random.RandomState(seed)
    if isinstance(seed, np.random.RandomState):
        return seed
    raise ValueError(f"{seed!r} cannot be used to seed a numpy.random.RandomState instance")


class _Scratch:
    """Device buffers of one Lloyd run (allocated once, reused every iteration)."""

    def __init__(self, N: int, K: int, D: int, device, precision_mode: int):
        self.N, self.K, self.D = N, K, D
        self.mode = precision_mode
        self.labels = [torch.full((N,), -1, dtype=torch.int32, device=device) for _ in range(2)]
        self.centers = [new_padded(K, D, device, zero=True) for _ in range(2)]
        self.sums = new_padded(K, D, device, zero=True)
        self.counts = torch.zeros(K, dtype=torch.int32, device=device)
        self.n_changed = torch.zeros(1, dtype=torch.int32, device=device)
        self.stats = torch.zeros(2 + K, dtype=torch.float64, device=device)
        if precision_mode == 1:
            self.ws_assign = workspace(_lib.query("gdr_kmeans_assign_tc_ws_bytes", N, K, D), device)
        else:
            self.ws_assign = workspace(_lib.query("gdr_kmeans_assign_ws_bytes", N, K, D, 0), device)
        self.tc = None           # TcOperand of the centred X (tensor-core mode)
        self.n_refined = torch.zeros(1, dtype=torch.int32, device=device)
        self.ws_seg = workspace(_lib.query("gdr_segment_sum_ws_bytes", N, K, D), device)
        self.ws_misc = workspace(
            max(_lib.query("gdr_inertia_ws_bytes", N, D), _lib.query("gdr_kmeans_relocate_ws_bytes", N, K, D)),
            device)
        self.host = torch.empty(4, dtype=torch.float64).pin_memory()
        self.host_i = torch.empty(1, dtype=torch.int32).pin_memory()


class TcOperand:
    """Cached TF32 hi/lo split of X for the tensor-core E-step (X is constant across the
    Lloyd iterations, so the split is done once per fit)."""

    def __init__(self, X: torch.Tensor):
        N, D = X.shape
        self.N, self.D = N, D
        self.buf = workspace(_lib.query("gdr_kmeans_tc_xsplit_bytes", N, D), X.device)
        _lib.call("gdr_kmeans_tc_prepare", N, D, ptr(X), X.stride(0), ptr(self.buf), self.buf.numel(), stream())


def assign_labels(X: torch.Tensor, C: torch.Tensor, labels: torch.Tensor, *, labels_prev=None,
                  n_changed=None, best=None, precision_mode: int = 0, ws: Optional[torch.Tensor] = None,
                  tc_operand: Optional[TcOperand] = None, n_refined=None):
    """E-step: labels[i] = argmin_j |c_j|^2 - 2 x_i.c_j (first index wins).  X, C must be
    row-padded (see _dev.padded_rows).  With ``tc_operand`` the tcgen05 3xTF32 kernel runs
    on the cached split and ambiguous rows are re-scored in exact fp32."""
    N, D = X.shape
    K = C.shape[0]
    if tc_operand is not None:
        if ws is None:
            ws = workspace(_lib.query("gdr_kmeans_assign_tc_ws_bytes", N, K, D), X.device)
        _lib.call("gdr_kmeans_assign_tc", N, K, D, ptr(X), X.stride(0), ptr(tc_operand.buf), ptr(C), C.stride(0),
                  ptr(labels), ptr(labels_prev), ptr(n_changed), ptr(best), ptr(n_refined), ptr(ws), ws.numel(),
                  stream())
        return labels
    if ws is None:
        ws = workspace(_lib.query("gdr_kmeans_assign_ws_bytes", N, K, D, precision_mode), X.device)
    _lib.call("gdr_kmeans_assign", N, K, D, ptr(X), X.stride(0), ptr(C), C.stride(0), ptr(labels),
              ptr(labels_prev), ptr(n_changed), ptr(best), int(precision_mode), ptr(ws), ws.numel(),
              stream())
    return labels


def segment_sum(X: torch.Tensor, labels: torch.Tensor, K: int, *, sums=None, counts=None,
                ws: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-cluster row sums (ascending row order, deterministic) and member counts."""
    N, D = X.shape
    if sums is None:
        sums = new_padded(K, D, X.device, zero=True)
    if counts is None:
        counts = torch.zeros(K, dtype=torch.int32, device=X.device)
    if ws is None:
        ws = workspace(_lib.query("gdr_segment_sum_ws_bytes", N, K, D), X.device)
    _lib.call("gdr_segment_sum", N, K, D, ptr(X), X.stride(0), ptr(labels), ptr(sums), sums.stride(0),
              ptr(counts), ptr(ws), ws.numel(), stream())
    return sums, counts


def means_of_sums(sums: torch.Tensor, counts: torch.Tensor, empty_nan: bool) -> torch.Tensor:
    """sums[c] / counts[c] from segment_sum's (sums, counts).  ``empty_nan``: gdr_kmeans_finalize in mean mode (fp32
    division, an empty cluster gives a NaN row; a padded [K, D] view), else the division by counts.clamp_min(1) of
    distill_recsys.py:635 (an empty segment gives a zero row)."""
    if not empty_nan:
        return sums / counts.clamp_min(1).unsqueeze(1).to(sums.dtype)
    K, D = sums.shape
    out = new_padded(K, D, sums.device)
    stats = torch.zeros(2 + K, dtype=torch.float64, device=sums.device)
    _lib.call("gdr_kmeans_finalize", K, D, ptr(sums), sums.stride(0), ptr(counts), 0, 0, ptr(out),
              out.stride(0), ptr(stats), 1, stream())
    return out


def cluster_means(features: torch.Tensor, labels: torch.Tensor, n_clusters: int) -> torch.Tensor:
    """feat_syn[c] = mean(features[labels == c]); an empty cluster gives a NaN row.

    Replaces the O(n*N) Python loop at clustgdd_agent_transduct.py:121-125
    (clustgdd_agent_induct.py:143-152)."""
    X = padded_rows(features.to(torch.float32))
    lab = labels.to(device=X.device, dtype=torch.int32).contiguous()
    sums, counts = segment_sum(X, lab, int(n_clusters))
    return means_of_sums(sums, counts, empty_nan=True)


def segment_mean_pool(emb: torch.Tensor, assign: torch.Tensor, n_segments: int) -> torch.Tensor:
    """index_add_ + bincount().clamp_min(1) mean pooling of distill_recsys.py:628-636."""
    X = padded_rows(emb.to(torch.float32))
    lab = assign.to(device=X.device, dtype=torch.int32).contiguous()
    sums, counts = segment_sum(X, lab, int(n_segments))
    return means_of_sums(sums, counts, empty_nan=False)


class KMeans:
    """GPU Lloyd k-means with scikit-learn's KMeans interface (dense float32 input).

    Differences from sklearn that are part of the contract:
      * ``algorithm`` must be "lloyd"; sample weights are not supported (the reference
        never passes them);
      * ``init`` may be an array (parity mode), "random" (rows picked by
        ``RandomState(random_state).permutation``) or "k-means++" (greedy D^2 seeding on the
        device, host RNG — same distribution as sklearn, not the same stream);
      * ``precision`` selects the E-step kernel: "fp32" exact SIMT, "tc" tcgen05 3xTF32
        screen + exact re-score of ambiguous rows.
    Inputs may be numpy arrays (copied to ``device``) or CUDA tensors; fitted attributes
    come back in the same kind.
    """

    def __init__(self, n_clusters=8, *, init="k-means++", n_init="auto", max_iter=300, tol=1e-4,
                 verbose=0, random_state=None, copy_x=True, algorithm="lloyd", precision="auto",
                 device=None):
        self.n_clusters = n_clusters
        self.init = init
        self.n_init = n_init
        self.max_iter = max_iter
        self.tol = tol
        self.verbose = verbose
        self.random_state = random_state
        self.copy_x = copy_x
        self.algorithm = algorithm
        self.precision = precision
        self.device = device

    # -- helpers -------------------------------------------------------------------
    def _mode(self, D: Optional[int] = None) -> int:
        """0 = exact fp32 SIMT E-step, 1 = tcgen05 3xTF32 screen + exact re-score.  "auto" picks
        the tensor-core kernel whenever the feature width fits its shared-memory plan (D <= 128);
        both produce the same labels (tests/test_gpu_tc.py)."""
        if self.precision not in ("fp32", "tc", "auto"):
            raise ValueError("precision must be 'auto', 'fp32' or 'tc'")
        if self.precision == "auto":
            return 1 if (D is not None and D <= 128) else 0
        return 1 if self.precision == "tc" else 0

    def _to_device(self, X):
        self._numpy_io = not isinstance(X, torch.Tensor)
        if self._numpy_io:
            X = np.asarray(X)
            if X.ndim != 2:
                raise ValueError(f"Expected 2D array, got {X.ndim}D array instead")
            dev = device_of(self.device)
            Xd = torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)).to(dev)
        else:
            if not X.is_cuda:
                raise ValueError("torch input must live on a CUDA device (no CPU path)")
            if X.dim() != 2:
                raise ValueError(f"Expected 2D tensor, got {X.dim()}D")
            Xd = X.to(torch.float32)
        return Xd

    def _out(self, t: torch.Tensor):
        return t.cpu().numpy() if self._numpy_io else t

    def _init_centers(self, Xc: torch.Tensor, mean: torch.Tensor, rs) -> torch.Tensor:
        N, D = Xc.shape
        K = self.n_clusters
        init = self.init
        C0 = new_padded(K, D, Xc.device, zero=True)
        if isinstance(init, str):
            if init == "random":
                seeds = torch.from_numpy(rs.permutation(N)[:K].astype(np.int64)).to(Xc.device)
                C0.copy_(Xc[seeds])
            elif init == "k-means++":
                from .kmeans_init import kmeans_plusplus_device
                C0.copy_(kmeans_plusplus_device(Xc, K, rs))
            else:
                raise ValueError(f"init should be 'k-means++', 'random' or an array, got {init!r}")
        else:
            arr = init if isinstance(init, torch.Tensor) else torch.from_numpy(
                np.ascontiguousarray(np.asarray(init), dtype=np.float32))
            if tuple(arr.shape) != (K, D):
                raise ValueError(
                    f"The shape of the initial centers {tuple(arr.shape)} does not match "
                    f"the number of clusters {K} / features {D}.")
            C0.copy_(arr.to(device=Xc.device, dtype=torch.float32))
            # init -= X_mean  (sklearn/_kmeans.py:1492-1493)
            _lib.call("gdr_add_row_vector", K, D, ptr(C0), C0.stride(0), ptr(mean), -1.0, stream())
        return C0

    # -- the Lloyd driver (sklearn/_kmeans.py:630-758) ----------------------------------
    def _lloyd(self, Xc: torch.Tensor, C0: torch.Tensor, tol_abs: float, S: _Scratch):
        N, D = Xc.shape
        K = self.n_clusters
        cur, nxt = 0, 1
        S.centers[cur].copy_(C0)
        lab_new, lab_old = 0, 1
        S.labels[lab_old].fill_(-1)
        strict = False
        n_iter = 0
        for i in range(int(self.max_iter)):
            n_iter = i + 1
            S.n_changed.zero_()
            ev = getattr(self, "_assign_events", None)
            if ev is not None:  # bench.py: CUDA-event pair around the dominant kernel
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            assign_labels(Xc, S.centers[cur], S.labels[lab_new], labels_prev=S.labels[lab_old],
                          n_changed=S.n_changed, precision_mode=S.mode, ws=S.ws_assign, tc_operand=S.tc,
                          n_refined=S.n_refined if S.tc is not None else None)
            if ev is not None:
                e1.record()
                ev.append((e0, e1))
            segment_sum(Xc, S.labels[lab_new], K, sums=S.sums, counts=S.counts, ws=S.ws_seg)
            self._finalize(S, cur, nxt)
            S.host[:2].copy_(S.stats[:2], non_blocking=True)
            S.host_i.copy_(S.n_changed, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            shift_tot, n_empty, n_changed = float(S.host[0]), int(S.host[1]), int(S.host_i[0])
            if n_empty > 0:
                # _relocate_empty_clusters_dense (sklearn/_k_means_common.pyx:167-211)
                _lib.call("gdr_kmeans_relocate", N, K, D, ptr(Xc), Xc.stride(0), ptr(S.centers[cur]),
                          S.centers[cur].stride(0), ptr(S.labels[lab_new]), ptr(S.sums), S.sums.stride(0),
                          ptr(S.counts), ptr(S.ws_misc), S.ws_misc.numel(), stream())
                self._finalize(S, cur, nxt)
                shift_tot = float(S.stats[0].item())
            if self.verbose:
                print(f"Iteration {i}, center shift {shift_tot:.6g}, labels changed {n_changed}.")
            cur, nxt = nxt, cur
            if n_changed == 0:
                strict = True
                break
            if shift_tot <= tol_abs:
                break
            lab_new, lab_old = lab_old, lab_new
        labels = S.labels[lab_new]
        if not strict:
            # rerun the E-step so that labels match the final centres (:742-754)
            assign_labels(Xc, S.centers[cur], labels, precision_mode=S.mode, ws=S.ws_assign, tc_operand=S.tc)
        inertia_dev = S.stats[0:1]
        _lib.call("gdr_inertia", N, D, ptr(Xc), Xc.stride(0), ptr(S.centers[cur]), S.centers[cur].stride(0),
                  ptr(labels), ptr(inertia_dev), ptr(S.ws_misc), S.ws_misc.numel(), stream())
        inertia = float(inertia_dev.item())
        return labels.clone(), inertia, S.centers[cur].clone(), n_iter

    def _lloyd_native(self, Xc: torch.Tensor, C0: torch.Tensor, tol_abs: float, mode: int):
        """One Lloyd run inside libgdr_b200 (gdr_kmeans_lloyd): same control flow as
        ``_lloyd`` below, but the ~20 launches per iteration are issued from C++."""
        N, D = Xc.shape
        K = int(self.n_clusters)
        centers = new_padded(K, D, Xc.device, zero=True)
        centers.copy_(C0)
        labels = torch.empty(N, dtype=torch.int32, device=Xc.device)
        ws = workspace(_lib.query("gdr_kmeans_lloyd_ws_bytes", N, K, D, mode), Xc.device)
        import ctypes
        inertia = ctypes.c_double(0.0)
        n_iter = ctypes.c_int32(0)
        info = (ctypes.c_int32 * 2)()
        _lib.call("gdr_kmeans_lloyd", N, K, D, ptr(Xc), Xc.stride(0), ptr(centers), centers.stride(0), ptr(labels),
                  int(self.max_iter), float(tol_abs), mode, ctypes.addressof(inertia), ctypes.addressof(n_iter),
                  ctypes.addressof(info), int(bool(self.verbose)), ptr(ws), ws.numel(), stream())
        self._strict_convergence = bool(info[0])
        self._relocations = int(info[1])
        return labels, float(inertia.value), centers, int(n_iter.value)

    @staticmethod
    def _finalize(S: _Scratch, cur: int, nxt: int):
        _lib.call("gdr_kmeans_finalize", S.K, S.D, ptr(S.sums), S.sums.stride(0), ptr(S.counts),
                  ptr(S.centers[cur]), S.centers[cur].stride(0), ptr(S.centers[nxt]),
                  S.centers[nxt].stride(0), ptr(S.stats), 0, stream())

    # -- public API ----------------------------------------------------------------
    def fit(self, X, y=None, sample_weight=None):
        if sample_weight is not None:
            raise NotImplementedError("sample_weight is not supported (the reference never passes it)")
        if self.algorithm not in ("lloyd", "auto", "full"):
            raise ValueError("only algorithm='lloyd' is implemented")
        Xd = self._to_device(X)
        N, D = Xd.shape
        K = int(self.n_clusters)
        if K <= 0:
            raise ValueError("n_clusters must be > 0")
        if N < K:
            raise ValueError(f"n_samples={N} should be >= n_clusters={K}.")
        dev = Xd.device
        mode = self._mode(D)
        rs = _check_random_state(self.random_state)

        # X -= X.mean(0) ; tol' = mean(var(X, axis=0)) * tol   (:1487-1489, :285-293)
        Xin = padded_rows(Xd)
        Xc = new_padded(N, D, dev)
        mean = torch.empty(D, dtype=torch.float32, device=dev)
        var_mean = torch.zeros(1, dtype=torch.float64, device=dev)
        ws = workspace(_lib.query("gdr_center_columns_ws_bytes", N, D), dev)
        _lib.call("gdr_center_columns", N, D, ptr(Xin), Xin.stride(0), ptr(mean), ptr(var_mean), ptr(Xc),
                  Xc.stride(0), ptr(ws), ws.numel(), stream())
        tol_abs = 0.0 if self.tol == 0 else float(var_mean.item()) * float(self.tol)
        self._tol = tol_abs

        init_is_array = not isinstance(self.init, str)
        n_init = self.n_init
        if n_init == "auto":
            n_init = 1 if (init_is_array or self.init == "k-means++") else 10
        if init_is_array:
            n_init = 1
        stepwise = getattr(self, "_assign_events", None) is not None  # Python loop only when instrumented
        if stepwise:
            S = _Scratch(N, K, D, dev, mode)
            if mode == 1:
                S.tc = TcOperand(Xc)
        best = None
        for _ in range(int(n_init)):
            C0 = self._init_centers(Xc, mean, rs)
            if stepwise:
                labels, inertia, centers, n_iter = self._lloyd(Xc, C0, tol_abs, S)
            else:
                labels, inertia, centers, n_iter = self._lloyd_native(Xc, C0, tol_abs, mode)
            if best is None or inertia < best[1]:
                best = (labels, inertia, centers, n_iter)
        labels, inertia, centers, n_iter = best
        # best_centers += X_mean (:1546)
        _lib.call("gdr_add_row_vector", K, D, ptr(centers), centers.stride(0), ptr(mean), 1.0, stream())
        self._centers_dev = centers
        self._labels_dev = labels
        self.cluster_centers_ = self._out(centers.contiguous() if pad4(D) == D else centers.clone().contiguous())
        self.labels_ = self._out(labels)
        self.inertia_ = inertia
        self.n_iter_ = n_iter
        self.n_features_in_ = D
        return self

    def fit_predict(self, X, y=None, sample_weight=None):
        return self.fit(X, sample_weight=sample_weight).labels_

    def predict(self, X):
        Xd = self._to_device(X)
        if Xd.shape[1] != self.n_features_in_:
            raise ValueError("X has a different number of features than the fitted model")
        Xp = padded_rows(Xd)
        labels = torch.empty(Xd.shape[0], dtype=torch.int32, device=Xd.device)
        assign_labels(Xp, padded_rows(self._centers_dev), labels, precision_mode=0)
        return self._out(labels)


class MiniBatchKMeans(KMeans):
    """scikit-learn's MiniBatchKMeans on the GPU — the estimator behind ``MiniBatchKMeans(n_clusters, random_state,
    batch_size)`` at clustgdd_agent_transduct.py:102-103, clustgdd_agent_induct.py:131-132 and
    distill_recsys.py:173-176.

    Control flow and arithmetic follow sklearn/cluster/_kmeans.py:2056-2224 (``fit``), :1566-1685 (``_mini_batch_step``),
    :1974-2053 (EWA early stopping, random reassignment) and _k_means_minibatch.pyx:56-110 (centre update):
    no mean-centring, validation subset + ``init_size`` subset for the initialisation, ``max_iter * N // batch`` steps of
    [sample a batch with replacement -> E-step on the batch -> per-centre running mean -> reassignment of starved
    centres], stop on ``max_no_improvement`` steps without a better smoothed inertia (or ``tol``), final E-step over all
    rows.  The random numbers come from numpy's RandomState on the host in the order sklearn draws them (``randint`` for
    the subsets, the k-means++ draws, ``choice(p=...)`` as cumsum + searchsorted per step, ``choice(replace=False)`` for the
    reassignments); every distance, assignment and update runs in libgdr_b200.  The E-step labels are exact up to the
    1e-6 margin band, so a trajectory can part from sklearn's at a near-tie: parity is judged on WCSS."""

    def __init__(self, n_clusters=8, *, init="k-means++", max_iter=100, batch_size=1024, verbose=0,
                 compute_labels=True, random_state=None, tol=0.0, max_no_improvement=10, init_size=None,
                 n_init="auto", reassignment_ratio=0.01, precision="auto", device=None):
        super().__init__(n_clusters=n_clusters, init=init, n_init=n_init, max_iter=max_iter, tol=tol, verbose=verbose,
                         random_state=random_state, precision=precision, device=device)
        self.batch_size, self.compute_labels, self.max_no_improvement = batch_size, compute_labels, max_no_improvement
        self.init_size, self.reassignment_ratio = init_size, reassignment_ratio

    # -- E-step + inertia of a row block against given centres (sklearn _labels_inertia) --
    @staticmethod
    def _labels_inertia(Xp: torch.Tensor, C: torch.Tensor, labels: torch.Tensor, mode: int = 0, tc=None):
        assign_labels(Xp, C, labels, precision_mode=0, tc_operand=tc if mode == 1 else None)
        return MiniBatchKMeans._inertia(Xp, C, labels)

    @staticmethod
    def _inertia(Xp: torch.Tensor, C: torch.Tensor, labels: torch.Tensor):
        out = torch.zeros(1, dtype=torch.float64, device=Xp.device)
        ws = workspace(_lib.query("gdr_inertia_ws_bytes", Xp.shape[0], Xp.shape[1]), Xp.device)
        _lib.call("gdr_inertia", Xp.shape[0], Xp.shape[1], ptr(Xp), Xp.stride(0), ptr(C), C.stride(0), ptr(labels), ptr(out),
                  ptr(ws), ws.numel(), stream())
        return out

    def _check_fit_args(self, N: int):
        """The argument checks of fit that depend on the data only through N."""
        K = int(self.n_clusters)
        if K <= 0:
            raise ValueError("n_clusters must be > 0")
        if N < K:
            raise ValueError(f"n_samples={N} should be >= n_clusters={K}.")
        if self.reassignment_ratio < 0:
            raise ValueError(f"reassignment_ratio should be >= 0, got {self.reassignment_ratio} instead.")

    def _mb_init(self, rows, N: int, D: int, dev, rs, init_size: int) -> torch.Tensor:
        """_init_centroids (sklearn/_kmeans.py:985-1060) on an ``init_size`` random subset (``rows``: see minibatch_loop)."""
        K = int(self.n_clusters)
        Xi = rows(rs.randint(0, N, init_size).astype(np.int64)) if init_size < N else rows(None)
        C0 = new_padded(K, D, dev, zero=True)
        if isinstance(self.init, str):
            if self.init == "k-means++":
                from .kmeans_init import kmeans_plusplus_device
                C0.copy_(kmeans_plusplus_device(Xi, K, rs))
            elif self.init == "random":
                n_i = Xi.shape[0]
                seeds = rs.choice(n_i, size=K, replace=False, p=np.ones(n_i, dtype=np.float32) / np.float32(n_i))
                C0.copy_(Xi[torch.from_numpy(np.asarray(seeds, dtype=np.int64)).to(dev)])
            else:
                raise ValueError(f"init should be 'k-means++', 'random' or an array, got {self.init!r}")
        else:
            arr = self.init if isinstance(self.init, torch.Tensor) else torch.from_numpy(
                np.ascontiguousarray(np.asarray(self.init), dtype=np.float32))
            if tuple(arr.shape) != (K, D):
                raise ValueError(f"The shape of the initial centers {tuple(arr.shape)} does not match "
                                 f"the number of clusters {K} / features {D}.")
            C0.copy_(arr.to(device=dev, dtype=torch.float32))
        return C0

    def fit(self, X, y=None, sample_weight=None):
        if sample_weight is not None:
            raise NotImplementedError("sample_weight is not supported (the reference never passes it)")
        Xd = self._to_device(X)
        N, D = Xd.shape
        self._check_fit_args(N)
        dev = Xd.device
        rs = _check_random_state(self.random_state)
        Xp = padded_rows(Xd.contiguous())

        def rows(idx):
            return Xp if idx is None else padded_rows(Xp[torch.from_numpy(idx).to(dev)].contiguous())

        def assemble(idx, C, labels_b):
            Xb = padded_rows(Xp[torch.from_numpy(idx).to(dev, non_blocking=True)].contiguous())
            assign_labels(Xb, C, labels_b, precision_mode=0)
            return Xb

        def var_mean():
            vm = torch.zeros(1, dtype=torch.float64, device=dev)
            mean = torch.empty(D, dtype=torch.float32, device=dev)
            scratch = new_padded(N, D, dev)
            ws = workspace(_lib.query("gdr_center_columns_ws_bytes", N, D), dev)
            _lib.call("gdr_center_columns", N, D, ptr(Xp), Xp.stride(0), ptr(mean), ptr(vm), ptr(scratch), scratch.stride(0),
                      ptr(ws), ws.numel(), stream())
            return float(vm.item())

        centers, ewa = minibatch_loop(self, N, D, dev, rs, rows, assemble, var_mean)
        self._centers_dev = centers
        self.n_features_in_ = D
        self.cluster_centers_ = self._out(centers.contiguous() if pad4(D) == D else centers.clone().contiguous())
        if self.compute_labels:
            labels = torch.empty(N, dtype=torch.int32, device=dev)
            mode = self._mode(D)
            tc = TcOperand(Xp) if mode == 1 else None
            self.inertia_ = float(self._labels_inertia(Xp, centers, labels, mode=mode, tc=tc).item())
            self._labels_dev = labels
            self.labels_ = self._out(labels)
        else:
            self.inertia_ = (ewa if ewa is not None else 0.0) * N
        return self


def minibatch_loop(est: MiniBatchKMeans, N: int, D: int, dev, rs, rows, assemble, var_mean):
    """The body of ``MiniBatchKMeans.fit`` between the argument checks and the final E-step, shared by the one-GPU
    estimator and ``parallel.DistMiniBatchKMeans``.  Every host draw, the EWA / early-stop logic, the centre update and
    the reassignment are here and run on replicated data; the rows of X enter through three seams:
      rows(idx)                      padded rows ``idx`` (numpy int64) of X, or X itself for ``idx`` None;
      assemble(idx, centers, labels) the padded batch rows X[idx], with ``labels[j]`` = the exact-fp32 label
                                     (precision_mode 0) of row j against ``centers``;
      var_mean()                     the mean of X's column variances (only called for tol > 0).
    Sets ``est.n_steps_`` and ``est.n_iter_``; returns (centres [K, D] padded, smoothed batch inertia or None)."""
    K = int(est.n_clusters)
    batch = min(int(est.batch_size), N)
    init_size = est.init_size
    if init_size is None:
        init_size = 3 * batch
        if init_size < K:
            init_size = 3 * K
    elif init_size < K:
        init_size = 3 * K
    init_size = min(int(init_size), N)
    init_is_array = not isinstance(est.init, str)
    n_init = est.n_init
    if n_init == "auto":
        n_init = 1 if (init_is_array or est.init == "k-means++") else 3
    if init_is_array:
        n_init = 1
    tol_abs = 0.0
    if est.tol > 0:       # _tolerance (:285-293): mean of the column variances * tol
        tol_abs = var_mean() * float(est.tol)

    # validation set for the initialisation (:2110-2112)
    X_valid = rows(rs.randint(0, N, init_size).astype(np.int64))
    lab_valid = torch.empty(X_valid.shape[0], dtype=torch.int32, device=dev)
    best_inertia, centers = None, None
    for _ in range(int(n_init)):
        cand = est._mb_init(rows, N, D, dev, rs, init_size)
        inertia = float(est._labels_inertia(X_valid, cand, lab_valid).item())
        if best_inertia is None or inertia < best_inertia:
            centers, best_inertia = cand, inertia
    centers_new = new_padded(K, D, dev, zero=True)
    counts = torch.zeros(K, dtype=torch.float32, device=dev)
    ewa, ewa_min, no_improvement, n_since = None, None, 0, 0
    n_steps = (int(est.max_iter) * N) // batch
    # RandomState.choice(n, size, p=w / w.sum(), replace=True): cdf = p.cumsum(); cdf /= cdf[-1];
    # cdf.searchsorted(random_sample(size), side="right") — the same table, built once
    w32 = np.ones(N, dtype=np.float32)
    cdf = (w32 / np.sum(w32)).astype(np.float64).cumsum()
    cdf /= cdf[-1]
    labels_b = torch.empty(batch, dtype=torch.int32, device=dev)
    host = torch.empty(2, dtype=torch.float64).pin_memory()
    step, any_zero = -1, True          # counts start at zero: the first step always reassigns
    for step in range(n_steps):
        Xb = assemble(cdf.searchsorted(rs.random_sample(batch), side="right").astype(np.int64), centers, labels_b)
        # _random_reassign (:2039-2053): every 10 * n_clusters samples, or as soon as a centre has no weight
        n_since += batch
        inertia_dev = est._inertia(Xb, centers, labels_b)
        _lib.call("gdr_minibatch_update", batch, K, D, ptr(Xb), Xb.stride(0), ptr(labels_b), ptr(centers), centers.stride(0),
                  ptr(centers_new), centers_new.stride(0), ptr(counts), stream())
        # the reassignment decision looks at the counts BEFORE this step's update in sklearn (the flag is an argument
        # of _mini_batch_step), so it is taken from the previous step's read-back
        reassign = any_zero or n_since >= 10 * K
        if reassign:
            n_since = 0
            if est.reassignment_ratio > 0:
                to_re = counts < float(est.reassignment_ratio) * counts.max()
                n_re = int(to_re.sum().item())
                if n_re > 0.5 * batch:
                    keep = torch.argsort(counts)[int(0.5 * batch):]
                    to_re[keep] = False
                    n_re = int(to_re.sum().item())
                if n_re:
                    picks = torch.from_numpy(np.asarray(rs.choice(batch, replace=False, size=n_re), dtype=np.int64)).to(dev)
                    centers_new[to_re] = Xb[picks]
                if n_re and n_re < K:
                    counts[to_re] = counts[~to_re].min()
        host[0:1].copy_(inertia_dev, non_blocking=True)
        host[1:2].copy_((counts == 0).any().to(torch.float64).reshape(1), non_blocking=True)
        csd = float(((centers_new - centers) ** 2).sum().item()) if tol_abs > 0 else 0.0
        centers, centers_new = centers_new, centers
        torch.cuda.current_stream().synchronize()
        any_zero = bool(host[1] > 0)
        # _mini_batch_convergence (:1974-2037)
        b_inertia = float(host[0]) / batch
        if step == 0:
            continue
        if ewa is None:
            ewa = b_inertia
        else:
            alpha = min(batch * 2.0 / (N + 1), 1.0)
            ewa = ewa * (1 - alpha) + b_inertia * alpha
        if est.verbose:
            print(f"Minibatch step {step + 1}/{n_steps}: mean batch inertia: {b_inertia}, ewa inertia: {ewa}")
        if tol_abs > 0.0 and csd <= tol_abs:
            break
        if ewa_min is None or ewa < ewa_min:
            no_improvement, ewa_min = 0, ewa
        else:
            no_improvement += 1
        if est.max_no_improvement is not None and no_improvement >= est.max_no_improvement:
            break
    est.n_steps_ = step + 1
    est.n_iter_ = int(np.ceil(((step + 1) * batch) / N))
    return centers, ewa


def standard_scale(X: torch.Tensor) -> torch.Tensor:
    """StandardScaler(with_mean=True, with_std=True).fit_transform (distill_recsys.py:172):
    mean / population variance in fp64, scale = sqrt(var) with zero variance -> 1,
    result fp32((x - fp32(mean)) / fp32(scale))."""
    X = X.to(torch.float32)
    if not X.is_cuda:
        raise ValueError("standard_scale needs a CUDA tensor (no CPU path)")
    N, D = X.shape
    Xin = X if X.stride(1) == 1 else X.contiguous()
    out = torch.empty((N, D), dtype=torch.float32, device=X.device)
    ws = workspace(_lib.query("gdr_standard_scale_ws_bytes", N, D), X.device)
    _lib.call("gdr_standard_scale", N, D, ptr(Xin), Xin.stride(0), ptr(out), out.stride(0), 0, 0, ptr(ws),
              ws.numel(), stream())
    return out


def kmeans_cluster(X, n_clusters: int, seed: int, minibatch: bool = True, batch_size: int = 2048,
                   init="k-means++", device=None, precision: str = "auto"):
    """distill_recsys.py:158-181 — returns (labels int64[N], centers f32[K, D]) as numpy.

    z-scores the columns, then clusters: MiniBatchKMeans(n_clusters, random_state=seed, batch_size, n_init="auto") when
    ``minibatch`` and more than 20 000 rows, else KMeans(n_clusters, random_state=seed, n_init="auto") — the reference's
    rule (:173-178).  ``init`` (an array, or "random") is an extension for parity runs with pinned centres."""
    if n_clusters <= 0:
        raise ValueError("n_clusters must be > 0")
    Xn = np.asarray(X)
    if n_clusters >= Xn.shape[0]:
        n_clusters = max(1, min(n_clusters, Xn.shape[0]))
    dev = device_of(device)
    Xd = torch.from_numpy(np.ascontiguousarray(Xn, dtype=np.float32)).to(dev)
    Xs = standard_scale(Xd)
    if minibatch and Xn.shape[0] > 20000:
        km = MiniBatchKMeans(n_clusters=n_clusters, random_state=seed, batch_size=batch_size, n_init="auto", init=init,
                             precision=precision)
    else:
        km = KMeans(n_clusters=n_clusters, random_state=seed, n_init="auto", init=init, precision=precision)
    labels = km.fit_predict(Xs)
    return labels.cpu().numpy().astype(np.int64), km.cluster_centers_.cpu().numpy().astype(np.float32)
