"""Joint-count path on B200 (SURVEY.md section 8(f)-4): mutual-information / symmetrical-uncertainty
matrices of discrete columns, and the two reference selectors that consume them.

Host-side mirror of ``fast_select.mutual_information`` (mutual_information.py:117-196),
``fast_select.mRMR`` (mRMR.py:30-152) and ``fast_select.CFS`` (CFS.py:246-429): same names,
parameters, validation and fitted attributes.  The pairwise statistics -- all of them, including
the p x p redundancy matrix the reference leaves to the CPU (mutual_information.py:191-193) --
come from one tensor-core GEMM over the reduced one-hot rows of the columns plus a finishing
kernel (fastselect_b200/csrc/joint.cu) through the C ABI; the greedy searches that follow are
O(p k) host work, as in the reference.  With ``pairs="selected"`` the estimators skip the p x p matrix
and ask for the k + 1 columns their search reads (fs_joint_columns), which is what lets them run on
genotype-scale p.  There is no CPU fallback.
"""
from __future__ import annotations

import math

import numpy as np
from sklearn.base import BaseEstimator, TransformerMixin
from sklearn.feature_selection import SelectorMixin
from sklearn.utils.validation import check_is_fitted, check_X_y, validate_data

from . import _native
from ._shard import dist_info, joint_sharded

_NO_GPU_MI = "backend='gpu' requested but CUDA not available"                                   # mutual_information.py:150
_NO_GPU_MRMR = ("GPU backend was selected, but no usable sm_100 GPU / CUDA driver was found. "
                "Please ensure you have an NVIDIA B200 with the latest drivers.")               # mRMR.py:60-64
_NO_GPU_CFS = "backend='gpu', but no CUDA-enabled GPU is available."                            # CFS.py:347
_NO_CPU = ("fastselect_b200 implements only the GPU backend of the joint-count path; "
           "backend='cpu' is not available (use the reference package for CPU runs).")
MAX_STATES = _native.FS_DISTINCT_CAP        # distinct values per column on the tensor-core path


def _validate_discrete(arr, name):
    """mutual_information.py:13-22: integer codes, none negative."""
    arr = np.asarray(arr)
    if not np.issubdtype(arr.dtype, np.integer):
        raise ValueError(f"{name} must be an integer-coded array (got {arr.dtype}). "
                         "Discretise continuous data before calling this function.")
    if arr.size and arr.min() < 0:
        raise ValueError(f"{name} contains negative values; expected 0..K-1 codes.")
    return arr


def _resolve_backend(backend, message):
    if backend == "cpu":
        raise NotImplementedError(_NO_CPU)
    if backend not in ("auto", "gpu"):
        raise ValueError("backend must be one of 'auto', 'gpu', or 'cpu'")
    if _native.device_count() < 1:
        raise RuntimeError(message)


def _stack_for_upload(x, y):
    """[x | y] in the narrowest element type the library takes that holds every value exactly;
    only the partition of the samples by value matters on the device."""
    lo = min(int(x.min()), int(y.min()))
    hi = max(int(x.max()), int(y.max()))
    if 0 <= lo and hi <= 255:
        dt = np.uint8
    elif -(1 << 24) <= lo and hi <= (1 << 24):
        dt = np.float32
    elif -(1 << 53) <= lo and hi <= (1 << 53):
        dt = np.float64
    else:
        raise ValueError("integer codes beyond 2^53 cannot be uploaded exactly")
    out = np.empty((x.shape[0], x.shape[1] + 1), dt)
    out[:, :-1] = x
    out[:, -1] = y
    return out


def _open_discrete(codes):
    """A data set over the integer matrix ``codes`` ([n, q]) with every column typed discrete."""
    n, q = codes.shape
    if n < 2:
        raise ValueError(f"need at least 2 samples, got {n}")
    arith = _native.FS_ARITH_F64 if codes.dtype == np.float64 else _native.FS_ARITH_F32
    ds = _native.Dataset(codes, np.zeros(n, np.int32), 1)
    try:
        _, _, cnt = ds.column_stats()
        if int(cnt.max()) > MAX_STATES:
            bad = int(np.argmax(cnt > MAX_STATES))
            raise ValueError(f"GPU backend supports up to {MAX_STATES} unique states/bins "
                             f"(column {bad} has more).")
        ds.set_features(np.ones(q, np.uint8), np.ones(q, np.float32), arith)
    except BaseException:
        ds.close()
        raise
    return ds


def joint_matrix(codes, kind, log_base=1.0, stats_out=None):
    """Pairwise statistic of every column pair of the integer matrix ``codes`` ([n, q]): float64
    ``[q, q]`` with a zero diagonal.  One process per GPU: every rank uploads the matrix, computes a
    band of rows balanced over the upper triangle, and ONE allreduce sums the bands.  ``stats_out``
    (a dict) receives this rank's ``fs_stats``."""
    codes = np.asarray(codes)
    q = codes.shape[1]
    with _open_discrete(codes) as ds:

        def compute_band(lo, hi, out_ptr):
            res = ds.joint_matrix(kind, log_base, pos_begin=lo, pos_end=hi, out_device_ptr=out_ptr,
                                  want_stats=stats_out is not None)
            if stats_out is not None:
                res, st = res
                stats_out.update(st)
            return res

        _, world = dist_info()
        nccl = False
        if world > 1:
            import torch.distributed as dist

            nccl = dist.get_backend() == "nccl"
        return joint_sharded(q, compute_band, device_buffers=nccl)


class JointColumns:
    """One data set held open for a whole fit: ``columns(positions)`` returns the statistic of each
    position of the integer matrix ``codes`` ([n, q]) against every position, float64
    ``[len(positions), q]`` -- bitwise the rows of :func:`joint_matrix`, without the q x q matrix.  The
    first call encodes the columns; later calls reuse the encoding.  Runs on this process's GPU with no
    communication: under ``enable_distributed`` / ``set_gpus`` every rank computes the same columns."""

    def __init__(self, codes, kind, log_base=1.0):
        self.kind, self.log_base = kind, log_base
        self._ds = _open_discrete(np.asarray(codes))

    def columns(self, positions):
        return self._ds.joint_columns(self.kind, self.log_base, positions)

    def close(self):
        self._ds.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def open_joint_columns(codes, kind, log_base=1.0):
    """The GPU behind ``pairs="selected"``: a :class:`JointColumns` over ``codes``."""
    return JointColumns(codes, kind, log_base)


_PAIRS = ("all", "selected")


def _check_pairs(pairs):
    if pairs not in _PAIRS:
        raise ValueError(f"pairs must be 'all' or 'selected' (got {pairs!r}).")


def calculate_mi_matrices(X, y, *, backend="auto", unit="bit"):
    """(relevance [p], redundancy [p, p]) of integer-coded data, float64 (mutual_information.py:158-196).
    Redundancy is symmetric with a zero diagonal (:53, :58-62)."""
    X = np.asarray(X)
    y = np.asarray(y)
    if X.ndim != 2 or y.ndim != 1 or X.shape[0] != y.shape[0]:
        raise ValueError("X must be 2-D and y 1-D with matching sample size")
    X = _validate_discrete(X, "X")
    y = _validate_discrete(y, "y")
    _resolve_backend(backend, _NO_GPU_MI)
    return _mi_matrices(X, y, math.log(2.0) if unit == "bit" else 1.0)


def _mi_matrices(X, y, log_base):
    """I(f; y) and I(f; g) of integer matrices whose VALUES are the states (any integers)."""
    p = X.shape[1]
    m = joint_matrix(_stack_for_upload(X, y), _native.FS_JOINT_MI, log_base)
    return m[p, :p].copy(), np.ascontiguousarray(m[:p, :p])


def calculate_mi_single_pair(x1, x2, *, backend="auto", unit="bit"):
    """I(x1; x2) of two integer-coded vectors (mutual_information.py:117-155)."""
    x1 = np.asarray(x1)
    x2 = np.asarray(x2)
    if x1.ndim != 1 or x2.ndim != 1 or x1.shape != x2.shape:
        raise ValueError("x1 and x2 must be 1-D arrays of equal length")
    x1 = _validate_discrete(x1.ravel(), "x1")
    x2 = _validate_discrete(x2.ravel(), "x2")
    _resolve_backend(backend, _NO_GPU_MI)
    log_base = math.log(2.0) if unit == "bit" else 1.0
    m = joint_matrix(_stack_for_upload(x1[:, None], x2), _native.FS_JOINT_MI, log_base)
    return float(m[0, 1])


class mRMR(BaseEstimator, TransformerMixin):
    """Minimum-redundancy maximum-relevance selection on discrete data (drop-in for
    ``fast_select.mRMR``, GPU backend; mRMR.py:30-152).

    ``method``: 'MID' scores ``I(f; y) - mean I(f; S)``, 'MIQ' the quotient (:114-117).

    ``pairs`` chooses what the fit returns.  ``"all"`` (the reference's behaviour) computes the whole
    p x p redundancy matrix and keeps it as ``redundancy_matrix_``.  ``"selected"`` computes only the
    columns the greedy search reads -- relevance, then one column per selected feature -- and keeps
    those as ``redundancy_columns_`` (float64 ``[k, p]``, row i = ``I(top_features_[i]; .)``, equal to
    ``redundancy_matrix_[top_features_]``); ``redundancy_matrix_`` is not set.  Everything else is
    identical bit for bit.  Because the two differ in what they return, the choice is the caller's and
    is never made automatically; use ``"selected"`` when p x p float64 does not fit (p = 100 000 is 80 GB)."""

    def __init__(self, n_features_to_select: int, method: str = "MID", backend: str = "gpu", pairs: str = "all"):
        self.n_features_to_select = n_features_to_select
        self.method = method
        self.backend = backend
        self.pairs = pairs
        if self.method not in ["MID", "MIQ"]:
            raise ValueError("Method must be either 'MID' or 'MIQ'.")
        _check_pairs(self.pairs)
        if self.backend not in ["cpu", "gpu"]:
            raise ValueError("Backend must be either 'cpu' or 'gpu'.")
        if self.backend == "cpu":
            raise NotImplementedError(_NO_CPU)
        if _native.device_count() < 1:
            raise RuntimeError(_NO_GPU_MRMR)

    def fit(self, X, y):
        X, y = validate_data(self, X, y, dtype=None, y_numeric=True, ensure_2d=True)
        self.n_features_in_ = X.shape[1]
        if not (0 < self.n_features_to_select <= self.n_features_in_):
            raise ValueError("n_features_to_select must be a positive integer less "
                             "than or equal to the number of features.")
        # the reference recodes X and y against the sorted union of their values (:90-92); the
        # statistics only depend on which samples share a value, so the data goes up as it is
        self.unique_vals_ = np.unique(np.concatenate([np.unique(X), np.unique(y)]))
        for arr, name in ((X, "X"), (y, "y")):          # what _validate_discrete sees there: the codes keep X's dtype
            if not np.issubdtype(arr.dtype, np.integer):
                raise ValueError(f"{name} must be an integer-coded array (got {arr.dtype}). "
                                 "Discretise continuous data before calling this function.")
        _check_pairs(self.pairs)
        for attr in ("redundancy_matrix_", "redundancy_columns_"):
            self.__dict__.pop(attr, None)
        if self.pairs == "all":
            relevance, redundancy = _mi_matrices(X, y, math.log(2.0))
            self.relevance_scores_ = relevance
            self.redundancy_matrix_ = redundancy
            self.top_features_ = self._select(relevance, redundancy, self.n_features_to_select, self.method)
        else:
            p = X.shape[1]
            with open_joint_columns(_stack_for_upload(X, y), _native.FS_JOINT_MI, math.log(2.0)) as src:
                relevance = src.columns([p])[0, :p].copy()
                fetched = []

                def column(f):
                    fetched.append(src.columns([f])[0, :p])
                    return fetched[-1]

                self.relevance_scores_ = relevance
                self.top_features_ = self._select_columns(relevance, column, self.n_features_to_select, self.method)
            self.redundancy_columns_ = np.stack(fetched)
        self.feature_importances_ = self.relevance_scores_
        return self

    @staticmethod
    def _select(relevance, redundancy, n_select, method):
        """Greedy forward selection of mRMR.py:102-131 on the full redundancy matrix."""
        return mRMR._select_columns(relevance, lambda f: redundancy[:, f], n_select, method)

    @staticmethod
    def _select_columns(relevance, column, n_select, method):
        """Greedy forward selection of mRMR.py:102-131: start at the most relevant feature, then
        repeatedly take the best MID / MIQ score; candidates that ``np.isclose`` to the best score
        are separated by the smaller mean redundancy.  ``column(f)`` is ``redundancy[:, f]``; it is
        asked once for every selected feature, in selection order."""
        p = relevance.size
        selected = np.zeros(n_select, dtype=np.int32)
        remaining = np.ones(p, dtype=bool)
        first = int(np.argmax(relevance))
        selected[0] = first
        remaining[first] = False
        red_sum = column(first).copy()
        for i in range(1, n_select):
            idx = np.flatnonzero(remaining)
            mean_red = red_sum[idx] / i
            if method == "MID":
                scores = relevance[idx] - mean_red
            else:
                scores = relevance[idx] / (mean_red + 1e-9)
            cand = idx[np.isclose(scores, np.max(scores), atol=1e-12)]
            best = cand[np.argmin(red_sum[cand] / i)] if cand.size > 1 else cand[0]
            selected[i] = best
            remaining[best] = False
            red_sum += column(best)
        return selected

    def transform(self, X):
        """Reduce X to the selected features (mRMR.py:138-147)."""
        check_is_fitted(self)
        X = validate_data(self, X, reset=False, dtype=None)
        return X[:, self.top_features_]

    def fit_transform(self, X, y):
        self.fit(X, y)
        return self.transform(X)


def _cfs_merit(sum_r_cf, k, sum_r_ff):
    """CFS.py:11-23, elementwise on arrays of candidate sums."""
    if k == 0:
        return np.zeros_like(np.asarray(sum_r_cf, np.float64))
    r_cf_avg = sum_r_cf / k
    r_ff_avg = (2.0 * sum_r_ff) / (k * (k - 1)) if k > 1 else np.zeros_like(np.asarray(sum_r_ff, np.float64))
    denom = np.sqrt(k + k * (k - 1) * r_ff_avg)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(denom > 1e-12, (k * r_cf_avg) / denom, 0.0)


def _best_first_search(r_cf, r_ff, min_r_cf=0.1):
    """Greedy forward search of CFS.py:114-162 on the full correlation matrix."""
    return _best_first_search_columns(r_cf, lambda s: r_ff[:, s], min_r_cf)


def _best_first_search_columns(r_cf, column, min_r_cf=0.1):
    """Greedy forward search of CFS.py:114-162: grow the subset by the candidate with the largest
    merit while the merit strictly improves.  The sums are formed in the reference's order (the
    subset's own terms first, then the candidate's) so that ties fall the same way.  ``column(s)`` is
    ``r_ff[:, s]``; it is only asked for features already in the subset."""
    p = r_cf.size
    first = int(np.argmax(r_cf))
    if r_cf[first] < min_r_cf:
        return []
    selected = [first]
    current = float(r_cf[first])
    eligible = ~(r_cf.astype(np.float64) < min_r_cf)     # the reference compares in float64 (numba promotion)
    while True:
        k = len(selected) + 1
        base_cf = 0.0
        for s in selected:
            base_cf += float(r_cf[s])
        base_ff = 0.0
        for a in selected:
            for b in selected:
                if a < b:
                    base_ff += float(column(b)[a])
        sum_cf = base_cf + r_cf.astype(np.float64)
        sum_ff = np.full(p, base_ff)
        for s in selected:
            sum_ff = sum_ff + column(s).astype(np.float64)
        merit = _cfs_merit(sum_cf, k, sum_ff)
        ok = eligible.copy()
        ok[selected] = False
        if not ok.any():
            break
        merit = np.where(ok, merit, -np.inf)
        best = int(np.argmax(merit))             # first index of the largest merit, as the scan at :127-154
        if merit[best] > current:
            selected.append(best)
            current = float(merit[best])
        else:
            break
    return selected


def _prune_redundant(selected, r_cf, r_ff):
    """Redundancy filter of CFS.py:106-112 on the full correlation matrix."""
    return _prune_redundant_columns(selected, r_cf, lambda s: r_ff[:, s])


def _prune_redundant_columns(selected, r_cf, column):
    """Redundancy filter of CFS.py:106-112: visit the chosen features from the most to the least
    class-correlated (stable, so equal correlations keep their index order) and keep one only if no
    feature kept so far is at least as correlated with it as the class is.  ``column(s)`` is
    ``r_ff[:, s]`` and is only asked for features in ``selected``."""
    selected = np.asarray(selected, dtype=int)
    order = selected[np.argsort(-r_cf[selected], kind="stable")]
    kept = []
    for f in order.tolist():
        if kept and bool((np.array([column(k)[f] for k in kept]) >= r_cf[f]).any()):
            continue
        kept.append(f)
    return kept


def _subset_merit(selected, r_cf, column):
    """CFS.py:406-409 merit of the final subset: the float32 sums of the subset's ``r_cf`` and of the
    upper triangle of its ``r_ff`` block, formed as ``np.sum`` forms them on the full matrix."""
    k = len(selected)
    if k == 0:
        return 0.0
    block = np.empty((k, k), np.float32)
    for j, b in enumerate(selected):
        block[:, j] = column(b)[selected]
    sum_r_cf = np.sum(r_cf[selected])
    sum_r_ff = np.sum(np.triu(block, k=1))
    return float(_cfs_merit(np.float64(sum_r_cf), k, np.float64(sum_r_ff)))


class CFS(BaseEstimator, SelectorMixin):
    """Correlation-based feature selection with symmetrical uncertainty (drop-in for
    ``fast_select.CFS``, GPU backend; CFS.py:246-429).  Continuous columns are binned with
    ``KBinsDiscretizer`` on the host exactly as the reference does; the correlations of all pairs
    come from the tensor-core joint-count kernels; ``n_bins`` and the number of distinct values of
    a discrete column must not exceed 16 (the reference's own GPU kernel stops at 32, CFS.py:349-350).

    ``pairs`` chooses what the fit returns.  ``"all"`` (the reference's behaviour) computes every
    feature-feature correlation and keeps the p x p matrix as ``r_ff_``.  ``"selected"`` computes the
    class column (``r_cf_``) and one column per feature the forward search accepts, and does not set
    ``r_ff_``; ``selected_indices_``, ``support_mask_``, ``merit_`` and ``r_cf_`` are identical bit for
    bit.  Because the two differ in what they return, the choice is the caller's and is never made
    automatically; use ``"selected"`` when p x p does not fit."""

    def __init__(self, n_bins=10, strategy="uniform", backend="auto", n_jobs=-1, pairs="all"):
        self.n_bins = n_bins
        self.strategy = strategy
        self.backend = backend
        self.n_jobs = n_jobs
        self.pairs = pairs

    def fit(self, X, y):
        feature_names = np.asarray(X.columns) if hasattr(X, "columns") else None
        X, y = check_X_y(X, y, dtype=None, ensure_min_samples=2)
        self.n_features_in_ = X.shape[1]
        if feature_names is not None:
            self.feature_names_in_ = feature_names
        codes, n_states = self._encode(X)
        unique_y, y_encoded = np.unique(y, return_inverse=True)
        if self.backend == "cpu":
            raise NotImplementedError(_NO_CPU)
        if self.backend not in ("auto", "gpu"):
            raise ValueError("backend must be one of 'auto', 'gpu', or 'cpu'")
        _check_pairs(self.pairs)
        if _native.device_count() < 1:
            raise RuntimeError(_NO_GPU_CFS)
        if len(unique_y) > MAX_STATES or (n_states.size and int(n_states.max()) > MAX_STATES):
            raise ValueError(f"GPU backend supports up to {MAX_STATES} unique states/bins.")
        p = self.n_features_in_
        self.__dict__.pop("r_ff_", None)
        if self.pairs == "all":
            su = joint_matrix(_stack_for_upload(codes, y_encoded), _native.FS_JOINT_SU)
            r_cf = su[p, :p].astype(np.float32)                      # the reference's arrays are float32 (:88, :95)
            r_ff = np.ascontiguousarray(su[:p, :p], dtype=np.float32)
            self.r_cf_, self.r_ff_ = r_cf, r_ff
            self._search(r_cf, lambda s: r_ff[:, s])
        else:
            with open_joint_columns(_stack_for_upload(codes, y_encoded), _native.FS_JOINT_SU) as src:
                self.r_cf_ = src.columns([p])[0, :p].astype(np.float32)
                cache = {}

                def column(s):
                    if s not in cache:
                        cache[s] = src.columns([s])[0, :p].astype(np.float32)
                    return cache[s]

                self._search(self.r_cf_, column)
        return self

    def _search(self, r_cf, column):
        """Best-first search, redundancy filter and merit (CFS.py:375-409); ``column(s)`` is ``r_ff[:, s]``."""
        p = r_cf.size
        selected = _best_first_search_columns(r_cf, column)
        selected = np.sort(np.array(selected, dtype=int))
        self.selected_indices_ = np.sort(np.array(_prune_redundant_columns(selected, r_cf, column), dtype=int))
        self.support_mask_ = np.zeros(p, dtype=bool)
        if len(self.selected_indices_) > 0:
            self.support_mask_[self.selected_indices_] = True
        self.merit_ = _subset_merit(self.selected_indices_, r_cf, column)

    def _encode(self, X):
        """CFS.py:319-334: floating columns -> ``n_bins`` ordinal bins, other columns -> the rank of
        each value among the column's distinct values."""
        from sklearn.preprocessing import KBinsDiscretizer

        p = X.shape[1]
        is_cont = np.array([np.issubdtype(X[:, i].dtype, np.floating) for i in range(p)])
        codes = np.zeros(X.shape, dtype=np.int32)
        n_states = np.zeros(p, dtype=np.int32)
        cont = np.flatnonzero(is_cont)
        if cont.size:
            disc = KBinsDiscretizer(n_bins=self.n_bins, encode="ordinal", strategy=self.strategy, subsample=None)
            codes[:, cont] = disc.fit_transform(X[:, cont]).astype(np.int32)
            n_states[cont] = self.n_bins
        for i in np.flatnonzero(~is_cont):
            vals, inv = np.unique(X[:, i], return_inverse=True)
            codes[:, i] = inv
            n_states[i] = len(vals)
        return codes, n_states

    def _get_support_mask(self):
        check_is_fitted(self)
        return self.support_mask_

    def transform(self, X):
        """Reduce X to the selected features; DataFrames keep their labels (CFS.py:411-429)."""
        check_is_fitted(self)
        if hasattr(X, "iloc"):
            return X.iloc[:, self.support_mask_]
        return X[:, self.support_mask_]
