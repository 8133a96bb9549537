"""MDR (multifactor dimensionality reduction) on B200: exhaustive one- and two-locus search for the column
combination whose high-risk / low-risk cell labelling best separates a binary class, scored by
cross-validated balanced accuracy.

The name and outline follow ``fast_select.MDR`` (k-way combinations, stratified k-fold cross-validation,
balanced accuracy, 3-state genotypes), but the exact semantics are this project's own (DESIGN.md, "MDR")
and have not been checked against the reference implementation.  The scan over all combinations runs in
fastselect_b200/csrc/mdr.cu through the C ABI; the host only assigns folds, ranks the few fold winners and
builds the final model from exact cell counts.  There is no CPU fallback.
"""
from __future__ import annotations

import numpy as np
from sklearn.base import BaseEstimator, ClassifierMixin, TransformerMixin
from sklearn.model_selection import StratifiedKFold
from sklearn.utils.validation import check_is_fitted, validate_data

from . import _native

MAX_STATES = 3
_NO_GPU = "MDR needs a usable sm_100 GPU (NVIDIA B200); none was found."
_NO_CPU = ("fastselect_b200 implements only the GPU backend of MDR; backend='cpu' is not available "
           "(use the reference package for CPU runs).")


def make_folds(y_enc, cv, random_state):
    """fold[i] in [0, cv): StratifiedKFold, shuffled only when a random_state is given."""
    shuffle = random_state is not None
    skf = StratifiedKFold(n_splits=cv, shuffle=shuffle, random_state=random_state if shuffle else None)
    fold = np.empty(y_enc.size, np.int32)
    for f, (_, test) in enumerate(skf.split(np.zeros((y_enc.size, 1)), y_enc)):
        fold[test] = f
    return fold


def decode_combinations(idx, p, order):
    """Combination indices -> positions, int64 ``[m, order]``.  Order 2: the lexicographic rank of (a, b),
    a < b, i.e. ``idx = a * p - a * (a + 1) / 2 + (b - a - 1)``."""
    idx = np.asarray(idx, np.int64).reshape(-1)
    if order == 1:
        return idx[:, None].copy()
    # first index of row a: off(a) = a * p - a * (a + 1) / 2; a from the quadratic, then exact integer fix-ups
    q = 2.0 * p - 1.0
    a = np.floor((q - np.sqrt(np.maximum(q * q - 8.0 * idx, 0.0))) / 2.0).astype(np.int64)
    a = np.clip(a, 0, max(p - 2, 0))

    def off(v):
        return v * p - v * (v + 1) // 2

    while True:
        lo = off(a) > idx
        hi = off(a + 1) <= idx
        if not (lo.any() or hi.any()):
            break
        a = a - lo + hi
    return np.stack([a, idx - off(a) + a + 1], axis=1)


def encode_combinations(combos, p):
    """Inverse of :func:`decode_combinations` (positions ``[m, order]`` -> indices)."""
    combos = np.asarray(combos, np.int64)
    if combos.shape[1] == 1:
        return combos[:, 0].copy()
    a, b = combos[:, 0], combos[:, 1]
    return a * p - a * (a + 1) // 2 + (b - a - 1)


def fold_scores(tables):
    """Training and test balanced accuracy of every fold from ``[m, cv, 2, 9]`` cell counts, float64
    ``[m, cv]`` each: the integer rule and the single division of the kernel."""
    t = np.asarray(tables, np.int64)
    alls = t.sum(1)                                       # [m, 2, 9]
    m, cv = t.shape[:2]
    train = np.empty((m, cv))
    test = np.empty((m, cv))
    for f in range(cv):
        e0, e1 = t[:, f, 0], t[:, f, 1]
        t0, t1 = alls[:, 0] - e0, alls[:, 1] - e1
        M0, M1, N0, N1 = e0.sum(1), e1.sum(1), t0.sum(1), t1.sum(1)
        high = t1 * N0[:, None] > t0 * N1[:, None]
        TP, TN = np.where(high, t1, 0).sum(1), np.where(high, 0, t0).sum(1)
        tp, tn = np.where(high, e1, 0).sum(1), np.where(high, 0, e0).sum(1)
        train[:, f] = (TP * N0 + TN * N1).astype(np.float64) / (2 * N1 * N0).astype(np.float64)
        test[:, f] = (tp * M0 + tn * M1).astype(np.float64) / (2 * M1 * M0).astype(np.float64)
    return train, test


def _fold_mean(v):
    acc = np.zeros(v.shape[0])
    for f in range(v.shape[1]):                          # sequential, in fold order, as the kernel sums
        acc = acc + v[:, f]
    return acc / v.shape[1]


def _upload_array(X):
    """X in an element type the library takes that keeps every distinct value distinct."""
    if X.dtype in (np.uint8, np.int8, np.float32, np.float64):
        return X
    if X.dtype == np.bool_:
        return X.astype(np.uint8)
    if np.issubdtype(X.dtype, np.integer):
        lo, hi = (int(X.min()), int(X.max())) if X.size else (0, 0)
        if 0 <= lo and hi <= 255:
            return X.astype(np.uint8)
        if -128 <= lo and hi <= 127:
            return X.astype(np.int8)
        if -(1 << 53) <= lo and hi <= (1 << 53):
            return X.astype(np.float64)
        raise ValueError("integer values beyond 2^53 cannot be uploaded exactly")
    return X.astype(np.float64)


class MDRData:
    """One data set held open for a fit: X ([n, p]) with the binary class ``y_enc`` on this process's GPU.
    ``n_states`` holds every column's number of distinct values (from the device's column scan; values
    above 16 read as 17).  Under ``enable_distributed`` / ``set_gpus`` every rank runs its own scan."""

    def __init__(self, X, y_enc):
        x = _upload_array(np.asarray(X))
        self._ds = _native.Dataset(x, np.asarray(y_enc, np.int32), 2)
        try:
            _, _, cnt = self._ds.column_stats()
            self.n_states = cnt.astype(np.int64)
            arith = _native.FS_ARITH_F64 if x.dtype == np.float64 else _native.FS_ARITH_F32
            p = x.shape[1]
            self._ds.set_features(np.ones(p, np.uint8), np.ones(p, np.float32), arith)
        except BaseException:
            self._ds.close()
            raise

    def scan(self, fold, order, n_top, want_all=False):
        return self._ds.mdr_scan(fold, order, n_top, want_all=want_all)

    def tables(self, fold, order, combos):
        return self._ds.mdr_tables(fold, order, combos)

    def interaction_scan(self, n_top, want_all=False):
        return self._ds.interaction_scan(n_top, want_all=want_all)

    def close(self):
        self._ds.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def open_mdr(X, y_enc):
    """The GPU behind :class:`MDR`: an :class:`MDRData` over ``X`` and ``y_enc``."""
    return MDRData(X, y_enc)


class MDR(BaseEstimator, ClassifierMixin, TransformerMixin):
    """Multifactor dimensionality reduction over every combination of ``order`` (1 or 2) columns.

    Every column must hold at most 3 distinct values (genotypes 0/1/2, or any 3 numbers); ``y`` exactly 2
    labels, ``classes_[1]`` being the case class.  Samples go to ``cv`` folds by ``StratifiedKFold``
    (shuffled with ``random_state`` when one is given).  Per combination and fold, a cell is high-risk when
    its case / control ratio in the training folds exceeds the overall training ratio; the combination is
    scored by the balanced accuracy of that labelling on the training folds and on the held-out fold.

    ``best_combination_`` is the fold winner (highest training balanced accuracy of a fold) that wins the
    most folds (``cv_consistency_``), then has the higher mean test balanced accuracy, then the lower
    combination index.  ``top_combinations_`` lists the ``n_top`` best by mean test balanced accuracy.
    ``predict`` labels a sample ``classes_[1]`` when its cell of the best combination is high-risk on all
    samples; values not seen in ``fit`` are low-risk.  ``transform`` keeps the best combination's columns.
    The semantics are this project's own and have not been checked against ``fast_select.MDR``."""

    def __init__(self, order=2, cv=5, n_top=100, random_state=None, backend="auto"):
        self.order = order
        self.cv = cv
        self.n_top = n_top
        self.random_state = random_state
        self.backend = backend

    def _check_params(self):
        if isinstance(self.order, bool) or self.order not in (1, 2):
            raise ValueError(f"order must be 1 or 2 (got {self.order!r}).")
        if isinstance(self.cv, bool) or not isinstance(self.cv, (int, np.integer)) or not 2 <= self.cv <= 10:
            raise ValueError(f"cv must be an integer in [2, 10] (got {self.cv!r}).")
        if (isinstance(self.n_top, bool) or not isinstance(self.n_top, (int, np.integer))
                or not 1 <= self.n_top <= _native.FS_MDR_MAX_TOP):
            raise ValueError(f"n_top must be an integer in [1, {_native.FS_MDR_MAX_TOP}] (got {self.n_top!r}).")
        if self.backend == "cpu":
            raise NotImplementedError(_NO_CPU)
        if self.backend not in ("auto", "gpu"):
            raise ValueError("backend must be one of 'auto', 'gpu', or 'cpu'")

    def fit(self, X, y):
        X, y = validate_data(self, X, y, dtype=None, ensure_min_samples=2)
        if not (np.issubdtype(X.dtype, np.number) or X.dtype == np.bool_):
            raise ValueError(f"X must be numeric (got {X.dtype}).")
        self._check_params()
        order, cv = int(self.order), int(self.cv)
        classes, y_enc = np.unique(y, return_inverse=True)
        if classes.size != 2:
            raise ValueError(f"MDR needs exactly 2 classes in y (got {classes.size}).")
        if int(np.bincount(y_enc, minlength=2).min()) < cv:
            raise ValueError(f"each class needs at least cv = {cv} samples.")
        p = X.shape[1]
        if p < order:
            raise ValueError(f"order {order} needs at least {order} features (got {p}).")
        if _native.device_count() < 1:
            raise RuntimeError(_NO_GPU)
        fold = make_folds(y_enc, cv, self.random_state)
        n_combos = p if order == 1 else p * (p - 1) // 2
        with open_mdr(X, y_enc) as src:
            bad = np.flatnonzero(np.asarray(src.n_states) > MAX_STATES)
            if bad.size:
                raise ValueError(f"MDR supports columns with at most {MAX_STATES} distinct values "
                                 f"(column {int(bad[0])} has more).")
            res = src.scan(fold, order, min(int(self.n_top), n_combos))
            fbest = np.asarray(res["fold_best"], np.int64)[:cv]
            cand = np.unique(fbest)
            cand_tables = src.tables(fold, order, decode_combinations(cand, p, order))
        train, test = fold_scores(cand_tables)
        mean_train, mean_test = _fold_mean(train), _fold_mean(test)
        cvc = np.array([int(np.sum(fbest == c)) for c in cand])
        k = min(range(cand.size), key=lambda i: (-cvc[i], -mean_test[i], cand[i]))
        full = cand_tables[k].sum(0)                      # [2, 9] over all samples
        high = full[1] * full[0].sum() > full[0] * full[1].sum()
        best = tuple(int(v) for v in decode_combinations(cand[k:k + 1], p, order)[0])

        self.classes_ = classes
        self.best_combination_ = best
        self.cv_consistency_ = int(cvc[k])
        self.train_balanced_accuracy_ = float(mean_train[k])
        self.test_balanced_accuracy_ = float(mean_test[k])
        self.top_combinations_ = decode_combinations(res["top_idx"], p, order)
        self.top_train_balanced_accuracy_ = np.asarray(res["top_train"], np.float64)
        self.top_test_balanced_accuracy_ = np.asarray(res["top_test"], np.float64)
        self.fold_best_combinations_ = decode_combinations(fbest, p, order)
        self.feature_values_ = [np.unique(X[:, f]) for f in best]
        self.high_risk_ = high.reshape(3, 3)[:, 0].copy() if order == 1 else high.reshape(3, 3)
        return self

    def _cells(self, X):
        """Cell of every sample under the best combination, -1 where a value was not seen in fit."""
        cell = np.zeros(X.shape[0], np.int64)
        seen = np.ones(X.shape[0], bool)
        for j, f in enumerate(self.best_combination_):
            vals = self.feature_values_[j]
            col = X[:, f]
            pos = np.clip(np.searchsorted(vals, col), 0, vals.size - 1)
            seen &= vals[pos] == col
            cell = cell * 3 + pos
        if len(self.best_combination_) == 1:
            cell = cell * 3
        return np.where(seen, cell, -1)

    def predict(self, X):
        check_is_fitted(self)
        X = validate_data(self, X, reset=False, dtype=None)
        cell = self._cells(X)
        table = np.broadcast_to(self.high_risk_[:, None], (3, 3)) if self.high_risk_.ndim == 1 else self.high_risk_
        risk = np.zeros(cell.size, bool)
        ok = cell >= 0
        risk[ok] = table.reshape(-1)[cell[ok]]
        return np.where(risk, self.classes_[1], self.classes_[0])

    def transform(self, X):
        check_is_fitted(self)
        X = validate_data(self, X, reset=False, dtype=None)
        return X[:, list(self.best_combination_)]
