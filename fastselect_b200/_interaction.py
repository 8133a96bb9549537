"""Two-locus interaction test after BOOST (Wan et al., AJHG 2010): a KSA screen of every column pair on the
GPU, then an exact likelihood-ratio test of the listed pairs on the host.

The screen runs in fastselect_b200/csrc/mdr.cu (``fs_interaction_scan``) on MDR's bit-planes with a single
fold, so it takes MDR's inputs: columns with at most 3 distinct values and a binary class.  The statistic
``L_KSA`` of the Kirkwood superposition approximation bounds the likelihood-ratio statistic ``G`` of the
no-three-way-interaction log-linear model from above, so a pair left out of the list cannot have a larger
``G`` than the last listed ``L_KSA``.  The semantics are this project's own (DESIGN.md section 11).  There is
no CPU fallback.
"""
from __future__ import annotations

import numpy as np
from scipy.stats import chi2
from sklearn.base import BaseEstimator
from sklearn.utils.validation import validate_data

from . import _mdr, _native

IPF_TOL = 1e-9              # fitted margins within IPF_TOL * N of the observed ones
IPF_MAX_CYCLES = 10_000
_NO_GPU = "PairwiseInteraction needs a usable sm_100 GPU (NVIDIA B200); none was found."
_NO_CPU = ("fastselect_b200 implements only the GPU backend of PairwiseInteraction; backend='cpu' is not "
           "available.")


def open_interaction(X, y_enc):
    """The GPU behind :class:`PairwiseInteraction`: an :class:`~fastselect_b200._mdr.MDRData` over ``X`` and
    ``y_enc``."""
    return _mdr.MDRData(X, y_enc)


def _ratio(obs, fit):
    return np.divide(obs, fit, out=np.zeros_like(obs), where=fit > 0)


def no_three_way_fit(n, tol=IPF_TOL, max_cycles=IPF_MAX_CYCLES):
    """Maximum-likelihood fit of the no-three-way-interaction model to tables ``n`` (float64 ``[m, I, J, K]``):
    iterative proportional fitting of the AB, AY and BY margins from mu = 1, until every fitted margin is
    within ``tol * N`` of the observed one.  Raises ``RuntimeError`` after ``max_cycles`` cycles."""
    n = np.asarray(n, np.float64)
    nij, nik, njk = n.sum(3), n.sum(2), n.sum(1)
    lim = tol * n.sum((1, 2, 3))
    mu = np.ones_like(n)
    for _ in range(max_cycles):
        mu = mu * _ratio(nij, mu.sum(3))[:, :, :, None]
        mu = mu * _ratio(nik, mu.sum(2))[:, :, None, :]
        mu = mu * _ratio(njk, mu.sum(1))[:, None, :, :]
        err = np.maximum(np.maximum(np.abs(mu.sum(3) - nij).max((1, 2)), np.abs(mu.sum(2) - nik).max((1, 2))),
                         np.abs(mu.sum(1) - njk).max((1, 2)))
        if np.all(err <= lim):
            return mu
    raise RuntimeError(f"iterative proportional fitting did not converge in {max_cycles} cycles")


def lr_statistic(tables):
    """Likelihood-ratio statistic G of the no-three-way model for ``[m, 2, 9]`` class tables (entry
    ``[q, k, i * 3 + j]``): ``2 sum_{n > 0} n log(n / mu)``, clamped at 0, float64 ``[m]``."""
    t = np.asarray(tables, np.int64)
    n = t.reshape(-1, 2, 3, 3).transpose(0, 2, 3, 1).astype(np.float64)      # [m, i, j, k]
    if n.shape[0] == 0:
        return np.zeros(0)
    mu = no_three_way_fit(n)
    pos = n > 0
    terms = np.zeros_like(n)
    terms[pos] = n[pos] * np.log(n[pos] / mu[pos])
    return np.maximum(2.0 * terms.sum((1, 2, 3)), 0.0)


def p_values(G, dof):
    """chi-square upper tail of G with dof degrees of freedom; 1 where dof = 0."""
    dof = np.asarray(dof, np.int64)
    return np.where(dof > 0, chi2.sf(G, np.maximum(dof, 1)), 1.0)


class PairwiseInteraction(BaseEstimator):
    """Test of the two-locus interaction of every column pair with respect to a binary class.

    Every column must hold at most 3 distinct values (genotypes 0/1/2, or any 3 numbers); ``y`` exactly 2
    labels, ``classes_[1]`` being the case class.  A sample's state in a column is the rank of its value among
    the column's distinct values.  For every pair the GPU computes ``L_KSA``, the BOOST screening statistic of
    its 3 x 3 x 2 table, and keeps the ``n_top`` largest (lower pair index first on ties).  For those pairs the
    host fits the no-three-way-interaction log-linear model (margins AB, AY, BY) by iterative proportional
    fitting and tests it against the saturated model: ``G = 2 sum n log(n / mu)`` with
    ``(V_a - 1)(V_b - 1)`` degrees of freedom, V being a column's number of distinct values.

    Fitted attributes: ``classes_``; ``pairs_`` (int64 ``[m, 2]``, column indices, by ``L_KSA`` descending);
    ``ksa_statistic_``, ``statistic_`` (G), ``dof_``, ``p_values_`` (``[m]``); ``bound_``, the last listed
    ``L_KSA`` (0 when every pair is listed): since ``G <= L_KSA``, no unlisted pair has a larger G, up to
    rounding; ``n_pairs_tested_`` = p (p - 1) / 2, for a multiple-testing correction of the user's choice (none
    is applied).  The semantics are this project's own."""

    def __init__(self, n_top=100, backend="auto"):
        self.n_top = n_top
        self.backend = backend

    def _check_params(self):
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
        classes, y_enc = np.unique(y, return_inverse=True)
        if classes.size != 2:
            raise ValueError(f"PairwiseInteraction needs exactly 2 classes in y (got {classes.size}).")
        p = X.shape[1]
        if p < 2:
            raise ValueError(f"PairwiseInteraction needs at least 2 features (got {p}).")
        if _native.device_count() < 1:
            raise RuntimeError(_NO_GPU)
        n_pairs = p * (p - 1) // 2
        n_top = min(int(self.n_top), n_pairs)
        with open_interaction(X, y_enc) as src:
            n_states = np.asarray(src.n_states, np.int64)
            bad = np.flatnonzero(n_states > _mdr.MAX_STATES)
            if bad.size:
                raise ValueError(f"PairwiseInteraction supports columns with at most {_mdr.MAX_STATES} distinct "
                                 f"values (column {int(bad[0])} has more).")
            res = src.interaction_scan(n_top)
        pairs = _mdr.decode_combinations(res["top_idx"], p, 2)
        ksa = np.asarray(res["top_ksa"], np.float64)
        G = lr_statistic(res["top_tables"])
        dof = (n_states[pairs[:, 0]] - 1) * (n_states[pairs[:, 1]] - 1)

        self.classes_ = classes
        self.pairs_ = pairs
        self.ksa_statistic_ = ksa
        self.statistic_ = G
        self.dof_ = dof
        self.p_values_ = p_values(G, dof)
        self.bound_ = float(ksa[-1]) if n_top < n_pairs else 0.0
        self.n_pairs_tested_ = n_pairs
        return self
