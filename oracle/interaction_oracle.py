"""numpy restatement of this project's pairwise interaction test (fastselect_b200/_interaction.py,
``fs_interaction_scan`` in fastselect_b200/csrc/mdr.cu).

TEST INFRASTRUCTURE ONLY.  The semantics are this project's own (DESIGN.md section 11).  ``ksa`` forms L_KSA in
the kernel's operation order (cells in (i, j, k) order, products left to right, no fused multiply-add); the
kernel's ``log`` is not numpy's, so the values agree to rounding, not bitwise.  ``lr_test`` fits the
no-three-way model table by table with plain loops, independently of the estimator's vectorised code.
"""
from __future__ import annotations

import math

import numpy as np
from scipy.stats import chi2

from oracle import mdr_oracle as M


def tables(codes, y):
    """Class tables of every pair: int64 ``[n_pairs, 2, 9]``, entry ``[q, k, i * 3 + j]``."""
    return M.segment_tables(codes, np.asarray(y), np.zeros(codes.shape[0], np.int64), 1, 2)


def ksa(tab):
    """L_KSA of every table of ``tab`` (``[m, 2, 9]``), float64 ``[m]``."""
    t = np.asarray(tab, np.int64)
    m = t.shape[0]
    n = t.reshape(m, 2, 3, 3).transpose(0, 2, 3, 1)            # [m, i, j, k]
    nij, nik, njk = n.sum(3), n.sum(2), n.sum(1)
    ni, nj, nk = n.sum((2, 3)), n.sum((1, 3)), n.sum((1, 2))
    N = nk.sum(1).astype(np.float64)
    f = np.float64
    q = np.zeros((m, 3, 3, 2))
    eta = np.zeros(m)
    for i in range(3):
        for j in range(3):
            for k in range(2):
                ok = (nij[:, i, j] > 0) & (nik[:, i, k] > 0) & (njk[:, j, k] > 0)
                num = nij[:, i, j].astype(f) * nik[:, i, k].astype(f) * njk[:, j, k].astype(f)
                den = ni[:, i].astype(f) * nj[:, j].astype(f) * nk[:, k].astype(f)
                q[:, i, j, k] = np.where(ok, num / np.where(ok, den, 1.0), 0.0)
                eta = eta + q[:, i, j, k]
    L = np.zeros(m)
    for i in range(3):
        for j in range(3):
            for k in range(2):
                c = n[:, i, j, k].astype(f)
                pos = c > 0
                r = (c * eta) / np.where(pos, N * q[:, i, j, k], 1.0)
                L = L + np.where(pos, c * np.log(np.where(pos, r, 1.0)), 0.0)
    return 2.0 * L


def lr_test(tab, n_a, n_b, tol=1e-9, max_cycles=10_000):
    """(G, dof, p) of one ``[2, 9]`` table: IPF of the AB, AY and BY margins from mu = 1, written cell by cell."""
    n = [[[int(tab[k][i * 3 + j]) for k in range(2)] for j in range(3)] for i in range(3)]
    N = sum(n[i][j][k] for i in range(3) for j in range(3) for k in range(2))
    mu = [[[1.0, 1.0] for _ in range(3)] for _ in range(3)]
    ab = [[n[i][j][0] + n[i][j][1] for j in range(3)] for i in range(3)]
    ay = [[sum(n[i][j][k] for j in range(3)) for k in range(2)] for i in range(3)]
    by = [[sum(n[i][j][k] for i in range(3)) for k in range(2)] for j in range(3)]

    def scale(obs, fit):
        return obs / fit if fit > 0 else 0.0

    for _ in range(max_cycles):
        for i in range(3):
            for j in range(3):
                s = scale(ab[i][j], mu[i][j][0] + mu[i][j][1])
                mu[i][j] = [mu[i][j][0] * s, mu[i][j][1] * s]
        for i in range(3):
            for k in range(2):
                s = scale(ay[i][k], sum(mu[i][j][k] for j in range(3)))
                for j in range(3):
                    mu[i][j][k] *= s
        for j in range(3):
            for k in range(2):
                s = scale(by[j][k], sum(mu[i][j][k] for i in range(3)))
                for i in range(3):
                    mu[i][j][k] *= s
        err = max([abs(mu[i][j][0] + mu[i][j][1] - ab[i][j]) for i in range(3) for j in range(3)]
                  + [abs(sum(mu[i][j][k] for j in range(3)) - ay[i][k]) for i in range(3) for k in range(2)]
                  + [abs(sum(mu[i][j][k] for i in range(3)) - by[j][k]) for j in range(3) for k in range(2)])
        if err <= tol * N:
            break
    else:
        raise RuntimeError("IPF did not converge")
    G = 0.0
    for i in range(3):
        for j in range(3):
            for k in range(2):
                if n[i][j][k] > 0:
                    G += n[i][j][k] * math.log(n[i][j][k] / mu[i][j][k])
    G = max(2.0 * G, 0.0)
    dof = (n_a - 1) * (n_b - 1)
    return G, dof, (float(chi2.sf(G, dof)) if dof > 0 else 1.0)


def top_list(values, n_top):
    """Indices of the n_top largest values, largest first, lower index first on ties."""
    return np.lexsort((np.arange(values.size), -values))[:n_top]


def fit(X, y, n_top=100):
    """The fitted attributes of ``fastselect_b200.PairwiseInteraction`` computed from scratch."""
    X = np.asarray(X)
    classes, y_enc = np.unique(y, return_inverse=True)
    codes, n_states = M.cells(X)
    p = X.shape[1]
    n_pairs = p * (p - 1) // 2
    tab = tables(codes, y_enc)
    L = ksa(tab)
    top = top_list(L, min(n_top, n_pairs))
    pairs = M.decode(top, p, 2)
    res = [lr_test(tab[q], n_states[a], n_states[b]) for q, (a, b) in zip(top, pairs)]
    return dict(classes_=classes, pairs_=pairs, ksa_statistic_=L[top],
                statistic_=np.array([r[0] for r in res]), dof_=np.array([r[1] for r in res], np.int64),
                p_values_=np.array([r[2] for r in res]), bound_=float(L[top[-1]]) if top.size < n_pairs else 0.0,
                n_pairs_tested_=n_pairs)


class Source:
    """Stands in for ``fastselect_b200._mdr.MDRData`` behind ``_interaction.open_interaction`` in CPU tests."""

    def __init__(self, X, y_enc):
        self.X = np.asarray(X)
        self.y = np.asarray(y_enc)
        self.codes, self.n_states = M.cells(self.X)
        self.calls = []

    def interaction_scan(self, n_top, want_all=False):
        self.calls.append("interaction_scan")
        tab = tables(self.codes, self.y)
        L = ksa(tab)
        top = top_list(L, n_top)
        out = dict(top_idx=top.astype(np.int64), top_ksa=L[top], top_tables=tab[top])
        if want_all:
            out["all_ksa"] = L
        return out

    def close(self):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
