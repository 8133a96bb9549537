"""numpy restatement of this project's MDR (fastselect_b200/_mdr.py, fastselect_b200/csrc/mdr.cu).

TEST INFRASTRUCTURE ONLY.  The semantics are this project's own (DESIGN.md, "MDR"); they have not been
checked against ``fast_select.MDR``.  Every number here is formed the way the kernel forms it -- integer
counts, one float64 division per balanced accuracy, means summed in fold order -- so the results are
bitwise comparable.
"""
from __future__ import annotations

import numpy as np


def cells(X):
    """Rank of every value among its column's sorted distinct values, int64 ``[n, p]``; distinct counts ``[p]``."""
    X = np.asarray(X)
    out = np.empty(X.shape, np.int64)
    n_states = np.empty(X.shape[1], np.int64)
    for f in range(X.shape[1]):
        vals, inv = np.unique(X[:, f], return_inverse=True)
        out[:, f] = inv
        n_states[f] = vals.size
    return out, n_states


def n_combinations(p, order):
    return p if order == 1 else p * (p - 1) // 2


def encode(a, b, p):
    """Lexicographic rank of the pairs (a, b), a < b, among the pairs of p positions."""
    a = np.asarray(a, np.int64)
    return a * p - a * (a + 1) // 2 + (np.asarray(b, np.int64) - a - 1)


def decode(idx, p, order):
    """Combination indices -> positions, int64 ``[m, order]`` (inverse of :func:`encode`)."""
    idx = np.asarray(idx, np.int64).reshape(-1)
    if order == 1:
        return idx[:, None].copy()
    out = np.empty((idx.size, 2), np.int64)
    for q, t in enumerate(idx.tolist()):
        a = 0
        while (a + 1) * p - (a + 1) * (a + 2) // 2 <= t:
            a += 1
        out[q] = (a, t - (a * p - a * (a + 1) // 2) + a + 1)
    return out


def segment_tables(codes, y, fold, cv, order):
    """Cell counts of every combination in every segment s = 2 * fold + class: int64 ``[n_combos, 2 cv, 9]``,
    cell va * 3 + vb.  Pairs come from one one-hot product per segment."""
    n, p = codes.shape
    nc = n_combinations(p, order)
    out = np.zeros((nc, 2 * cv, 9), np.int64)
    onehot = np.zeros((n, 3 * p), np.float32)
    onehot[np.arange(n)[:, None], 3 * np.arange(p)[None, :] + codes] = 1.0
    if order == 2:
        ia, ib = np.triu_indices(p, 1)
    for f in range(cv):
        for c in range(2):
            rows = onehot[(fold == f) & (y == c)]
            if order == 1:
                out[:, 2 * f + c, 0::3] = rows.sum(0).reshape(p, 3).astype(np.int64)      # cell va * 3
            else:
                prod = (rows.T @ rows).reshape(p, 3, p, 3)
                t = prod[ia, :, ib, :]                       # [pairs, 3 (va), 3 (vb)]
                out[:, 2 * f + c, :] = np.rint(t).astype(np.int64).reshape(-1, 9)
    return out


def fold_scores(tables):
    """Training and test balanced accuracy of every fold from ``[m, 2 cv, 9]`` segment tables: two float64
    ``[m, cv]`` arrays."""
    tables = np.asarray(tables, np.int64)
    m, nseg, _ = tables.shape
    cv = nseg // 2
    all0 = tables[:, 0::2].sum(1)
    all1 = tables[:, 1::2].sum(1)
    train = np.empty((m, cv))
    test = np.empty((m, cv))
    for f in range(cv):
        e0, e1 = tables[:, 2 * f], tables[:, 2 * f + 1]
        t0, t1 = all0 - e0, all1 - e1
        M0, M1 = e0.sum(1), e1.sum(1)
        N0, N1 = t0.sum(1), t1.sum(1)
        high = t1 * N0[:, None] > t0 * N1[:, None]
        TP = np.where(high, t1, 0).sum(1)
        TN = np.where(high, 0, t0).sum(1)
        tp = np.where(high, e1, 0).sum(1)
        tn = np.where(high, 0, e0).sum(1)
        train[:, f] = (TP * N0 + TN * N1).astype(np.float64) / (2 * N1 * N0).astype(np.float64)
        test[:, f] = (tp * M0 + tn * M1).astype(np.float64) / (2 * M1 * M0).astype(np.float64)
    return train, test


def fold_mean(v):
    """Mean over the folds summed in fold order (not np.sum's pairwise order)."""
    acc = np.zeros(v.shape[0])
    for f in range(v.shape[1]):
        acc = acc + v[:, f]
    return acc / v.shape[1]


def top_list(mean_test, n_top):
    """Indices of the n_top highest mean test values, highest first, lower index first on ties."""
    idx = np.arange(mean_test.size)
    return np.lexsort((idx, -mean_test))[:n_top]


def fold_best(train):
    """Per fold, the first index of the highest training value."""
    return np.array([int(np.argmax(train[:, f])) for f in range(train.shape[1])], np.int64)


def best_combination(fbest, mean_test_of):
    """Among the fold bests: highest CV consistency, then higher mean test, then lower index."""
    cand = sorted(set(fbest.tolist()))
    cvc = {c: int(np.sum(fbest == c)) for c in cand}
    best = min(cand, key=lambda c: (-cvc[c], -mean_test_of(c), c))
    return best, cvc[best]


def high_risk(tables_one):
    """High-risk cells of one combination on all samples from its ``[2 cv, 9]`` segment tables: bool ``[9]``."""
    t0 = tables_one[0::2].sum(0)
    t1 = tables_one[1::2].sum(0)
    return t1 * t0.sum() > t0 * t1.sum()


def scan(X, y_enc, fold, cv, order):
    """Everything the kernel computes for all combinations: dict of segment tables, per-fold and mean BAs."""
    codes, _ = cells(X)
    tables = segment_tables(codes, np.asarray(y_enc), np.asarray(fold), cv, order)
    train, test = fold_scores(tables)
    return dict(tables=tables, train=train, test=test, mean_train=fold_mean(train), mean_test=fold_mean(test))


def fit(X, y, order=2, cv=5, n_top=100, random_state=None):
    """The fitted attributes of ``fastselect_b200.MDR`` computed from scratch (folds from the estimator's
    own fold assignment)."""
    from fastselect_b200._mdr import make_folds

    X = np.asarray(X)
    classes, y_enc = np.unique(y, return_inverse=True)
    fold = make_folds(y_enc, cv, random_state)
    s = scan(X, y_enc, fold, cv, order)
    p = X.shape[1]
    top = top_list(s["mean_test"], min(n_top, n_combinations(p, order)))
    fb = fold_best(s["train"])
    best, cvc = best_combination(fb, lambda c: s["mean_test"][c])
    cols = tuple(int(v) for v in decode([best], p, order)[0])
    return dict(classes_=classes, best_combination_=cols, cv_consistency_=cvc,
                train_balanced_accuracy_=float(s["mean_train"][best]), test_balanced_accuracy_=float(s["mean_test"][best]),
                top_combinations_=decode(top, p, order), top_train_balanced_accuracy_=s["mean_train"][top],
                top_test_balanced_accuracy_=s["mean_test"][top], fold_best_combinations_=decode(fb, p, order),
                feature_values_=[np.unique(X[:, c]) for c in cols],
                high_risk_=high_risk(s["tables"][best]).reshape(3, 3)[:, 0] if order == 1
                else high_risk(s["tables"][best]).reshape(3, 3))


class Source:
    """Stands in for ``fastselect_b200._mdr.MDRData`` (the GPU hook) in CPU tests."""

    def __init__(self, X, y_enc):
        self.X = np.asarray(X)
        self.y = np.asarray(y_enc)
        self.codes, self.n_states = cells(self.X)
        self.calls = []

    def scan(self, fold, order, n_top, want_all=False):
        self.calls.append("scan")
        cv = int(np.max(fold)) + 1
        tables = segment_tables(self.codes, self.y, np.asarray(fold), cv, order)
        train, test = fold_scores(tables)
        mt, me = fold_mean(train), fold_mean(test)
        top = top_list(me, n_top)
        out = dict(top_idx=top.astype(np.int64), top_train=mt[top], top_test=me[top], fold_best=fold_best(train))
        if want_all:
            out.update(all_train=mt, all_test=me)
        return out

    def tables(self, fold, order, combos):
        self.calls.append("tables")
        combos = np.asarray(combos, np.int64).reshape(-1, order)
        cv = int(np.max(fold)) + 1
        out = np.zeros((combos.shape[0], cv, 2, 9), np.int64)
        fold = np.asarray(fold)
        for q, cmb in enumerate(combos):
            g = self.codes[:, cmb[0]] * 3 + (self.codes[:, cmb[1]] if order == 2 else 0)
            for f in range(cv):
                for c in range(2):
                    out[q, f, c] = np.bincount(g[(fold == f) & (self.y == c)], minlength=9)
        return out

    def close(self):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
