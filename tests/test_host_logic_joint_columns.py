"""CPU: host side of ``pairs="selected"`` (fastselect_b200/_mi.py) -- mRMR and CFS driven by the columns
their greedy searches ask for, with the GPU hook (``_mi.open_joint_columns``) replaced by the oracle or by
the rows of a given matrix.  They must reproduce the reference's selections (tests/golden/joint_vectors.npz)
and pick exactly what the full-matrix searches of the parent implementation (copied below, unchanged)
pick, planted ties included."""
import os

import numpy as np
import pytest
from sklearn.base import clone

import fastselect_b200 as fsb
from fastselect_b200 import _mi, _native

HERE = os.path.dirname(os.path.abspath(__file__))
DATA_MRMR = ("mrmr_fixture", "mrmr_dup", "geno", "states")
DATA_CFS = ("cfs_fixture", "geno", "states", "mrmr_fixture")


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(HERE, "golden", "joint_vectors.npz"))


def oracle_full(codes, kind, log_base):
    from oracle import ref_oracle as R

    codes = np.asarray(codes)
    xc = np.stack([np.unique(codes[:, f], return_inverse=True)[1] for f in range(codes.shape[1])], axis=1)
    q = xc.shape[1]
    if kind == _native.FS_JOINT_MI:
        vec, mat = R.mi_matrices(xc[:, :-1], xc[:, -1], unit="nat")
        vec, mat = vec / log_base, mat / log_base
    else:
        vec, mat = R.su_matrices(xc[:, :-1], xc[:, -1])
    full = np.zeros((q, q))
    full[:q - 1, :q - 1] = mat
    full[q - 1, :q - 1] = vec
    full[:q - 1, q - 1] = vec
    return full


class FakeColumns:
    """Stands in for _mi.JointColumns: rows of a [q, q] matrix; records what is asked."""

    def __init__(self, full, log):
        self.full, self.log = full, log

    def columns(self, positions):
        positions = list(np.atleast_1d(positions))
        self.log.append(positions)
        return self.full[positions].copy()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        pass


@pytest.fixture
def hooks(monkeypatch):
    """Both GPU hooks served from one source: the oracle (default) or a fixed [p + 1, p + 1] matrix."""
    state = {"full": None, "calls": [], "matrix_calls": 0}

    def source(codes, kind, log_base):
        return state["full"] if state["full"] is not None else oracle_full(codes, kind, log_base)

    def fake_open(codes, kind, log_base=1.0):
        return FakeColumns(source(codes, kind, log_base), state["calls"])

    def fake_matrix(codes, kind, log_base=1.0, stats_out=None):
        state["matrix_calls"] += 1
        return source(codes, kind, log_base)

    monkeypatch.setattr(_mi, "open_joint_columns", fake_open)
    monkeypatch.setattr(_mi, "joint_matrix", fake_matrix)
    monkeypatch.setattr(_native, "device_count", lambda: 1)
    return state


# --- the parent implementation's full-matrix searches, verbatim: the yardstick of the column-driven ones ---
def ref_mrmr_select(relevance, redundancy, n_select, method):
    p = relevance.size
    selected = np.zeros(n_select, dtype=np.int32)
    remaining = np.ones(p, dtype=bool)
    first = int(np.argmax(relevance))
    selected[0] = first
    remaining[first] = False
    red_sum = redundancy[:, first].copy()
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
        red_sum += redundancy[:, best]
    return selected


def ref_best_first_search(r_cf, r_ff, min_r_cf=0.1):
    p = r_cf.size
    first = int(np.argmax(r_cf))
    if r_cf[first] < min_r_cf:
        return []
    selected = [first]
    current = float(r_cf[first])
    eligible = ~(r_cf.astype(np.float64) < min_r_cf)
    while True:
        k = len(selected) + 1
        base_cf = 0.0
        for s in selected:
            base_cf += float(r_cf[s])
        base_ff = 0.0
        for a in selected:
            for b in selected:
                if a < b:
                    base_ff += float(r_ff[a, b])
        sum_cf = base_cf + r_cf.astype(np.float64)
        sum_ff = np.full(p, base_ff)
        for s in selected:
            sum_ff = sum_ff + r_ff[:, s].astype(np.float64)
        merit = _mi._cfs_merit(sum_cf, k, sum_ff)
        ok = eligible.copy()
        ok[selected] = False
        if not ok.any():
            break
        merit = np.where(ok, merit, -np.inf)
        best = int(np.argmax(merit))
        if merit[best] > current:
            selected.append(best)
            current = float(merit[best])
        else:
            break
    return selected


def ref_cfs_fit(r_cf, r_ff):
    selected = np.sort(np.array(ref_best_first_search(r_cf, r_ff), dtype=int))
    order = selected[np.argsort(-r_cf[selected], kind="stable")]
    kept = []
    for f in order.tolist():
        if kept and bool((r_ff[f, kept] >= r_cf[f]).any()):
            continue
        kept.append(f)
    kept = np.sort(np.array(kept, dtype=int))
    k = len(kept)
    merit = 0.0
    if k:
        merit = float(_mi._cfs_merit(np.float64(np.sum(r_cf[kept])), k,
                                     np.float64(np.sum(np.triu(r_ff[np.ix_(kept, kept)], k=1)))))
    return kept, merit


@pytest.mark.parametrize("method", ["MID", "MIQ"])
def test_mrmr_selected_reproduces_the_reference(g, hooks, method):
    for data in DATA_MRMR:
        x, y = g[f"X_{data}"], g[f"y_{data}"]
        ref = g[f"mrmr_top_{method}_{data}"]
        hooks["calls"].clear()
        est = fsb.mRMR(n_features_to_select=len(ref), method=method, backend="gpu", pairs="selected").fit(x, y)
        assert np.array_equal(est.top_features_, ref), (data, method)
        np.testing.assert_allclose(est.relevance_scores_, g[f"mi_rel_bit_{data}"], rtol=1e-9, atol=1e-14)
        assert est.feature_importances_ is est.relevance_scores_ and est.n_features_in_ == x.shape[1]
        assert np.array_equal(est.unique_vals_, np.unique(np.concatenate([np.unique(x), np.unique(y)])))
        assert not hasattr(est, "redundancy_matrix_")
        assert est.redundancy_columns_.shape == (len(ref), x.shape[1]) and est.redundancy_columns_.dtype == np.float64
        np.testing.assert_allclose(est.redundancy_columns_, g[f"mi_red_bit_{data}"][ref], rtol=1e-9, atol=1e-14)
        # the class column, then one column per selected feature in selection order
        assert hooks["calls"] == [[x.shape[1]]] + [[int(f)] for f in ref]
        assert hooks["matrix_calls"] == 0
        assert np.array_equal(est.transform(x), x[:, ref])


def test_cfs_selected_reproduces_the_reference(g, hooks):
    for data in DATA_CFS:
        x, y = g[f"X_{data}"], g[f"y_{data}"]
        est = fsb.CFS(backend="gpu", pairs="selected").fit(x, y)
        assert np.array_equal(est.selected_indices_, g[f"cfs_sel_{data}"]), data
        assert est.merit_ == pytest.approx(float(g[f"cfs_merit_{data}"][0]), rel=1e-5, abs=1e-6)
        assert est.r_cf_.dtype == np.float32
        np.testing.assert_allclose(est.r_cf_, g[f"cfs_rcf_{data}"], rtol=0, atol=1e-6)
        assert not hasattr(est, "r_ff_")
        assert est.support_mask_.sum() == len(est.selected_indices_)
        assert np.array_equal(est.transform(x), x[:, g[f"cfs_sel_{data}"]])
    assert hooks["matrix_calls"] == 0


def test_selected_and_all_agree_on_the_golden_data(g, hooks):
    """Same source for both modes: every shared attribute is bitwise equal."""
    for data in DATA_MRMR:
        x, y = g[f"X_{data}"], g[f"y_{data}"]
        for method in ("MID", "MIQ"):
            a = fsb.mRMR(5, method, "gpu").fit(x, y)
            s = fsb.mRMR(5, method, "gpu", pairs="selected").fit(x, y)
            assert np.array_equal(a.top_features_, s.top_features_)
            assert np.array_equal(a.relevance_scores_, s.relevance_scores_)
            assert np.array_equal(a.redundancy_matrix_[a.top_features_], s.redundancy_columns_)
            assert not hasattr(a, "redundancy_columns_")
    for data in DATA_CFS:
        x, y = g[f"X_{data}"], g[f"y_{data}"]
        a = fsb.CFS(backend="gpu").fit(x, y)
        s = fsb.CFS(backend="gpu", pairs="selected").fit(x, y)
        assert np.array_equal(a.selected_indices_, s.selected_indices_)
        assert np.array_equal(a.support_mask_, s.support_mask_)
        assert np.array_equal(a.r_cf_, s.r_cf_) and a.merit_ == s.merit_


def planted_matrix(rs, p, levels):
    """Symmetric [p + 1, p + 1] matrix (position p = the class) drawn from a few levels, so that scores,
    redundancies and merits tie exactly in many places."""
    m = rs.choice(levels, (p + 1, p + 1))
    m = np.triu(m, 1)
    m = m + m.T
    return m


@pytest.mark.parametrize("seed", range(12))
def test_mrmr_columns_pick_what_the_full_matrix_search_picks(hooks, seed):
    rs = np.random.RandomState(seed)
    p = 40
    full = planted_matrix(rs, p, np.array([0.0, 0.125, 0.25, 0.5, 0.75]))
    full[p, :p] = full[:p, p] = rs.choice([0.5, 0.75, 1.0], p)          # ties in relevance too
    hooks["full"] = full
    x = rs.randint(0, 3, (20, p)).astype(np.uint8)
    y = rs.randint(0, 2, 20)
    for method in ("MID", "MIQ"):
        k = 1 + seed % 15
        want = ref_mrmr_select(full[p, :p].copy(), np.ascontiguousarray(full[:p, :p]), k, method)
        s = fsb.mRMR(k, method, "gpu", pairs="selected").fit(x, y)
        a = fsb.mRMR(k, method, "gpu", pairs="all").fit(x, y)
        assert np.array_equal(s.top_features_, want) and np.array_equal(a.top_features_, want)
        assert np.array_equal(s.redundancy_columns_, a.redundancy_matrix_[want])


@pytest.mark.parametrize("seed", range(12))
def test_cfs_columns_pick_what_the_full_matrix_search_picks(hooks, seed):
    rs = np.random.RandomState(100 + seed)
    p = 30
    full = planted_matrix(rs, p, np.array([0.0, 0.05, 0.1, 0.2, 0.3]))
    full[p, :p] = full[:p, p] = rs.choice([0.05, 0.1, 0.3, 0.4, 0.4], p)
    hooks["full"] = full
    x = rs.randint(0, 3, (20, p)).astype(np.uint8)
    y = rs.randint(0, 2, 20)
    r_cf = full[p, :p].astype(np.float32)
    r_ff = np.ascontiguousarray(full[:p, :p], dtype=np.float32)
    kept, merit = ref_cfs_fit(r_cf, r_ff)
    hooks["calls"].clear()
    s = fsb.CFS(backend="gpu", pairs="selected").fit(x, y)
    a = fsb.CFS(backend="gpu").fit(x, y)
    for est in (s, a):
        assert np.array_equal(est.selected_indices_, kept) and est.merit_ == merit
    assert np.array_equal(s.r_cf_, a.r_cf_)
    # the class column first, then one column per accepted feature, none asked twice
    asked = [c[0] for c in hooks["calls"]]
    assert asked[0] == p and len(asked) == len(set(asked))
    assert set(kept.tolist()) <= set(asked[1:])


def test_pairs_validation_and_params(hooks):
    with pytest.raises(ValueError, match="pairs must be 'all' or 'selected'"):
        fsb.mRMR(n_features_to_select=2, pairs="some")
    x = np.arange(24).reshape(8, 3) % 3
    y = np.arange(8) % 2
    with pytest.raises(ValueError, match="pairs must be 'all' or 'selected'"):
        fsb.CFS(backend="gpu", pairs="diagonal").fit(x, y)
    m = fsb.mRMR(n_features_to_select=2, pairs="selected")
    assert m.get_params()["pairs"] == "selected" and clone(m).pairs == "selected"
    assert fsb.mRMR(n_features_to_select=2).get_params()["pairs"] == "all"
    c = fsb.CFS(pairs="selected")
    assert c.get_params()["pairs"] == "selected" and clone(c).pairs == "selected"
    assert fsb.CFS().get_params()["pairs"] == "all"


def test_refit_in_the_other_mode_drops_the_other_attribute(g, hooks):
    x, y = g["X_geno"], g["y_geno"]
    est = fsb.mRMR(3, "MID", "gpu").fit(x, y)
    est.set_params(pairs="selected").fit(x, y)
    assert not hasattr(est, "redundancy_matrix_") and est.redundancy_columns_.shape == (3, x.shape[1])
    est.set_params(pairs="all").fit(x, y)
    assert not hasattr(est, "redundancy_columns_") and est.redundancy_matrix_.shape == (x.shape[1],) * 2
    c = fsb.CFS(backend="gpu").fit(x, y)
    c.set_params(pairs="selected").fit(x, y)
    assert not hasattr(c, "r_ff_")
