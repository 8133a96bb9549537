"""GPU: MDR (fs_mdr_scan / fs_mdr_tables, fastselect_b200.MDR) against the numpy oracle (oracle/mdr_oracle.py).
Balanced accuracies are ratios of exact integers with one float64 division and fold-ordered means, so every
comparison is BITWISE."""
import numpy as np
import pytest

import fastselect_b200 as fsb
from fastselect_b200 import _mdr, _native
from oracle import mdr_oracle as O
from datasets import epistatic_genotypes

pytestmark = pytest.mark.gpu

DTYPES = [np.uint8, np.int8, np.float32]
ODD = {np.uint8: (0, 1, 200), np.int8: (-7, 0, 3), np.float32: (3.5, -7.0, 1e6)}


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def make_data(seed, n, p, dtype, cv):
    """3-state columns over odd values, one constant and two 2-valued columns, about 10 % cases."""
    rs = np.random.RandomState(seed)
    vals = np.array(ODD[dtype], dtype)
    X = vals[rs.randint(0, 3, (n, p))]
    X[:, 3] = vals[1]                                          # constant
    X[:, 5] = vals[rs.randint(0, 2, n)]                        # 2-valued
    X[:, p - 1] = vals[1 + rs.randint(0, 2, n)]
    y = np.zeros(n, np.int64)
    risk = (X[:, 1] == vals[2]) & (X[:, 7] != vals[0])
    n_case = max(int(round(0.1 * n)), cv)
    order = np.argsort(~risk + rs.rand(n) * 0.5, kind="stable")
    y[order[:n_case]] = 1
    return X, y


def check_scan(src, X, y, fold, cv, order, feat_idx=None, n_top=64):
    Xs = X if feat_idx is None else X[:, feat_idx]
    want = O.scan(Xs, y, fold, cv, order)
    nc = O.n_combinations(Xs.shape[1], order)
    n_top = min(n_top, nc)
    got = src._ds.mdr_scan(fold, order, n_top, feat_idx=feat_idx, want_all=True)
    assert np.array_equal(bits(got["all_train"]), bits(want["mean_train"]))
    assert np.array_equal(bits(got["all_test"]), bits(want["mean_test"]))
    top = O.top_list(want["mean_test"], n_top)
    assert np.array_equal(got["top_idx"], top)
    assert np.array_equal(bits(got["top_test"]), bits(want["mean_test"][top]))
    assert np.array_equal(bits(got["top_train"]), bits(want["mean_train"][top]))
    assert np.array_equal(got["fold_best"], O.fold_best(want["train"]))
    return want, got


@pytest.mark.parametrize("order", [1, 2])
@pytest.mark.parametrize("cv", [2, 3, 5, 10])
@pytest.mark.parametrize("n", [33, 127, 4095, 4097, 9001])
def test_scan_bitwise(native, n, cv, order):
    dtype = DTYPES[(n + cv) % 3]
    X, y = make_data(n * 31 + cv, n, 40, dtype, cv)
    fold = _mdr.make_folds(y, cv, n)
    with _mdr.MDRData(X, y) as src:
        want, got = check_scan(src, X, y, fold, cv, order)
        again = src._ds.mdr_scan(fold, order, min(64, O.n_combinations(40, order)), want_all=True)
        for k in got:
            assert np.array_equal(np.asarray(got[k]).view(np.int64), np.asarray(again[k]).view(np.int64)), k
        # unsorted column list, then the tables of some combinations in both operand orders
        idx = np.random.RandomState(n).permutation(40)[:29]
        check_scan(src, X, y, fold, cv, order, feat_idx=idx)
        codes, _ = O.cells(X[:, idx])
        combos = np.array([[0, 1], [5, 2], [28, 3], [7, 19]])[:, :order]
        tabs = src._ds.mdr_tables(fold, order, combos, feat_idx=idx)
        ref = O.Source(X[:, idx], y).tables(fold, order, combos)
        assert np.array_equal(tabs, ref)


def test_ties_top_list_and_fold_best(native):
    """Few samples and copied columns: many exactly equal scores; ranking must follow the index."""
    rs = np.random.RandomState(5)
    base = rs.randint(0, 3, (48, 9)).astype(np.uint8)
    X = base[:, rs.randint(0, 9, 70)]
    y = np.array([0, 1] * 24)
    for cv in (2, 3):
        fold = _mdr.make_folds(y, cv, None)
        with _mdr.MDRData(X, y) as src:
            want, _ = check_scan(src, X, y, fold, cv, 2, n_top=2048)
            assert np.unique(want["mean_test"]).size < want["mean_test"].size // 4
            check_scan(src, X, y, fold, cv, 1, n_top=70)


@pytest.mark.parametrize("order", [1, 2])
def test_estimator_equals_oracle(native, order):
    X, y = make_data(11, 2000, 120, np.int8, 5)
    est = fsb.MDR(order=order, cv=5, n_top=300, random_state=3).fit(X, y)
    want = O.fit(X, y, order, 5, 300, 3)
    for k, v in want.items():
        got = getattr(est, k)
        if isinstance(v, list):
            assert all(np.array_equal(a, b) for a, b in zip(got, v)) and len(got) == len(v), k
        elif isinstance(v, float):
            assert bits(got) == bits(v), k
        else:
            assert np.array_equal(np.asarray(got), np.asarray(v)), k


def test_c_abi_rejections(native):
    X, y = make_data(2, 200, 12, np.uint8, 5)
    fold = _mdr.make_folds(y, 5, None)
    with _mdr.MDRData(X, y) as src:
        ds = src._ds
        with pytest.raises(ValueError, match="order"):
            ds.mdr_scan(fold, 3, 1)
        with pytest.raises(ValueError, match="n_top"):
            ds.mdr_scan(fold, 2, 67)                            # 66 pairs
        with pytest.raises(ValueError, match="n_top"):
            ds.mdr_scan(fold, 1, 0)
        with pytest.raises(ValueError, match="n_folds"):
            ds.mdr_scan(np.arange(200) % 11, 1, 1)
        bad = fold.copy()
        bad[y == 1] = 0                                         # folds 1.. hold no case
        with pytest.raises(ValueError, match="no sample of class"):
            ds.mdr_scan(bad, 2, 1)
        neg = fold.copy()
        neg[0] = -1
        with pytest.raises(ValueError, match="fold"):
            ds.mdr_scan(neg, 2, 1)
        with pytest.raises(ValueError, match="combination"):
            ds.mdr_tables(fold, 2, [[3, 3]])
        with pytest.raises(ValueError):
            ds.mdr_scan(fold, 2, 1, feat_idx=[0, 12])
    X4 = X.copy()
    X4[0, 4] = 9
    with _mdr.MDRData(X4, y) as src:
        with pytest.raises(ValueError, match="at most 3"):
            src._ds.mdr_scan(fold, 2, 1)
        src._ds.mdr_scan(fold, 2, 1, feat_idx=[0, 1, 2])        # the 4-state column is not scanned
    y3 = y.copy()
    y3[0] = 2
    with _native.Dataset(X, y3, 3) as ds:
        ds.set_features(np.ones(12, np.uint8), np.ones(12, np.float32), _native.FS_ARITH_F32)
        with pytest.raises(ValueError, match="2 classes"):
            ds.mdr_scan(fold, 2, 1)
    with pytest.raises(ValueError, match="at most 3"):
        fsb.MDR().fit(X4, y)


def test_planted_interaction_at_c3_shape(native):
    X, y = epistatic_genotypes(42, 4000, 100_000)
    est = fsb.MDR().fit(X, y)
    assert est.best_combination_ == (25, 75)
    assert est.cv_consistency_ == 5
    assert tuple(est.top_combinations_[0]) == (25, 75)
    rs = np.random.RandomState(1)
    idx = np.concatenate([[75], rs.choice(np.setdiff1d(np.arange(100_000), [25, 75]), 2000, replace=False), [25]])
    rs.shuffle(idx)
    fold = _mdr.make_folds(y, 5, None)
    with _mdr.MDRData(X, y) as src:
        check_scan(src, X, y, fold, 5, 2, feat_idx=idx, n_top=100)


def test_encoding_is_shared_with_the_joint_path(native):
    """joint_columns, mdr_scan, joint_matrix and mdr_scan again on one column list of one data set: each result
    is bitwise the same call's on a freshly opened data set, and the second scan packs nothing."""
    X, y = make_data(7, 3001, 30, np.uint8, 5)
    fold = _mdr.make_folds(y, 5, None)
    idx = np.random.RandomState(7).permutation(30)[:24]
    calls = [lambda ds: ds.joint_columns(0, 1.0, [0, 5, 23], feat_idx=idx),
             lambda ds: ds.mdr_scan(fold, 2, 50, feat_idx=idx, want_all=True, want_stats=True),
             lambda ds: ds.joint_matrix(1, 1.0, feat_idx=idx),
             lambda ds: ds.mdr_scan(fold, 2, 50, feat_idx=idx, want_all=True, want_stats=True)]
    fresh = []
    for call in calls:
        with _mdr.MDRData(X, y) as src:
            fresh.append(call(src._ds))
    with _mdr.MDRData(X, y) as src:
        got = [call(src._ds) for call in calls]
    for i in (0, 2):
        assert np.array_equal(bits(got[i]), bits(fresh[i])), i
    for i in (1, 3):
        for k in fresh[i][0]:
            assert np.array_equal(np.asarray(got[i][0][k]).view(np.int64), np.asarray(fresh[i][0][k]).view(np.int64)), k
    # the first scan packs the planes (encode done by joint_columns); the second only scans and merges
    assert got[1][1]["launches"] == got[3][1]["launches"] + 1
    assert got[3][1]["ms_gather"] < 0.05, got[3][1]


def test_encoding_of_the_joint_path_keeps_the_mdr_limit(native):
    X, y = make_data(8, 400, 12, np.uint8, 5)
    X[0, 4] = 9                                                 # 4 states: a joint column, not an MDR one
    fold = _mdr.make_folds(y, 5, None)
    with _mdr.MDRData(X, y) as src:
        src._ds.joint_columns(0, 1.0, [4])
        with pytest.raises(ValueError, match="at most 3"):
            src._ds.mdr_scan(fold, 2, 1)


def test_scan_after_a_rebuild_of_the_working_set(native):
    X, y = make_data(9, 1500, 20, np.int8, 3)
    fold = _mdr.make_folds(y, 3, None)
    with _mdr.MDRData(X, y) as src:
        first = src._ds.mdr_scan(fold, 2, 40, want_all=True)
        src._ds.joint_columns(0, 1.0, [1], feat_idx=np.arange(0, 20, 3))
        again = src._ds.mdr_scan(fold, 2, 40, want_all=True)
    for k in first:
        assert np.array_equal(np.asarray(first[k]).view(np.int64), np.asarray(again[k]).view(np.int64)), k
