"""GPU: the pairwise interaction screen (fs_interaction_scan, fastselect_b200.PairwiseInteraction) against the
numpy oracle (oracle/interaction_oracle.py).  Tables are exact integers and compared exactly; L_KSA goes
through float64 log, whose CUDA and numpy implementations differ in the last bits, so it is compared within
rtol 1e-11 / atol 1e-11 N, and the top list is checked for consistency under that tolerance."""
import numpy as np
import pytest

import fastselect_b200 as fsb
from fastselect_b200 import _mdr, _native
from oracle import interaction_oracle as O
from oracle import mdr_oracle as M
from datasets import epistatic_genotypes

pytestmark = pytest.mark.gpu

DTYPES = [np.uint8, np.int8, np.float32]
ODD = {np.uint8: (0, 1, 200), np.int8: (-7, 0, 3), np.float32: (3.5, -7.0, 1e6)}


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def make_data(seed, n, p, dtype):
    """3-state columns over odd values, one constant and two 2-valued columns, about 10 % cases."""
    rs = np.random.RandomState(seed)
    vals = np.array(ODD[dtype], dtype)
    X = vals[rs.randint(0, 3, (n, p))]
    X[:, 3] = vals[1]                                          # constant
    X[:, 5] = vals[rs.randint(0, 2, n)]                        # 2-valued
    X[:, p - 1] = vals[1 + rs.randint(0, 2, n)]
    y = np.zeros(n, np.int64)
    risk = (X[:, 1] == vals[2]) & (X[:, 7] != vals[0])
    order = np.argsort(~risk + rs.rand(n) * 0.5, kind="stable")
    y[order[:max(int(round(0.1 * n)), 2)]] = 1
    return X, y


def check_scan(ds, X, y, feat_idx=None, n_top=64):
    """One scan against the oracle: every L_KSA within tolerance, the listed tables exactly, the list
    consistent.  Returns the scan's result."""
    Xs = X if feat_idx is None else X[:, feat_idx]
    codes, _ = M.cells(Xs)
    tab = O.tables(codes, y)
    want = O.ksa(tab)
    n_top = min(n_top, want.size)
    got = ds.interaction_scan(n_top, feat_idx=feat_idx, want_all=True)
    n = X.shape[0]
    tol = 1e-11 * n
    np.testing.assert_allclose(got["all_ksa"], want, rtol=1e-11, atol=tol)
    top, ksa = got["top_idx"], got["top_ksa"]
    assert np.unique(top).size == n_top
    assert np.array_equal(bits(ksa), bits(got["all_ksa"][top]))
    assert np.all(ksa[:-1] >= ksa[1:])
    same = ksa[:-1] == ksa[1:]
    assert np.all(top[:-1][same] < top[1:][same])
    must = np.flatnonzero(want > ksa[-1] + tol + 1e-11 * abs(ksa[-1]))
    assert np.isin(must, top).all()
    assert np.array_equal(got["top_tables"], tab[top])
    return got


@pytest.mark.parametrize("n", [33, 127, 4095, 4097, 9001])
def test_scan_against_oracle(native, n):
    dtype = DTYPES[n % 3]
    X, y = make_data(n * 17, n, 40, dtype)
    with _mdr.MDRData(X, y) as src:
        got = check_scan(src._ds, X, y)
        again = src._ds.interaction_scan(64, want_all=True)
        for k in got:
            assert np.array_equal(np.asarray(got[k]).view(np.int64), np.asarray(again[k]).view(np.int64)), k
        idx = np.random.RandomState(n).permutation(40)[:29]    # unsorted column list
        check_scan(src._ds, X, y, feat_idx=idx, n_top=406)


def test_ties_from_copied_columns(native):
    rs = np.random.RandomState(5)
    base = rs.randint(0, 3, (48, 9)).astype(np.uint8)
    X = base[:, rs.randint(0, 9, 70)]
    y = np.array([0, 1] * 24)
    with _mdr.MDRData(X, y) as src:
        got = check_scan(src._ds, X, y, n_top=2048)
    assert np.unique(got["all_ksa"]).size < got["all_ksa"].size // 4


def test_mdr_interleaved(native):
    """MDR scans before and after an interaction scan on one data set: bitwise the same, and the interaction
    scan between them is the one a fresh data set gives."""
    X, y = make_data(3, 3001, 30, np.int8)
    fold = _mdr.make_folds(y, 5, None)
    with _mdr.MDRData(X, y) as src:
        fresh = src._ds.interaction_scan(50, want_all=True)
    with _mdr.MDRData(X, y) as src:
        ds = src._ds
        m1 = ds.mdr_scan(fold, 2, 50, want_all=True)
        got = ds.interaction_scan(50, want_all=True)
        m2 = ds.mdr_scan(fold, 2, 50, want_all=True)
        tabs = ds.mdr_tables(fold, 2, [[1, 7], [0, 29]])
    for k in m1:
        assert np.array_equal(np.asarray(m1[k]).view(np.int64), np.asarray(m2[k]).view(np.int64)), k
    for k in fresh:
        assert np.array_equal(np.asarray(got[k]).view(np.int64), np.asarray(fresh[k]).view(np.int64)), k
    assert np.array_equal(tabs, M.Source(X, y).tables(fold, 2, [[1, 7], [0, 29]]))


def test_estimator_equals_oracle(native):
    X, y = make_data(11, 2000, 60, np.int8)
    est = fsb.PairwiseInteraction(n_top=300).fit(X, y)
    want = O.fit(X, y, 300)
    assert np.array_equal(est.classes_, want["classes_"])
    assert np.array_equal(est.pairs_, want["pairs_"])
    assert np.array_equal(est.dof_, want["dof_"])
    assert est.n_pairs_tested_ == want["n_pairs_tested_"]
    np.testing.assert_allclose(est.ksa_statistic_, want["ksa_statistic_"], rtol=1e-11, atol=1e-11 * 2000)
    np.testing.assert_allclose(est.bound_, want["bound_"], rtol=1e-11, atol=1e-11 * 2000)
    np.testing.assert_allclose(est.statistic_, want["statistic_"], rtol=1e-7, atol=1e-7)
    np.testing.assert_allclose(est.p_values_, want["p_values_"], rtol=1e-6, atol=1e-300)
    assert np.all(est.statistic_ <= est.ksa_statistic_ + 1e-9 * 2000)


def test_c_abi_rejections(native):
    X, y = make_data(2, 200, 12, np.uint8)
    with _mdr.MDRData(X, y) as src:
        ds = src._ds
        with pytest.raises(ValueError, match="n_top"):
            ds.interaction_scan(67)                             # 66 pairs
        with pytest.raises(ValueError, match="n_top"):
            ds.interaction_scan(0)
        with pytest.raises(ValueError, match="pair"):
            ds.interaction_scan(1, feat_idx=[4])
        with pytest.raises(ValueError):
            ds.interaction_scan(1, feat_idx=[0, 12])
    with _mdr.MDRData(np.tile(X, (1, 8)), y) as src:            # 96 columns, 4560 pairs
        with pytest.raises(ValueError, match="n_top"):
            src._ds.interaction_scan(_native.FS_MDR_MAX_TOP + 1)
    X4 = X.copy()
    X4[0, 4] = 9
    with _mdr.MDRData(X4, y) as src:
        with pytest.raises(ValueError, match="at most 3"):
            src._ds.interaction_scan(1)
        src._ds.interaction_scan(1, feat_idx=[0, 1, 2])          # the 4-state column is not scanned
    y3 = y.copy()
    y3[0] = 2
    with _native.Dataset(X, y3, 3) as ds:
        ds.set_features(np.ones(12, np.uint8), np.ones(12, np.float32), _native.FS_ARITH_F32)
        with pytest.raises(ValueError, match="2 classes"):
            ds.interaction_scan(1)
    with pytest.raises(ValueError, match="at most 3"):
        fsb.PairwiseInteraction().fit(X4, y)


def test_planted_interaction_at_c3_shape(native):
    X, y = epistatic_genotypes(42, 4000, 100_000)
    est = fsb.PairwiseInteraction().fit(X, y)
    assert tuple(est.pairs_[0]) == (25, 75)
    assert est.n_pairs_tested_ == 4_999_950_000
    assert est.p_values_[0] < 0.05 / est.n_pairs_tested_
    assert np.all(est.statistic_ <= est.ksa_statistic_ + 1e-9 * 4000)
    rs = np.random.RandomState(1)
    idx = np.concatenate([[75], rs.choice(np.setdiff1d(np.arange(100_000), [25, 75]), 2000, replace=False), [25]])
    rs.shuffle(idx)
    with _mdr.MDRData(X, y) as src:
        got = check_scan(src._ds, X, y, feat_idx=idx, n_top=100)
    top = _mdr.decode_combinations(got["top_idx"][:1], idx.size, 2)[0]
    assert sorted(idx[top].tolist()) == [25, 75]
