"""CPU: host side of MDR (fastselect_b200/_mdr.py) with the GPU hook (``_mdr.open_mdr``) served by the numpy
oracle (oracle/mdr_oracle.py): hand-computed balanced accuracies, the combination index, the ranking and tie
rules, the final model, and every parameter check."""
import pickle

import numpy as np
import pytest
from sklearn.base import clone

import fastselect_b200 as fsb
from fastselect_b200 import _mdr, _native
from oracle import mdr_oracle as O


@pytest.fixture
def hook(monkeypatch):
    opened = []

    def fake_open(X, y_enc):
        src = O.Source(X, y_enc)
        opened.append(src)
        return src

    monkeypatch.setattr(_mdr, "open_mdr", fake_open)
    monkeypatch.setattr(_native, "device_count", lambda: 1)
    return opened


def assert_fitted_equal(est, want):
    for k, v in want.items():
        got = getattr(est, k)
        if isinstance(v, list):
            assert len(got) == len(v)
            for a, b in zip(got, v):
                assert np.array_equal(a, b), k
        elif isinstance(v, float):
            assert np.float64(got).view(np.int64) == np.float64(v).view(np.int64), k
        else:
            assert np.array_equal(np.asarray(got), np.asarray(v)), k


def test_xor_pair_is_perfect(hook):
    rs = np.random.RandomState(0)
    X = rs.randint(0, 2, (200, 4)).astype(np.uint8)
    y = X[:, 1] ^ X[:, 3]
    est = fsb.MDR(order=2, cv=5).fit(X, y)
    assert est.best_combination_ == (1, 3)
    assert est.train_balanced_accuracy_ == 1.0 and est.test_balanced_accuracy_ == 1.0
    assert est.cv_consistency_ == 5
    assert tuple(est.top_combinations_[0]) == (1, 3) and est.top_test_balanced_accuracy_[0] == 1.0
    assert np.array_equal(est.predict(X), y)


def test_constant_column_scores_one_half():
    y = np.array([0, 1] * 10)
    s = O.scan(np.full((20, 1), 7.0), y, np.arange(20) % 2 * 0 + (np.arange(20) // 2) % 2, 2, 1)
    assert np.all(s["train"] == 0.5) and np.all(s["test"] == 0.5)


def test_ratio_tie_is_low_risk():
    # fold 0 (test): nothing in cell 0; training (fold 1): cell 0 holds 2 cases / 4 controls, cell 1 holds
    # 1 case / 2 controls -> both ratios equal N1 / N0 = 3 / 6, so both cells are low-risk
    t = np.zeros((1, 2, 2, 9), np.int64)
    t[0, 1, 0, 0], t[0, 1, 1, 0] = 4, 2
    t[0, 1, 0, 1], t[0, 1, 1, 1] = 2, 1
    t[0, 0, 0, 1], t[0, 0, 1, 1] = 3, 2
    train, _ = _mdr.fold_scores(t)
    assert train[0, 0] == 0.5                          # all low-risk: TN = N0, TP = 0
    seg = t.reshape(1, 4, 9)
    assert np.array_equal(O.fold_scores(seg)[0], train)
    t[0, 1, 1, 0] = 3                                  # one more case in cell 0: high-risk now
    train, _ = _mdr.fold_scores(t)
    # training of fold 0 is fold 1: N1 = 4, N0 = 6; TP = 3 (cell 0), TN = 2 (cell 1)
    assert train[0, 0] == (3 * 6 + 2 * 4) / (2 * 4 * 6)


@pytest.mark.parametrize("p", [2, 3, 17, 1000])
def test_combination_index_round_trip(p):
    a, b = np.triu_indices(p, 1)
    idx = _mdr.encode_combinations(np.stack([a, b], 1), p)
    assert np.array_equal(idx, np.arange(p * (p - 1) // 2))
    assert np.array_equal(_mdr.decode_combinations(idx, p, 2), np.stack([a, b], 1))
    assert np.array_equal(O.decode(idx[::97], p, 2), np.stack([a, b], 1)[::97])
    assert np.array_equal(_mdr.decode_combinations(np.arange(p), p, 1)[:, 0], np.arange(p))


def test_large_index_decode():
    p = 100_000
    combos = np.array([[0, 1], [25, 75], [99_998, 99_999], [50_000, 50_001], [3, 99_999]])
    assert np.array_equal(_mdr.decode_combinations(_mdr.encode_combinations(combos, p), p, 2), combos)


def planted(seed=3, n=300, p=12):
    rs = np.random.RandomState(seed)
    X = rs.randint(0, 3, (n, p)).astype(np.int8)
    y = ((X[:, 2] == 1) & (X[:, min(5, p - 1)] == 1)).astype(int)
    flip = rs.rand(n) < 0.2
    y[flip] = 1 - y[flip]
    return X, y


@pytest.mark.parametrize("order", [1, 2])
@pytest.mark.parametrize("cv,rs", [(2, None), (3, 7), (5, None), (10, 1)])
def test_estimator_equals_oracle(hook, order, cv, rs):
    X, y = planted()
    est = fsb.MDR(order=order, cv=cv, n_top=20, random_state=rs).fit(X, y)
    assert_fitted_equal(est, O.fit(X, y, order, cv, 20, rs))
    assert hook[-1].calls == ["scan", "tables"]


def test_ties_from_duplicated_columns(hook):
    X, y = planted()
    X = np.concatenate([X, X[:, [5, 2]], X[:, [2]]], axis=1)      # 12 <- 5, 13 <- 2, 14 <- 2
    est = fsb.MDR(order=2, cv=5, n_top=50).fit(X, y)
    want = O.fit(X, y, 2, 5, 50)
    assert_fitted_equal(est, want)
    assert est.best_combination_ == (2, 5)                          # lowest index among the exact copies
    top = [tuple(c) for c in est.top_combinations_[:6]]
    assert top[:4] == [(2, 5), (2, 12), (5, 13), (5, 14)]           # equal scores: index order
    s = O.scan(X, np.unique(y, return_inverse=True)[1], _mdr.make_folds(y, 5, None), 5, 2)
    assert len(set(s["mean_test"][_mdr.encode_combinations(np.array(top[:4]), 15)].tolist())) == 1


def test_predict_transform_unseen_refit_clone_pickle(hook):
    X, y = planted()
    labels = np.where(y == 1, "case", "ctrl")
    est = fsb.MDR(order=2, cv=3).fit(X, labels)
    assert list(est.classes_) == ["case", "ctrl"]                    # classes_[1] = "ctrl" is the case class here
    a, b = est.best_combination_
    assert np.array_equal(est.transform(X), X[:, [a, b]])
    pred = est.predict(X)
    va = np.searchsorted(est.feature_values_[0], X[:, a])
    vb = np.searchsorted(est.feature_values_[1], X[:, b])
    assert np.array_equal(pred == est.classes_[1], est.high_risk_[va, vb])
    Z = X.copy()
    Z[:4, a] = 9                                                    # unseen value: low-risk
    assert np.all(est.predict(Z)[:4] == est.classes_[0])
    est2 = pickle.loads(pickle.dumps(est))
    assert np.array_equal(est2.predict(X), pred)
    assert not any(isinstance(v, (_native.Dataset, _mdr.MDRData)) for v in vars(est).values())
    c = clone(est)
    assert c.get_params() == est.get_params() and not hasattr(c, "best_combination_")
    est.set_params(order=1).fit(X, y)                              # refit replaces every attribute
    assert len(est.best_combination_) == 1 and est.high_risk_.shape == (3,)
    assert_fitted_equal(est, O.fit(X, y, 1, 3, 100))
    assert est.top_combinations_.shape == (12, 1)                   # n_top clamps to the 12 combinations


def test_value_errors(hook):
    X, y = planted(n=60, p=4)
    X4 = X.copy()
    X4[0, 1] = 7                                                    # a 4th state
    with pytest.raises(ValueError, match="at most 3"):
        fsb.MDR().fit(X4, y)
    with pytest.raises(ValueError, match="2 classes"):
        fsb.MDR().fit(X, np.arange(60) % 3)
    y_few = np.zeros(60, int)
    y_few[:4] = 1
    with pytest.raises(ValueError, match="at least cv"):
        fsb.MDR(cv=5).fit(X, y_few)
    fsb.MDR(cv=4).fit(X, y_few)
    for bad in (1, 11, 2.5, True):
        with pytest.raises(ValueError, match="cv"):
            fsb.MDR(cv=bad).fit(X, y)
    for bad in (0, 3):
        with pytest.raises(ValueError, match="order"):
            fsb.MDR(order=bad).fit(X, y)
    for bad in (0, -1, _native.FS_MDR_MAX_TOP + 1):
        with pytest.raises(ValueError, match="n_top"):
            fsb.MDR(n_top=bad).fit(X, y)
    with pytest.raises(ValueError, match="numeric"):
        fsb.MDR().fit(X.astype(str).astype(object), y)
    with pytest.raises(ValueError):
        fsb.MDR().fit(np.where(X == 0, np.nan, X), y)
    with pytest.raises(ValueError, match="at least 2 features"):
        fsb.MDR(order=2).fit(X[:, :1], y)


def test_backends(hook, monkeypatch):
    X, y = planted(n=60, p=4)
    with pytest.raises(NotImplementedError):
        fsb.MDR(backend="cpu").fit(X, y)
    with pytest.raises(ValueError, match="backend"):
        fsb.MDR(backend="tpu").fit(X, y)
    monkeypatch.setattr(_native, "device_count", lambda: 0)
    with pytest.raises(RuntimeError):
        fsb.MDR().fit(X, y)


def test_upload_keeps_values_distinct():
    assert _mdr._upload_array(np.array([[0, 255]], np.int64)).dtype == np.uint8
    assert _mdr._upload_array(np.array([[-7, 3]], np.int64)).dtype == np.int8
    big = np.array([[-(1 << 40), 1 << 40, 5]], np.int64)
    assert np.array_equal(_mdr._upload_array(big).astype(np.int64), big)
    with pytest.raises(ValueError):
        _mdr._upload_array(np.array([[0, (1 << 60) + 1]], np.int64))
    assert _mdr._upload_array(np.array([[1.5]], np.float16)).dtype == np.float64


def test_folds_are_stratified_and_deterministic():
    y = np.array([0] * 13 + [1] * 7)
    f1 = _mdr.make_folds(y, 3, None)
    assert np.array_equal(f1, _mdr.make_folds(y, 3, None))
    for f in range(3):
        assert set(y[f1 == f]) == {0, 1}
    assert not np.array_equal(_mdr.make_folds(y, 3, 0), _mdr.make_folds(y, 3, 1))
