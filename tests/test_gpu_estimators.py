"""GPU: the estimator API end to end against the reference's own outputs (golden vectors)
and the behavioural contract of the reference's tests (tests/test_multisurf.py,
test_surf.py, test_relieff.py, test_turf.py)."""
import pickle

import numpy as np
import pytest

import fastselect_b200 as fsb
from oracle import ref_oracle as R

pytestmark = pytest.mark.gpu

CLS = {"MultiSURF": fsb.MultiSURF, "SURF": fsb.SURF, "ReliefF": fsb.ReliefF}


def test_estimators_match_reference_vectors(native, golden):
    arrays, meta = golden
    checked = 0
    for m in meta:
        if m["idx"] < 0 or m["algo"].startswith("TuRF"):
            continue
        x, y = arrays[f"X_{m['data']}"], arrays[f"y_{m['data']}"]
        ref = arrays[f"scores_{m['idx']}"]
        est = CLS[m["algo"]](n_features_to_select=min(3, x.shape[1]), backend="gpu", **m["params"]).fit(x, y)
        assert est.effective_backend_ == "gpu"
        assert np.array_equal(est.is_discrete_, arrays[f"isd_{m['idx']}"]), m
        assert est.feature_importances_.dtype == np.float32
        scale = max(1.0, float(np.abs(ref).max()))
        # SURVEY 8(c)(3): rtol 1e-5, atol 1e-7 * max(1, max|W|) against the reference's own float32 outputs
        np.testing.assert_allclose(est.feature_importances_, ref, rtol=1e-5, atol=1e-7 * scale, err_msg=str(m))
        top = np.argsort(ref)[::-1][:len(est.top_features_)]
        if not np.array_equal(est.top_features_, top):
            # 8(c)(4): adjacent reference weights closer than 2e-7 * max|W| are inside the reference's own noise
            gaps = np.abs(np.diff(np.sort(ref)[::-1][: len(top) + 1]))
            assert gaps.min() < 2e-7 * scale, m
        checked += 1
    assert checked >= 70


def test_readme_quickstart_top15(native, golden):
    from sklearn.datasets import make_classification

    arrays, _ = golden
    x, y = make_classification(n_samples=500, n_features=1000, n_informative=20, n_redundant=100, random_state=42)
    # the golden vectors were made with the scikit-learn of this image; a different RNG stream must be
    # noticed (the fixture regenerated with tests/golden/make_golden.py), not skipped over
    assert np.allclose([x.sum(), np.abs(x).sum(), float(y.sum())], arrays["readme_xsum"]), \
        "make_classification produced a different matrix than the one the golden vectors were made from"

    est = fsb.MultiSURF(n_features_to_select=15, backend="gpu").fit(x, y)
    np.testing.assert_allclose(est.feature_importances_, arrays["readme_scores"], rtol=1e-5,
                               atol=1e-7 * max(1.0, float(np.abs(arrays["readme_scores"]).max())))
    assert np.array_equal(est.top_features_, arrays["readme_top"])
    assert est.transform(x).shape == (500, 15)


def test_turf_matches_reference(native, golden):
    arrays, meta = golden
    for m in meta:
        if not m["algo"].startswith("TuRF"):
            continue
        base = m["algo"].split(":")[1]
        x, y = arrays[f"X_{m['data']}"], arrays[f"y_{m['data']}"]
        t = fsb.TuRF(CLS[base](n_features_to_select=5, backend="gpu", **m["params"]),
                     n_features_to_select=m["turf"]["n"], pct_remove=m["turf"]["pct"]).fit(x, y)
        ref = arrays[f"scores_{m['idx']}"]
        np.testing.assert_allclose(t.feature_importances_, ref, rtol=1e-5, atol=1e-7 * max(1.0, float(np.abs(ref).max())))
        assert np.array_equal(t.top_features_, arrays[f"top_{m['idx']}"]), m


def test_turf_resident_path_equals_refit_path(native):
    """TuRF's device-resident column-subset scoring gives the scores a from-scratch fit of
    X[:, active] gives (TuRF.py:110-111)."""
    from datasets import mixed

    x, y = mixed(51, 120, 40, 2)
    t = fsb.TuRF(fsb.MultiSURF(backend="gpu"), n_features_to_select=6, pct_remove=0.25).fit(x, y)

    class Refit(fsb.MultiSURF):      # same estimator, but not recognised as resident-capable
        pass

    active = np.arange(40)
    scores = fsb.MultiSURF(backend="gpu", n_features_to_select=1).fit(x, y).feature_importances_
    while len(active) > 6:
        k = max(1, int(len(active) * 0.25))
        if len(active) - k < 6:
            k = len(active) - 6
        active = np.delete(active, np.argsort(scores)[:k])
        scores = fsb.MultiSURF(backend="gpu", n_features_to_select=1).fit(x[:, active], y).feature_importances_
    assert np.array_equal(t.top_features_, np.sort(active))


def test_int8_genotypes_equal_float_input(native):
    from datasets import epistatic_genotypes

    x, y = epistatic_genotypes(7, 300, 500)
    a = fsb.MultiSURF(n_features_to_select=5, backend="gpu").fit(x, y)
    b = fsb.MultiSURF(n_features_to_select=5, backend="gpu").fit(x.astype(np.float64), y)
    assert np.array_equal(a.feature_importances_, b.feature_importances_)
    assert a.is_discrete_.all()
    c = fsb.SURF(n_features_to_select=5, backend="gpu", use_star=True).fit(x, y)
    d = fsb.SURF(n_features_to_select=5, backend="gpu", use_star=True).fit(x.astype(np.float64), y)
    assert np.array_equal(c.feature_importances_, d.feature_importances_)


def test_behavioural_contract(native, capsys):
    x = np.array([[1.1, 5.0, 10, 3.0], [1.2, 4.0, 10, 3.0], [2.3, 6.0, 10, 3.0], [2.5, 5.5, 10, 3.0],
                  [1.5, 4.5, 20, 3.0], [8.8, 5.0, 20, 3.0], [8.9, 4.0, 20, 3.0], [9.5, 6.0, 20, 3.0],
                  [10.5, 4.5, 20, 3.0], [10.5, 4.5, 10, 3.0]], dtype=np.float32)
    y = np.array([0] * 5 + [1] * 5, dtype=np.int32)
    m = fsb.MultiSURF(n_features_to_select=1, backend="gpu", discrete_limit=4).fit(x, y)
    assert set(m.top_features_) == {0} and abs(m.feature_importances_[3]) < 1e-7   # test_multisurf.py:36-45
    assert fsb.MultiSURF(n_features_to_select=3, backend="gpu").fit_transform(x, y).shape == (10, 3)
    fsb.MultiSURF(n_features_to_select=2, backend="gpu", use_star=True, verbose=True).fit(x, y)
    assert "Running MultiSURF*" in capsys.readouterr().out
    fsb.SURF(n_features_to_select=2, backend="gpu", verbose=True).fit(x, y)
    out = capsys.readouterr().out
    assert "Running SURF on the GPU now..." in out and "Feature scoring completed." in out
    # single-class y: all scores <= 0 (test_multisurf.py:193-205); ReliefF returns zeros
    s = fsb.MultiSURF(n_features_to_select=2, backend="gpu").fit(x, np.zeros(10)).feature_importances_
    assert (s <= 0).all()
    r = fsb.ReliefF(n_features_to_select=2, backend="gpu").fit(x, np.zeros(10))
    assert not r.feature_importances_.any() and r.top_features_.tolist() == [0, 1]
    with pytest.warns(UserWarning, match="smallest class size"):
        fsb.ReliefF(n_features_to_select=2, n_neighbors=5, backend="gpu").fit(x, y)
    # discrete_limit (test_multisurf.py:96-110)
    xd = np.array([[i, i % 3] for i in range(11)] * 2, dtype=np.float32)
    yd = np.array([0] * 11 + [1] * 11, dtype=np.int32)
    assert fsb.MultiSURF(discrete_limit=10, backend="gpu", n_features_to_select=2).fit(xd, yd).is_discrete_.tolist() == [False, True]
    assert fsb.MultiSURF(discrete_limit=12, backend="gpu", n_features_to_select=2).fit(xd, yd).is_discrete_.tolist() == [True, True]
    # wide discrete columns (more distinct values than the device scan tracks)
    xw = np.array([[i % 20, i % 3, (i * 7) % 19] for i in range(60)], dtype=np.float64)
    yw = (np.arange(60) % 2).astype(np.int64)
    est = fsb.SURF(discrete_limit=25, backend="gpu", n_features_to_select=2).fit(xw, yw)
    assert est.is_discrete_.all()
    want = R.fit_surf(xw, yw, 25, False, 2)[0]
    np.testing.assert_allclose(est.feature_importances_, want, rtol=1e-5, atol=1e-7)
    # fitted estimators pickle and refit identically
    m2 = pickle.loads(pickle.dumps(m))
    assert np.array_equal(m2.feature_importances_, m.feature_importances_)
    assert np.array_equal(m2.fit(x, y).feature_importances_, m.feature_importances_)


@pytest.mark.parametrize("cls", [fsb.MultiSURF, fsb.SURF, fsb.ReliefF])
def test_sklearn_estimator_checks(native, cls):
    """The reference runs sklearn's check_estimator with the default backend='auto'
    (tests/test_multisurf.py:78-83), i.e. through the GPU path on a GPU box."""
    from sklearn.utils.estimator_checks import check_estimator

    check_estimator(cls())


def test_sklearn_estimator_checks_turf(native):
    from sklearn.utils.estimator_checks import check_estimator

    check_estimator(fsb.TuRF(fsb.MultiSURF()))


def test_turf_on_genotypes_matches_oracle_driven_turf(native):
    """Config C5 geometry at reduced size: TuRF(MultiSURF, pct 0.1) on int8 genotypes with the
    data set resident on the GPU, against the same pruning loop driven by the CPU oracle."""
    from datasets import epistatic_genotypes

    x, y = epistatic_genotypes(44, 300, 600)
    t = fsb.TuRF(fsb.MultiSURF(backend="gpu"), n_features_to_select=10, pct_remove=0.1).fit(x, y)

    xf = x.astype(np.float32)
    active = np.arange(600)
    scores = R.fit_multisurf(xf, y)[0]
    first = scores.copy()
    while len(active) > 10:
        k = max(1, int(len(active) * 0.1))
        if len(active) - k < 10:
            k = len(active) - 10
        active = np.delete(active, np.argsort(scores)[:k])
        scores = R.fit_multisurf(xf[:, active], y)[0]
    # `first` comes from the oracle's REFERENCE-ARITHMETIC entry (float32 accumulators summed in the
    # reference's order: up to 7.7e-7 * max|W| away from the exact value, DESIGN.md section 5), hence 2e-6
    np.testing.assert_allclose(t.feature_importances_, first, rtol=1e-5, atol=2e-6 * np.abs(first).max())
    assert np.array_equal(t.top_features_, np.sort(active))


def test_non_integer_labels_follow_the_reference_cpu_semantics(native):
    """Labels are only compared for equality (MultiSURF.py:216), so y = {0.2, 0.7} must score like y = {0, 1}
    (the reference's CPU semantics; its own GPU branch truncates with astype(int32), MultiSURF.py:424, which
    would merge these two classes).  SURF keeps the reference's truncation on every backend (SURF.py:363,371)."""
    from datasets import mixed

    x, y = mixed(51, 160, 24, 2)
    yf = np.where(y == 0, 0.2, 0.7)
    a = fsb.MultiSURF(n_features_to_select=4, backend="gpu").fit(x, y)
    b = fsb.MultiSURF(n_features_to_select=4, backend="gpu").fit(x, yf)
    assert np.array_equal(a.feature_importances_, b.feature_importances_)
    r = fsb.ReliefF(n_features_to_select=4, n_neighbors=5, backend="gpu").fit(x, yf)
    r0 = fsb.ReliefF(n_features_to_select=4, n_neighbors=5, backend="gpu").fit(x, y)
    assert np.array_equal(r.feature_importances_, r0.feature_importances_)


def test_wide_integer_input_is_narrowed_not_converted(native):
    """np.random.randint returns int64: the estimators narrow it to int8 before validation (values
    unchanged) instead of letting sklearn convert it to float32; the scores are those of the int8 matrix."""
    from datasets import epistatic_genotypes

    x8, y = epistatic_genotypes(52, 300, 200)
    a = fsb.MultiSURF(n_features_to_select=5, backend="gpu").fit(x8, y)
    b = fsb.MultiSURF(n_features_to_select=5, backend="gpu").fit(x8.astype(np.int64), y)
    assert np.array_equal(a.feature_importances_, b.feature_importances_)
    t = fsb.TuRF(fsb.MultiSURF(backend="gpu", n_features_to_select=5), n_features_to_select=8, pct_remove=0.3).fit(x8.astype(np.int64), y)
    t0 = fsb.TuRF(fsb.MultiSURF(backend="gpu", n_features_to_select=5), n_features_to_select=8, pct_remove=0.3).fit(x8, y)
    assert np.array_equal(t.top_features_, t0.top_features_)


def test_staged_upload_of_pageable_views(native, monkeypatch):
    """fs_dataset_create copies a PAGEABLE source through page-locked blocks with a pool of host threads
    (dataset.cu); contiguous arrays, row-strided views and the driver's own staging must give the same fit."""
    rs = np.random.RandomState(11)
    n, p = 300, 40000                                          # 12 MB of int8: above the staging threshold
    y = rs.randint(0, 2, n)
    wide = rs.randint(0, 3, (n, p + 64)).astype(np.int8)
    wide[:, 7] = (y + rs.randint(0, 2, n)) % 3
    view = wide[:, :p]                                         # row stride p + 64
    assert not view.flags["C_CONTIGUOUS"]
    fit = lambda a: fsb.MultiSURF(n_features_to_select=5, backend="gpu").fit(a, y).feature_importances_
    w_view, w_copy = fit(view), fit(np.ascontiguousarray(view))
    monkeypatch.setenv("FS_B200_NO_STAGED_UPLOAD", "1")
    w_driver = fit(view)
    assert np.array_equal(w_view, w_copy) and np.array_equal(w_view, w_driver)
    assert np.argmax(w_view) == 7


def test_accumulation_kernels_agree_many_tiles(native, monkeypatch):
    """More target tiles than one launch of the merged-plane accumulation kernel takes (117 tiles of <= 224 rows
    > 112): the launches add into the same exact column sums.  Both it and the paired kernel (one launch) must
    match the oracle to the exactness of the one-hot path (see test_gpu_onehot_exact.py)."""
    from test_gpu_onehot_exact import oracle_multisurf

    rs = np.random.RandomState(12)
    n, p = 26000, 48
    y = rs.randint(0, 3, n)
    x = rs.randint(0, 3, (n, p)).astype(np.int8)
    x[:, 5] = (y + rs.randint(0, 2, n)) % 3
    assert sum(-(-int(c) // 224) for c in np.bincount(y)) > 112
    want, _, atol = oracle_multisurf(x, y, False, np.arange(n))
    for mode in ("3", "1"):
        monkeypatch.setenv("FS_B200_ACCUM_PAIR", mode)
        # the float64 sums fit() divides by n and rounds to float32
        with native.Dataset(x, y.astype(np.int32), 3) as ds:
            ds.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F32)
            w, st = ds.score(native.FS_MULTISURF, want_stats=True)
        assert st["n_tensor_cols"] == p and st["ops_accum_tensor"] > 0
        assert np.abs(w - want).max() <= atol, (mode, np.abs(w - want).max(), atol)
        assert np.argmax(fsb.MultiSURF(n_features_to_select=3, backend="gpu").fit(x, y).feature_importances_) == 5
