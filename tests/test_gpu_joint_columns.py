"""GPU: the column path of the joint-count statistics (fs_joint_columns) and ``pairs="selected"`` of mRMR /
CFS.  Rows from the column path must be BITWISE the rows of fs_joint_matrix (same marginals, same operand
order, same finishing arithmetic), a repeated call must reuse the encoding, and the estimators must give
the same fitted attributes in both modes -- at a size whose p x p matrix would not fit on the device too.

Tolerances against the float64 oracle: MI rtol 1e-11 (as tests/test_gpu_joint.py)."""
import numpy as np
import pytest

import fastselect_b200 as fsb
from fastselect_b200 import _native
from oracle import ref_oracle as R
from test_gpu_joint import CASES, many_states, open_codes

pytestmark = pytest.mark.gpu
KINDS = [(0, np.log(2.0)), (0, 1.0), (1, 1.0)]
KIND_IDS = ["mi_bit", "mi_nat", "su"]


def assert_rows_match(ds, kind, base, feat_idx=None):
    full = ds.joint_matrix(kind, base, feat_idx=feat_idx)
    q = full.shape[0]
    cols = ds.joint_columns(kind, base, np.arange(q), feat_idx=feat_idx)
    assert cols.shape == (q, q) and cols.dtype == np.float64
    assert np.array_equal(cols.view(np.int64), full.view(np.int64))
    rev = np.arange(q)[::-1].copy()                       # any order, repeated positions
    pick = np.concatenate([rev[:5], rev[:2]])
    assert np.array_equal(ds.joint_columns(kind, base, pick, feat_idx=feat_idx).view(np.int64),
                          full[pick].view(np.int64))


@pytest.mark.parametrize("name,make", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("kind,base", KINDS, ids=KIND_IDS)
def test_columns_are_the_matrix_rows_bitwise(native, name, make, kind, base):
    x, y = make()
    with open_codes(native, np.concatenate([x, y[:, None]], axis=1)) as ds:
        assert_rows_match(ds, kind, base)


@pytest.mark.parametrize("n", [127, 4095, 4097, 9001, 20000])
@pytest.mark.parametrize("kind,base", KINDS, ids=KIND_IDS)
def test_columns_at_odd_and_multi_chunk_sample_counts(native, n, kind, base):
    """odd n, n not a multiple of 128, and n over one 4096-sample chunk of the count kernel (up to 5)."""
    x, y = many_states(n, n, 37)
    xa = np.concatenate([x, y[:, None]], axis=1)
    with open_codes(native, xa) as ds:
        assert_rows_match(ds, kind, base)
        idx = np.random.RandomState(n).permutation(xa.shape[1])[:23]
        assert_rows_match(ds, kind, base, feat_idx=idx)


def test_genotype_columns_across_chunks(native):
    rs = np.random.RandomState(8)
    x = rs.randint(0, 3, (13001, 300)).astype(np.uint8)
    x[:, 7] = 1                                           # constant column
    with open_codes(native, x) as ds:
        assert_rows_match(ds, 0, np.log(2.0))
        assert_rows_match(ds, 1, 1.0)


def test_second_call_reuses_the_encoding(native):
    x, y = many_states(3, 5000, 64)
    xa = np.concatenate([x, y[:, None]], axis=1)
    with open_codes(native, xa) as ds:
        first, st1 = ds.joint_columns(0, 1.0, [64], want_stats=True)
        second, st2 = ds.joint_columns(0, 1.0, [5], want_stats=True)
        third, st3 = ds.joint_columns(0, 1.0, [64], want_stats=True)
        assert np.array_equal(first, third)
        # first: encode + marginals + one count + one finish; later: count + finish only
        assert st1["launches"] >= 4
        for st in (st2, st3):
            assert st["launches"] == 2 and st["n_chunks"] == 1
            assert st["ms_gather"] < 0.05, st
        # a position with 17 reduced rows' worth in one call: two count launches
        st4 = ds.joint_columns(0, 1.0, [14, 29, 44], want_stats=True)[1]     # 15 + 15 + 15 reduced rows
        assert st4["n_chunks"] == 3 and st4["launches"] == 6
        # a different column list rebuilds, and the old one is rebuilt again after it
        idx = np.arange(0, 65, 2)
        _, st5 = ds.joint_columns(0, 1.0, [1], feat_idx=idx, want_stats=True)
        assert st5["launches"] > 2
        _, st6 = ds.joint_columns(0, 1.0, [64], want_stats=True)
        assert st6["launches"] > 2
        # the matrix path on the same list shares the working set and leaves the cache valid
        full = ds.joint_matrix(0, 1.0)
        again, st7 = ds.joint_columns(0, 1.0, [64], want_stats=True)
        assert st7["launches"] == 2 and np.array_equal(again[0], full[64]) and np.array_equal(again, first)


def test_invalid_arguments(native):
    x, y = many_states(4, 200, 10)
    with open_codes(native, np.concatenate([x, y[:, None]], axis=1)) as ds:
        with pytest.raises(ValueError, match="outside"):
            ds.joint_columns(0, 1.0, [11])
        with pytest.raises(ValueError, match="outside"):
            ds.joint_columns(0, 1.0, [-1])
        with pytest.raises(ValueError, match="outside"):
            ds.joint_columns(0, 1.0, [3], feat_idx=[0, 1, 2])
        with pytest.raises(ValueError, match="log_base must be positive"):
            ds.joint_columns(0, 0.0, [0])
        with pytest.raises(ValueError, match="unknown kind"):
            ds.joint_columns(2, 1.0, [0])
    with _native.Dataset(np.random.RandomState(0).rand(30, 3).astype(np.float32), np.zeros(30, np.int32), 1) as ds:
        ds.set_features(np.zeros(3, np.uint8), np.ones(3, np.float32), _native.FS_ARITH_F32)
        with pytest.raises(ValueError, match="not a discrete column"):
            ds.joint_columns(0, 1.0, [0])


def check_mrmr_modes(x, y, k, method):
    a = fsb.mRMR(k, method, "gpu").fit(x, y)
    s = fsb.mRMR(k, method, "gpu", pairs="selected").fit(x, y)
    assert np.array_equal(a.top_features_, s.top_features_)
    assert np.array_equal(a.relevance_scores_.view(np.int64), s.relevance_scores_.view(np.int64))
    assert np.array_equal(a.unique_vals_, s.unique_vals_) and a.n_features_in_ == s.n_features_in_
    assert np.array_equal(a.redundancy_matrix_[a.top_features_].view(np.int64), s.redundancy_columns_.view(np.int64))
    assert not hasattr(s, "redundancy_matrix_") and s.feature_importances_ is s.relevance_scores_
    return s


def check_cfs_modes(x, y):
    a = fsb.CFS(backend="gpu").fit(x, y)
    s = fsb.CFS(backend="gpu", pairs="selected").fit(x, y)
    assert np.array_equal(a.selected_indices_, s.selected_indices_)
    assert np.array_equal(a.support_mask_, s.support_mask_)
    assert np.array_equal(a.r_cf_, s.r_cf_) and a.merit_ == s.merit_
    assert not hasattr(s, "r_ff_")
    return s


def test_estimators_selected_equals_all_on_the_golden_data(native):
    import os

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "joint_vectors.npz"))
    for data in ("mrmr_fixture", "mrmr_dup", "geno", "states"):
        x, y = g[f"X_{data}"], g[f"y_{data}"]
        for method in ("MID", "MIQ"):
            ref = g[f"mrmr_top_{method}_{data}"]
            s = check_mrmr_modes(x, y, len(ref), method)
            assert np.array_equal(s.top_features_, ref), (data, method)
    for data in ("cfs_fixture", "geno", "states", "mrmr_fixture"):
        s = check_cfs_modes(g[f"X_{data}"], g[f"y_{data}"])
        assert np.array_equal(s.selected_indices_, g[f"cfs_sel_{data}"]), data


def test_estimators_selected_equals_all_on_genotypes(native):
    rs = np.random.RandomState(33)
    n, p = 3000, 4000
    x = rs.randint(0, 3, (n, p)).astype(np.uint8)
    y = ((x[:, 10] + x[:, 2000] + (rs.random_sample(n) < 0.3)) > 2).astype(np.uint8)
    x[:, 3999] = x[:, 10]                                   # an exact duplicate of a relevant column
    for method in ("MID", "MIQ"):
        s = check_mrmr_modes(x, y, 25, method)
        assert {10, 2000} <= set(s.top_features_.tolist()) | {3999}
    check_cfs_modes(x, y)


def test_mrmr_selected_at_a_size_whose_matrix_does_not_fit(native):
    """4000 x 200 000 genotypes: the p x p float64 matrix would be 320 GB."""
    rs = np.random.RandomState(44)
    n, p = 4000, 200_000
    x = rs.randint(0, 3, (n, p), dtype=np.uint8)
    y = ((x[:, 123_456] == 2) ^ (rs.random_sample(n) < 0.1)).astype(np.uint8)
    est = fsb.mRMR(n_features_to_select=20, pairs="selected").fit(x, y)
    assert est.top_features_[0] == 123_456
    assert est.redundancy_columns_.shape == (20, p)
    cols = rs.choice(p, 64, replace=False)
    xi = x[:, cols].astype(np.int32)
    rel = R.mi_matrices(xi, y.astype(np.int32), want_matrix=False)[0]
    np.testing.assert_allclose(est.relevance_scores_[cols], rel, rtol=1e-11, atol=1e-15)
    for i in range(2):
        f = int(est.top_features_[i])
        red = R.mi_matrices(xi, x[:, f].astype(np.int32), want_matrix=False)[0]
        red[cols == f] = 0.0
        np.testing.assert_allclose(est.redundancy_columns_[i, cols], red, rtol=1e-11, atol=1e-15)
