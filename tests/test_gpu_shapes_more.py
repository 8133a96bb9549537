"""GPU: the benchmark shapes round 1 left untested (VERDICT round 1, "What's missing" 1-2 and the
production-path gap):

* C4 = SURF and SURF* on 20 000 x 50 000 mixed columns, float64 X (SURF.py:131-218, :330-372);
* C5 = 20 000 x 500 000 int8 genotypes: the oracle on 16 targets at full width for TuRF's first pass,
  and for the second pass (450 000 active columns, TuRF.py:99-113) the incrementally updated resident
  distance slab bit-exact against oracle distances;
* the PRODUCTION entry point (fs_score over a contiguous internal row range: class-aligned tiles,
  skipped K blocks, paired epilogue) against the oracle's weights for exactly those rows on C3 and C4
  -- fs_debug_rows runs the same plan on runs of consecutive internal rows of its targets.

Each test body also runs at a reduced shape so that a failure localises quickly."""
import numpy as np
import pytest

from datasets import epistatic_genotypes
from oracle import ref_oracle as R
from test_gpu_shapes_full import make_c4

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def atol_for(ref):
    return 1e-7 * max(1.0, float(np.abs(ref).max()))


# --------------------------------------------------------------------------- #
# C4: SURF / SURF*
# --------------------------------------------------------------------------- #
def surf_preprocess(x64, h):
    """SURF.fit's preprocessing (SURF.py:347-355) for the C4 layout: the genotype half is discrete
    (3 values <= discrete_limit), the Gaussian half is not; ranges from the float64 matrix, discrete -> 1."""
    p = x64.shape[1]
    isd = np.arange(p) < h
    ranges = x64.max(axis=0) - x64.min(axis=0)
    ranges[isd] = 1.0
    ranges[ranges == 0] = 1.0
    return isd, (1.0 / ranges).astype(np.float32)


def check_surf_rows(out, y, targets, use_star):
    """SURF.py:151-195 re-derived from the distance rows: d float32-rounded; threshold = the float32
    mean of the row (incl. d_ii = 0) / (n - 1), here only to float32 resolution (its exact summation
    order is the oracle's business); near = d < T strict; sum_f W_i[f] = sum_near_miss d - sum_near_hit d
    (+ sum_far_hit d - sum_far_miss d), no count normalisation."""
    d, thresh, mask = out["dist"], out["thresh"], out["mask"]
    n = d.shape[1]
    y = np.asarray(y)
    checksum = scale = 0.0
    for r, i in enumerate(targets):
        row = d[r]
        assert np.array_equal(row, row.astype(np.float32).astype(np.float64))
        np.testing.assert_allclose(thresh[r], row.sum() / (n - 1), rtol=1e-5)
        others = np.arange(n) != i
        near = (row < thresh[r]) & others
        hit = (y == y[i]) & others
        want = np.zeros(n, np.int8)
        want[near & hit] = 1
        want[near & ~hit & others] = 2
        if use_star:
            want[~near & ~hit & others] = 3
            want[~near & hit] = 4
        assert np.array_equal(mask[r], want), int(i)
        s = row[want == 2].sum() - row[want == 1].sum() + row[want == 4].sum() - row[want == 3].sum()
        checksum += s
        scale += row[want != 0].sum()
    # the distances are float32-rounded sums of the terms the weights add up exactly
    assert abs(out["wsum"].sum() - checksum) <= 2e-7 * max(scale, 1.0), (out["wsum"].sum(), checksum, scale)


def run_c4_surf(native, n, p, n_targets, use_star):
    x32, y = make_c4(n, p)
    x = x32.astype(np.float64)               # SURF validates X to float64 (SURF.py:330-332)
    del x32
    h = p // 2
    isd, recip = surf_preprocess(x, h)
    y32 = y.astype(np.int32)
    rs = np.random.RandomState(2)
    tg = np.sort(rs.choice(n, n_targets, replace=False))
    sub = tg[::8]
    with native.Dataset(x, y32, 2) as ds:
        ds.set_features(isd, recip, native.FS_ARITH_F64)
        full, st = ds.score(native.FS_SURF, use_star=use_star, want_stats=True)
        got = ds.debug_rows(native.FS_SURF, tg, use_star=use_star)
        got8 = ds.debug_rows(native.FS_SURF, sub, use_star=use_star)
        perm = ds.row_order()
        # production path: 16 contiguous internal rows straddling the class boundary
        cut = int((y32 == 0).sum())
        r0 = max(0, cut - 8)
        prod = ds.score(native.FS_SURF, use_star=use_star, row_begin=r0, row_end=r0 + 16)
    assert np.isfinite(full).all() and full.shape == (p,)
    assert st["n_tensor_cols"] == h and st["n_general_cols"] == p - h
    check_surf_rows(got, y, tg, use_star)
    want = R.surf_targets(x, y32, recip, isd, use_star, sub, sum_mode=2)
    # float32-rounded float64 sums of p terms in two different orders: equal unless on a rounding boundary
    np.testing.assert_allclose(got8["dist"], want["dist"], rtol=2e-7, atol=0)
    np.testing.assert_allclose(got8["thresh"], want["thresh"], rtol=3e-6)
    same = got8["mask"] == want["mask"]
    if not same.all():
        # a pair may only differ where its float32 distance sits within rounding of the threshold
        bad = np.argwhere(~same)
        for r, j in bad:
            assert abs(got8["dist"][r, j] - got8["thresh"][r]) <= 3e-6 * got8["thresh"][r], (r, j)
        assert len(bad) <= 2
    else:
        np.testing.assert_allclose(got8["wsum"], want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * len(sub))
    rows = perm[r0:r0 + 16]
    want_p = R.surf_targets(x, y32, recip, isd, use_star, rows, sum_mode=2, want_mask=False, want_dist=False)
    np.testing.assert_allclose(prod, want_p["wsum"], rtol=RTOL, atol=atol_for(want_p["wsum"]) * 16)


@pytest.mark.parametrize("use_star", [False, True])
def test_c4_reduced_shape_surf(native, use_star):
    run_c4_surf(native, 700, 1200, 64, use_star)


@pytest.mark.parametrize("use_star", [False, True])
def test_c4_full_shape_surf_mixed_float64(native, use_star):
    """C4: SURF / SURF* on 20 000 x 50 000 mixed columns (25 000 genotype + 25 000 Gaussian), float64 X."""
    run_c4_surf(native, 20_000, 50_000, 32, use_star)


# --------------------------------------------------------------------------- #
# production path (fs_score row range) vs the oracle on C3 / C4
# --------------------------------------------------------------------------- #
def run_c3_production_rows(native, n, p):
    x, y = epistatic_genotypes(42, n, p)
    isd = np.ones(p, bool)
    recip = np.full(p, 0.5, np.float32)
    cut = int((y == 0).sum())
    with native.Dataset(x, y.astype(np.int32), 2) as ds:
        ds.set_features(isd, recip, native.FS_ARITH_F32)
        perm = ds.row_order()
        ranges = [(0, 16), (max(0, cut - 8), cut + 8), (n - 16, n)]
        got = [ds.score(native.FS_MULTISURF, row_begin=a, row_end=b) for a, b in ranges]
        got_star = ds.score(native.FS_MULTISURF, use_star=True, row_begin=ranges[1][0], row_end=ranges[1][1])
    for (a, b), g in zip(ranges, got):
        want = R.multisurf_targets_bytes(x, y, False, perm[a:b], want_mask=False, want_dist=False)
        np.testing.assert_allclose(g, want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * (b - a))
    a, b = ranges[1]
    want = R.multisurf_targets_bytes(x, y, True, perm[a:b], want_mask=False, want_dist=False)
    np.testing.assert_allclose(got_star, want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * (b - a))


def test_c3_reduced_production_rows(native):
    run_c3_production_rows(native, 900, 1300)


def test_c3_full_shape_production_rows_match_oracle(native):
    """C3 at full width: fs_score over 16-row internal ranges (first rows, across the class boundary,
    last rows) against the oracle's weights for row_order()[rows]."""
    run_c3_production_rows(native, 4000, 100_000)


def run_c4_production_rows(native, n, p):
    x, y = make_c4(n, p)
    h = p // 2
    ranges_ = (x.max(axis=0) - x.min(axis=0)).astype(np.float32)
    ranges_[ranges_ == 0] = 1
    recip = (1.0 / ranges_).astype(np.float32)
    isd = np.arange(p) < h
    cut = int((y == 0).sum())
    a, b = max(0, cut - 8), cut + 8
    with native.Dataset(x, y.astype(np.int32), 2) as ds:
        ds.set_features(isd, recip, native.FS_ARITH_F32)
        perm = ds.row_order()
        got = ds.score(native.FS_MULTISURF, use_star=True, row_begin=a, row_end=b)
    want = R.multisurf_targets(x, y, recip, isd, True, perm[a:b], want_mask=False, want_dist=False)
    np.testing.assert_allclose(got, want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * (b - a))


def test_c4_reduced_production_rows(native):
    run_c4_production_rows(native, 600, 1000)


def test_c4_full_shape_production_rows_match_oracle(native):
    run_c4_production_rows(native, 20_000, 50_000)


# --------------------------------------------------------------------------- #
# C5: TuRF's first and second pass at 20 000 x 500 000
# --------------------------------------------------------------------------- #
def make_c5_like(n, p):
    """bench.py's C5 generator (int8 genotypes in independent 1000-row blocks, epistatic label)."""
    x = np.empty((n, p), np.int8)
    for b0 in range(0, n, 1000):
        b1 = min(b0 + 1000, n)
        x[b0:b1] = np.random.default_rng([44, b0 // 1000]).integers(0, 3, size=(b1 - b0, p), dtype=np.int8)
    rs = np.random.RandomState(44)
    y = np.zeros(n, np.int64)
    y[(x[:, 25] == 1) & (x[:, 75] == 1)] = 1
    need = n // 2 - int(y.sum())
    if need > 0:
        y[rs.choice(np.flatnonzero(y == 0), need, replace=False)] = 1
    return x, y


def run_c5(native, n, p, n_targets=16):
    x, y = make_c5_like(n, p)
    isd = np.ones(p, bool)
    recip = np.full(p, 0.5, np.float32)
    rs = np.random.RandomState(3)
    tg = np.sort(rs.choice(n, n_targets, replace=False))
    with native.Dataset(x, y.astype(np.int32), 2) as ds:          # int8 end to end
        ds.set_features(isd, recip, native.FS_ARITH_F32)
        perm = ds.row_order()
        inv = np.empty(n, np.int64)
        inv[perm] = np.arange(n)
        # ---- first pass: all p columns (what TuRF.fit scores first, TuRF.py:87)
        w1 = ds.score(native.FS_MULTISURF)
        got1 = ds.debug_rows(native.FS_MULTISURF, tg)
        want1 = R.multisurf_targets_bytes(x, y, False, tg)
        assert np.array_equal(got1["dist"], want1["dist"])
        assert np.array_equal(got1["thresh"], want1["thresh"])
        assert np.array_equal(got1["mask"], want1["mask"])
        np.testing.assert_allclose(got1["wsum"], want1["wsum"], rtol=RTOL, atol=atol_for(want1["wsum"]) * n_targets)
        # the production pass leaves the full slab resident (fs_debug_rows above dropped it: score again)
        w1b = ds.score(native.FS_MULTISURF)
        assert np.array_equal(w1, w1b)
        for q, t in enumerate(tg):
            row, info = ds.debug_slab(int(inv[t]), 1)
            assert info == (0, n, p)
            assert np.array_equal(row[0][inv], want1["dist"][q].astype(np.int32)), int(t)
        # ---- second pass: drop the worst 10 % (TuRF.py:99-106); the slab is updated by subtraction
        n_remove = max(1, int(p * 0.1))
        worst = np.argsort(w1)[:n_remove]
        active = np.delete(np.arange(p), worst)
        w2, st2 = ds.score(native.FS_MULTISURF, feat_idx=active, want_stats=True)
        # incremental update: far fewer tensor operations than a full distance pass over the active columns
        assert 0 < st2["ops_dist_tensor"] < 0.3 * 4.0 * n * n * active.size
        want2 = R.multisurf_targets_bytes(x, y, False, tg, cols=active)
        for q, t in enumerate(tg):
            row, info = ds.debug_slab(int(inv[t]), 1)
            assert info == (0, n, active.size)
            d_gpu = row[0][inv]                       # original sample order
            d_ref = want2["dist"][q].astype(np.int32)
            keep = np.arange(n) != t                  # the slab also holds d_ii = 0 structurally
            assert np.array_equal(d_gpu[keep], d_ref[keep]), int(t)
            assert d_gpu[t] == 0
        got2 = ds.debug_rows(native.FS_MULTISURF, tg, feat_idx=active)
        assert np.array_equal(got2["mask"], want2["mask"])
        np.testing.assert_allclose(got2["wsum"], want2["wsum"], rtol=RTOL, atol=atol_for(want2["wsum"]) * n_targets)
    assert w2.shape == (active.size,) and np.isfinite(w2).all()
    return w1, w2, active


def test_c5_reduced_shape_two_turf_passes(native):
    run_c5(native, 1200, 3000)


def test_c5_full_shape_two_turf_passes_match_oracle(native):
    """C5: MultiSURF at 20 000 x 500 000 int8 -- oracle on 16 targets at full width for the first pass;
    second pass (450 000 active columns): the incrementally updated slab bit-exact against oracle
    distances, masks identical, weights within tolerance.  The two planted SNPs survive the pruning."""
    w1, w2, active = run_c5(native, 20_000, 500_000)
    assert {25, 75} <= set(active.tolist())
    top2 = set(active[np.argsort(w2)[::-1][:2]].tolist())
    assert top2 == {25, 75}
