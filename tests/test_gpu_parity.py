"""GPU: parity of the CUDA path (through the C ABI) with the CPU oracle and with the
reference's own outputs (golden vectors).  Integer work is compared bit-exactly,
floating-point weights with the reference's own tolerance (tests/test_surf.py:74-80:
rtol 1e-5, atol 1e-7 scaled by max|W|)."""
import numpy as np
import pytest

from datasets import epistatic_genotypes, gaussian, genotype, mixed
from oracle import ref_oracle as R

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def atol_for(ref):
    return 1e-7 * max(1.0, float(np.abs(ref).max()))


def open_multisurf(native, x, y, dl=10):
    x32, recip, isd = R.multisurf_prep(x, dl)
    yc = np.unique(y, return_inverse=True)[1]
    ds = native.Dataset(x32, yc.astype(np.int32), int(yc.max()) + 1)
    ds.set_features(isd, recip, native.FS_ARITH_F32)
    return ds, (x32, yc.astype(np.int64), recip, isd)


def open_surf(native, x, y, dl=10):
    x64, recip, isd = R.surf_prep(x, dl)
    y32 = np.asarray(y).astype(np.int32)
    yc = np.unique(y32, return_inverse=True)[1]
    ds = native.Dataset(x64, yc.astype(np.int32), int(yc.max()) + 1)
    ds.set_features(isd, recip, native.FS_ARITH_F64)
    return ds, (x64, y32, recip, isd)


def open_relieff(native, x, y, dl=10):
    x32, y_enc, cp, recip, isd = R.relieff_prep(x, y, dl)
    ds = native.Dataset(x32, y_enc, len(cp))
    ds.set_features(isd, recip, native.FS_ARITH_F32)
    return ds, (x32, y_enc, recip, isd, cp)


DATA = {
    "geno2": lambda: genotype(21, 150, 90, 2),
    "geno3": lambda: genotype(22, 131, 70, 3),
    "gauss2": lambda: gaussian(23, 160, 75, 2),
    "gauss4": lambda: gaussian(24, 129, 33, 4),
    "mixed3": lambda: mixed(25, 140, 64, 3),
    "mixed2": lambda: mixed(26, 200, 130, 2),
    "tiny": lambda: mixed(27, 7, 5, 2),
    "one_feature": lambda: gaussian(28, 40, 1, 2),
}


@pytest.mark.parametrize("name", list(DATA))
@pytest.mark.parametrize("star", [False, True])
def test_multisurf_rows_match_oracle(native, name, star):
    x, y = DATA[name]()
    n = x.shape[0]
    ds, args = open_multisurf(native, x, y)
    with ds:
        tg = np.arange(n)
        got = ds.debug_rows(native.FS_MULTISURF, tg, use_star=star)
        want = R.multisurf_targets(*args, star, tg)
        isd = args[3]
        if isd.all():      # integer distances: bit-exact
            assert np.array_equal(got["dist"], want["dist"])
            assert np.array_equal(got["thresh"], want["thresh"])
        else:
            np.testing.assert_allclose(got["dist"], want["dist"], rtol=1e-13, atol=1e-13)
            np.testing.assert_allclose(got["thresh"], want["thresh"], rtol=1e-13)
        assert np.array_equal(got["mask"], want["mask"])          # identical neighbour sets
        np.testing.assert_allclose(got["wsum"], want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * n)
        # the production entry point over the full row range gives the same sums
        full = ds.score(native.FS_MULTISURF, use_star=star)
        np.testing.assert_allclose(full, want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * n)


@pytest.mark.parametrize("name", list(DATA))
@pytest.mark.parametrize("star", [False, True])
def test_surf_rows_match_oracle(native, name, star):
    x, y = DATA[name]()
    n = x.shape[0]
    ds, args = open_surf(native, x, y)
    with ds:
        tg = np.arange(n)
        got = ds.debug_rows(native.FS_SURF, tg, use_star=star)
        want = R.surf_targets(*args, star, tg, sum_mode=2)
        assert np.array_equal(got["dist"], want["dist"])          # float32-rounded distances
        np.testing.assert_allclose(got["thresh"], want["thresh"], rtol=1e-15)
        assert np.array_equal(got["mask"], want["mask"])
        np.testing.assert_allclose(got["wsum"], want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * n)
        full = ds.score(native.FS_SURF, use_star=star)
        np.testing.assert_allclose(full, want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * n)


@pytest.mark.parametrize("name", ["geno2", "geno3", "gauss2", "gauss4", "mixed3", "mixed2", "one_feature"])
@pytest.mark.parametrize("k", [1, 5, 30])
@pytest.mark.parametrize("ties", ["reference", "index"])
def test_relieff_rows_match_oracle(native, monkeypatch, name, k, ties):
    """ties='reference': candidates tied at the k-th distance are taken in the order numba's
    quicksort leaves them (what the reference does; oracle tie_mode 0).  ties='index':
    FS_B200_RELIEFF_TIES=index takes them by sample index (oracle tie_mode 1)."""
    x, y = DATA[name]()
    n = x.shape[0]
    if k >= n:
        pytest.skip("k >= n")
    if ties == "index":
        monkeypatch.setenv("FS_B200_RELIEFF_TIES", "index")
    else:
        monkeypatch.delenv("FS_B200_RELIEFF_TIES", raising=False)
    ds, args = open_relieff(native, x, y)
    x32, y_enc, recip, isd, cp = args
    with ds:
        tg = np.arange(n)
        got = ds.debug_rows(native.FS_RELIEFF, tg, k=k, class_probs=cp)
        want = R.relieff_targets(x32, y_enc, recip, isd, k, cp, tg, tie_mode=0 if ties == "reference" else 1)
        assert np.array_equal(got["dist"], want["dist"])
        assert np.array_equal(got["mask"], want["mask"])          # identical neighbour sets
        np.testing.assert_allclose(got["wsum"], want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * n)
        full = ds.score(native.FS_RELIEFF, k=k, class_probs=cp)
        np.testing.assert_allclose(full, want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * n)


@pytest.mark.parametrize("k", [1, 10])
def test_relieff_reference_ties_beyond_shared_memory(native, monkeypatch, k):
    """n = 26 000 genotypes: a row's (distance, index) pairs take 208 000 bytes, more than the
    tie replay stages in shared memory, so the quicksort runs on global scratch.  18 targets
    spread over the classes (all of them would need a 5 GB distance output)."""
    monkeypatch.delenv("FS_B200_RELIEFF_TIES", raising=False)
    x, y = genotype(41, 26_000, 24, 3)
    ds, (x32, y_enc, recip, isd, cp) = open_relieff(native, x, y)
    tg = []
    for c in range(len(cp)):
        idx = np.flatnonzero(y_enc == c)
        tg.append(idx[np.linspace(0, idx.size - 1, 6).astype(np.int64)])
    tg = np.concatenate(tg)
    with ds:
        got = ds.debug_rows(native.FS_RELIEFF, tg, k=k, class_probs=cp)
    want = R.relieff_targets(x32, y_enc, recip, isd, k, cp, tg, tie_mode=0)
    other = R.relieff_targets(x32, y_enc, recip, isd, k, cp, tg, tie_mode=1, want_dist=False)
    assert np.array_equal(got["dist"], want["dist"])
    assert np.array_equal(got["mask"], want["mask"])
    np.testing.assert_allclose(got["wsum"], want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * tg.size)
    assert not np.array_equal(want["mask"], other["mask"])      # the tie order decides neighbours


def test_surf_mean_uses_the_reference_summation_order(native, golden):
    """gauss2_long: the float32 row sum decides two neighbour pairs; only the order the
    reference's compiled code uses (oracle sum_mode 2) reproduces the reference scores."""
    arrays, meta = golden
    x, y = arrays["X_gauss2_long"], arrays["y_gauss2_long"]
    ds, args = open_surf(native, x, y)
    with ds:
        got = ds.debug_rows(native.FS_SURF, np.arange(x.shape[0]))
    want = R.surf_targets(*args, False, np.arange(x.shape[0]), sum_mode=2)
    other = R.surf_targets(*args, False, np.arange(x.shape[0]), sum_mode=1)
    assert np.array_equal(got["thresh"], want["thresh"])
    assert np.array_equal(got["mask"], want["mask"])
    assert not np.array_equal(want["mask"], other["mask"])      # the case is discriminating


def test_relieff_without_ties_matches_the_reference_order(native):
    """On continuous data there are no distance ties, so the reference's quicksort order
    and the index tie rule select the same neighbours."""
    x, y = gaussian(31, 220, 40, 3)
    ds, (x32, y_enc, recip, isd, cp) = open_relieff(native, x, y)
    with ds:
        got = ds.score(native.FS_RELIEFF, k=7, class_probs=cp) / 220
    want = R.relieff_scores(x32, y_enc, recip, isd, 7, cp, tie_mode=0)
    np.testing.assert_allclose(got, want, rtol=RTOL, atol=2e-6 * np.abs(want).max())


def test_row_range_partials_add_up(native):
    """Target-row sharding: partial sums over a partition of the rows equal the full sum."""
    x, y = mixed(32, 333, 50, 3)
    ds, _ = open_multisurf(native, x, y)
    with ds:
        full = ds.score(native.FS_MULTISURF, use_star=True)
        parts = [ds.score(native.FS_MULTISURF, use_star=True, row_begin=a, row_end=b)
                 for a, b in ((0, 100), (100, 101), (101, 333))]
        np.testing.assert_allclose(sum(parts), full, rtol=1e-12, atol=1e-12)
        empty = ds.score(native.FS_MULTISURF, row_begin=5, row_end=5)
        assert not empty.any()


def test_column_subset_equals_fit_on_sliced_matrix(native):
    """fs_score(feat_idx) == scoring X[:, feat_idx] from scratch (what TuRF relies on)."""
    x, y = mixed(33, 150, 60, 2)
    keep = np.array([0, 3, 4, 7, 29, 30, 31, 45, 58, 59])
    ds, _ = open_surf(native, x, y)
    with ds:
        sub = ds.score(native.FS_SURF, use_star=True, feat_idx=keep)
    ds2, _ = open_surf(native, x[:, keep], y)
    with ds2:
        ref = ds2.score(native.FS_SURF, use_star=True)
    np.testing.assert_allclose(sub, ref, rtol=1e-12, atol=1e-12)


def test_repeat_scores_are_bitwise_identical(native):
    x, y = mixed(34, 180, 70, 3)
    ds, _ = open_multisurf(native, x, y)
    with ds:
        a = ds.score(native.FS_MULTISURF)
        b = ds.score(native.FS_MULTISURF)
    assert np.array_equal(a, b)


def test_column_scan_matches_numpy(native):
    x, _ = mixed(35, 97, 41, 2)
    x[:, 6] = np.arange(97) % 17          # 17 distinct values: over the cap
    x[:, 7] = np.arange(97) % 16          # exactly at the cap
    for dt in (np.float64, np.float32):
        xd = x.astype(dt)
        with native.Dataset(xd, np.zeros(97, np.int32), 1) as ds:
            cmin, cmax, cnt = ds.column_stats()
        assert np.array_equal(cmin, xd.min(axis=0).astype(np.float64))
        assert np.array_equal(cmax, xd.max(axis=0).astype(np.float64))
        want = np.array([np.unique(xd[:, f]).size for f in range(41)])
        assert np.array_equal(cnt, np.minimum(want, native.FS_DISTINCT_CAP + 1))
    g = (np.arange(97 * 5).reshape(97, 5) % 3).astype(np.int8) - 1
    with native.Dataset(g, np.zeros(97, np.int32), 1) as ds:
        cmin, cmax, cnt = ds.column_stats()
    assert cmin.tolist() == [-1] * 5 and cmax.tolist() == [1] * 5 and cnt.tolist() == [3] * 5


def _mixed_cardinality_genotypes(seed, n, p):
    """0/1/2 genotypes with some 2-valued, 4-valued and constant columns mixed in (exercises the
    general encode path and one-hot rows of unequal width next to the 0/1/2 fast path)."""
    x, y = epistatic_genotypes(seed, n, p)
    rs = np.random.RandomState(seed + 1)
    x[:, 5::17] = rs.randint(0, 2, x[:, 5::17].shape)
    x[:, 9::23] = rs.randint(0, 4, x[:, 9::23].shape)
    x[:, 11::29] = 1
    return x, y


@pytest.mark.parametrize("rows", [None, (130, 517)])
def test_incremental_distance_update_equals_full_recompute(native, monkeypatch, rows):
    """TuRF iterations: the resident distance slab is updated by subtracting the removed columns
    (exact integers) -- scores must be bitwise those of a from-scratch computation, for a full
    fit (symmetric tiles) and for a row shard."""
    n, p = 700, 1500
    x, y = _mixed_cardinality_genotypes(37, n, p)
    isd = np.ones(p, bool)
    recip = np.ones(p, np.float32)
    rs = np.random.RandomState(5)
    a1 = np.sort(rs.choice(p, int(p * 0.9), replace=False))
    a2 = np.sort(rs.choice(a1, int(a1.size * 0.9), replace=False))
    kw = {} if rows is None else dict(row_begin=rows[0], row_end=rows[1])

    def run():
        with native.Dataset(x, y.astype(np.int32), 2) as ds:
            ds.set_features(isd, recip, native.FS_ARITH_F32)
            out = [ds.score(native.FS_MULTISURF, want_stats=True, **kw)]
            out.append(ds.score(native.FS_MULTISURF, feat_idx=a1, want_stats=True, **kw))
            out.append(ds.score(native.FS_MULTISURF, feat_idx=a2, want_stats=True, **kw))
            out.append(ds.score(native.FS_MULTISURF, use_star=True, feat_idx=a2, want_stats=True, **kw))   # slab reused
        return out

    inc = run()
    monkeypatch.setenv("FS_B200_INCREMENTAL", "0")
    full = run()
    for (wi, si), (wf, sf) in zip(inc, full):
        assert np.array_equal(wi, wf)
    assert inc[0][1]["ops_dist_tensor"] == full[0][1]["ops_dist_tensor"]
    assert 0 < inc[1][1]["ops_dist_tensor"] < 0.5 * full[1][1]["ops_dist_tensor"]
    assert 0 < inc[2][1]["ops_dist_tensor"] < 0.5 * full[2][1]["ops_dist_tensor"]
    assert inc[3][1]["ops_dist_tensor"] == 0 and full[3][1]["ops_dist_tensor"] > 0


def _balanced_2_and_4_valued(seed, n, p):
    """As many 2-valued as 4-valued byte columns and nothing else: two reduced one-hot rows per column ON
    AVERAGE with identity value codes, which is not the 0/1/2 case the lean encoder hard-codes."""
    rs = np.random.RandomState(seed)
    x = np.empty((n, p), np.int8)
    x[:, 0::2] = rs.randint(0, 2, x[:, 0::2].shape)
    x[:, 1::2] = rs.randint(0, 4, x[:, 1::2].shape)
    y = ((x[:, 1] >= 2) ^ (rs.random_sample(n) < 0.2)).astype(np.int64)
    return x, y


@pytest.mark.parametrize("make", [lambda: _mixed_cardinality_genotypes(38, 400, 333), lambda: _balanced_2_and_4_valued(39, 300, 128)],
                         ids=["mixed", "balanced_2_4"])
def test_general_encode_path_matches_oracle(native, make):
    """Columns with 2, 3 and 4 values and constants on the one-hot path (reduced planes of unequal
    width): distances, masks and weights against the oracle."""
    x, y = make()
    xf = x.astype(np.float32)
    x32, recip, isd = R.multisurf_prep(xf, 10)
    tg = np.arange(0, x.shape[0], 3)
    with native.Dataset(x, y.astype(np.int32), 2) as ds:
        ds.set_features(isd, recip, native.FS_ARITH_F32)
        got = ds.debug_rows(native.FS_MULTISURF, tg, use_star=True)
    want = R.multisurf_targets(x32, y.astype(np.int64), recip, isd, True, tg)
    assert np.array_equal(got["dist"], want["dist"])
    assert np.array_equal(got["mask"], want["mask"])
    np.testing.assert_allclose(got["wsum"], want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * tg.size)


def test_chunked_target_rows_give_the_same_result(native, monkeypatch):
    """A 16 MB slab budget at n = 3000 (rows of round_up(n, 128) = 3072 samples) splits the target rows into chunks:
    3072 x 15 bytes per row (float64 and int32 distances, selection, masks) gives 256-row chunks on mixed data,
    3072 x 7 bytes (no float64 slab) 768-row chunks on genotypes.  Mixed data must match the single-chunk run;
    genotypes must match the oracle to the exactness of the one-hot path (see test_gpu_onehot_exact.py)."""
    from test_gpu_onehot_exact import oracle_multisurf

    n = 3000
    x, y = mixed(36, n, 40, 2)
    g, gy = epistatic_genotypes(36, n, 40)
    ds, _ = open_multisurf(native, x, y)
    with ds:
        a = ds.score(native.FS_MULTISURF, use_star=True)
    monkeypatch.setenv("FS_B200_CHUNK_MB", "16")
    ds, _ = open_multisurf(native, x, y)
    with ds:
        b, st = ds.score(native.FS_MULTISURF, use_star=True, want_stats=True)
    assert st["n_chunks"] == 12, st["n_chunks"]
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12)
    with native.Dataset(g, gy.astype(np.int32), 2) as ds:
        ds.set_features(np.ones(40, bool), np.ones(40, np.float32), native.FS_ARITH_F32)
        for star in (False, True):
            w, st = ds.score(native.FS_MULTISURF, use_star=star, want_stats=True)
            assert st["n_chunks"] == 4 and st["n_general_cols"] == 0, st
            want, _, atol = oracle_multisurf(g, gy, star, ds.row_order())
            assert np.abs(w - want).max() <= atol, (star, np.abs(w - want).max(), atol)


def test_c3_shape_subset_of_targets(native):
    """Config C3 geometry at reduced p (genotypes int8, epistatic labels): exact integer
    distances / identical masks / weights for a random subset of targets, and the two
    planted SNPs rank first."""
    x, y = epistatic_genotypes(42, 1500, 1200)
    xf = x.astype(np.float32)
    x32, recip, isd = R.multisurf_prep(xf, 10)
    assert isd.all()
    yc = y.astype(np.int64)
    rs = np.random.RandomState(0)
    tg = np.sort(rs.choice(1500, 256, replace=False))
    with native.Dataset(x, y.astype(np.int32), 2) as ds:          # int8 end to end
        ds.set_features(isd, recip, native.FS_ARITH_F32)
        got = ds.debug_rows(native.FS_MULTISURF, tg)
        full = ds.score(native.FS_MULTISURF) / 1500
    want = R.multisurf_targets(x32, yc, recip, isd, False, tg)
    assert np.array_equal(got["dist"], want["dist"])
    assert np.array_equal(got["thresh"], want["thresh"])
    assert np.array_equal(got["mask"], want["mask"])
    np.testing.assert_allclose(got["wsum"], want["wsum"], rtol=RTOL, atol=atol_for(want["wsum"]) * 256)
    assert set(np.argsort(full)[::-1][:2]) == {25, 75}
