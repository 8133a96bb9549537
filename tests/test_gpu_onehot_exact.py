"""GPU: the one-hot tensor-core GEMMs of the production path held to the exactness DESIGN.md (sections 2 and 4)
promises on genotype data, at the tile, K-block, class and launch edges where their host plans branch.

* Accumulation: ``fs_score`` over contiguous internal row ranges (class-aligned tiles, skipped K blocks) with each
  kernel -- ``FS_B200_ACCUM_PAIR`` = 3 (merged-plane CTA pairs, the default for 0/1/2 columns), 1 (paired epilogue),
  0 (one thread per one-hot row, the default for every other value count) -- and ``fs_debug_rows`` on scattered
  targets (mixed tiles), against the CPU oracle's weights at a tolerance derived from the number formats
  (``exact_tolerance``) instead of rtol 1e-5: a single miscounted (target, sample, feature) triple fails.
* Distances: the resident slab of ``tc_dist_pair_kernel`` (symmetric mirrored tiles for the full range, plain tiles
  for a range off the 128-row grid, the incremental subtract update) bitwise against exact integer distances.

The CPU tests at the end check the tolerance argument with exact rational arithmetic and check that every case
reaches the edge it is listed for (tile counts, launches, one-hot row blocks, L2 bands, K-block remainders)."""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest

from datasets import epistatic_genotypes
from oracle import ref_oracle as R

# host-plan constants of tc_accum.cu / tc_dist.cu that the cases below are built around
MERGED_BN, PAIRED_BN = 224, 240                 # target rows per tile: merged-plane kernel / paired and rows kernels
MERGED_MAX_TILES, MAX_TILES = 112, 256          # tile descriptors per launch
KS = 256                                        # samples per K block (128 bytes of FP4 nibbles)
BM = 128                                        # one-hot rows per block
L2_BAND_N, L2_BAND_GROUPS = 8192, 12            # merged kernel: groups of two tiles in bands of twelve for n > 8192
ORACLE_BLOCK = 256                              # targets per oracle call; the block sums are added exactly
MODES = ("3", "1", "0")


# --------------------------------------------------------------------------- #
# reference and tolerance
# --------------------------------------------------------------------------- #
def _term_bound(mask):
    """Upper bound of |one target's weight term| per mask row.  MultiSURF: |m / n_miss - h / n_hit| <= 1; MultiSURF*
    subtracts far misses from m but still divides by the near-miss count, so |m| / n_miss can exceed 1."""
    near = (mask == R.NEAR_MISS).sum(axis=1)
    far = (mask == R.FAR_MISS).sum(axis=1)
    return np.maximum(1.0, (near + far) / np.maximum(near, 1))


def exact_tolerance(n, nt, term_sum, block):
    """Largest distance between the GPU weights and the oracle's allowed by the arithmetic of both.

    GPU: a per-target coefficient c is held as C = round(c * 2^52) and multiplied by integer counts |t| <= n in
    int64, so each (target, mask) pair errs by at most n * 2^-53.  Oracle: one float64 division per term and a
    float64 sum over at most ``block`` terms (the block sums are added exactly), at most block * sum|term| * 2^-53.
    Both bounds are taken with a factor of four to spare."""
    atol = (nt * n + min(block, nt) * term_sum) * 2.0 ** -51
    # one miscounted (target, sample, feature) triple moves a weight by at least 1 / (n - 1)
    assert atol < 0.01 / n, (atol, n, nt)
    return atol


def oracle_multisurf(codes, y, star, targets, cols=None, block=ORACLE_BLOCK):
    """CPU oracle weights of the (original-order) ``targets``, exact on integer counts, one float64 division per
    term; blocks of targets are summed in float64 by the oracle and the block sums added exactly (math.fsum).
    Returns (wsum, masks, atol)."""
    targets = np.asarray(targets, np.int64)
    parts, masks, term_sum = [], [], 0.0
    for b0 in range(0, targets.size, block):
        out = R.multisurf_targets_bytes(codes, y, star, targets[b0:b0 + block], cols=cols, want_dist=False)
        parts.append(out["wsum"])
        masks.append(out["mask"])
        term_sum += float(_term_bound(out["mask"]).sum())
    parts = np.array(parts)
    wsum = np.array([math.fsum(parts[:, f]) for f in range(parts.shape[1])])
    return wsum, np.concatenate(masks), exact_tolerance(codes.shape[0], targets.size, term_sum, block)


def oracle_surf(codes, y, star, targets):
    """SURF / SURF* on genotypes: discrete terms +-1 (range 1), so the weights are integers."""
    p = codes.shape[1]
    out = R.surf_targets(codes.astype(np.float64), y.astype(np.int32), np.ones(p, np.float32), np.ones(p, np.uint8),
                         star, np.asarray(targets, np.int64), sum_mode=2, want_dist=False)
    assert np.array_equal(out["wsum"], np.round(out["wsum"]))
    return out["wsum"], out["mask"]


def exact_distances(codes, rows):
    """Mismatch counts of the samples ``rows`` against every sample, as exact float64 one-hot products."""
    d = np.full((len(rows), codes.shape[0]), float(codes.shape[1]))
    for v in np.unique(codes):
        e = (codes == v).astype(np.float64)
        d -= e[rows] @ e.T
    return d.astype(np.int64)


# --------------------------------------------------------------------------- #
# data
# --------------------------------------------------------------------------- #
def _genotypes(seed, p, class_sizes):
    """0/1/2 int8 genotypes in which every column holds all three values, labels with the given class sizes in
    shuffled sample order, column 0 tied to the label."""
    rs = np.random.RandomState(seed)
    y = np.repeat(np.arange(len(class_sizes)), class_sizes)
    rs.shuffle(y)
    n = y.size
    x = rs.randint(0, 3, (n, p)).astype(np.int8)
    x[:, 0] = (y + rs.randint(0, 2, n)) % 3
    x[:3] = np.arange(3, dtype=np.int8)[:, None]
    return x, y.astype(np.int64)


def _mixed_cardinality_genotypes(seed, n, p):
    """0/1/2 genotypes with some 2-valued, 4-valued and constant columns mixed in (exercises the
    general encode path and one-hot rows of unequal width next to the 0/1/2 fast path)."""
    x, y = epistatic_genotypes(seed, n, p)
    rs = np.random.RandomState(seed + 1)
    x[:, 5::17] = rs.randint(0, 2, x[:, 5::17].shape)
    x[:, 9::23] = rs.randint(0, 4, x[:, 9::23].shape)
    x[:, 11::29] = 1
    return x, y


def _balanced_2_and_4_valued(seed, n, p):
    """As many 2-valued as 4-valued byte columns and nothing else: two reduced one-hot rows per column ON
    AVERAGE with identity value codes, which is not the 0/1/2 case the lean encoder hard-codes."""
    rs = np.random.RandomState(seed)
    x = np.empty((n, p), np.int8)
    x[:, 0::2] = rs.randint(0, 2, x[:, 0::2].shape)
    x[:, 1::2] = rs.randint(0, 4, x[:, 1::2].shape)
    y = ((x[:, 1] >= 2) ^ (rs.random_sample(n) < 0.2)).astype(np.int64)
    return x, y


def _odd_split(n):
    """Two classes; the first ends on an odd sample, off every 256-sample K block."""
    a = (n // 2) | 1
    return [a, n - a]


ENCODINGS = {
    "i8_012": lambda g: g,
    "u8_012": lambda g: g.astype(np.uint8),
    "i8_m101": lambda g: g - 1,
    "i8_123": lambda g: g + 1,
    "f32_012": lambda g: g.astype(np.float32),
}


class Case:
    """One data set of the accumulation sweep.  ``make`` returns (int8 genotype codes, labels); ``cross`` is a row
    range across a class boundary that starts off the 128-row grid; ``edge`` names what the case reaches (checked
    on the CPU by test_cases_reach_their_edges)."""

    def __init__(self, edge, make, cross, encoding="i8_012", surf=False):
        self.edge, self.make, self.cross, self.encoding, self.surf = edge, make, cross, encoding, surf


CASES = {}
for _n in (255, 256, 257, 511, 513):
    _s = _odd_split(_n)
    CASES[f"kblock_n{_n}"] = Case("kblock", functools.partial(_genotypes, _n, 40, _s), (_s[0] - 37, min(_n, _s[0] + 200)),
                                  surf=True)
for _p in (64, 65, 150):
    CASES[f"mblocks_p{_p}"] = Case("mblocks", functools.partial(_genotypes, _p, _p, [301, 299]), (264, 500))
CASES["class_tails"] = Case("class_tails", functools.partial(_genotypes, 7, 30, [31, 1, 2, 33, 933]), (5, 300), surf=True)
CASES["launch_150x40"] = Case("launch", functools.partial(_genotypes, 8, 24, [40] * 150), (3, 1003))
CASES["launch_300x20"] = Case("launch", functools.partial(_genotypes, 9, 24, [20] * 300), (3, 1003))
CASES["l2_n8192"] = Case("l2_off", functools.partial(_genotypes, 10, 40, [4096, 4096]), (4059, 4296))
CASES["l2_n8193"] = Case("l2_bands", functools.partial(_genotypes, 11, 40, [4096, 4097]), (4059, 4296))
for _e in ENCODINGS:
    CASES[f"enc_{_e}"] = Case("encoding", functools.partial(_genotypes, 12, 65, [257, 256]), (220, 457), encoding=_e)
CASES["mixed_cardinality"] = Case("not_v3", functools.partial(_mixed_cardinality_genotypes, 38, 400, 333), None)
CASES["balanced_2_4"] = Case("not_v3", functools.partial(_balanced_2_and_4_valued, 39, 300, 128), None)


@functools.lru_cache(maxsize=4)
def case_data(name):
    """(matrix as uploaded, int8 codes, labels, class starts in internal order, row ranges)."""
    c = CASES[name]
    codes, y = c.make()
    codes.setflags(write=False)
    starts = np.concatenate([[0], np.cumsum(np.bincount(y))])
    n = codes.shape[0]
    cross = c.cross
    if cross is None:
        b = int(starts[1])
        a = b - 37 if (b - 37) % 128 else b - 38
        cross = (a, min(n, b + 150))
    ranges = [(0, n), cross, (int(starts[1]), int(starts[1]) + 1), (n - 1, n)]
    return ENCODINGS[c.encoding](codes), codes, y, starts, ranges


def three_valued(codes):
    return all(np.unique(codes[:, f]).size == 3 for f in range(codes.shape[1]))


def scattered_targets(n):
    rs = np.random.RandomState(n)
    return np.sort(rs.choice(n, min(n, 150), replace=False))


@functools.lru_cache(maxsize=64)
def ref_multisurf(name, star, a, b, perm_key):
    codes, y = CASES[name].make()
    perm = np.frombuffer(perm_key, np.int64)
    return oracle_multisurf(codes, y, star, perm[a:b])


@functools.lru_cache(maxsize=64)
def ref_multisurf_targets(name, star, tg_key):
    codes, y = CASES[name].make()
    return oracle_multisurf(codes, y, star, np.frombuffer(tg_key, np.int64))


def _accum_params():
    out = []
    for name in CASES:
        codes, _ = CASES[name].make()
        for mode in (MODES if three_valued(codes) else ("default",)):
            out.append(pytest.param(name, mode, id=f"{name}-{mode}"))
    return out


def _set_mode(monkeypatch, mode):
    if mode == "default":
        monkeypatch.delenv("FS_B200_ACCUM_PAIR", raising=False)
    else:
        monkeypatch.setenv("FS_B200_ACCUM_PAIR", mode)


# --------------------------------------------------------------------------- #
# accumulation sweep
# --------------------------------------------------------------------------- #
@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _accum_params())
def test_multisurf_weights_are_exact(native, monkeypatch, name, mode):
    """MultiSURF and MultiSURF*: fs_score over [0, n) (symmetric distances), a range across a class boundary off the
    128-row grid, one row and the last row, then fs_debug_rows on scattered targets, against the oracle."""
    _set_mode(monkeypatch, mode)
    x, codes, y, starts, ranges = case_data(name)
    n, p = codes.shape
    with native.Dataset(x, y.astype(np.int32), starts.size - 1) as ds:
        ds.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F32)
        perm = ds.row_order()
        assert np.array_equal(y[perm], np.repeat(np.arange(starts.size - 1), np.diff(starts)))   # class-sorted
        for a, b in ranges:
            for star in (False, True):
                got, st = ds.score(native.FS_MULTISURF, use_star=star, row_begin=a, row_end=b, want_stats=True)
                assert st["n_general_cols"] == 0 and st["n_tensor_cols"] > 0 and st["ops_accum_tensor"] > 0, st
                want, _, atol = ref_multisurf(name, star, a, b, perm.tobytes())
                err = np.abs(got - want).max()
                assert err <= atol, (name, mode, star, (a, b), err, atol)
        tg = scattered_targets(n)
        for star in (False, True):
            got = ds.debug_rows(native.FS_MULTISURF, tg, use_star=star)
            want, mask, atol = ref_multisurf_targets(name, star, tg.tobytes())
            assert np.array_equal(got["mask"], mask)
            err = np.abs(got["wsum"] - want).max()
            assert err <= atol, (name, mode, star, "debug_rows", err, atol)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", [k for k, c in CASES.items() if c.surf])
def test_surf_weights_are_exact_integers(native, monkeypatch, name, mode):
    """SURF and SURF* on genotypes: coefficients +-1, so the fixed-point sums are exact and the weights must equal
    the oracle's integers (while sum |t| * 2^26 < 2^53, i.e. n <= 8192)."""
    _set_mode(monkeypatch, mode)
    x, codes, y, starts, ranges = case_data(name)
    n, p = codes.shape
    assert n <= 8192
    with native.Dataset(x, y.astype(np.int32), starts.size - 1) as ds:
        ds.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F64)
        perm = ds.row_order()
        for a, b in ranges:
            for star in (False, True):
                got, st = ds.score(native.FS_SURF, use_star=star, row_begin=a, row_end=b, want_stats=True)
                assert st["n_tensor_cols"] == p and st["ops_accum_tensor"] > 0, st
                want, _ = oracle_surf(codes, y, star, perm[a:b])
                assert np.array_equal(got, want), (name, mode, star, (a, b), np.abs(got - want).max())
        tg = scattered_targets(n)
        for star in (False, True):
            got = ds.debug_rows(native.FS_SURF, tg, use_star=star)
            want, mask = oracle_surf(codes, y, star, tg)
            assert np.array_equal(got["mask"], mask)
            assert np.array_equal(got["wsum"], want), (name, mode, star, "debug_rows")


# --------------------------------------------------------------------------- #
# distance sweep
# --------------------------------------------------------------------------- #
def _check_slab(ds, codes, perm, inv, a, b, cols=None):
    slab, info = ds.debug_slab(a, b - a)
    sub = codes if cols is None else np.ascontiguousarray(codes[:, cols])
    varying = int((sub.min(axis=0) != sub.max(axis=0)).sum())              # constant columns have no one-hot rows
    assert info == (a, b - a, varying)
    assert np.all(slab[np.arange(b - a), np.arange(a, b)] == 0)            # d_ii = 0
    want = exact_distances(sub, perm[a:b])
    got = slab[:, inv]                                                     # original sample order
    bad = np.argwhere(got != want)
    assert bad.size == 0, (a, b, bad[:5].tolist(), got[tuple(bad[0])], want[tuple(bad[0])])


def _dist_ranges(n):
    return [(0, n), (37, 37 + min(300, n - 37))]


@pytest.mark.gpu
@pytest.mark.parametrize("p", [1, 127, 128, 129, 300])
@pytest.mark.parametrize("n", [129, 255, 256, 257, 513])
def test_distance_slab_is_exact(native, n, p):
    """The slab fs_score leaves resident, for [0, n) (symmetric: half of the super-blocks mirrored) and for a range
    starting at row 37 (not symmetric, off the 128-row grid), n around the 256-row super-block and p around the
    128-byte K block (2p reduced one-hot rows)."""
    codes, y = _genotypes(100 + n, p, _odd_split(n))
    with native.Dataset(codes, y.astype(np.int32), 2) as ds:
        ds.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F32)
        perm = ds.row_order()
        inv = np.empty(n, np.int64)
        inv[perm] = np.arange(n)
        for a, b in _dist_ranges(n):
            _, st = ds.score(native.FS_MULTISURF, row_begin=a, row_end=b, want_stats=True)
            assert st["n_chunks"] == 1 and st["ops_dist_tensor"] > 0
            _check_slab(ds, codes, perm, inv, a, b)


def _mixed_columns(seed, n, p):
    """Genotypes with a constant column, two {0, 2} columns and a 4-valued column: an odd number of reduced
    one-hot rows (sum over columns of values - 1)."""
    codes, y = _genotypes(seed, p, _odd_split(n))
    rs = np.random.RandomState(seed + 1)
    codes[:, 1] = 1
    codes[:, 2] = 2 * rs.randint(0, 2, n)
    codes[:, 3] = 2 * rs.randint(0, 2, n)
    codes[:, 4] = rs.randint(0, 4, n)
    return codes, y


def _reduced_rows(codes):
    return sum(np.unique(codes[:, f]).size - 1 for f in range(codes.shape[1]))


@pytest.mark.gpu
@pytest.mark.parametrize("n,p", [(257, 129), (513, 300)])
def test_distance_slab_mixed_cardinality_is_exact(native, n, p):
    codes, y = _mixed_columns(200 + n, n, p)
    assert _reduced_rows(codes) % 2 == 1
    with native.Dataset(codes, y.astype(np.int32), 2) as ds:
        ds.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F32)
        perm = ds.row_order()
        inv = np.empty(n, np.int64)
        inv[perm] = np.arange(n)
        for a, b in _dist_ranges(n):
            ds.score(native.FS_MULTISURF, row_begin=a, row_end=b)
            _check_slab(ds, codes, perm, inv, a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [257, 513])
def test_incremental_slab_equals_exact_distances_of_kept_columns(native, n):
    """TuRF's update: after scoring all 700 columns, scoring without 129 of them subtracts their distances from the
    resident slab (symmetric with mirrored tiles for [0, n), plain for a range off the 128-row grid)."""
    p = 700
    codes, y = _genotypes(300 + n, p, _odd_split(n))
    rs = np.random.RandomState(n)
    removed = np.concatenate([[0, p - 1], rs.choice(np.arange(1, p - 1), 127, replace=False)])
    kept = np.setdiff1d(np.arange(p), removed)
    with native.Dataset(codes, y.astype(np.int32), 2) as ds:
        ds.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F32)
        perm = ds.row_order()
        inv = np.empty(n, np.int64)
        inv[perm] = np.arange(n)
        for a, b in _dist_ranges(n):
            _, full = ds.score(native.FS_MULTISURF, row_begin=a, row_end=b, want_stats=True)
            _check_slab(ds, codes, perm, inv, a, b)
            _, inc = ds.score(native.FS_MULTISURF, feat_idx=kept, row_begin=a, row_end=b, want_stats=True)
            # subtracting 258 one-hot rows (2 K blocks) instead of recomputing 1142 (5 K blocks) of 1400 (6 K blocks)
            assert 0 < inc["ops_dist_tensor"] < 0.5 * full["ops_dist_tensor"], (inc["ops_dist_tensor"], full["ops_dist_tensor"])
            _check_slab(ds, codes, perm, inv, a, b, cols=kept)


# --------------------------------------------------------------------------- #
# CPU: the tolerance argument and the edges the cases reach
# --------------------------------------------------------------------------- #
def _exact_weights(codes, y, star, targets, masks):
    """The oracle's weights in rational arithmetic from its own masks: per target sum over near misses (minus far
    misses) / n_miss - sum over near hits / n_hit, a count of 0 leaving its sum undivided."""
    p = codes.shape[1]
    w = [Fraction(0)] * p
    fixed = [0] * p                      # the GPU's arithmetic: round(c * 2^52) times integer counts, in integers
    for t, i in enumerate(targets):
        m = masks[t]
        diff = (codes != codes[i]).astype(np.int64)
        hit = diff[m == R.NEAR_HIT].sum(axis=0)
        miss = diff[m == R.NEAR_MISS].sum(axis=0) - diff[m == R.FAR_MISS].sum(axis=0)
        n_hit, n_miss = int((m == R.NEAR_HIT).sum()), int((m == R.NEAR_MISS).sum())
        ch = Fraction(1, max(n_hit, 1))
        cm = Fraction(1, max(n_miss, 1))
        Ch, Cm = round(ch * 2 ** 52), round(cm * 2 ** 52)
        for f in range(p):
            w[f] += cm * int(miss[f]) - ch * int(hit[f])
            fixed[f] += Cm * int(miss[f]) - Ch * int(hit[f])
    return w, [Fraction(v, 2 ** 52) for v in fixed]


@pytest.mark.parametrize("star", [False, True])
def test_exact_tolerance_covers_oracle_and_fixed_point(star):
    """On 60 x 12 genotypes with a class of one sample (no hits): the oracle's float64 weights (blocks of 16 targets,
    block sums added exactly) and the GPU's fixed-point arithmetic both stay within exact_tolerance of the weights
    computed in rational arithmetic -- each within its own half of the bound."""
    codes, y = _genotypes(5, 12, [1, 25, 34])
    n, p = codes.shape
    targets = np.arange(n)
    want, masks, atol = oracle_multisurf(codes, y, star, targets, block=16)
    assert (masks == R.FAR_MISS).any() == star
    exact, fixed = _exact_weights(codes, y, star, targets, masks)
    term_sum = float(_term_bound(masks).sum())
    oracle_err = max(abs(Fraction(float(want[f])) - exact[f]) for f in range(p))
    fixed_err = max(abs(fixed[f] - exact[f]) for f in range(p))
    assert oracle_err <= Fraction(16 * term_sum) * Fraction(1, 2 ** 51)
    assert fixed_err <= Fraction(n * n, 2 ** 51)
    assert oracle_err + fixed_err <= Fraction(atol)
    assert max(abs(v) for v in exact) > 1                               # not a trivially small case


def _tiles(starts, a, b, bn):
    """Row counts of the tiles make_plan cuts [a, b) into: class-aligned, at most bn rows each."""
    out = []
    for c in range(starts.size - 1):
        lo, hi = max(a, starts[c]), min(b, starts[c + 1])
        out += [min(bn, hi - r) for r in range(lo, hi, bn)]
    return out


def test_cases_reach_their_edges():
    """Recompute each case's structural claim from its class sizes, p and n."""
    seen = set()
    for name, c in CASES.items():
        x, codes, y, starts, ranges = case_data(name)
        n, p = codes.shape
        sizes = np.diff(starts)
        merged, paired = _tiles(starts, 0, n, MERGED_BN), _tiles(starts, 0, n, PAIRED_BN)
        a, b = ranges[1]
        assert a % 128 != 0 and 0 < a < b <= n and any(a < s < b for s in starts), name
        if c.edge == "kblock":
            assert starts.size == 3 and starts[1] % 2 == 1 and starts[1] % KS != 0
            seen.add(("last_kblock_rows", n % KS))
            seen.add(("odd_n", n % 2))
        elif c.edge == "mblocks":
            k_rows = 2 * p
            seen.add(("m_blocks", -(-k_rows // BM), k_rows % BM))
        elif c.edge == "class_tails":
            assert sorted(sizes)[:4] == [1, 2, 31, 33]
            tails = [r for r in merged + paired if r % 16]
            assert {1, 2, 31, 33, 933 % MERGED_BN, 933 % PAIRED_BN} <= set(tails), tails
            assert starts[2] - starts[1] == 1 and ranges[2] == (starts[1], starts[1] + 1)   # the target without hits
            seen.add("class_tails")
        elif c.edge == "launch":
            launches_m = -(-len(merged) // MERGED_MAX_TILES)
            launches_p = -(-len(paired) // MAX_TILES)
            assert len(merged) > MERGED_MAX_TILES and launches_m in (2, 3)
            seen.add(("launches", launches_m, launches_p))
        elif c.edge in ("l2_off", "l2_bands"):
            groups = -(-len(merged) // 2)
            assert (n > L2_BAND_N) == (c.edge == "l2_bands")
            if c.edge == "l2_bands":
                assert groups > L2_BAND_GROUPS and groups % L2_BAND_GROUPS != 0, groups
                seen.add(("l2_groups", groups))
        elif c.edge == "encoding":
            assert np.array_equal(x.astype(np.int64) - {"i8_m101": -1, "i8_123": 1}.get(c.encoding, 0), codes)
            seen.add(("encoding", x.dtype.str, int(x.min())))
        elif c.edge == "not_v3":
            counts = {np.unique(codes[:, f]).size for f in range(p)}
            assert counts - {3}, counts
            seen.add(("not_v3", tuple(sorted(counts))))
        if c.edge != "not_v3":
            assert three_valued(codes), name
    # the table of edges: last K block of 255 / 0 / 1 samples, odd n; one-hot row blocks 1, 2 (a 2-row partial
    # block) and 3; merged 2 and 3 launches, paired 1 and 2; 19 L2 groups (one band of 12 and a remainder);
    # the lean encoder's byte inputs and the general encoder's
    assert {("last_kblock_rows", 255), ("last_kblock_rows", 0), ("last_kblock_rows", 1), ("odd_n", 1)} <= seen
    assert {("m_blocks", 1, 0), ("m_blocks", 2, 2), ("m_blocks", 3, 44)} <= seen
    assert {("launches", 2, 1), ("launches", 3, 2), ("l2_groups", 19), "class_tails"} <= seen
    assert {("encoding", "|i1", 0), ("encoding", "|u1", 0), ("encoding", "|i1", -1), ("encoding", "|i1", 1),
            ("encoding", "<f4", 0)} <= seen
    assert {("not_v3", (1, 2, 3, 4)), ("not_v3", (2, 4))} <= seen
