"""GPU: the CUDA-core scoring path (dist_general.cu, select.cu, accum_general.cu) held to an exact reference at the
tile, chunk, row-block and neighbour-list edges where its host plans branch.

The data are dyadic: continuous values k/8 in [0, 4] with 0 and 4 in every column (range 4, 1/range = 0.25 exactly),
optional "compare" columns (dyadic values flagged discrete, 33 distinct: the FP32/FP64 compare chunks) and 0/1/2
genotype columns (the one-hot path, so distances are Dc + Dd), with one sample duplicated.  On such data every
per-feature term is exact in float32 and float64, every distance is exact in any summation order, MultiSURF's sums
of d and d^2 and SURF's float32 row sum are exact (while n * p * 32 < 2^24), so distances, thresholds and neighbour
masks must equal the CPU oracle's bit for bit:

* Selection: ``fs_debug_rows`` on scattered targets -- distances, thresholds and masks of MultiSURF(*) and SURF(*).
* SURF and SURF*: coefficients +-1, so the general accumulation is exact on both instantiations (float32 tiles of at
  most 128 multiples of 1/8, the float32 image ``x - min`` at any row offset, the float64 kernel); weights bitwise.
  ``FS_ARITH_F32`` runs SURF on the kernels MultiSURF and ReliefF use, which makes it the exact probe of those.
* MultiSURF(*): float32 coefficients, so a per-feature bound derived from the kernel's arithmetic.
* ReliefF: masks bitwise against the oracle's reference tie order (``tie_mode=0``), weights within a float64 bound,
  neighbour lists longer than the 256-entry stage, more than 64 classes, small classes, k = n - 1, the tie replay
  in shared memory and in its global scratch.

The CPU tests at the end check the dyadic claims, the bounds, and that every case reaches the edge it is listed for."""
import functools

import numpy as np
import pytest

from oracle import ref_oracle as R

# host-plan constants of dist_general.cu / accum_general.cu / select.cu / score.cu the cases are built around
TILE = 64                                       # dist_general_kernel: 64 x 64 distance tiles
CHUNK_COLS = {"f32": 32, "f64": 16}             # columns per 128-byte chunk
ACC_ROWS, ACC_WANT_CHUNKS = 16, 128             # accum_general: register block of target rows; row chunks wanted
GATHER_STAGE = 256                              # ReliefF gathers: neighbour-list entries staged per round
TIE_SMEM_BYTES = 200 * 1024                     # relieff_ties_kernel: shared-memory row (pairs + class counters)
CHUNK_MB_DEFAULT = 6144                         # score.cu chunk_rows budget
DISTINCT_CAP = 16                               # more distinct values than this: a compare column
DYADIC_STEPS = 32                               # continuous values k / 8, k = 0..32
RECIP = 0.25                                    # 1 / range of every continuous column
U = 2.0 ** -53                                  # float64 unit roundoff


def rows_per_cta(R_):
    return max(ACC_ROWS, -(-(-(-R_ // ACC_WANT_CHUNKS)) // ACC_ROWS) * ACC_ROWS)


def chunk_rows(n, have_general, have_tensor, relieff, budget_mb=CHUNK_MB_DEFAULT):
    ldn = -(-n // 128) * 128
    per_row = ldn * ((8 if have_general else 0) + (4 if have_tensor else 0) + 1 + (2 if have_tensor else 0)
                     + (8 if relieff else 0))
    return max(128, budget_mb * (1 << 20) // per_row // 128 * 128)


def n_chunks(n, R_, have_general, have_tensor, relieff, budget_mb=CHUNK_MB_DEFAULT):
    rmax = min(chunk_rows(n, have_general, have_tensor, relieff, budget_mb), -(-R_ // 128) * 128)
    return -(-R_ // rmax)


def tie_storage(n, n_classes):
    return "shared" if n * 8 + 4 * n_classes <= TIE_SMEM_BYTES else "global"


# --------------------------------------------------------------------------- #
# data
# --------------------------------------------------------------------------- #
class Data:
    """Dyadic continuous | compare | genotype columns, labels 0..C-1 with the given class sizes (shuffled)."""

    def __init__(self, seed, p_cont, p_cmp, p_geno, class_sizes):
        rs = np.random.RandomState(seed)
        y = np.repeat(np.arange(len(class_sizes)), class_sizes)
        rs.shuffle(y)
        n = y.size
        cont = rs.randint(0, DYADIC_STEPS + 1, (n, p_cont)) / 8.0
        cont[0], cont[1] = 0.0, 4.0                                      # range exactly 4
        if p_cont:
            cont[2:, 0] = np.minimum(4.0, y[2:] % 3 * 1.5 + rs.randint(0, 9, n - 2) / 8.0)   # a relevant column
        cmp = rs.randint(0, DYADIC_STEPS + 1, (n, p_cmp)) / 8.0
        cmp[:DYADIC_STEPS + 1] = (np.arange(DYADIC_STEPS + 1) / 8.0)[:, None]              # all 33 values
        geno = rs.randint(0, 3, (n, p_geno)).astype(np.float64)
        geno[:3] = np.arange(3)[:, None]
        if p_geno:
            geno[3:, 0] = (y[3:] + rs.randint(0, 2, n - 3)) % 3
        x = np.hstack([cont, cmp, geno])
        x[n - 1] = x[n // 2]                                             # a duplicated sample
        self.x, self.y = x, y.astype(np.int32)
        self.n, self.p = x.shape
        self.p_cont, self.p_cmp, self.p_geno = p_cont, p_cmp, p_geno
        self.n_classes = len(class_sizes)
        self.sizes = np.bincount(y, minlength=self.n_classes)
        self.isd = np.array([False] * p_cont + [True] * (p_cmp + p_geno))
        self.recip = np.where(self.isd, 1.0, RECIP).astype(np.float32)
        self.starts = np.concatenate([[0], np.cumsum(self.sizes)])       # class starts in internal (sorted) order
        self.class_probs = (self.sizes / n).astype(np.float32)
        self.x32 = self.x.astype(np.float32)
        assert np.array_equal(self.x32, self.x)
        assert self.n * self.p * 32 < 2 ** 24, (self.n, self.p)          # float32 sums of distances stay exact

    def terms(self, i):
        """Exact per-feature terms of sample i against every sample: [n, p] float64."""
        t = np.abs(self.x - self.x[i])
        t[:, ~self.isd] *= RECIP
        t[:, self.isd] = t[:, self.isd] != 0
        return t

    def dataset(self, native, arith):
        ds = native.Dataset(self.x, self.y, self.n_classes)
        ds.set_features(self.isd, self.recip, native.FS_ARITH_F64 if arith == "f64" else native.FS_ARITH_F32)
        return ds


@functools.lru_cache(maxsize=None)
def data(seed, p_cont, p_cmp, p_geno, sizes):
    d = Data(seed, p_cont, p_cmp, p_geno, sizes)
    d.key = (seed, p_cont, p_cmp, p_geno, sizes)
    return d


def scattered(n, m, seed):
    """min(n, m) sorted targets; the duplicated pair (n // 2, n - 1) is always among them."""
    rs = np.random.RandomState(seed)
    rest = np.setdiff1d(np.arange(n), [n // 2, n - 1])
    return np.sort(np.concatenate([rs.choice(rest, min(n, m) - 2, replace=False), [n // 2, n - 1]])).astype(np.int64)


# --------------------------------------------------------------------------- #
# oracle
# --------------------------------------------------------------------------- #
@functools.lru_cache(maxsize=64)
def oracle(key, algo, star, tg_key, k=0, tie_mode=0):
    d = data(*key)
    tg = np.frombuffer(tg_key, np.int64)
    if algo == "multisurf":
        return R.multisurf_targets(d.x32, d.y.astype(np.int64), d.recip, d.isd, star, tg)
    if algo == "surf":
        return R.surf_targets(d.x, d.y, d.recip, d.isd, star, tg, sum_mode=2)
    return R.relieff_targets(d.x32, d.y, d.recip, d.isd, k, d.class_probs, tg, tie_mode=tie_mode)


def _weighted_term_sums(d, targets, W):
    """S_f = sum over targets t and samples j of |W[t, j]| * term_f(targets[t], j), float64.  Every value is a
    multiple of 1/8 in [0, 4], so sum_j |W_tj| * term_f is taken as (|W| @ one-hot of the value levels) times the
    term of each level against the target's value."""
    levels = np.arange(DYADIC_STEPS + 1) / 8.0
    codes = np.rint(d.x * 8).astype(np.int64)
    onehot = np.zeros((d.n, d.p, levels.size))
    np.put_along_axis(onehot, codes[:, :, None], 1.0, axis=2)
    onehot = onehot.reshape(d.n, -1)
    S = np.zeros(d.p)
    for b0 in range(0, len(targets), 512):
        tg = np.asarray(targets[b0:b0 + 512])
        A = (np.abs(W[b0:b0 + 512]) @ onehot).reshape(len(tg), d.p, levels.size)
        T = np.abs(levels[None, None, :] - d.x[tg][:, :, None])
        T[:, ~d.isd] *= RECIP
        T[:, d.isd] = T[:, d.isd] != 0
        S += (A * T).sum(axis=(0, 2))
    return S


def multisurf_tolerance(d, targets, masks):
    """Per-feature bound of |GPU - oracle| for MultiSURF(*): the general accumulation rounds each coefficient to
    float32 and adds a 128-sample tile of products in float32 (129 roundings of at most 2^-24 of the tile's sum of
    |c| * t), then float64 folds, partials and the oracle's float64 sums (slack); the one-hot columns' fixed-point
    coefficients err by at most n * 2^-53 per target and mask."""
    hit = masks == R.NEAR_HIT
    miss = (masks == R.NEAR_MISS) | (masks == R.FAR_MISS)
    nh = np.maximum(hit.sum(axis=1), 1)
    nm = np.maximum((masks == R.NEAR_MISS).sum(axis=1), 1)
    W = hit / nh[:, None] + miss / nm[:, None]
    S = _weighted_term_sums(d, targets, W)
    return (129 * 2.0 ** -24 + 2.0 ** -40) * S + len(targets) * d.n * 2.0 ** -52


def relieff_weights(d, k, masks, targets):
    """ReliefF neighbour weights [targets, n] from the masks (ReliefF.py:177-216): 1/h_found per hit,
    P(c) / (1 - P(c_i)) / k per miss of class c (magnitudes)."""
    denom = 1.0 - d.class_probs[d.y[targets]].astype(np.float64)
    denom[denom == 0.0] = 1.0
    hits = masks == R.NEAR_HIT
    W = hits / np.maximum(hits.sum(axis=1), 1)[:, None]
    return W + (masks == R.NEAR_MISS) * (d.class_probs[d.y].astype(np.float64)[None, :] / denom[:, None] / k)


def relieff_chain(d, k, R_, n_chunks_=1):
    """Longest chain of float64 roundings between an exact term and a weight: the gathers' per-CTA fma chains
    (rows per CTA x list length), the partial and chunk reductions, and the oracle's per-target and target sums."""
    cap = min(d.n_classes * k, d.n)
    return rows_per_cta(R_) * cap + R_ + n_chunks_ + d.n_classes + R_ + 8


def relieff_tolerance(d, k, targets, masks, n_chunks_=1):
    S = _weighted_term_sums(d, targets, relieff_weights(d, k, masks, np.asarray(targets)))
    return relieff_chain(d, k, len(targets), n_chunks_) * 2.0 * U * S


def relieff_min_change(d, k):
    """Smallest weight change of one wrong neighbour on a feature where the two candidates differ: the smallest
    neighbour weight times the smallest nonzero term (2^-5 on a continuous column)."""
    denom = 1.0 - float(d.class_probs.min())
    w_miss = float(d.class_probs.min()) / max(denom, 1e-300) / k
    w_hit = 1.0 / min(k, d.n)
    return min(w_miss, w_hit) * RECIP / 8


# --------------------------------------------------------------------------- #
# cases
# --------------------------------------------------------------------------- #
def _dist_params():
    out = []
    for n in (63, 64, 65, 129, 255):
        for arith, ps in (("f32", (1, 31, 32, 33, 100)), ("f64", (15, 16, 17))):
            for p in ps:
                for mixed in (False, True):
                    out.append(pytest.param(n, arith, p, mixed, id=f"n{n}-{arith}-p{p}-{'mixed' if mixed else 'cont'}"))
    return out


def dist_data(n, p, mixed):
    a = (n // 2) | 1
    return data(1000 + n + 7 * p, p, 17 if mixed else 0, 5 if mixed else 0, (a, n - a))


# production fs_score: (n, continuous, compare, genotype columns, class sizes)
PROD = {
    "n100": (100, 70, 17, 6, (41, 59)),
    "n300": (300, 70, 17, 6, (133, 100, 67)),
    "n2100": (2100, 40, 17, 6, (1001, 1099)),
    "n4200": (4200, 40, 17, 6, (2049, 2151)),
}


def prod_data(name, cmp):
    n, pc, pm, pg, sizes = PROD[name]
    return data(2000 + n, pc, pm if cmp else 0, pg, sizes)


def prod_ranges(d):
    """[0, n) (mirrored tiles), a range across a class boundary off the 64-row grid, one row, the last row."""
    b = int(d.starts[1])
    a = b - 37 if (b - 37) % TILE else b - 38
    return [(0, d.n), (a, min(d.n, b + 150)), (b, b + 1), (d.n - 1, d.n)]


# ReliefF: name -> (edge, seed, continuous, genotype columns, class sizes, k, production range or None)
def _classes(c, size, last):
    """c classes: c - 1 of ``size`` samples and one of ``last``."""
    return tuple([size] * (c - 1) + [last])


RELIEFF = {
    "list_c3_k100": ("list_gt_stage", 31, 24, 6, (150, 140, 130), 100, "all"),
    "list_c2_k200": ("list_gt_stage", 32, 24, 6, (260, 231), 200, "all"),
    "list_c70_k5": ("list_gt_stage", 33, 16, 6, _classes(69, 9, 12), 5, "all"),
    "classes_65": ("many_classes", 34, 16, 6, _classes(65, 8, 13), 3, "all"),
    "small_classes": ("small_classes", 35, 24, 6, (1, 4, 5, 150, 3), 4, "all"),
    "k_n_minus_1": ("k_n_minus_1", 36, 24, 6, (33, 37), 69, "all"),
    "prod_r2100": ("rows_gt_2048", 37, 24, 6, (700, 650, 750), 10, "all"),
    "global_ties_c70": ("global_ties", 38, 8, 4, _classes(70, 376, 56), 5, None),
}


def relieff_data(name):
    _, seed, pc, pg, sizes, k, _ = RELIEFF[name]
    return data(seed, pc, 0, pg, sizes), k


def relieff_targets(name):
    d, _ = relieff_data(name)
    return scattered(d.n, 18 if d.n > 10000 else 48, 7 + d.n)


CHUNK_N, CHUNK_MB = 3000, 16


def chunk_data():
    return data(4000, 24, 0, 6, (1499, 1501))


def chunk_relieff_data():
    return data(4001, 16, 0, 4, (1100, 900, 1000)), 4


# --------------------------------------------------------------------------- #
# GPU: distances, thresholds, masks
# --------------------------------------------------------------------------- #
def _check_rows(native, ds, d, algo, star, tg, arith):
    got = ds.debug_rows(native.FS_MULTISURF if algo == "multisurf" else native.FS_SURF, tg, use_star=star)
    want = oracle(d.key, algo, star, tg.tobytes())
    tag = (d.n, d.p, arith, algo, star)
    bad = np.argwhere(got["dist"] != want["dist"])
    assert bad.size == 0, (tag, "dist", bad[:4].tolist())
    assert np.array_equal(got["thresh"], want["thresh"]), (tag, "thresh")
    assert np.array_equal(got["mask"], want["mask"]), (tag, "mask", np.argwhere(got["mask"] != want["mask"])[:4].tolist())
    if algo == "surf":
        assert np.array_equal(got["wsum"], want["wsum"]), (tag, np.abs(got["wsum"] - want["wsum"]).max())
    else:
        tol = multisurf_tolerance(d, tg, want["mask"])
        assert np.all(np.abs(got["wsum"] - want["wsum"]) <= tol), (tag, np.abs(got["wsum"] - want["wsum"]).max())


@pytest.mark.gpu
@pytest.mark.parametrize("n,arith,p,mixed", _dist_params())
def test_distances_thresholds_masks_are_exact(native, n, arith, p, mixed):
    """fs_debug_rows on scattered targets (the duplicated pair included, several 64-row tiles where n allows):
    distances, thresholds and masks of MultiSURF(*) and SURF(*) bitwise, SURF weights bitwise, MultiSURF weights
    within the float32-coefficient bound."""
    d = dist_data(n, p, mixed)
    tg = scattered(n, 100, n + p)
    with d.dataset(native, arith) as ds:
        for algo in ("multisurf", "surf"):
            for star in (False, True):
                _check_rows(native, ds, d, algo, star, tg, arith)


# --------------------------------------------------------------------------- #
# GPU: production fs_score
# --------------------------------------------------------------------------- #
def _prod_params():
    return [pytest.param(name, arith, cmp, id=f"{name}-{arith}-{'cmp' if cmp else 'nocmp'}")
            for name in PROD for arith in ("f32", "f64") for cmp in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,arith,cmp", _prod_params())
def test_production_surf_bitwise_and_multisurf_bounded(native, name, arith, cmp):
    """fs_score over [0, n) (mirrored tiles; for n > 2048 32- and 48-row CTAs with a partial block), a range across
    a class boundary off the 64-row grid, one row and the last row.  SURF(*) bitwise (F64 without compare columns:
    the float32 image at row offsets; with them the float64 kernel; F32: the float32 kernel and compare chunks),
    MultiSURF(*) within the float32-coefficient bound."""
    d = prod_data(name, cmp)
    key = d.key
    with d.dataset(native, arith) as ds:
        perm = ds.row_order()
        assert np.array_equal(d.y[perm], np.repeat(np.arange(d.n_classes), d.sizes))
        for a, b in prod_ranges(d):
            tg = perm[a:b].astype(np.int64)
            for star in (False, True):
                got, st = ds.score(native.FS_SURF, use_star=star, row_begin=a, row_end=b, want_stats=True)
                assert st["n_general_cols"] == d.p_cont + d.p_cmp and st["n_chunks"] == 1, st
                want = oracle(key, "surf", star, tg.tobytes())
                assert np.array_equal(got, want["wsum"]), (name, arith, cmp, "surf", star, (a, b),
                                                           np.abs(got - want["wsum"]).max())
                got = ds.score(native.FS_MULTISURF, use_star=star, row_begin=a, row_end=b)
                want = oracle(key, "multisurf", star, tg.tobytes())
                tol = multisurf_tolerance(d, tg, want["mask"])
                err = np.abs(got - want["wsum"])
                assert np.all(err <= tol), (name, arith, cmp, "multisurf", star, (a, b), err.max(), tol[err.argmax()])


@pytest.mark.gpu
def test_chunked_surf_bitwise_and_relieff_bounded(native, monkeypatch):
    """FS_B200_CHUNK_MB=16 at n = 3000: the target rows run in several chunks, the later ones at row0 != 0 of the
    float32 image (SURF, F64) and of the float32 matrix (SURF, F32; ReliefF)."""
    monkeypatch.setenv("FS_B200_CHUNK_MB", str(CHUNK_MB))
    d = chunk_data()
    key = d.key
    assert d.n == CHUNK_N
    for arith in ("f64", "f32"):
        with d.dataset(native, arith) as ds:
            perm = ds.row_order()
            for a, b in ((0, d.n), (77, d.n - 5)):
                tg = perm[a:b].astype(np.int64)
                got, st = ds.score(native.FS_SURF, use_star=True, row_begin=a, row_end=b, want_stats=True)
                assert st["n_chunks"] == n_chunks(d.n, b - a, True, True, False, CHUNK_MB) > 1, st
                want = oracle(key, "surf", True, tg.tobytes())
                assert np.array_equal(got, want["wsum"]), (arith, (a, b), np.abs(got - want["wsum"]).max())
    d, k = chunk_relieff_data()
    rkey = d.key
    with d.dataset(native, "f32") as ds:
        perm = ds.row_order()
        tg = perm.astype(np.int64)
        got, st = ds.score(native.FS_RELIEFF, k=k, class_probs=d.class_probs, want_stats=True)
        nc = n_chunks(d.n, d.n, True, True, True, CHUNK_MB)
        assert st["n_chunks"] == nc > 1, st
        want = oracle(rkey, "relieff", False, tg.tobytes(), k, 0)
        tol = relieff_tolerance(d, k, tg, want["mask"], nc)
        err = np.abs(got - want["wsum"])
        assert np.all(err <= tol), (err.max(), tol[err.argmax()])


# --------------------------------------------------------------------------- #
# GPU: ReliefF
# --------------------------------------------------------------------------- #
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RELIEFF))
def test_relieff_masks_bitwise_weights_bounded(native, monkeypatch, name):
    """fs_debug_rows on scattered targets: masks bitwise against the reference tie order, weights within the
    float64 bound; then production fs_score over [0, n) within the bound."""
    monkeypatch.delenv("FS_B200_RELIEFF_TIES", raising=False)
    d, k = relieff_data(name)
    key = d.key
    tg = relieff_targets(name)
    with d.dataset(native, "f32") as ds:
        got = ds.debug_rows(native.FS_RELIEFF, tg, k=k, class_probs=d.class_probs)
        want = oracle(key, "relieff", False, tg.tobytes(), k, 0)
        assert np.array_equal(got["dist"], want["dist"]), name
        bad = np.nonzero((got["mask"] != want["mask"]).any(axis=1))[0]
        assert bad.size == 0, (name, "targets with other neighbours", tg[bad][:8].tolist())
        tol = relieff_tolerance(d, k, tg, want["mask"])
        err = np.abs(got["wsum"] - want["wsum"])
        assert np.all(err <= tol), (name, err.max(), tol[err.argmax()])
        if RELIEFF[name][6] == "all":
            perm = ds.row_order()
            got, st = ds.score(native.FS_RELIEFF, k=k, class_probs=d.class_probs, want_stats=True)
            assert st["n_chunks"] == 1
            want = oracle(key, "relieff", False, perm.astype(np.int64).tobytes(), k, 0)
            tol = relieff_tolerance(d, k, perm, want["mask"])
            err = np.abs(got - want["wsum"])
            assert np.all(err <= tol), (name, "fs_score", err.max(), tol[err.argmax()])


@pytest.mark.gpu
def test_relieff_index_ties_above_64_classes(native, monkeypatch):
    """FS_B200_RELIEFF_TIES=index on 70 classes: sample-index tie order, the oracle's tie_mode=1."""
    monkeypatch.setenv("FS_B200_RELIEFF_TIES", "index")
    d, k = relieff_data("list_c70_k5")
    key = d.key
    tg = relieff_targets("list_c70_k5")
    with d.dataset(native, "f32") as ds:
        got = ds.debug_rows(native.FS_RELIEFF, tg, k=k, class_probs=d.class_probs)
    want = oracle(key, "relieff", False, tg.tobytes(), k, 1)
    assert np.array_equal(got["mask"], want["mask"])
    tol = relieff_tolerance(d, k, tg, want["mask"])
    assert np.all(np.abs(got["wsum"] - want["wsum"]) <= tol)


# --------------------------------------------------------------------------- #
# CPU: the dyadic claims, the bounds, and the edges the cases reach
# --------------------------------------------------------------------------- #
def test_oracle_distances_are_exact_sums():
    """On dyadic data the oracle's distances (float64, float32 for SURF / ReliefF) equal the exact float64 sums
    of the terms, whatever their order; the duplicated sample is at distance exactly 0."""
    d = data(5, 33, 17, 5, (31, 40))
    tg = np.arange(d.n, dtype=np.int64)
    exact = np.array([d.terms(i).sum(axis=1) for i in tg])
    exact[tg, tg] = 0.0
    for algo in ("multisurf", "surf", "relieff"):
        want = oracle(d.key, algo, False, tg.tobytes(), 3, 0)
        assert np.array_equal(want["dist"], exact), algo
    assert exact[d.n // 2, d.n - 1] == 0.0
    assert np.array_equal(exact.astype(np.float32), exact)
    assert np.array_equal(exact[:, ::-1].sum(axis=1), exact.sum(axis=1))


@pytest.mark.parametrize("star", [False, True])
def test_surf_oracle_weights_equal_exact_sums_of_masks(star):
    """SURF(*) weights of the oracle equal the sums, taken exactly, of +-terms over its own masks."""
    d = data(6, 31, 17, 5, (40, 57))
    tg = np.arange(d.n, dtype=np.int64)
    want = oracle(d.key, "surf", star, tg.tobytes())
    sign = {R.NEAR_HIT: -1.0, R.NEAR_MISS: 1.0, R.FAR_MISS: -1.0, R.FAR_HIT: 1.0}
    w = np.zeros(d.p)
    for t, i in enumerate(tg):
        c = np.zeros(d.n)
        for code, s in sign.items():
            c[want["mask"][t] == code] = s
        w += c @ d.terms(i)
    assert (want["mask"] == R.FAR_HIT).any() == star
    assert np.array_equal(want["wsum"], w)
    assert np.array_equal(w * 32, np.round(w * 32))                   # multiples of 2^-5: exact in float64


def _all_data():
    out = [dist_data(n, p, mixed) for n in (63, 64, 65, 129, 255) for p in (1, 15, 16, 17, 31, 32, 33, 100)
           for mixed in (False, True)]
    out += [prod_data(name, cmp) for name in PROD for cmp in (False, True)]
    out += [chunk_data(), chunk_relieff_data()[0]] + [relieff_data(name)[0] for name in RELIEFF]
    return out


def test_every_case_meets_the_exactness_bound():
    """n * p * 32 < 2^24 (the float32 row sums and tile sums of multiples of 1/8 are exact), every continuous
    column spans [0, 4] in steps of 1/8, compare columns have more than 16 distinct values, genotype columns 3."""
    for d in _all_data():
        assert d.n * d.p * 32 < 2 ** 24
        cont = d.x[:, :d.p_cont]
        assert np.all(cont.min(axis=0) == 0) and np.all(cont.max(axis=0) == 4)
        assert np.array_equal(cont * 8, np.round(cont * 8))
        for f in range(d.p_cont, d.p_cont + d.p_cmp):
            assert np.unique(d.x[:, f]).size == DYADIC_STEPS + 1 > DISTINCT_CAP
        for f in range(d.p_cont + d.p_cmp, d.p):
            assert np.unique(d.x[:, f]).size == 3
        assert np.array_equal(d.x[d.n - 1], d.x[d.n // 2])
        # a 128-sample float32 tile of +-|a - b| (<= 4, multiples of 1/8) stays below 2^24 / 8
        assert 128 * 4 * 8 < 2 ** 24


def test_cases_reach_their_edges():
    """Recompute each case's structural claim from the mirrored host-plan constants."""
    seen = set()
    for n in (63, 64, 65, 129, 255):
        seen.add(("tiles", -(-n // TILE), n % TILE))
        tg = scattered(n, 100, n)
        seen.add(("target_tiles", -(-tg.size // TILE)))
    for arith, ps in (("f32", (1, 31, 32, 33, 100)), ("f64", (15, 16, 17))):
        for p in ps:
            fc = CHUNK_COLS[arith]
            seen.add((arith, -(-p // fc), p % fc))
    for arith in ("f32", "f64"):
        seen.add(("cmp_chunks", arith, -(-17 // CHUNK_COLS[arith]), 17 % CHUNK_COLS[arith]))
    assert {("tiles", 1, 63), ("tiles", 1, 0), ("tiles", 2, 1), ("tiles", 3, 1), ("tiles", 4, 63)} <= seen
    assert {("target_tiles", 1), ("target_tiles", 2)} <= seen
    assert {("f32", 1, 1), ("f32", 1, 31), ("f32", 1, 0), ("f32", 2, 1), ("f32", 4, 4)} <= seen
    assert {("f64", 1, 15), ("f64", 1, 0), ("f64", 2, 1), ("cmp_chunks", "f32", 1, 17), ("cmp_chunks", "f64", 2, 1)} <= seen

    # production: n < 128, n % 128 != 0, R > 2048 with 32- and 48-row CTAs ending in a partial 16-row block
    rows = {}
    for name in PROD:
        d = prod_data(name, True)
        (a0, b0), (a, b), one, last = prod_ranges(d)
        assert (a0, b0) == (0, d.n) and a % TILE and any(a < s < b for s in d.starts) and one[1] - one[0] == 1
        assert last == (d.n - 1, d.n)
        rows[d.n] = (rows_per_cta(d.n), d.n % rows_per_cta(d.n) % ACC_ROWS)
        assert n_chunks(d.n, d.n, True, True, False) == 1
    assert min(rows) < 128 and any(n % 128 for n in rows)
    assert rows[2100] == (32, 4) and rows[4200] == (48, 8)

    # chunks: 12 SURF chunks of 256 rows and 24 ReliefF chunks of 128 rows at FS_B200_CHUNK_MB=16
    assert chunk_data().n == CHUNK_N
    assert n_chunks(CHUNK_N, CHUNK_N, True, True, False, CHUNK_MB) == 12
    assert n_chunks(CHUNK_N, CHUNK_N - 82, True, True, False, CHUNK_MB) == 12
    assert n_chunks(CHUNK_N, CHUNK_N, True, True, True, CHUNK_MB) == 24

    # ReliefF
    for name, (edge, _, _, _, sizes, k, _) in RELIEFF.items():
        d, _ = relieff_data(name)
        cap = min(d.n_classes * k, d.n)
        if edge == "list_gt_stage":
            seen.add(("stage_rounds", -(-cap // GATHER_STAGE)))
            assert cap > GATHER_STAGE
        elif edge == "many_classes":
            assert d.n_classes == 65
        elif edge == "small_classes":
            assert {1, k, k + 1} <= set(sizes)
            seen.add("small_classes")
        elif edge == "k_n_minus_1":
            assert k == d.n - 1 and cap == d.n
        elif edge == "rows_gt_2048":
            assert d.n > 2048 and rows_per_cta(d.n) > ACC_ROWS and d.n % rows_per_cta(d.n) % ACC_ROWS
        elif edge == "global_ties":
            assert d.n_classes == 70 and relieff_targets(name).size == 18
        seen.add(("ties", tie_storage(d.n, d.n_classes), d.n_classes > 64))
    assert {("stage_rounds", 2)} <= seen
    assert {("ties", "shared", True), ("ties", "global", True), ("ties", "shared", False)} <= seen
    assert tie_storage(25599, 2) == "shared" and tie_storage(25600, 2) == "global"


@functools.lru_cache(maxsize=None)
def _relieff_case_tolerance(name):
    d, k = relieff_data(name)
    key = d.key
    tg = relieff_targets(name)
    want = oracle(key, "relieff", False, tg.tobytes(), k, 0)
    return d, k, relieff_tolerance(d, k, tg, want["mask"])


@pytest.mark.parametrize("name", list(RELIEFF))
def test_relieff_tolerance_is_discriminating(name):
    """The float64 bound is below half the smallest change one wrong neighbour can make (and of order
    2^-45 times the weighted term sums), on the debug targets and over all n targets."""
    d, k, tol = _relieff_case_tolerance(name)
    assert tol.max() < 0.5 * relieff_min_change(d, k), (tol.max(), relieff_min_change(d, k))
    if RELIEFF[name][6] == "all" and d.n <= 700:
        tg = np.arange(d.n, dtype=np.int64)
        want = oracle(d.key, "relieff", False, tg.tobytes(), k, 0)
        tol = relieff_tolerance(d, k, tg, want["mask"])
        assert tol.max() < 0.5 * relieff_min_change(d, k), (tol.max(), relieff_min_change(d, k))


def test_multisurf_tolerance_is_discriminating_on_single_rows():
    """For one target the float32-coefficient bound is below half the smallest change one wrong neighbour makes
    (1 / max(n_hit, n_miss) times a term of 2^-5)."""
    for name in ("n100", "n300"):
        d = prod_data(name, True)
        key = d.key
        for i in (0, d.n // 3, d.n - 1):
            for star in (False, True):
                tg = np.array([i], np.int64)
                want = oracle(key, "multisurf", star, tg.tobytes())
                nh, nm, _ = want["counts"][0]
                tol = multisurf_tolerance(d, tg, want["mask"])
                assert tol.max() < 0.5 * RECIP / 8 / max(nh, nm, 1), (name, i, tol.max(), nh, nm)


def test_70_classes_separate_the_tie_orders():
    """On the 70-class case the reference tie order and the sample-index order pick different neighbours, and the
    weights differ by far more than the tolerance: a replay that fell back to index order would fail."""
    d, k, tol = _relieff_case_tolerance("list_c70_k5")
    tg = relieff_targets("list_c70_k5")
    ref = oracle(d.key, "relieff", False, tg.tobytes(), k, 0)
    idx = oracle(d.key, "relieff", False, tg.tobytes(), k, 1)
    differ = (ref["mask"] != idx["mask"]).any(axis=1)
    assert differ.mean() > 0.5, differ.mean()
    assert np.abs(ref["wsum"] - idx["wsum"]).max() > 1e3 * tol.max()
