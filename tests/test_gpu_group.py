"""GPU: the multi-GPU group (include/fastselect_b200.h, "Multi-GPU group") with the ranks EMULATED on one
GPU -- one fs_comm + fs_dataset per rank, arenas mapped by raw pointer, one host thread and one CUDA
stream per rank, the library's own device-side barriers between them.  Checks that a collective
fs_score returns on every rank the value a single data set returns for all rows: bitwise for one-hot
(genotype) columns, whose accumulation is sharded by columns and tiled exactly like a single-GPU pass;
to float64 rounding where continuous columns add partial sums over the ranks' rows.  Also the
single-process multi-GPU entry (fs_multi_*), which on a one-GPU box runs with one rank."""
import threading

import numpy as np
import pytest

from datasets import epistatic_genotypes, mixed
from oracle import ref_oracle as R

pytestmark = pytest.mark.gpu


def balanced_starts(n, world, align=4):
    base, extra = divmod(n, world)
    return [(r * base + min(r, extra)) // align * align for r in range(world)] + [n]


class EmulatedGroup:
    """`world` ranks of one group on device 0 of this process."""

    def __init__(self, native, x, y_enc, n_classes, world, with_x, monkeypatch):
        import torch

        monkeypatch.setenv("FS_B200_BARRIER_TIMEOUT_S", "10")
        self.native, self.world = native, world
        n, p = x.shape
        self.starts = balanced_starts(n, world)
        self.streams = [torch.cuda.Stream(device=0) for _ in range(world)]
        self.comms = [native.Comm(r, world, 0) for r in range(world)]
        need = native.Comm.required_bytes(n, p, x.dtype, world, with_x=with_x)
        for c in self.comms:
            c.reserve(need)
        ptrs = [c.arena for c in self.comms]
        for c in self.comms:
            c.connect(raw_ptrs=ptrs)
        self.sets = [None] * world
        if with_x:      # sharded upload: collective, one thread per rank
            self.run(lambda r: self._create(r, x, y_enc, n_classes))
        else:
            for r in range(world):
                self.sets[r] = native.Dataset(x, y_enc, n_classes, device=0, stream=self.streams[r].cuda_stream)

    def _create(self, r, x, y_enc, n_classes):
        self.sets[r] = self.native.Dataset(x, y_enc, n_classes, stream=self.streams[r].cuda_stream, comm=self.comms[r])

    def run(self, fn):
        out, err = [None] * self.world, [None] * self.world

        def work(r):
            try:
                out[r] = fn(r)
            except BaseException as e:      # noqa: BLE001 -- re-raised on the main thread
                err[r] = e

        th = [threading.Thread(target=work, args=(r,)) for r in range(self.world)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        for e in err:
            if e is not None:
                raise e
        return out

    def set_features(self, isd, recip, arith):
        for r, ds in enumerate(self.sets):
            ds.set_features(isd, recip, arith)
            ds.attach_comm(self.comms[r], self.starts)

    def score(self, algo, **kw):
        return self.run(lambda r: self.sets[r].score(algo, row_begin=self.starts[r], row_end=self.starts[r + 1], **kw))

    def close(self):
        for ds in self.sets:
            if ds is not None:
                ds.close()
        for c in self.comms:
            c.close()


def _mixed_cardinality_genotypes(seed, n, p):
    x, y = epistatic_genotypes(seed, n, p)
    rs = np.random.RandomState(seed + 1)
    x[:, 5::17] = rs.randint(0, 2, x[:, 5::17].shape)
    x[:, 9::23] = rs.randint(0, 4, x[:, 9::23].shape)
    x[:, 11::29] = 1
    return x, y


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("lean", [True, False], ids=["genotype012", "mixed_cardinality"])
@pytest.mark.parametrize("with_x", [False, True], ids=["full_upload", "sharded_upload"])
def test_group_scores_equal_single_rank_bitwise_on_onehot_columns(native, monkeypatch, world, lean, with_x):
    n, p = 900, 700
    x, y = epistatic_genotypes(39, n, p) if lean else _mixed_cardinality_genotypes(39, n, p)
    isd, recip = np.ones(p, bool), np.ones(p, np.float32)
    y32 = y.astype(np.int32)
    rs = np.random.RandomState(5)
    a1 = np.sort(rs.choice(p, int(p * 0.9), replace=False))
    a2 = np.sort(rs.choice(a1, int(a1.size * 0.9), replace=False))
    calls = [dict(algo=native.FS_MULTISURF), dict(algo=native.FS_MULTISURF, use_star=True),
             dict(algo=native.FS_MULTISURF, feat_idx=a1), dict(algo=native.FS_MULTISURF, feat_idx=a2),     # TuRF: incremental slab
             dict(algo=native.FS_SURF, use_star=True, feat_idx=a2), dict(algo=native.FS_SURF)]
    with native.Dataset(x, y32, 2) as plain:
        plain.set_features(isd, recip, native.FS_ARITH_F32)
        want = [plain.score(**c) for c in calls]
    g = EmulatedGroup(native, x, y32, 2, world, with_x, monkeypatch)
    try:
        g.set_features(isd, recip, native.FS_ARITH_F32)
        for c, w in zip(calls, want):
            c = dict(c)
            got = g.score(c.pop("algo"), **c)
            for r in range(world):
                assert np.array_equal(got[r], w), (r, c)
        # sharding the accumulation by columns can be switched off: partial sums over the ranks' rows, same value
        monkeypatch.setenv("FS_B200_FEATURE_SHARD", "0")
        got = g.score(native.FS_MULTISURF, use_star=True)
        for r in range(world):
            np.testing.assert_allclose(got[r], want[1], rtol=1e-12, atol=1e-9)
            assert np.array_equal(got[r], got[0])
    finally:
        g.close()


@pytest.mark.parametrize("world", [2, 4])
def test_group_scores_on_mixed_columns_and_relieff(native, monkeypatch, world):
    """Continuous columns and ReliefF accumulate partial sums over the rank's rows; the ranks' vectors are
    added in rank order: identical on every rank, equal to the single-rank value to float64 rounding."""
    x, y = mixed(41, 640, 90, 3)
    x32, recip, isd = R.multisurf_prep(x, 10)
    yc = np.unique(y, return_inverse=True)[1].astype(np.int32)
    cp = (np.bincount(yc) / yc.size).astype(np.float32)
    calls = [dict(algo=native.FS_MULTISURF, use_star=True), dict(algo=native.FS_SURF),
             dict(algo=native.FS_RELIEFF, k=5, class_probs=cp)]
    with native.Dataset(x32, yc, 3) as plain:
        plain.set_features(isd, recip, native.FS_ARITH_F32)
        want = [plain.score(**c) for c in calls]
    g = EmulatedGroup(native, x32, yc, 3, world, True, monkeypatch)
    try:
        g.set_features(isd, recip, native.FS_ARITH_F32)
        for c, w in zip(calls, want):
            c = dict(c)
            got = g.score(c.pop("algo"), **c)
            for r in range(world):
                np.testing.assert_allclose(got[r], w, rtol=1e-11, atol=1e-11)
                assert np.array_equal(got[r], got[0])
    finally:
        g.close()


def test_group_barrier_times_out_instead_of_hanging(native, monkeypatch):
    """A rank that never joins the collective call: the others fail with TimeoutError after
    FS_B200_BARRIER_TIMEOUT_S instead of spinning forever."""
    monkeypatch.setenv("FS_B200_BARRIER_TIMEOUT_S", "1.5")
    x, y = epistatic_genotypes(40, 600, 300)
    g = EmulatedGroup(native, x, y.astype(np.int32), 2, 2, False, monkeypatch)
    monkeypatch.setenv("FS_B200_BARRIER_TIMEOUT_S", "1.5")
    try:
        g.comms[0].close(); g.comms[1].close()
        g.comms = [native.Comm(r, 2, 0) for r in range(2)]          # re-created with the short timeout
        need = native.Comm.required_bytes(600, 300, x.dtype, 2, with_x=False)
        for c in g.comms:
            c.reserve(need)
        for c in g.comms:
            c.connect(raw_ptrs=[q.arena for q in g.comms])
        g.set_features(np.ones(300, bool), np.ones(300, np.float32), native.FS_ARITH_F32)
        with pytest.raises(TimeoutError):
            g.sets[0].score(native.FS_MULTISURF, row_begin=g.starts[0], row_end=g.starts[1])      # rank 1 never calls
    finally:
        g.close()


def test_single_process_multi_gpu_entry(native, monkeypatch):
    """fs_multi_* through the estimator (FASTSELECT_B200_GPUS): all visible GPUs, one process.  On a
    one-GPU box this runs a single rank; on a multi-GPU box the result must equal the one-GPU fit."""
    import fastselect_b200 as fsb

    x, y = epistatic_genotypes(43, 1200, 900)
    one = fsb.MultiSURF(n_features_to_select=5, backend="gpu").fit(x, y)
    n_dev = native.device_count()
    with native.MultiDataset(x, y.astype(np.int32), 2, list(range(n_dev))) as md:
        assert md.world == n_dev
        md.set_features(np.ones(900, bool), np.full(900, 0.5, np.float32), native.FS_ARITH_F32)
        w = md.score(native.FS_MULTISURF)
    assert np.array_equal((w / 1200).astype(np.float32), one.feature_importances_)
    if n_dev > 1:
        monkeypatch.setenv("FASTSELECT_B200_GPUS", str(n_dev))
        many = fsb.MultiSURF(n_features_to_select=5, backend="gpu").fit(x, y)
        assert np.array_equal(many.feature_importances_, one.feature_importances_)
        assert np.array_equal(many.top_features_, one.top_features_)
        t1 = fsb.TuRF(fsb.MultiSURF(backend="gpu", n_features_to_select=5), n_features_to_select=20, pct_remove=0.2).fit(x, y)
        monkeypatch.delenv("FASTSELECT_B200_GPUS")
        t0 = fsb.TuRF(fsb.MultiSURF(backend="gpu", n_features_to_select=5), n_features_to_select=20, pct_remove=0.2).fit(x, y)
        assert np.array_equal(t0.top_features_, t1.top_features_)


# ---- a call's distance plan across buffers: the slab of a collective call lives in the rank's arena, that of any
# other call in the data set's own buffer.  A slab cached in one of them must never seed an incremental update or
# a reuse in the other.

def _turf_columns(p):
    rs = np.random.RandomState(5)
    a1 = np.sort(rs.choice(p, int(p * 0.9), replace=False))
    a2 = np.sort(rs.choice(a1, int(a1.size * 0.9), replace=False))
    a3 = np.sort(rs.choice(a2, int(a2.size * 0.9), replace=False))
    return a1, a2, a3


def _fresh(native, x, y32, **call):
    """Score and slab of one call on a data set that has never scored before."""
    with native.Dataset(x, y32, 2) as ds:
        ds.set_features(np.ones(x.shape[1], bool), np.ones(x.shape[1], np.float32), native.FS_ARITH_F32)
        w = ds.score(native.FS_MULTISURF, **call)
        lo = call.get("row_begin", 0)
        hi = call.get("row_end", x.shape[0])
        return w, ds.debug_slab(lo, hi - lo)


def test_group_then_alone_recomputes_the_slab(native, monkeypatch):
    n, p = 900, 700
    x, y = epistatic_genotypes(47, n, p)
    y32 = y.astype(np.int32)
    a1, a2, a3 = _turf_columns(p)
    g = EmulatedGroup(native, x, y32, 2, 2, False, monkeypatch)
    try:
        g.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F32)
        for cols in (None, a1):                   # a1: incremental update of the arena slab
            want, _ = _fresh(native, x, y32, feat_idx=cols)
            for got in g.score(native.FS_MULTISURF, feat_idx=cols):
                assert np.array_equal(got, want)
        ds = g.sets[0]
        ds.attach_comm(None, None)
        # alone, on the rows and a subset of the columns the arena slab was cached for, then on all rows
        for call in (dict(feat_idx=a2, row_begin=g.starts[0], row_end=g.starts[1]), dict(feat_idx=a3)):
            want, (want_slab, want_info) = _fresh(native, x, y32, **call)
            assert np.array_equal(ds.score(native.FS_MULTISURF, **call), want)
            lo, hi = call.get("row_begin", 0), call.get("row_end", n)
            got_slab, got_info = ds.debug_slab(lo, hi - lo)
            assert got_info == want_info and np.array_equal(got_slab, want_slab)
    finally:
        g.close()


def test_alone_then_group_recomputes_the_slab(native, monkeypatch):
    n, p = 900, 700
    x, y = epistatic_genotypes(48, n, p)
    y32 = y.astype(np.int32)
    isd, recip = np.ones(p, bool), np.ones(p, np.float32)
    a1, a2, _ = _turf_columns(p)
    fresh = EmulatedGroup(native, x, y32, 2, 2, False, monkeypatch)
    try:
        fresh.set_features(isd, recip, native.FS_ARITH_F32)
        want = fresh.score(native.FS_MULTISURF, feat_idx=a2)
    finally:
        fresh.close()
    g = EmulatedGroup(native, x, y32, 2, 2, False, monkeypatch)
    try:
        # each rank alone caches the slab of all columns over its shard in its own buffer
        for r, ds in enumerate(g.sets):
            ds.set_features(isd, recip, native.FS_ARITH_F32)
            w, _ = _fresh(native, x, y32, row_begin=g.starts[r], row_end=g.starts[r + 1])
            assert np.array_equal(ds.score(native.FS_MULTISURF, row_begin=g.starts[r], row_end=g.starts[r + 1]), w)
            ds.attach_comm(g.comms[r], g.starts)
        got = g.score(native.FS_MULTISURF, feat_idx=a1)
        assert np.array_equal(got[0], got[1])
        got = g.score(native.FS_MULTISURF, feat_idx=a2)
        for r in range(2):
            assert np.array_equal(got[r], want[r])
    finally:
        g.close()


def test_score_after_joint_columns_rebuilds_the_working_set(native):
    n, p = 900, 700
    x, y = epistatic_genotypes(49, n, p)
    y32 = y.astype(np.int32)
    a1, _, _ = _turf_columns(p)
    want, (want_slab, want_info) = _fresh(native, x, y32, feat_idx=a1)
    with native.Dataset(x, y32, 2) as ds:
        ds.set_features(np.ones(p, bool), np.ones(p, np.float32), native.FS_ARITH_F32)
        ds.score(native.FS_MULTISURF)
        # the joint path builds the working set of a1 without distance operands
        ds.joint_columns(native.FS_JOINT_MI, 2.0, [0, 3], feat_idx=a1)
        assert np.array_equal(ds.score(native.FS_MULTISURF, feat_idx=a1), want)
        got_slab, got_info = ds.debug_slab(0, n)
        assert got_info == want_info and np.array_equal(got_slab, want_slab)


# (launches, n_chunks) of every call of a TuRF-like sequence: all columns, then two shrinking subsets.  A
# working set or operand built twice, or a slab recomputed where it could be updated, changes the counts.
TURF_LAUNCHES_ALONE = [(8, 1), (9, 1), (9, 1)]
TURF_LAUNCHES_GROUP = [[(18, 1)] * 2, [(17, 1)] * 2, [(17, 1)] * 2]     # per rank


def test_turf_sequence_launch_counts(native, monkeypatch):
    n, p = 900, 700
    x, y = epistatic_genotypes(50, n, p)
    y32 = y.astype(np.int32)
    isd, recip = np.ones(p, bool), np.ones(p, np.float32)
    a1, a2, _ = _turf_columns(p)
    seq = (None, a1, a2)
    with native.Dataset(x, y32, 2) as ds:
        ds.set_features(isd, recip, native.FS_ARITH_F32)
        alone = [ds.score(native.FS_MULTISURF, feat_idx=c, want_stats=True)[1] for c in seq]
    g = EmulatedGroup(native, x, y32, 2, 2, False, monkeypatch)
    try:
        g.set_features(isd, recip, native.FS_ARITH_F32)
        group = [[s for _, s in g.score(native.FS_MULTISURF, feat_idx=c, want_stats=True)] for c in seq]
    finally:
        g.close()
    got_alone = [(s["launches"], s["n_chunks"]) for s in alone]
    got_group = [[(s["launches"], s["n_chunks"]) for s in ranks] for ranks in group]
    assert (got_alone, got_group) == (TURF_LAUNCHES_ALONE, TURF_LAUNCHES_GROUP), repr((got_alone, got_group))
