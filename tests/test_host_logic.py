"""CPU: host-side logic of the package -- parameter validation and error behaviour of the
estimator mirror, TuRF's pruning schedule (ports of the behaviours in the reference's
tests/test_turf.py, tests/test_multisurf.py:121-178), the C ABI surface, and the
multi-process row sharding (gloo, world_size 2)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
from sklearn.base import BaseEstimator
from sklearn.exceptions import NotFittedError

import fastselect_b200 as fsb
from fastselect_b200 import _native
from fastselect_b200._shard import shard_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HAVE_GPU = _native.device_count() > 0

X = np.random.RandomState(0).rand(12, 5)
Y = np.arange(12) % 2


@pytest.mark.parametrize("cls", [fsb.MultiSURF, fsb.SURF, fsb.ReliefF])
def test_parameter_validation_messages(cls):
    for bad in (-1, 0, 100):
        with pytest.raises(ValueError, match="must be > 0 and <= n_features"):
            cls(n_features_to_select=bad, backend="gpu").fit(X, Y)
    with pytest.raises(ValueError, match="must be in"):
        cls(n_features_to_select=1.1, backend="gpu").fit(X, Y)
    with pytest.raises(TypeError, match="must be an int or a float"):
        cls(n_features_to_select="hi", backend="gpu").fit(X, Y)
    with pytest.raises(ValueError, match="backend must be one of"):
        cls(backend="tpu").fit(X, Y)
    with pytest.raises(ValueError, match="contains NaN"):
        xn = X.copy()
        xn[0, 0] = np.nan
        cls(backend="gpu").fit(xn, Y)
    with pytest.raises(NotFittedError):
        cls().transform(X)
    with pytest.raises(NotImplementedError, match="only the GPU backend"):
        cls(n_features_to_select=2, backend="cpu").fit(X, Y)


def test_relieff_n_neighbors_validation():
    for k in (0, 12, 50):
        with pytest.raises(ValueError, match="n_neighbors"):
            fsb.ReliefF(n_neighbors=k, backend="gpu").fit(X, Y)


@pytest.mark.skipif(HAVE_GPU, reason="needs a box WITHOUT a GPU")
def test_gpu_backend_fails_loudly_without_a_gpu():
    """No silent CPU fallback: MultiSURF.py:399-403 / SURF.py:341-342 messages."""
    with pytest.raises(RuntimeError, match="no compatible NVIDIA GPU"):
        fsb.MultiSURF(backend="gpu").fit(X, Y)
    with pytest.raises(RuntimeError, match="no CUDA-enabled GPU is available"):
        fsb.SURF(backend="gpu").fit(X, Y)
    with pytest.raises(RuntimeError):
        fsb.ReliefF(backend="auto").fit(X, Y)
    with pytest.raises(RuntimeError):
        fsb.MultiSURF(backend="auto").fit(X, Y)          # 'auto' does not fall back either
    with pytest.raises(RuntimeError, match="no usable NVIDIA sm_100"):
        _native.Dataset(X, Y.astype(np.int32), 2)


def test_relieff_single_class_early_return_needs_no_gpu():
    r = fsb.ReliefF(n_features_to_select=2).fit(X, np.zeros(12))
    assert not r.feature_importances_.any() and r.top_features_.tolist() == [0, 1]


def test_c_abi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "fastselect_b200.h")).read()
    declared = set(re.findall(r"FS_API\s+[\w\s\*]+?\b(fs_\w+)\s*\(", header))
    assert {"fs_score", "fs_dataset_create", "fs_debug_rows", "fs_device_count"} <= declared
    lib = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.fs_abi_version() == _native.FS_ABI_VERSION
    out = subprocess.run(["nm", "-D", "--defined-only", _native.LIB_PATH], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert declared <= exported
    assert not [s for s in exported if "fso_" in s], "the oracle must not be linked into the product"


# Every C entry point that can fail inside turns that failure into a return code and a message; a null
# handle is rejected before any device work, so this runs without a GPU.
_NULL_HANDLE_CALLS = [
    ("fs_score", (None, 0, 0, 0, None, None, 0, 0, 0, None, 0, None), -1, "fs_score: null pointer"),
    ("fs_debug_rows", (None, 0, 0, 0, None, None, 0, None, 0, None, None, None, None), -1,
     "fs_debug_rows: invalid argument"),
    ("fs_debug_slab", (None, 0, 1, None, None), -1, "fs_debug_slab: invalid argument"),
    ("fs_joint_matrix", (None, 0, 1.0, None, 0, 0, 0, None, 0, None), -1, "fs_joint_matrix: null pointer"),
    ("fs_joint_tables", (None, None, 0, None, 0, None), -1, "fs_joint_tables: invalid argument"),
    ("fs_joint_columns", (None, 0, 1.0, None, 0, None, 0, None, 0, None), -1, "fs_joint_columns: null pointer"),
    ("fs_mdr_scan", (None, None, 0, 2, None, 2, 1, None, None, None, None, None, None, None), -1, "mdr: null pointer"),
    ("fs_mdr_tables", (None, None, 0, 2, None, 2, None, 0, None), -1, "mdr: null pointer"),
    ("fs_dataset_create", (None, None, 0, 1, 1, 1, None, 2, 0, None), -1, "fs_dataset_create: null pointer"),
    ("fs_dataset_create_device", (None, None, 0, 1, 1, 1, None, 2, 0, None), -1,
     "fs_dataset_create_device: null pointer"),
    ("fs_dataset_create_group", (None, None, None, 0, 1, 1, 1, None, 2, None), -1,
     "fs_dataset_create_group: null pointer"),
    ("fs_dataset_attach_comm", (None, None, None), -1, "fs_dataset_attach_comm: null data set"),
    ("fs_comm_create", (None, 0, 1, 0), -1, "fs_comm_create: null pointer"),
    ("fs_comm_reserve", (None, 0, None, None), -1, "fs_comm_reserve: null communicator"),
    ("fs_comm_connect", (None, None, None), -5, "fs_comm_connect: reserve the arena first"),
    ("fs_multi_create", (None, None, 0, 1, 1, 1, None, 2, None, 1), -1, "fs_multi_create: null pointer"),
    ("fs_multi_score", (None, 0, 0, 0, None, None, 0, None, None), -1, "fs_multi_score: null pointer"),
]


@pytest.mark.parametrize("name,args,code,message", _NULL_HANDLE_CALLS, ids=[c[0] for c in _NULL_HANDLE_CALLS])
def test_c_entry_points_reject_a_null_handle(name, args, code, message):
    lib = _native.load()
    assert getattr(lib, name)(*args) == code
    assert lib.fs_last_error().decode().startswith(message)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "fastselect_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                hits = re.findall(r"(?:from|import)\s+oracle|libfs_oracle|fso_\w+\s*\(|#include[^\n]*oracle|ref_oracle", src)
                assert not hits, (os.path.join(dirpath, f), hits)


# ---------------------------------------------------------------------------
# TuRF (behaviours of the reference's tests/test_turf.py with the same mock)
# ---------------------------------------------------------------------------
class MockReliefEstimator(BaseEstimator):
    def __init__(self):
        pass

    def fit(self, X, y):
        self.n_features_in_ = X.shape[1]
        self.feature_importances_ = np.linspace(1.0, 0.0, self.n_features_in_)
        return self


def _data(n=50, p=100):
    rs = np.random.RandomState(0)
    return rs.rand(n, p), rs.randint(0, 2, n)


def test_turf_selects_the_requested_number_sorted():
    x, y = _data()
    t = fsb.TuRF(MockReliefEstimator(), n_features_to_select=10, pct_remove=0.1).fit(x, y)
    assert len(t.top_features_) == 10
    assert np.array_equal(t.top_features_, np.arange(10))          # sorted surviving indices
    assert t.feature_importances_.shape == (100,)
    assert t.transform(x).shape == (50, 10)
    assert t.fit_transform(x, y).shape == (50, 10)


def test_turf_never_overshoots_and_honours_n_iterations():
    x, y = _data(p=23)
    t = fsb.TuRF(MockReliefEstimator(), n_features_to_select=7, pct_remove=0.5).fit(x, y)
    assert len(t.top_features_) == 7
    t = fsb.TuRF(MockReliefEstimator(), n_features_to_select=2, pct_remove=0.1, n_iterations=3).fit(x, y)
    assert len(t.top_features_) == 23 - 2 - 2 - 1                   # max(1, int(len * 0.1)) per iteration
    t = fsb.TuRF(MockReliefEstimator(), n_features_to_select=30).fit(x, y)
    assert len(t.top_features_) == 23                               # nothing to remove


def test_turf_schedule_of_config_c5():
    """p = 500 000, pct 0.1 -> 10 features: 109 fits, sum of p_t = 5 000 376 (SURVEY.md 3.4)."""
    t = fsb.TuRF(MockReliefEstimator(), n_features_to_select=10, pct_remove=0.1)
    n_active, fits, total = 500_000, 1, 500_000
    while n_active > 10:
        n_active -= t._n_to_remove(n_active)
        fits += 1
        total += n_active
    assert (fits, total) == (109, 5_000_376)


def test_turf_errors_and_verbose(capsys):
    x, y = _data(p=12)
    for pct in (0.0, 1.0, -0.5, 1.5):
        with pytest.raises(ValueError, match="pct_remove must be between 0 and 1"):
            fsb.TuRF(MockReliefEstimator(), pct_remove=pct).fit(x, y)
    with pytest.raises(NotFittedError):
        fsb.TuRF(MockReliefEstimator()).transform(x)
    fsb.TuRF(MockReliefEstimator(), n_features_to_select=10, pct_remove=0.1, verbose=True).fit(x, y)
    assert "Iteration 0: 11 features remaining." in capsys.readouterr().out


# ---------------------------------------------------------------------------
# row sharding
# ---------------------------------------------------------------------------
def test_shard_rows_partitions_every_row_once():
    for n in (2, 7, 100, 4000, 20001):
        for w in (1, 2, 3, 8):
            parts = [shard_rows(n, w, r) for r in range(w)]
            assert parts[0][0] == 0 and parts[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
            sizes = [b - a for a, b in parts]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_rows(10, 2, 2)


_WORKER = r"""
import os, sys
import numpy as np
import torch.distributed as dist
sys.path.insert(0, {root!r})
from fastselect_b200._shard import score_sharded, shard_rows, dist_info, enable_distributed, group_comm
from oracle import ref_oracle as R
from datasets import mixed

dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
# sharding across the process group is OPT-IN: without it a fit inside a torchrun job stays local
assert dist_info() == (0, 1)
enable_distributed()
assert dist_info() == (dist.get_rank(), 2)
assert group_comm(61, 18, np.float32, np.zeros(61, np.int32)) is None      # gloo: no multi-GPU group, allreduce path
x, y = mixed(3, 61, 18, 3)
x32, recip, isd = R.multisurf_prep(x, 10)
yc = np.unique(y, return_inverse=True)[1].astype(np.int64)
calls = []
def score_rows(lo, hi, out_ptr):          # the oracle stands in for the GPU kernel in this CPU test
    assert out_ptr is None
    calls.append((lo, hi))
    return R.multisurf_targets(x32, yc, recip, isd, True, np.arange(lo, hi), False, False)["wsum"]
total = score_sharded(61, 18, score_rows, device_buffers=False)
full = R.multisurf_targets(x32, yc, recip, isd, True, np.arange(61), False, False)["wsum"]
assert calls == [shard_rows(61, 2, dist.get_rank())], calls
np.testing.assert_allclose(total, full, rtol=1e-12, atol=1e-12)
print("rank", dist.get_rank(), "ok", calls)
dist.destroy_process_group()
"""


def test_two_rank_gloo_sharding_matches_single_process(tmp_path):
    import socket

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=port))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], env=env, stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
    assert "rank 0 ok [(0, 31)]" in outs[0] and "rank 1 ok [(31, 61)]" in outs[1]


def test_turf_selection_equals_argsort_prefix():
    """TuRF._worst: O(p) selection returns the set np.argsort(scores)[:k] (TuRF.py:104), ties included."""
    from fastselect_b200._turf import TuRF

    rs = np.random.RandomState(0)
    for trial in range(400):
        n = rs.randint(2, 80)
        s = rs.randint(0, 5, n).astype(np.float32) if trial % 2 else rs.standard_normal(n).astype(np.float32)
        k = rs.randint(1, n + 1)
        assert set(TuRF._worst(s, k).tolist()) == set(np.argsort(s)[:k].tolist())


def test_aligned_shards_partition_every_row_once():
    """shard_rows(align=4): the multi-GPU symmetric distance kernel wants shard starts that are
    multiples of 4; the shards must still cover every row exactly once."""
    from fastselect_b200._shard import shard_starts

    for n in (5, 61, 4000, 5656, 11312):
        for w in (1, 2, 3, 8):
            starts = shard_starts(n, w, align=4)
            assert starts[0] == 0 and starts[-1] == n and len(starts) == w + 1
            assert all(a <= b for a, b in zip(starts, starts[1:]))
            assert all(s % 4 == 0 for s in starts[:-1])
            assert [shard_rows(n, w, r, 4) for r in range(w)] == list(zip(starts, starts[1:]))


def test_group_shards_fall_on_distance_super_blocks():
    """group_shard_starts: a multi-GPU group's shards end on super-blocks of 256 target rows (the tile of the
    distance GEMM) when every rank gets at least four of them, stay within one super-block of the balanced
    split (the arena's slab is sized for ceil(n / world) + 256 rows), and cover every row exactly once."""
    from fastselect_b200._shard import group_shard_starts, shard_starts

    for n in (5, 61, 1000, 4000, 5656, 8000, 11312, 20000, 26000):
        for w in (1, 2, 3, 4, 8):
            starts = group_shard_starts(n, w)
            assert starts[0] == 0 and starts[-1] == n and len(starts) == w + 1
            rows = [b - a for a, b in zip(starts, starts[1:])]
            assert all(r >= 0 for r in rows) and max(rows) <= -(-n // w) + 256
            assert all(s % 4 == 0 for s in starts[:-1])
            if -(-n // 256) >= 4 * w:
                assert all(s % 256 == 0 for s in starts[:-1]) and min(rows) > 0
                # whole super-blocks per rank: the ranks' row super-blocks add up to ceil(n / 256), no more
                assert sum(-(-r // 256) for r in rows) == -(-n // 256)
            else:
                assert starts == shard_starts(n, w, 4)


def test_top_features_equal_the_reference_expression():
    """_ReliefBase._top == np.argsort(scores)[::-1][:k] (MultiSURF.py:443), ties included."""
    from fastselect_b200._relief import _ReliefBase

    rs = np.random.RandomState(1)
    for trial in range(300):
        p = rs.randint(9, 400)
        k = rs.randint(1, max(2, p // 8))
        s = (rs.randint(0, 50, p) / 7).astype(np.float32) if trial % 2 else rs.standard_normal(p).astype(np.float32)
        assert np.array_equal(_ReliefBase._top(s, k), np.argsort(s)[::-1][:k])


def test_bench_reference_arm_prints_the_contract_line():
    """bench.py --impl reference (the oracle port on the host cores) prints one JSON line with the
    keys the driver reads; tiny workload so that the CPU suite stays fast."""
    import json

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "300",
                          "--p", "400", "--steps", "1", "--warmup", "1"], capture_output=True, text=True, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "multisurf_fit_pair_features_per_s"
    assert line["unit"] == "sample-pair*features/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0 and line["vs_baseline"] is None


def test_bench_dump_outputs_are_reproducible_and_bounded(tmp_path):
    """bench.py --dump-outputs DIR: the last timed step's outputs as float32 / float64 .npy files, the same
    for the same arguments whatever --steps is, and a fixed sample of an output above its share of 64 MB."""
    def run(out, *args):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--warmup", "0",
                              "--dump-outputs", str(out), *args], capture_output=True, text=True, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        return {f.stem: np.load(f) for f in out.iterdir()}

    a = run(tmp_path / "a", "--n", "300", "--p", "400", "--steps", "1")
    b = run(tmp_path / "b", "--n", "300", "--p", "400", "--steps", "2")
    assert set(a) == set(b) == {"feature_importances"} and a["feature_importances"].shape == (400,)
    assert np.array_equal(a["feature_importances"], b["feature_importances"])
    j = run(tmp_path / "j", "--workload", "j1", "--n", "300", "--p", "2100", "--steps", "1")
    assert j["relevance"].shape == (2100,)
    assert j["redundancy"].ndim == 1 and 0 < j["redundancy"].size < 2100 * 2100       # 35 MB > 32 MB: sampled
    assert sum(f.stat().st_size for f in (tmp_path / "j").iterdir()) <= 64 << 20
    assert all(v.dtype in (np.float32, np.float64) for v in (*a.values(), *j.values()))


def test_turf_resident_scoring_keeps_the_base_estimators_validation():
    """The reference re-fits the base estimator on X[:, active] every iteration (TuRF.py:110-111), so an
    integer n_features_to_select of the BASE estimator above the remaining column count raises there;
    the resident path makes the same check before scoring a subset."""
    from fastselect_b200._turf import TuRF

    class FakeSession:
        def score(self, active=None):
            return np.zeros(5 if active is None else len(active), np.float32)

    scorer = TuRF._checked_scorer(FakeSession(), fsb.MultiSURF(n_features_to_select=4))
    assert scorer(np.arange(4)).shape == (4,)
    with pytest.raises(ValueError, match="must be > 0 and <= n_features"):
        scorer(np.arange(3))
    assert TuRF._checked_scorer(FakeSession(), fsb.MultiSURF(n_features_to_select=0.2))(np.arange(2)).shape == (2,)
