"""ctypes binding of libfastselect_b200.so (the C ABI declared in include/fastselect_b200.h).

There is no CPU fallback: if the shared library is missing or no sm_100 GPU is
usable, :func:`require_gpu` raises ``RuntimeError`` and nothing is computed.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

FS_RELIEFF, FS_SURF, FS_MULTISURF = 0, 1, 2
FS_U8, FS_I8, FS_F32, FS_F64 = 0, 1, 2, 3
FS_ARITH_F32, FS_ARITH_F64 = 0, 1
FS_JOINT_MI, FS_JOINT_SU = 0, 1
FS_DISTINCT_CAP = 16
FS_ABI_VERSION = 9
FS_MDR_MAX_TOP = 2048

_DTYPES = {np.dtype(np.uint8): FS_U8, np.dtype(np.int8): FS_I8,
           np.dtype(np.float32): FS_F32, np.dtype(np.float64): FS_F64}

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libfastselect_b200.so")


class FsStats(C.Structure):
    _fields_ = [("ms_total", C.c_float), ("ms_gather", C.c_float), ("ms_dist_tensor", C.c_float),
                ("ms_dist_general", C.c_float), ("ms_select", C.c_float), ("ms_accum_tensor", C.c_float),
                ("ms_accum_general", C.c_float), ("ms_reduce", C.c_float), ("launches", C.c_int32),
                ("n_chunks", C.c_int32), ("n_tensor_cols", C.c_int64), ("n_general_cols", C.c_int64),
                ("onehot_k", C.c_int64), ("pairs_selected", C.c_int64),
                ("ops_dist_tensor", C.c_double), ("ops_accum_tensor", C.c_double),
                ("ms_host_prep", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load():
    """Load the shared library (built in-tree by ``__graft_entry__.build()`` / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"fastselect_b200: {LIB_PATH} is missing - build it with "
            "`make -C fastselect_b200/csrc` (or __graft_entry__.build()). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.fs_last_error.restype = C.c_char_p
    lib.fs_device_count.restype = C.c_int
    lib.fs_abi_version.restype = C.c_int
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    lib.fs_dataset_create.argtypes = [C.POINTER(vp), vp, C.c_int, i64, i64, i64, vp, i32, i32, vp]
    lib.fs_dataset_create_device.argtypes = lib.fs_dataset_create.argtypes
    lib.fs_dataset_column_stats.argtypes = [vp, vp, vp, vp]
    lib.fs_dataset_set_features.argtypes = [vp, vp, vp, C.c_int]
    lib.fs_dataset_destroy.argtypes = [vp]
    lib.fs_dataset_row_order.argtypes = [vp, vp]
    lib.fs_score.argtypes = [vp, C.c_int, C.c_int, i32, vp, vp, i64, i64, i64, vp, C.c_int, C.POINTER(FsStats)]
    lib.fs_debug_rows.argtypes = [vp, C.c_int, C.c_int, i32, vp, vp, i64, vp, i64, vp, vp, vp, vp]
    lib.fs_comm_create.argtypes = [C.POINTER(vp), i32, i32, i32]
    lib.fs_comm_required_bytes.argtypes = [i64, i64, i32, i32, i32]
    lib.fs_comm_required_bytes.restype = C.c_uint64
    lib.fs_comm_reserve.argtypes = [vp, C.c_uint64, vp, C.POINTER(i32)]
    lib.fs_comm_connect.argtypes = [vp, vp, vp]
    lib.fs_comm_arena.argtypes = [vp]
    lib.fs_comm_arena.restype = vp
    lib.fs_comm_connected.argtypes = [vp]
    lib.fs_comm_destroy.argtypes = [vp]
    lib.fs_dataset_create_group.argtypes = [C.POINTER(vp), vp, vp, C.c_int, i64, i64, i64, vp, i32, vp]
    lib.fs_dataset_attach_comm.argtypes = [vp, vp, vp]
    lib.fs_multi_create.argtypes = [C.POINTER(vp), vp, C.c_int, i64, i64, i64, vp, i32, vp, i32]
    lib.fs_multi_world.argtypes = [vp]
    lib.fs_multi_column_stats.argtypes = [vp, vp, vp, vp]
    lib.fs_multi_set_features.argtypes = [vp, vp, vp, C.c_int]
    lib.fs_multi_score.argtypes = [vp, C.c_int, C.c_int, i32, vp, vp, i64, vp, C.POINTER(FsStats)]
    lib.fs_multi_destroy.argtypes = [vp]
    lib.fs_joint_matrix.argtypes = [vp, C.c_int, C.c_double, vp, i64, i64, i64, vp, C.c_int, C.POINTER(FsStats)]
    lib.fs_joint_tables.argtypes = [vp, vp, i64, vp, i64, vp]
    lib.fs_joint_columns.argtypes = [vp, C.c_int, C.c_double, vp, i64, vp, i64, vp, C.c_int, C.POINTER(FsStats)]
    lib.fs_debug_slab.argtypes = [vp, i64, i64, vp, vp]
    lib.fs_mdr_scan.argtypes = [vp, vp, i64, i32, vp, i32, i64, vp, vp, vp, vp, vp, vp, C.POINTER(FsStats)]
    lib.fs_mdr_tables.argtypes = [vp, vp, i64, i32, vp, i32, vp, i64, vp]
    lib.fs_interaction_scan.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, C.POINTER(FsStats)]
    if lib.fs_abi_version() != FS_ABI_VERSION:
        raise RuntimeError(f"fastselect_b200: {LIB_PATH} has ABI version {lib.fs_abi_version()}, "
                           f"this package needs {FS_ABI_VERSION}; rebuild it (make -C fastselect_b200/csrc)")
    _lib = lib
    return lib


def device_count() -> int:
    """Usable sm_100 GPUs; 0 when the library or a GPU is missing (never raises)."""
    try:
        return int(load().fs_device_count())
    except (RuntimeError, OSError):
        return 0


def _raise(rc, what):
    msg = load().fs_last_error().decode("utf-8", "replace")
    if rc == -2:
        raise RuntimeError(f"{what}: {msg}")
    if rc == -4:
        raise MemoryError(f"{what}: {msg}")
    if rc == -1:
        raise ValueError(f"{what}: {msg}")
    if rc == -6:
        raise TimeoutError(f"{what}: {msg}")
    raise RuntimeError(f"{what} failed ({rc}): {msg}")


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def _call(name, *args):
    """Call the C entry point ``name`` and raise on a non-zero return code."""
    rc = getattr(load(), name)(*args)
    if rc != 0:
        _raise(rc, name)
    return rc


def _columns(feat_idx, p):
    """(int64 array or None, n_kept) of a column list; None stands for all ``p`` columns."""
    if feat_idx is None:
        return None, p
    feat_idx = np.ascontiguousarray(feat_idx, np.int64)
    return feat_idx, feat_idx.size


def _folds(fold, n):
    """(int32 fold vector, n_folds) of a per-sample fold assignment."""
    fold = np.ascontiguousarray(fold, np.int32)
    if fold.shape != (n,):
        raise ValueError(f"fold must have one entry per sample ({n})")
    return fold, int(fold.max()) + 1 if fold.size else 0


def _stats(want_stats):
    """(FsStats or None, the matching pointer argument)."""
    stats = FsStats() if want_stats else None
    return stats, C.byref(stats) if stats is not None else None



def default_device() -> int:
    for key in ("FASTSELECT_B200_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(key)
        if v is not None and v.strip() != "":
            return int(v)
    return 0


class _DeviceData:
    """What :class:`Dataset` (``fs_dataset_*``) and :class:`MultiDataset` (``fs_multi_*``) share: the input
    checks, the handle's lifecycle, the column scan and the typing."""

    _prefix = ""

    @staticmethod
    def _matrix(x):
        if x.dtype not in _DTYPES:
            raise TypeError(f"unsupported dtype {x.dtype}")
        if x.ndim != 2:
            raise ValueError("x must be 2-D")
        if x.strides[1] != x.itemsize or x.strides[0] % x.itemsize or x.strides[0] < x.shape[1] * x.itemsize:
            x = np.ascontiguousarray(x)
        return x

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def close(self):
        if getattr(self, "_h", None):
            getattr(load(), self._prefix + "_destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def column_stats(self):
        cmin = np.empty(self.p, np.float64)
        cmax = np.empty(self.p, np.float64)
        cnt = np.empty(self.p, np.int32)
        _call(self._prefix + "_column_stats", self._h, _ptr(cmin), _ptr(cmax), _ptr(cnt))
        return cmin, cmax, cnt

    def set_features(self, is_discrete, recip, arith):
        is_discrete = np.ascontiguousarray(is_discrete, np.uint8)
        recip = np.ascontiguousarray(recip, np.float32)
        _call(self._prefix + "_set_features", self._h, _ptr(is_discrete), _ptr(recip), int(arith))


class Dataset(_DeviceData):
    """A device-resident data set (``fs_dataset``): upload + on-GPU column scan.

    Not stored on fitted estimators (they stay picklable); always used as a
    context manager so the device memory is released deterministically."""

    _prefix = "fs_dataset"

    def __init__(self, x: np.ndarray, y_enc: np.ndarray, n_classes: int, device: int | None = None,
                 stream: int = 0, comm: "Comm | None" = None):
        """``comm``: a connected multi-GPU communicator -- the upload is then COLLECTIVE: this rank copies
        only its 1 / world of the rows and the shards are replicated over NVLink (every rank passes the
        same ``x``)."""
        lib = load()
        x = self._matrix(x)
        self.n, self.p = x.shape
        self._keep = x
        y_enc = np.ascontiguousarray(y_enc, np.int32)
        h = C.c_void_p()
        dev = default_device() if device is None else device
        if comm is not None and comm.world > 1:
            rc = lib.fs_dataset_create_group(C.byref(h), comm._h, _ptr(x), _DTYPES[x.dtype], self.n, self.p,
                                             x.strides[0] // x.itemsize, _ptr(y_enc), int(n_classes),
                                             C.c_void_p(stream))
            dev = comm.device
        else:
            rc = lib.fs_dataset_create(C.byref(h), _ptr(x), _DTYPES[x.dtype], self.n, self.p,
                                       x.strides[0] // x.itemsize, _ptr(y_enc), int(n_classes), dev,
                                       C.c_void_p(stream))
        if rc != 0:
            _raise(rc, "fs_dataset_create")
        self.device = dev
        self.comm = None
        self.shard = None
        self._h = h
        self._keep = None

    def attach_comm(self, comm, row_starts):
        """Join a multi-GPU group (include/fastselect_b200.h): afterwards ``score`` over exactly this rank's
        shard ``[row_starts[rank], row_starts[rank + 1])`` is a COLLECTIVE call that returns the complete
        weight sums on every rank.  ``comm=None`` detaches."""
        if comm is None:
            self.comm, self.shard = None, None
            _call("fs_dataset_attach_comm", self._h, None, None)
        else:
            starts = np.ascontiguousarray(row_starts, np.int64)
            _call("fs_dataset_attach_comm", self._h, comm._h, _ptr(starts))
            self.comm = comm
            self.shard = (int(starts[comm.rank]), int(starts[comm.rank + 1]))

    def row_order(self):
        perm = np.empty(self.n, np.int64)
        _call("fs_dataset_row_order", self._h, _ptr(perm))
        return perm

    def score(self, algo, use_star=False, k=0, class_probs=None, feat_idx=None, row_begin=0, row_end=None,
              out_device_ptr=None, want_stats=False):
        """Partial weight sums (float64, before the final ``/ n``) of the target rows
        ``[row_begin, row_end)``.  With ``out_device_ptr`` the result is written to that
        device buffer (for an in-place NCCL allreduce) and ``None`` is returned."""
        row_end = self.n if row_end is None else row_end
        feat_idx, n_kept = _columns(feat_idx, self.p)
        cp = None if class_probs is None else np.ascontiguousarray(class_probs, np.float32)
        stats, stats_arg = _stats(want_stats)
        out = None
        if out_device_ptr is None:
            out = np.empty(n_kept, np.float64)
            dst, on_dev = _ptr(out), 0
        else:
            dst, on_dev = C.c_void_p(out_device_ptr), 1
        _call("fs_score", self._h, int(algo), int(bool(use_star)), int(k), _ptr(cp), _ptr(feat_idx), n_kept,
              int(row_begin), int(row_end), dst, on_dev, stats_arg)
        return (out, stats.as_dict()) if want_stats else out

    def joint_matrix(self, kind, log_base=1.0, feat_idx=None, pos_begin=0, pos_end=None, out_device_ptr=None,
                     want_stats=False):
        """Pairwise statistic (FS_JOINT_MI / FS_JOINT_SU) of the discrete columns ``feat_idx``: the
        float64 ``[n_kept, n_kept]`` matrix restricted to the pairs whose smaller position lies in
        ``[pos_begin, pos_end)`` (see include/fastselect_b200.h)."""
        feat_idx, n_kept = _columns(feat_idx, self.p)
        pos_end = n_kept if pos_end is None else pos_end
        stats, stats_arg = _stats(want_stats)
        out = None
        if out_device_ptr is None:
            out = np.empty((n_kept, n_kept), np.float64)
            dst, on_dev = _ptr(out), 0
        else:
            dst, on_dev = C.c_void_p(out_device_ptr), 1
        _call("fs_joint_matrix", self._h, int(kind), float(log_base), _ptr(feat_idx), n_kept, int(pos_begin),
              int(pos_end), dst, on_dev, stats_arg)
        return (out, stats.as_dict()) if want_stats else out

    def joint_columns(self, kind, log_base, positions, feat_idx=None, want_stats=False):
        """Rows ``positions`` of :meth:`joint_matrix` without the matrix: float64 ``[len(positions), n_kept]``,
        row i = statistic of position ``positions[i]`` against every position (0 at itself), bitwise equal
        to ``joint_matrix(kind, log_base, feat_idx)[positions]``.  The first call on a column list encodes
        it; later calls on the same list reuse the encoding (see include/fastselect_b200.h)."""
        positions = np.ascontiguousarray(np.atleast_1d(positions), np.int64)
        if positions.ndim != 1 or positions.size < 1:
            raise ValueError("positions must be a non-empty 1-D list of column positions")
        feat_idx, n_kept = _columns(feat_idx, self.p)
        stats, stats_arg = _stats(want_stats)
        out = np.empty((positions.size, n_kept), np.float64)
        _call("fs_joint_columns", self._h, int(kind), float(log_base), _ptr(feat_idx), n_kept, _ptr(positions),
              positions.size, _ptr(out), 0, stats_arg)
        return (out, stats.as_dict()) if want_stats else out

    def joint_tables(self, pairs, feat_idx=None):
        """Exact contingency tables of ``pairs`` (``[m, 2]`` positions in ``feat_idx``): int64
        ``[m, 16, 16]``, entry ``[q, va, vb]`` counting the samples with the va-th smallest value of
        the first column and the vb-th smallest value of the second."""
        pairs = np.ascontiguousarray(pairs, np.int64).reshape(-1, 2)
        feat_idx, n_kept = _columns(feat_idx, self.p)
        out = np.empty((pairs.shape[0], 16, 16), np.int64)
        _call("fs_joint_tables", self._h, _ptr(feat_idx), n_kept, _ptr(pairs), pairs.shape[0], _ptr(out))
        return out

    def mdr_scan(self, fold, order, n_top, feat_idx=None, want_all=False, want_stats=False):
        """MDR search over the combinations of order 1 or 2 of the positions of ``feat_idx`` (see
        include/fastselect_b200.h): ``fold`` ([n], original sample order) assigns every sample to one of
        ``max(fold) + 1`` cross-validation folds.  Returns a dict with ``top_idx`` (int64 ``[n_top]``),
        ``top_train`` / ``top_test`` (mean balanced accuracies), ``fold_best`` (int64 ``[n_folds]``) and, with
        ``want_all``, ``all_train`` / ``all_test`` (float64 ``[n_combos]``)."""
        fold, n_folds = _folds(fold, self.n)
        feat_idx, n_kept = _columns(feat_idx, self.p)
        n_combos = n_kept if order == 1 else n_kept * (n_kept - 1) // 2
        out = dict(top_idx=np.empty(n_top, np.int64), top_train=np.empty(n_top, np.float64),
                   top_test=np.empty(n_top, np.float64), fold_best=np.empty(max(n_folds, 1), np.int64))
        if want_all:
            out["all_train"] = np.empty(n_combos, np.float64)
            out["all_test"] = np.empty(n_combos, np.float64)
        stats, stats_arg = _stats(want_stats)
        _call("fs_mdr_scan", self._h, _ptr(feat_idx), n_kept, int(order), _ptr(fold), n_folds, int(n_top),
              _ptr(out["top_idx"]), _ptr(out["top_train"]), _ptr(out["top_test"]), _ptr(out["fold_best"]),
              _ptr(out.get("all_train")), _ptr(out.get("all_test")), stats_arg)
        return (out, stats.as_dict()) if want_stats else out

    def mdr_tables(self, fold, order, combos, feat_idx=None):
        """Exact cell counts of the combinations ``combos`` (``[m, order]`` positions in ``feat_idx``): int64
        ``[m, n_folds, 2, 9]``, entry ``[q, f, c, va * 3 + vb]`` counting the samples of fold f and class c whose
        values have ranks va / vb among their columns' distinct values (order 1: vb = 0)."""
        fold, n_folds = _folds(fold, self.n)
        combos = np.ascontiguousarray(combos, np.int64).reshape(-1, int(order))
        feat_idx, n_kept = _columns(feat_idx, self.p)
        out = np.empty((combos.shape[0], max(n_folds, 1), 2, 9), np.int64)
        _call("fs_mdr_tables", self._h, _ptr(feat_idx), n_kept, int(order), _ptr(fold), n_folds, _ptr(combos),
              combos.shape[0], _ptr(out))
        return out

    def interaction_scan(self, n_top, feat_idx=None, want_all=False, want_stats=False):
        """KSA screen of every pair of the positions of ``feat_idx`` (see include/fastselect_b200.h): returns a
        dict with ``top_idx`` (int64 ``[n_top]``, pair indices of :meth:`mdr_scan` order 2), ``top_ksa``
        (float64 ``[n_top]``, highest first), ``top_tables`` (int64 ``[n_top, 2, 9]``, entry ``[q, k, i * 3 + j]``
        counting the samples of class k with state i in the first and j in the second column) and, with
        ``want_all``, ``all_ksa`` (float64 ``[n_pairs]``)."""
        feat_idx, n_kept = _columns(feat_idx, self.p)
        out = dict(top_idx=np.empty(n_top, np.int64), top_ksa=np.empty(n_top, np.float64),
                   top_tables=np.empty((n_top, 2, 9), np.int64))
        if want_all:
            out["all_ksa"] = np.empty(n_kept * (n_kept - 1) // 2, np.float64)
        stats, stats_arg = _stats(want_stats)
        _call("fs_interaction_scan", self._h, _ptr(feat_idx), n_kept, int(n_top), _ptr(out["top_idx"]),
              _ptr(out["top_ksa"]), _ptr(out["top_tables"]), _ptr(out.get("all_ksa")), stats_arg)
        return (out, stats.as_dict()) if want_stats else out

    def debug_slab(self, row_begin, nrows):
        """Rows of the resident one-hot distance slab (internal row and sample order) as the last
        ``score`` call left it; returns (int32 [nrows, n], (first cached row, cached rows, columns))."""
        out = np.empty((nrows, self.n), np.int32)
        info = np.zeros(3, np.int64)
        _call("fs_debug_slab", self._h, int(row_begin), int(nrows), _ptr(out), _ptr(info))
        return out, tuple(int(v) for v in info)

    def debug_rows(self, algo, targets, use_star=False, k=0, class_probs=None, feat_idx=None):
        targets = np.ascontiguousarray(targets, np.int64)
        nt = targets.size
        feat_idx, n_kept = _columns(feat_idx, self.p)
        cp = None if class_probs is None else np.ascontiguousarray(class_probs, np.float32)
        dist = np.empty((nt, self.n), np.float64)
        thresh = np.empty(nt, np.float64)
        mask = np.empty((nt, self.n), np.int8)
        wsum = np.empty(n_kept, np.float64)
        _call("fs_debug_rows", self._h, int(algo), int(bool(use_star)), int(k), _ptr(cp), _ptr(feat_idx), n_kept,
              _ptr(targets), nt, _ptr(dist), _ptr(thresh), _ptr(mask), _ptr(wsum))
        return dict(dist=dist, thresh=thresh, mask=mask, wsum=wsum)


class Comm:
    """One rank of a multi-GPU group (``fs_comm``): its exchange arena and the mappings of the peers' arenas."""

    def __init__(self, rank: int, world: int, device: int):
        h = C.c_void_p()
        _call("fs_comm_create", C.byref(h), int(rank), int(world), int(device))
        self._h, self.rank, self.world, self.device = h, int(rank), int(world), int(device)

    @staticmethod
    def required_bytes(n, p, dtype, world, with_x=True) -> int:
        return int(load().fs_comm_required_bytes(int(n), int(p), _DTYPES[np.dtype(dtype)], int(world), int(bool(with_x))))

    def reserve(self, nbytes):
        """Make sure the arena holds ``nbytes``; returns (64-byte IPC handle, arena was re-allocated)."""
        handle = np.zeros(64, np.uint8)
        changed = C.c_int32(0)
        _call("fs_comm_reserve", self._h, C.c_uint64(int(nbytes)), _ptr(handle), C.byref(changed))
        return handle, bool(changed.value)

    @property
    def arena(self) -> int:
        return int(load().fs_comm_arena(self._h) or 0)

    @property
    def connected(self) -> bool:
        return bool(load().fs_comm_connected(self._h))

    def connect(self, handles=None, raw_ptrs=None):
        """Map the peers' arenas (``handles``: world x 64 bytes of CUDA IPC handles; ``raw_ptrs``: arena
        pointers of ranks inside this process).  Run a host-level barrier over all ranks afterwards."""
        hs = None if handles is None else np.ascontiguousarray(handles, np.uint8)
        rp = None
        if raw_ptrs is not None:
            rp = (C.c_void_p * self.world)(*[C.c_void_p(int(q)) for q in raw_ptrs])
        _call("fs_comm_connect", self._h, _ptr(hs), rp)

    def close(self):
        if getattr(self, "_h", None):
            load().fs_comm_destroy(self._h)
            self._h = None


class MultiDataset(_DeviceData):
    """A data set spread over several GPUs of THIS process (``fs_multi``: one host thread per GPU inside
    the library).  Same surface as :class:`Dataset` as far as the estimators use it; ``score`` always
    covers all target rows and returns the complete weight sums."""

    _prefix = "fs_multi"

    def __init__(self, x: np.ndarray, y_enc: np.ndarray, n_classes: int, devices):
        lib = load()
        x = self._matrix(x)
        self.n, self.p = x.shape
        y_enc = np.ascontiguousarray(y_enc, np.int32)
        devs = np.ascontiguousarray(devices, np.int32)
        h = C.c_void_p()
        _call("fs_multi_create", C.byref(h), _ptr(x), _DTYPES[x.dtype], self.n, self.p, x.strides[0] // x.itemsize,
              _ptr(y_enc), int(n_classes), _ptr(devs), int(devs.size))
        self._h = h
        self.world = int(lib.fs_multi_world(h))
        self.comm, self.shard = None, None

    def score(self, algo, use_star=False, k=0, class_probs=None, feat_idx=None, row_begin=0, row_end=None,
              out_device_ptr=None, want_stats=False):
        if out_device_ptr is not None or row_begin != 0 or (row_end is not None and row_end != self.n):
            raise ValueError("MultiDataset.score covers all target rows and returns a host vector")
        feat_idx, n_kept = _columns(feat_idx, self.p)
        cp = None if class_probs is None else np.ascontiguousarray(class_probs, np.float32)
        stats, stats_arg = _stats(want_stats)
        out = np.empty(n_kept, np.float64)
        _call("fs_multi_score", self._h, int(algo), int(bool(use_star)), int(k), _ptr(cp), _ptr(feat_idx), n_kept,
              _ptr(out), stats_arg)
        return (out, stats.as_dict()) if want_stats else out
