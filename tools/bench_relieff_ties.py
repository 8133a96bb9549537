"""Measure ReliefF's reference tie order (relieff_ties_kernel) on a B200.

ReliefF (k = 10) on 0/1/2 int8 genotypes, which take the tensor path, at n = 8 000, where a row's
(distance, index) pairs are staged in shared memory, and at n = 30 000, where they go to global
scratch.  With p = 200 columns the k-th distance is tied in nearly every target row, so nearly every
row is replayed.  Per shape, after one warm-up call, a fixed range of target rows is scored --calls
times (Dataset.score(row_begin, row_end, want_stats=True); CUDA events inside the library), then
once more per call with FS_B200_RELIEFF_TIES=index, which skips the replay.  Printed as one JSON
line: the GPU's name and power limit, median and all ms_select / ms_total per shape, and a SHA-256
of the weight sums; --out DIR also saves them as wsum_n<N>.npy, so that two builds can be compared
bit for bit.  --lib selects the shared library, so that two builds can alternate as separate
processes in one session.

Needs a B200; there is no CPU path.
Usage: python tools/bench_relieff_ties.py [--lib PATH] [--out DIR] [--calls N] [--rows R] [--n N ...]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fastselect_b200 import _native  # noqa: E402

P, K, SEED = 200, 10, 7


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, plim, clk = [s.strip() for s in out.split(",")]
    return dict(name=name, power_limit=plim, clocks_max_sm=clk)


def data(n):
    rs = np.random.RandomState(SEED)
    x = rs.randint(0, 3, (n, P)).astype(np.int8)
    y = rs.randint(0, 2, n).astype(np.int32)
    y[(x[:, 1] == 1) & (x[:, 3] == 1)] = 1
    class_probs = (np.bincount(y) / n).astype(np.float32)
    return x, y, class_probs


def run_shape(n, rows, calls):
    x, y, cp = data(n)
    r0 = n // 2 - rows // 2
    res = dict(n=n, p=P, k=K, row_begin=r0, row_end=r0 + rows)
    with _native.Dataset(x, y, len(cp)) as ds:
        ds.set_features(np.ones(P, bool), np.ones(P, np.float32), _native.FS_ARITH_F32)

        def score():
            return ds.score(_native.FS_RELIEFF, k=K, class_probs=cp, row_begin=r0, row_end=r0 + rows,
                            want_stats=True)

        wsum, _ = score()                                  # warm-up
        stats = []
        for _ in range(calls):
            w, st = score()
            assert np.array_equal(w, wsum)
            stats.append(st)
        os.environ["FS_B200_RELIEFF_TIES"] = "index"
        try:
            index = [score()[1] for _ in range(calls)]
        finally:
            del os.environ["FS_B200_RELIEFF_TIES"]
    for key in ("ms_select", "ms_total"):
        res[key] = float(np.median([s[key] for s in stats]))
        res[key + "_all"] = [round(s[key], 4) for s in stats]
    res["ms_select_index_ties"] = float(np.median([s["ms_select"] for s in index]))
    res["n_tensor_cols"] = stats[0]["n_tensor_cols"]
    res["wsum_sha256"] = hashlib.sha256(wsum.tobytes()).hexdigest()
    return res, wsum


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=_native.LIB_PATH, help="shared library to load")
    ap.add_argument("--out", default=None, help="directory for the weight sums (wsum_n<N>.npy)")
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--rows", type=int, default=2048)
    ap.add_argument("--n", type=int, nargs="+", default=[8000, 30_000])
    a = ap.parse_args()
    _native.LIB_PATH = os.path.abspath(a.lib)
    _native.load()
    if _native.device_count() < 1:
        raise SystemExit("bench_relieff_ties.py needs a B200")
    res = dict(lib=a.lib, gpu=gpu_info(), calls=a.calls, shapes=[])
    for n in a.n:
        r, wsum = run_shape(n, a.rows, a.calls)
        res["shapes"].append(r)
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            np.save(os.path.join(a.out, f"wsum_n{n}.npy"), wsum)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
