"""Measure the MDR scan (fs_mdr_scan) and the MDR fit on a B200.

Writes one JSON (default profiles/r04_mdr.json) with the GPU's name, power limit and maximum SM clock read in
the same run, and per shape (order 2, cv = 5, n_top = 100, 0/1/2 genotypes with a planted pair):
  * pack and scan kernel time per call (CUDA events inside the library, fs_stats), after a warm-up call;
    the pack is timed on the first call of a (column list, fold) pair, later calls reuse it;
  * pairs per second of the scan, and the POPC count derived from the shapes: n_pairs * W * 4, W being the
    words of a bit-plane row (every segment padded to whole words); no POPC peak is measured here, so no
    share of peak is reported;
  * at 4000 x 100 000 (C3), MDR().fit wall time from a numpy array and the combination it finds.

Needs a B200; there is no CPU path.  Usage: python tools/bench_mdr.py [--out FILE] [--quick] [--steps K]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import fastselect_b200 as fsb  # noqa: E402
from fastselect_b200 import _mdr, _native  # noqa: E402
from datasets import epistatic_genotypes  # noqa: E402


def gpu_info():
    q = "name,power.limit,power.max_limit,clocks.max.sm,memory.total"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, plim, pmax, clk, mem = [s.strip() for s in out.split(",")]
    return dict(name=name, power_limit=plim, power_max_limit=pmax, clocks_max_sm=clk, memory_total=mem)


def plane_words(y_enc, fold, cv):
    """Words of one bit-plane row: every (fold, class) segment padded to whole 32-bit words, then to 4 words."""
    seg = np.bincount(2 * fold + y_enc, minlength=2 * cv)
    w = int(np.sum((seg + 31) // 32))
    return (w + 3) // 4 * 4


def scan_shape(n, p, steps, cv=5):
    X, y = epistatic_genotypes(42, n, p)
    fold = _mdr.make_folds(y, cv, None)
    pairs = p * (p - 1) // 2
    W = plane_words(y, fold, cv)
    with _mdr.MDRData(X, y) as src:
        first, st0 = src._ds.mdr_scan(fold, 2, 100, want_stats=True)
        runs = []
        for _ in range(steps):
            t0 = time.perf_counter()
            out, st = src._ds.mdr_scan(fold, 2, 100, want_stats=True)
            runs.append(dict(wall_ms=1e3 * (time.perf_counter() - t0), total_ms=st["ms_total"],
                             pack_ms=st["ms_gather"], scan_ms=st["ms_dist_general"], merge_ms=st["ms_reduce"],
                             blocks=st["n_chunks"]))
            assert np.array_equal(out["top_idx"], first["top_idx"])
    scan_ms = float(np.median([r["scan_ms"] for r in runs]))
    top = _mdr.decode_combinations(first["top_idx"][:1], p, 2)[0]
    return dict(n=n, p=p, cv=cv, pairs=pairs, plane_words=W, popc=pairs * W * 4,
                first_call=dict(pack_ms=st0["ms_gather"], scan_ms=st0["ms_dist_general"], merge_ms=st0["ms_reduce"],
                                total_ms=st0["ms_total"]),
                runs=runs, scan_ms_median=scan_ms, pairs_per_s=pairs / (scan_ms * 1e-3),
                popc_per_s=pairs * W * 4 / (scan_ms * 1e-3), popc_share_of_peak="not measured",
                best_mean_test=float(first["top_test"][0]), top_pair=[int(v) for v in top])


def fit_c3(steps):
    X, y = epistatic_genotypes(42, 4000, 100_000)
    fsb.MDR().fit(X, y)                                   # warm-up
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        est = fsb.MDR().fit(X, y)
        times.append(time.perf_counter() - t0)
    return dict(shape=[4000, 100_000], fit_s=times, fit_s_median=float(np.median(times)),
                best_combination=list(est.best_combination_), cv_consistency=est.cv_consistency_,
                test_balanced_accuracy=est.test_balanced_accuracy_)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_mdr.json"))
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small shapes only (a smoke run of this script)")
    a = ap.parse_args()
    if _native.device_count() < 1:
        raise SystemExit("bench_mdr.py needs a B200")
    res = dict(gpu=gpu_info(), steps=a.steps)
    shapes = [(2000, 4000)] if a.quick else [(4000, 100_000), (20_000, 20_000)]
    res["scan"] = [scan_shape(n, p, a.steps) for n, p in shapes]
    if not a.quick:
        res["fit_c3"] = fit_c3(a.steps)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
