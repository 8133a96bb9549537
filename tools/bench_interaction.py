"""Measure the pairwise interaction screen (fs_interaction_scan) next to MDR's scan (fs_mdr_scan) on a B200.

Writes one JSON (default profiles/r05_interaction.json) with the GPU's name, power limit and maximum SM clock
read in the same run, and per shape (0/1/2 genotypes with a planted pair, n_top = 100):
  * scan kernel time per call of both scans on the same data set in the same process (CUDA events inside the
    library, fs_stats), after one warm-up call of each, the two calls alternating; the pack is timed on the
    first call of each (the planes of one fold and of MDR's five folds are different), later calls repack
    since the two alternate, so only ms_dist_general (the scan kernel) is compared;
  * pairs per second, and the AND + POPC count derived from the shapes: n_pairs * W * 4, W being the words of
    a bit-plane row (every segment padded to whole words, then to 4 words); no POPC peak is measured here, so
    no share of peak is reported;
  * at 4000 x 100 000 (C3), PairwiseInteraction().fit wall time from a numpy array, its first pair and p-value.

Needs a B200; there is no CPU path.  Usage: python tools/bench_interaction.py [--out FILE] [--quick] [--steps K]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import fastselect_b200 as fsb  # noqa: E402
from fastselect_b200 import _mdr, _native  # noqa: E402
from bench_mdr import gpu_info, plane_words  # noqa: E402
from datasets import epistatic_genotypes  # noqa: E402


def scan_shape(n, p, steps, cv=5, n_top=100):
    X, y = epistatic_genotypes(42, n, p)
    fold = _mdr.make_folds(y, cv, None)
    pairs = p * (p - 1) // 2
    W = {"interaction": plane_words(y, np.zeros(n, np.int64), 1), "mdr": plane_words(y, fold, cv)}
    calls = {"interaction": lambda ds: ds.interaction_scan(n_top, want_stats=True),
             "mdr": lambda ds: ds.mdr_scan(fold, 2, n_top, want_stats=True)}
    runs = {k: [] for k in calls}
    with _mdr.MDRData(X, y) as src:
        first = {k: call(src._ds) for k, call in calls.items()}             # warm-up, pack timed here
        for _ in range(steps):
            for k, call in calls.items():
                t0 = time.perf_counter()
                out, st = call(src._ds)
                runs[k].append(dict(wall_ms=1e3 * (time.perf_counter() - t0), total_ms=st["ms_total"],
                                    pack_ms=st["ms_gather"], scan_ms=st["ms_dist_general"],
                                    merge_ms=st["ms_reduce"], blocks=st["n_chunks"]))
                assert np.array_equal(out["top_idx"], first[k][0]["top_idx"])
    res = dict(n=n, p=p, pairs=pairs, n_top=n_top, mdr_cv=cv)
    for k in calls:
        scan_ms = float(np.median([r["scan_ms"] for r in runs[k]]))
        st0 = first[k][1]
        res[k] = dict(plane_words=W[k], popc=pairs * W[k] * 4,
                      first_call=dict(pack_ms=st0["ms_gather"], scan_ms=st0["ms_dist_general"],
                                      merge_ms=st0["ms_reduce"], total_ms=st0["ms_total"]),
                      runs=runs[k], scan_ms_median=scan_ms, pairs_per_s=pairs / (scan_ms * 1e-3),
                      popc_per_s=pairs * W[k] * 4 / (scan_ms * 1e-3), popc_share_of_peak="not measured",
                      top_pair=[int(v) for v in _mdr.decode_combinations(first[k][0]["top_idx"][:1], p, 2)[0]])
    res["interaction"]["top_ksa"] = float(first["interaction"][0]["top_ksa"][0])
    return res


def fit_c3(steps):
    X, y = epistatic_genotypes(42, 4000, 100_000)
    fsb.PairwiseInteraction().fit(X, y)                  # warm-up
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        est = fsb.PairwiseInteraction().fit(X, y)
        times.append(time.perf_counter() - t0)
    return dict(shape=[4000, 100_000], fit_s=times, fit_s_median=float(np.median(times)),
                first_pair=[int(v) for v in est.pairs_[0]], ksa=float(est.ksa_statistic_[0]),
                G=float(est.statistic_[0]), dof=int(est.dof_[0]), p_value=float(est.p_values_[0]),
                bound=est.bound_, n_pairs_tested=est.n_pairs_tested_)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_interaction.json"))
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small shapes only (a smoke run of this script)")
    a = ap.parse_args()
    if _native.device_count() < 1:
        raise SystemExit("bench_interaction.py needs a B200")
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
