"""Measure the column path of the joint-count statistics (fs_joint_columns) and mRMR(pairs="selected").

Writes one JSON (default profiles/joint_columns.json) with the GPU's name, power limit and maximum SM
clock read in the same run, and:
  * count / finish kernel time per call (CUDA events inside the library, fs_stats), warmed, on genotype
    data at 4000 x 100 000 and 20 000 x 200 000 and on 16-state columns at 4000 x 20 000 -- At is
    larger than the 126 MB L2 at every shape, so every call streams it from HBM;
    bytes model K * ceil(n / 2) over the count kernel's time, its share of 7.7 TB/s (data sheet), and
    the population-count model (one POPC per selected reduced row per 32 samples and At row, 16 per SM
    and clock) against the same time, the larger of the two being the bound;
  * mRMR(n_features_to_select=50, pairs="selected").fit from a numpy array at 4000 x 100 000, split
    into np.unique (unique_vals_), the upload copy, upload + column scan, encode, column calls and the
    rest of the host work;
  * pairs="all" vs pairs="selected" at 10 000 x 10 000 with k = 10, alternated;
  * parity: the selections of both modes at 10 000 x 10 000, and at 4000 x 100 000 the oracle on 64
    random columns against the class and against the first two selected features.

Needs a B200; there is no CPU path.  Usage: python tools/bench_joint_columns.py [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import fastselect_b200 as fsb  # noqa: E402
from fastselect_b200 import _mi, _native  # noqa: E402

HBM_BPS = 7.7e12           # HGX B200 data sheet, one GPU
POPC_PER_SM_CLK = 16
COUNT_SEL_BUCKETS = (1, 2, 4, 8, 16)      # template sizes of the count kernel (joint.cu)


def gpu_info():
    q = "name,power.limit,power.max_limit,clocks.max.sm,memory.total"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, plim, pmax, clk, mem = [s.strip() for s in out.split(",")]
    return dict(name=name, power_limit=plim, power_max_limit=pmax, clocks_max_sm=clk, memory_total=mem)


def genotypes(rng, n, p):
    return rng.integers(0, 3, (n, p), dtype=np.uint8)


def open_codes(codes):
    ds = _native.Dataset(codes, np.zeros(codes.shape[0], np.int32), 1)
    ds.set_features(np.ones(codes.shape[1], np.uint8), np.ones(codes.shape[1], np.float32), _native.FS_ARITH_F32)
    return ds


def kernel_times(codes, label, sm_clk_hz, sms, calls=40, positions_per_call=1):
    """Median per-call times of fs_joint_columns on one data set (one position per call, as the
    greedy searches ask)."""
    n, q = codes.shape
    rs = np.random.RandomState(0)
    with open_codes(codes) as ds:
        t0 = time.perf_counter()
        _, first = ds.joint_columns(0, 1.0, [q - 1], want_stats=True)
        first_wall = time.perf_counter() - t0
        for _ in range(5):                                   # warm
            ds.joint_columns(0, 1.0, rs.randint(0, q, positions_per_call))
        rows = []
        for _ in range(calls):
            pos = rs.randint(0, q, positions_per_call)
            t0 = time.perf_counter()
            _, st = ds.joint_columns(0, 1.0, pos, want_stats=True)
            rows.append((st["ms_dist_general"], st["ms_reduce"], st["ms_total"], st["ms_gather"],
                         (time.perf_counter() - t0) * 1e3, st["launches"], st["n_chunks"]))
        K = int(first["onehot_k"])
    a = np.array(rows)
    med = np.median(a, axis=0)
    ls = K // q if K % q == 0 else K / q
    sel = int(round(ls * positions_per_call))
    bucket = next(b for b in COUNT_SEL_BUCKETS if b >= sel)
    bytes_model = K * math.ceil(n / 2)
    count_s = med[0] * 1e-3
    t_mem = bytes_model / HBM_BPS
    popc = K * math.ceil(n / 32) * bucket
    t_popc = popc / (POPC_PER_SM_CLK * sms * sm_clk_hz)
    return dict(
        label=label, n=n, columns=q, reduced_rows_K=K, reduced_rows_per_position=ls, positions_per_call=positions_per_call,
        count_kernel_template_rows=bucket, calls=calls,
        first_call=dict(wall_ms=first_wall * 1e3, ms_encode_and_marginals=first["ms_gather"],
                        ms_count=first["ms_dist_general"], ms_finish=first["ms_reduce"], launches=first["launches"]),
        median_ms=dict(count=med[0], finish=med[1], device_total=med[2], encode=med[3], wall=med[4]),
        min_ms_count=float(a[:, 0].min()), max_ms_count=float(a[:, 0].max()),
        launches_per_call=int(med[5]), count_launches_per_call=int(med[6]),
        bytes_model=bytes_model, achieved_bytes_per_s=bytes_model / count_s, share_of_7_7_TBps=t_mem / count_s,
        popc_model=popc, popc_bound_ms=t_popc * 1e3, share_of_popc_bound=t_popc / count_s,
        bound="HBM" if t_mem >= t_popc else "population count",
    )


def mrmr_end_to_end(x, y, k):
    """One fit, timed by pieces through a timing subclass of the GPU hook."""
    rec = {"calls": []}

    class Timed(_mi.JointColumns):
        def __init__(self, *a, **kw):
            t0 = time.perf_counter()
            super().__init__(*a, **kw)
            rec["open_s"] = time.perf_counter() - t0

        def columns(self, positions):
            t0 = time.perf_counter()
            out, st = self._ds.joint_columns(self.kind, self.log_base, positions, want_stats=True)
            rec["calls"].append((time.perf_counter() - t0, st))
            return out

    saved = _mi.open_joint_columns
    _mi.open_joint_columns = lambda codes, kind, log_base=1.0: Timed(codes, kind, log_base)
    try:
        t0 = time.perf_counter()
        est = fsb.mRMR(n_features_to_select=k, pairs="selected").fit(x, y)
        total = time.perf_counter() - t0
    finally:
        _mi.open_joint_columns = saved
    t0 = time.perf_counter()
    np.unique(np.concatenate([np.unique(x), np.unique(y)]))
    uniq = time.perf_counter() - t0
    t0 = time.perf_counter()
    _mi._stack_for_upload(x, y)
    stack = time.perf_counter() - t0
    walls = np.array([c[0] for c in rec["calls"]])
    sts = [c[1] for c in rec["calls"]]
    encode_ms = sts[0]["ms_gather"]
    calls_s = float(walls.sum())
    return est, dict(
        n=x.shape[0], p=x.shape[1], k=k, fit_s=total, np_unique_s=uniq, stack_for_upload_s=stack,
        upload_and_column_scan_s=rec["open_s"], encode_first_call_ms=encode_ms,
        column_calls=len(walls), column_calls_wall_s=calls_s,
        column_calls_count_kernel_ms=float(sum(s["ms_dist_general"] for s in sts)),
        column_calls_finish_kernel_ms=float(sum(s["ms_reduce"] for s in sts)),
        column_calls_device_ms=float(sum(s["ms_total"] for s in sts)),
        host_rest_s=total - uniq - stack - rec["open_s"] - calls_s,
        note="np_unique_s and stack_for_upload_s are timed separately on the same arrays after the fit; "
             "host_rest_s = fit_s minus every other piece (the greedy loop, validation)",
    )


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "joint_columns.json"))
    ap.add_argument("--quick", action="store_true", help="small shapes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    if _native.device_count() < 1:
        raise SystemExit("bench_joint_columns: no usable sm_100 GPU")
    info = gpu_info()
    clk_hz = float(info["clocks_max_sm"].split()[0]) * 1e6
    sms = 148
    try:
        import torch

        sms = torch.cuda.get_device_properties(0).multi_processor_count
    except Exception:
        pass
    res = dict(gpu=info, sms=sms, hbm_datasheet_Bps=HBM_BPS, quick=args.quick)
    rng = np.random.default_rng(7)
    s = 20 if args.quick else 1

    # warm the library once (module load, pools)
    ds_warm = open_codes(genotypes(rng, 500, 100))
    ds_warm.joint_columns(0, 1.0, [0])
    ds_warm.close()

    shapes = [(4000, 100_000), (20_000, 200_000)]
    res["kernels"] = []
    for n, p in shapes:
        n_, p_ = max(n // s, 64), max(p // s, 64)
        codes = genotypes(rng, n_, p_ + 1)
        res["kernels"].append(kernel_times(codes, "genotype", clk_hz, sms))
        del codes
    n_, p_ = max(4000 // s, 64), max(20_000 // s, 64)
    codes = rng.integers(0, 16, (n_, p_ + 1), dtype=np.uint8)
    res["kernels"].append(kernel_times(codes, "16-state", clk_hz, sms))
    del codes

    # mRMR end to end + parity at 4000 x 100 000
    n_, p_ = max(4000 // s, 64), max(100_000 // s, 64)
    x = genotypes(rng, n_, p_)
    y = ((x[:, 17] == 2) ^ (rng.random(n_) < 0.2)).astype(np.uint8)
    mrmr_end_to_end(x[:200, :300], y[:200], 5)              # warm
    runs = []
    for _ in range(2):
        est, piece = mrmr_end_to_end(x, y, 50)
        runs.append(piece)
    res["mrmr_selected_end_to_end"] = runs
    from oracle import ref_oracle as R

    cols = np.random.RandomState(1).choice(p_, 64, replace=False)
    xi = x[:, cols].astype(np.int32)
    rel = R.mi_matrices(xi, y.astype(np.int32), want_matrix=False)[0]
    par = dict(n=n_, p=p_, columns=cols.tolist(), relevance_max_rel_err=float(np.max(
        np.abs(est.relevance_scores_[cols] - rel) / np.maximum(np.abs(rel), 1e-300))),
               relevance_max_abs_err=float(np.max(np.abs(est.relevance_scores_[cols] - rel))),
               relevance_allclose_rtol_1e_11_atol_1e_15=bool(np.allclose(est.relevance_scores_[cols], rel, rtol=1e-11, atol=1e-15)))
    for i in range(2):
        f = int(est.top_features_[i])
        red = R.mi_matrices(xi, x[:, f].astype(np.int32), want_matrix=False)[0]
        red[cols == f] = 0.0
        got = est.redundancy_columns_[i, cols]
        par[f"redundancy_of_selected_{i}_max_rel_err"] = float(np.max(np.abs(got - red) / np.maximum(np.abs(red), 1e-300)))
        par[f"redundancy_of_selected_{i}_max_abs_err"] = float(np.max(np.abs(got - red)))
    par["top_features_first_5"] = est.top_features_[:5].tolist()
    res["parity_4000x100000"] = par
    del x

    # pairs="all" vs pairs="selected" at J1's shape, alternated
    n_, p_ = max(10_000 // s, 64), max(10_000 // s, 64)
    x = genotypes(rng, n_, p_)
    y = ((x[:, 3] + x[:, 5000 % p_]) > 2).astype(np.uint8)
    fsb.mRMR(10, pairs="all").fit(x, y)
    fsb.mRMR(10, pairs="selected").fit(x, y)
    times = {"all": [], "selected": []}
    tops = {}
    for _ in range(3):
        for mode in ("all", "selected"):
            t0 = time.perf_counter()
            e = fsb.mRMR(10, pairs=mode).fit(x, y)
            times[mode].append(time.perf_counter() - t0)
            tops[mode] = e
    a, b = tops["all"], tops["selected"]
    res["j1_all_vs_selected"] = dict(
        n=n_, p=p_, k=10, fit_s=times, median_s={m: float(np.median(v)) for m, v in times.items()},
        same_top_features=bool(np.array_equal(a.top_features_, b.top_features_)),
        relevance_bitwise_equal=bool(np.array_equal(a.relevance_scores_, b.relevance_scores_)),
        redundancy_columns_bitwise_equal=bool(np.array_equal(a.redundancy_matrix_[a.top_features_], b.redundancy_columns_)),
    )
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print(json.dumps({k: res[k] for k in ("gpu", "j1_all_vs_selected")}, default=float))
    for kt in res["kernels"]:
        print(kt["label"], kt["n"], kt["columns"], "count ms", kt["median_ms"]["count"], "share HBM",
              kt["share_of_7_7_TBps"], "bound", kt["bound"])


if __name__ == "__main__":
    main()
