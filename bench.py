#!/usr/bin/env python
"""bench.py -- MultiSURF fit throughput (sample-pair*features/s) on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c3|c2|c4|c5|j1]
                    [--dump-outputs DIR]

A "step" is one pass of the scoring hot path (encode of the active columns, n x n
distances, neighbour selection, weight accumulation, reduction) over one synthetic data
set.  `value` is measured with the raw matrix already resident in HBM; `e2e` is the same
metric through the estimator API (`MultiSURF(backend='gpu').fit`) from host buffers, with
the host->device upload, the on-GPU column scan and the device->host read of the weights
inside the timed region.

The inputs are seeded: the same arguments give the same data on every run, so the outputs that
--dump-outputs writes can be compared between two builds.

Default workload (BASELINE.json configs[2], the config the metric's "1/2/4/8 B200" is
quoted on): MultiSURF on synthetic 0/1/2 genotypes, 4000 samples x 100000 SNPs, epistatic
label (SURVEY.md 8d C3).  With N > 1 GPUs (one process per GPU under torchrun) the target
rows are sharded across ranks and the partial weight vectors are combined by one NCCL
allreduce; weak scaling keeps the per-GPU work (rows_per_gpu x n x p) fixed by growing n
with sqrt(N).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (no __pycache__ of tests/ etc.)

METRIC = "multisurf_fit_pair_features_per_s"
UNIT = "sample-pair*features/s"
WORKLOAD_SHAPES = {"c3": (4000, 100_000), "c2": (10_000, 10_000), "c4": (20_000, 50_000), "c4surf": (20_000, 50_000),
                   "c5": (20_000, 500_000)}
DUMP_BYTES = 64 << 20


# --------------------------------------------------------------------------- #
# workloads (SURVEY.md 8d)
# --------------------------------------------------------------------------- #
def make_workload(name, n_gpus, scaling, n_override=None, p_override=None, rows=None):
    from datasets import epistatic_genotypes

    if name == "c5":
        return make_c5(n_override or 20_000, p_override or 500_000, rows)
    if name == "c3":
        n, p = 4000, 100_000
        algo, star = "MultiSURF", False
    elif name == "c2":
        n, p = 10_000, 10_000
        algo, star = "ReliefF", False
    elif name == "c4":
        n, p = 20_000, 50_000
        algo, star = "MultiSURF", True
    elif name == "c4surf":
        n, p = 20_000, 50_000
        algo, star = "SURF", True
    else:
        raise SystemExit(f"unknown workload {name}")
    if n_override:
        n = n_override
    if p_override:
        p = p_override
    if scaling == "weak" and n_gpus > 1:
        n = int(round(n * np.sqrt(n_gpus) / 8.0)) * 8
    if name == "c3":
        x, y = epistatic_genotypes(42, n, p)
        desc = f"C3: MultiSURF on int8 0/1/2 genotypes {n} samples x {p} SNPs, epistatic label"
    elif name == "c2":
        from sklearn.datasets import make_classification

        x, y = make_classification(n_samples=n, n_features=p, n_informative=20, n_redundant=100, random_state=42)
        desc = f"C2: ReliefF k=10 on continuous make_classification {n} x {p}"
    else:
        rs = np.random.RandomState(43)
        x = np.empty((n, p), np.float32)
        h = p // 2
        x[:, :h] = rs.randint(0, 3, (n, h))
        x[:, h:] = rs.standard_normal((n, p - h)).astype(np.float32)
        y = np.zeros(n, np.int64)
        y[(x[:, 25 % h] == 1) & (x[:, 75 % h] == 1)] = 1
        need = n // 2 - int(y.sum())
        y[rs.choice(np.flatnonzero(y == 0), need, replace=False)] = 1
        x[:, h] += 1.0 * y
        if name == "c4surf":
            x = x.astype(np.float64)           # SURF validates X to float64 (SURF.py:330-332)
            desc = f"C4: SURF* on mixed float64 {n} x {p} (half genotype, half gaussian)"
        else:
            desc = f"C4: MultiSURF* on mixed {n} x {p} (half genotype, half gaussian)"
    return dict(name=name, x=x, y=y, n=n, p=p, algo=algo, star=star, desc=desc)


def make_c5(n, p, rows=None):
    """SURVEY.md 8(d) C5: int8 0/1/2 genotypes n x p, epistatic label on SNPs 25 and 75, for
    TuRF(MultiSURF, pct_remove=0.1).  Generated in independent 1000-row blocks (seed = [44, block])
    so that the CPU arm can build just the first `rows` samples of the very same matrix."""
    m = n if rows is None else min(rows, n)
    x = np.empty((m, p), np.int8)
    for b0 in range(0, m, 1000):
        b1 = min(b0 + 1000, m)
        x[b0:b1] = np.random.default_rng([44, b0 // 1000]).integers(0, 3, size=(b1 - b0, p), dtype=np.int8)
    rs = np.random.RandomState(44)
    y = np.zeros(m, np.int64)
    y[(x[:, 25 % p] == 1) & (x[:, 75 % p] == 1)] = 1
    need = m // 2 - int(y.sum())
    if need > 0:
        y[rs.choice(np.flatnonzero(y == 0), need, replace=False)] = 1
    desc = f"C5: TuRF(MultiSURF, pct_remove=0.1) on int8 0/1/2 genotypes {n} samples x {p} SNPs, epistatic label"
    return dict(name="c5", x=x, y=y, n=n, p=p, algo="MultiSURF", star=False, desc=desc)


def turf_schedule(p, n_select=10, pct=0.1):
    """Column counts of every scoring pass of TuRF (TuRF.py:94-113): the first fit and one per iteration."""
    sizes, cur = [p], p
    while cur > n_select:
        k = max(1, int(cur * pct))
        if cur - k < n_select:
            k = cur - n_select
        cur -= k
        sizes.append(cur)
    return sizes


def make_estimator(w):
    import fastselect_b200 as fsb

    if w["algo"] == "ReliefF":
        return fsb.ReliefF(n_features_to_select=10, n_neighbors=10, backend="gpu")
    if w["algo"] == "SURF":
        return fsb.SURF(n_features_to_select=10, backend="gpu", use_star=w["star"])
    return fsb.MultiSURF(n_features_to_select=10, backend="gpu", use_star=w["star"])


# --------------------------------------------------------------------------- #
# clocks during the timed region
# --------------------------------------------------------------------------- #
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region: NVML polled every 2 ms from a side
    thread (the timed region of the default workload lasts ~25 ms, too short for nvidia-smi)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.max_mhz = index, threading.Event(), [], None
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _sample(self):
        if self.nvml is not None:
            n = self.nvml
            mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            try:
                mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            self.samples.append((mhz, mask))
            return 0.002
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout
        parts = [t.strip() for t in out.strip().split(",")]
        if len(parts) >= 6:
            self.max_mhz = float(parts[1])
            mask = sum(bit for bit, col in ((0x8, 2), (0x40, 3), (0x20, 4), (0x4, 5)) if parts[col].lower().startswith("active"))
            self.samples.append((float(parts[0]), mask))
        return 0.05

    def run(self):
        while not self.stop_flag.is_set():
            try:
                wait = self._sample()
            except Exception:
                wait = 0.05
            self.stop_flag.wait(wait)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        sm = sorted(m for m, _ in self.samples)
        mask = 0
        for _, m in self.samples:
            mask |= m
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": [nm for bit, nm in self.REASONS.items() if mask & bit], "samples": len(sm),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# --------------------------------------------------------------------------- #
# CPU baseline (oracle port on a bounded sample)
# --------------------------------------------------------------------------- #
def cpu_sample(w, units=2.0e10):
    """Bounded CPU sample of the workload: ALL n samples (the neighbour statistics depend on n) and the
    first p_s columns, p_s sized for about `units` sample-pair*features (~10 s on 16 host threads)."""
    n_s = min(w["n"], w["x"].shape[0])
    p_s = int(max(32, min(w["p"], units / (float(n_s) * n_s))))
    return w["x"][:n_s, :p_s], w["y"][:n_s], n_s, p_s


def run_cpu_port(w, xs, ys):
    """One timed pass of the oracle (C restatement of the reference CPU kernel, OpenMP over
    target instances like the reference's prange); returns (seconds, feature scores)."""
    from oracle import ref_oracle as R

    if w["algo"] == "ReliefF":
        x32, y_enc, cp, recip, isd = R.relieff_prep(xs, ys, 10)
        t0 = time.perf_counter()
        scores = R.relieff_scores(x32, y_enc, recip, isd, 10, cp, 0)
    elif w["algo"] == "SURF":
        x64, recip, isd = R.surf_prep(xs, 10)
        y32 = np.asarray(ys).astype(np.int32)
        t0 = time.perf_counter()
        scores = R.surf_scores(x64, y32, recip, isd, w["star"], sum_mode=2)
    else:
        x32, recip, isd = R.multisurf_prep(xs, 10)
        yc = np.unique(ys, return_inverse=True)[1].astype(np.int64)
        t0 = time.perf_counter()
        scores = R.multisurf_scores(x32, yc, recip, isd, w["star"])
    return time.perf_counter() - t0, scores


def cpu_baseline(w):
    from oracle import ref_oracle as R

    R.set_threads(os.cpu_count() or 1)
    xs, ys, n_s, p_s = cpu_sample(w)
    dt, _ = run_cpu_port(w, xs, ys)
    return {"value": n_s * n_s * p_s / dt, "unit": UNIT, "cores": R.max_threads(), "kind": "port",
            "sample": f"all {n_s} samples x first {p_s} features of the workload, one fit, {dt:.2f} s"}


def reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port: the
    reference is Python/Numba and does not travel to the GPU box) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_oracle as R

    R.build()
    R.set_threads(os.cpu_count() or 1)
    # the same n as the own arm's single-GPU workload; only as many columns as a bounded CPU step needs
    n_full, p_full = WORKLOAD_SHAPES[args.workload]
    n_full, p_full = args.n or n_full, args.p or p_full
    p_gen = int(max(32, min(p_full, 2.0e10 / (float(n_full) * n_full))))
    w = make_workload(args.workload, 1, "weak", n_full, p_gen)
    xs, ys, n_s, p_s = cpu_sample(w)
    for _ in range(args.warmup):
        run_cpu_port(w, xs[:200], ys[:200])
    t = 0.0
    for _ in range(args.steps):
        dt, scores = run_cpu_port(w, xs, ys)
        t += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"feature_importances": scores})
    value = args.steps * n_s * n_s * p_s / t
    desc = w["desc"].replace(f"x {p_gen}", f"x {p_full}")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64 (CPU)",
            "data": "synthetic",
            "config": {"workload": desc + f" -- CPU sample per step: all {n_s} samples x first {p_s} features "
                                          "(throughput in the same unit; the full width would take hours)",
                       "n": n_full, "p": p_full, "sample_n": n_s, "sample_p": p_s},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": R.max_threads(), "kind": "port",
                             "sample": f"all {n_s} samples x first {p_s} features per step"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def load_traffic(workload):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of each kernel from the
    committed `ncu --set full` capture of this workload (profiles/traffic.json), keyed by phase."""
    if workload is None:
        return {}
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(workload, {})
    except Exception:
        return {}


def dump_outputs(out_dir, outputs):
    """--dump-outputs: each output of the timed path's last step (a numpy array, or a torch tensor left on
    the device) as out_dir/<name>.npy in float32 or float64, DUMP_BYTES at most in all.  An output larger
    than its share is replaced by the flat sample of the entries at np.unique(default_rng(0).integers(0,
    size, share // 8)): fixed for a given shape, so two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(outputs)
    for name, a in outputs.items():
        size = int(np.prod(a.shape))
        if size * 8 > share:
            pos = np.unique(np.random.default_rng(0).integers(0, size, share // 8))
            if isinstance(a, np.ndarray):
                a = a.reshape(-1)[pos]
            else:
                import torch

                a = a.reshape(-1)[torch.from_numpy(pos).to(a.device)]
        a = np.asarray(a) if isinstance(a, np.ndarray) else a.cpu().numpy()
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# --------------------------------------------------------------------------- #
# own arm
# --------------------------------------------------------------------------- #
def init_ranks():
    """One process per GPU under torchrun (NCCL only carries the 64-byte arena handles); returns
    (rank, local_rank, world, barrier)."""
    import torch
    import torch.distributed as dist

    import fastselect_b200 as fsb
    from fastselect_b200 import _native

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    _native.load()
    if _native.device_count() < 1:
        raise SystemExit("bench.py: no usable sm_100 GPU (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    os.environ["FASTSELECT_B200_DEVICE"] = str(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        fsb.enable_distributed()          # every rank fits the SAME X, y: shard the fit across the group

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    return rank, local_rank, world, barrier


def load_peaks():
    """Roofline denominators: MEASURED_PEAKS.json (driver-written: HBM copy, cuBLAS bf16) and the FP4
    tensor peak measured with tools/fp4_peak.cu on this pool's B200 (profiles/r02_fp4_peak.json)."""
    peaks, fp4 = {}, {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    try:
        for sh in json.load(open(os.path.join(ROOT, "profiles", "r02_fp4_peak.json")))["shapes"]:
            if sh["cta_group"] == 1 and sh["n"] == 256:
                fp4 = {"burst": 1e3 * sh["burst_pops"], "sustained": 1e3 * sh["sustained_pops"]}
    except Exception:
        pass
    return peaks, fp4


def fp4_denominator(peaks, fp4, burst):
    if fp4:
        return fp4["burst" if burst else "sustained"], ("measured tcgen05 kind::mxf4 peak, %s (tools/fp4_peak.cu, profiles/r02_fp4_peak.json)"
                                                        % ("burst" if burst else "sustained 4 s"))
    bf16 = peaks.get("bf16_tflops" if burst else "bf16_tflops_sustained", 1590.0 if burst else 1400.0)
    return 4.0 * bf16, "4 x cuBLAS bf16 (no measured FP4 peak file)"


def parity_check(w, est_factory, weights, world, rank, barrier, n_targets=16):
    """The timed run's weights against (a) the other ranks' (must be identical), (b) a plain single-GPU
    run of the same data on rank 0 (bitwise for one-hot columns), (c) the CPU oracle on `n_targets`
    targets through fs_debug_rows on rank 0."""
    import torch
    import torch.distributed as dist

    import fastselect_b200 as fsb
    from fastselect_b200 import _native
    from oracle import ref_oracle as R

    out = {"ranks_identical": True}
    if world > 1:
        t = torch.from_numpy(weights.astype(np.float64)).cuda()
        hi, lo = t.clone(), t.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        out["ranks_identical"] = bool(torch.equal(hi, lo))
    if rank == 0:
        fsb.enable_distributed(False)              # a plain one-GPU session on rank 0; the other ranks wait
        try:
            R.set_threads(os.cpu_count() or 1)
            sess, _ = est_factory()._open_session(w["x"], w["y"])
            with sess:
                single = sess.score()
                tg = np.sort(np.random.RandomState(7).choice(w["n"], min(n_targets, w["n"]), replace=False))
                got = sess.ds.debug_rows(sess.algo, tg, use_star=sess.use_star, k=sess.k, class_probs=sess.class_probs)
                x_dev_dtype = w["x"]
            out["equals_single_gpu"] = "bitwise" if np.array_equal(single, weights) else (
                "allclose(rtol 1e-6)" if np.allclose(single, weights, rtol=1e-6, atol=1e-9) else "MISMATCH")
            if w["algo"] == "MultiSURF" and x_dev_dtype.dtype in (np.int8, np.uint8):
                want = R.multisurf_targets_bytes(w["x"], w["y"], w["star"], tg)
            elif w["algo"] == "MultiSURF":
                x32, recip, isd = R.multisurf_prep(w["x"], 10)
                want = R.multisurf_targets(x32, np.unique(w["y"], return_inverse=True)[1], recip, isd, w["star"], tg)
            elif w["algo"] == "SURF":
                x64, recip, isd = R.surf_prep(w["x"], 10)
                want = R.surf_targets(x64, np.asarray(w["y"]).astype(np.int32), recip, isd, w["star"], tg, sum_mode=2)
            else:
                x32, y_enc, cp, recip, isd = R.relieff_prep(w["x"], w["y"], 10)
                want = R.relieff_targets(x32, y_enc, recip, isd, 10, cp, tg, tie_mode=0)
            ok = bool(np.array_equal(got["mask"], want["mask"])) and bool(
                np.allclose(got["wsum"], want["wsum"], rtol=1e-5, atol=1e-7 * len(tg) * max(1.0, float(np.abs(want["wsum"]).max()))))
            exact = bool(np.array_equal(got["dist"], want["dist"]))
            out.update(oracle_targets=int(len(tg)), oracle_neighbour_sets_and_weights="ok" if ok else "MISMATCH",
                       oracle_distances="bit-exact" if exact else
                       ("allclose(rtol 2e-7)" if np.allclose(got["dist"], want["dist"], rtol=2e-7, atol=1e-12) else "MISMATCH"))
        finally:
            fsb.enable_distributed(world > 1)
    barrier()
    out["ok"] = bool(out["ranks_identical"]) and "MISMATCH" not in json.dumps(out)
    return out


def own_arm(args):
    import torch
    import torch.distributed as dist

    from fastselect_b200 import _native
    from fastselect_b200._shard import shard_rows

    rank, local_rank, world, barrier = init_ranks()
    if args.gpus != world and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
    w = make_workload(args.workload, world, args.scaling, args.n, args.p)
    n, p = w["n"], w["p"]
    est = make_estimator(w)
    peaks, fp4 = load_peaks()

    # ---- resident-data timing: the estimator's own session, kept open
    # host inputs live in pinned memory, so the e2e leg's upload runs at PCIe speed
    x_pinned = torch.from_numpy(w["x"]).pin_memory()
    x_in = x_pinned.numpy()
    sess, _ = est._open_session(x_in, w["y"])         # N > 1: collective (1 / N of X uploaded per rank, NVLink replication)
    collective = bool(sess.collective)
    lo, hi = sess.ds.shard if collective else shard_rows(n, world, rank, sess.row_align)
    buf = torch.empty(p, dtype=torch.float64, device=torch.device("cuda", local_rank))
    last_stats = {}

    def step():
        # set_features invalidates the cached working set: every step re-encodes the columns
        sess.ds.set_features(sess.is_discrete, sess.recip, sess.arith)
        nonlocal last_stats
        _, last_stats = sess.ds.score(sess.algo, sess.use_star, sess.k, sess.class_probs, None, lo, hi,
                                      out_device_ptr=buf.data_ptr(), want_stats=True)
        if world > 1 and not collective:
            dist.all_reduce(buf)          # fallback without peer access: partial sums over the rank's rows

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    agg = {}
    e0.record()
    for _ in range(args.steps):
        step()
        for k_, v in last_stats.items():
            agg[k_] = agg.get(k_, 0) + v
    e1.record()
    barrier()
    sampler.stop_flag.set()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"weight_sums": buf})
    units = float(n) * n * p
    value = units * args.steps / (ms / 1e3)
    weights = (buf.cpu().numpy() / n).astype(np.float32)
    sess.close()

    # ---- end to end through the estimator API from host buffers
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(2 if n * p <= 2_000_000_000 else 1):
        make_estimator(w).fit(x_in, w["y"])        # untimed full-size fits: device pool, arenas and pinned staging grown
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fitted = make_estimator(w).fit(x_in, w["y"])
    barrier()
    dt = time.perf_counter() - t0
    # the same from PAGEABLE host memory (what a caller's numpy array usually is)
    x_page = np.array(x_in)
    make_estimator(w).fit(x_page, w["y"])       # untimed: like the timed steps above, the pageable fit is measured warm
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        make_estimator(w).fit(x_page, w["y"])
    barrier()
    dt_page = (time.perf_counter() - t0) / e2e_steps
    del x_page
    tt = torch.tensor([dt, dt_page], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt, dt_page = float(tt[0].item()), float(tt[1].item())
    e2e_value = units * e2e_steps / dt
    rows_up = n // world if collective else n           # rows this rank copies over PCIe
    h2d = int(rows_up * x_in.shape[1] * x_in.itemsize + 4 * n + p * 5 + p * 4)
    d2h = int(p * (8 + 8 + 4) + p * 8)
    same = bool(np.array_equal(fitted.feature_importances_, weights))

    # ---- parity of the timed run (every rank takes part in the collectives; rank 0 runs the checks)
    w_in = dict(w, x=x_in)
    parity = parity_check(w_in, lambda: make_estimator(w), weights, world, rank, barrier) if not args.no_parity else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines (per-phase CUDA events from fs_stats, on the stream the kernels run on)
    steps = args.steps
    phases = {k_: agg.get(k_, 0.0) / steps for k_ in ("ms_gather", "ms_dist_tensor", "ms_dist_general", "ms_select",
                                                      "ms_accum_tensor", "ms_accum_general", "ms_reduce", "ms_total",
                                                      "ms_host_prep")}
    rows = hi - lo
    clk = sampler.summary()
    burst = (ms / steps) < 100.0          # millisecond-scale kernels: burst peak; second-scale steps: sustained
    fp4_peak, peak_src = fp4_denominator(peaks, fp4, burst)
    hbm = peaks.get("hbm_gbs", 6650.0)
    traffic = load_traffic(args.workload if world == 1 else None)
    st_avg = {k_: agg.get(k_, 0) / steps for k_ in ("n_tensor_cols", "n_general_cols", "onehot_k", "pairs_selected")}
    pt, pg, kk = st_avg["n_tensor_cols"], st_avg["n_general_cols"], st_avg["onehot_k"]
    kernels = {}
    # tensor kernels.  USEFUL operations = the contraction the algebra needs (2 per MAC): distances
    # rows x n x K over the reduced one-hot rows, halved when the symmetric half is skipped; accumulation
    # this rank's one-hot rows x all their (target, sample) pairs once.  ISSUED = what went to the tensor
    # pipe (tile padding included; fs_stats).  SURVEY 8(d)'s symmetric-free 3-plane figure (6 ops/u) beside.
    k_acc = kk / world if collective and w["algo"] != "ReliefF" else kk
    r_acc = n if collective and w["algo"] != "ReliefF" else rows
    useful = {"ms_dist_tensor": 2.0 * rows * n * kk * (0.5 if (world == 1 or collective) else 1.0),
              "ms_accum_tensor": 2.0 * k_acc * r_acc * n}
    for ph, key in (("ms_dist_tensor", "ops_dist_tensor"), ("ms_accum_tensor", "ops_accum_tensor")):
        if phases[ph] > 0 and agg.get(key, 0) > 0:
            sec = phases[ph] / 1e3
            ach = useful[ph] / sec / 1e12
            kernels[ph] = {"bound": "tensor", "achieved": ach, "peak": fp4_peak, "unit": "TOP/s fp4 (e2m1, exact integers)",
                           "frac": ach / fp4_peak, "issued_rate": agg[key] / steps / sec / 1e12,
                           "survey_algorithmic_rate": 6.0 * rows * n * pt / sec / 1e12, "traffic": traffic.get(ph)}
    if phases["ms_gather"] > 0 and kk > 0:
        # encode: raw columns read once; U (this rank's rows), Wd (all rows) and this rank's share of At as FP4
        # nibbles (K / 2 bytes per sample) and of codesT written once
        share = 1.0 / world if collective and w["algo"] != "ReliefF" else 1.0
        byts = n * pt * w["x"].itemsize * (1.0 + (share if share < 1 else 0.0)) + (rows + n) * kk / 2.0 + share * (n * kk / 2.0 + n * pt)
        gbs = byts / (phases["ms_gather"] / 1e3) / 1e9
        kernels["ms_gather"] = {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                                "traffic": traffic.get("ms_gather"), "note": "time includes the host-side working-set preparation (ms_host_prep)"}
    # CUDA-core kernels: FP32-lane issue rate (SURVEY 8d): 2 lane-instructions per (pair, continuous feature)
    # for distances, 2 per SELECTED pair and feature for the accumulation, against SMs x 128 lanes x clock
    clock_mhz = clk.get("sm_mhz") or clk.get("sm_max_mhz") or 1965.0
    issue_peak = 148 * 128 * clock_mhz * 1e6 / 1e12                       # T lane-instr/s at the clock sampled under load
    if phases["ms_dist_general"] > 0 and pg > 0:
        ach = 2.0 * rows * n * pg / (phases["ms_dist_general"] / 1e3) / 1e12
        kernels["ms_dist_general"] = {"bound": "fp32-issue", "achieved": ach, "peak": issue_peak, "unit": "T lane-instr/s",
                                      "frac": ach / issue_peak, "traffic": traffic.get("ms_dist_general"),
                                      "note": "2 algorithmic lane-instructions per (ordered pair, continuous feature); symmetric tiles evaluate half of the pairs"}
    if phases["ms_accum_general"] > 0 and pg > 0:
        if w["algo"] == "ReliefF":
            byts = st_avg["pairs_selected"] * pg * 4.0
            gbs = byts / (phases["ms_accum_general"] / 1e3) / 1e9
            kernels["ms_accum_general"] = {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                                           "traffic": traffic.get("ms_accum_general"),
                                           "note": "ReliefF sparse gather: bytes of the selected neighbours' rows (n k C p x 4); mostly L2 hits"}
        else:
            ach = 2.0 * st_avg["pairs_selected"] * pg / (phases["ms_accum_general"] / 1e3) / 1e12
            kernels["ms_accum_general"] = {"bound": "fp32-issue", "achieved": ach, "peak": issue_peak, "unit": "T lane-instr/s",
                                           "frac": ach / issue_peak, "traffic": traffic.get("ms_accum_general"),
                                           "note": "2 algorithmic lane-instructions per (selected pair, continuous feature)"}
    top = max((q for q in ("ms_dist_tensor", "ms_dist_general", "ms_accum_tensor", "ms_accum_general") if q in kernels),
              key=lambda q: phases[q])
    roof = dict(kernels[top], kernel=top,
                peak_source=peak_src if kernels[top]["bound"] == "tensor" else
                ("148 SMs x 128 FP32 lanes x %.0f MHz (SM clock sampled during the timed region)" % clock_mhz
                 if kernels[top]["bound"] == "fp32-issue" else "measured copy (MEASURED_PEAKS.json)"))

    # the CPU baseline is reported at N = 1 only (rank 0)
    cpu = cpu_baseline(w) if world == 1 and not os.environ.get("FS_BENCH_SKIP_CPU") else None   # (kernel experiments skip the CPU leg)
    sharding = f"target rows x{world}"
    if collective:
        sharding += (", symmetric distance tiles / neighbour masks / weight slices stored into the peers' arenas over NVLink, "
                     "accumulation sharded by one-hot columns, device-side barriers; 1/N of X uploaded per rank")
    elif world > 1:
        sharding += ", one NCCL allreduce"
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak",
            "vs_baseline": None, "dtype": "e2m1 (FP4) one-hot / exact FP32 accum (genotype), f32 terms + f64 accum (continuous)",
            "data": "synthetic",
            "config": {"workload": w["desc"], "n": n, "p": p, "algo": w["algo"] + ("*" if w["star"] else ""),
                       "rows_per_gpu": rows, "sharding": sharding,
                       "l2": "inputs larger than L2 (no flush needed)", "step": "encode + distances + select + accumulate"},
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "seconds_per_fit": dt / e2e_steps, "matches_resident_run": same,
                    "pageable_seconds_per_fit": dt_page, "pageable_value": units / dt_page,
                    "note": "value: X in pinned host memory; pageable_*: the same fit from an ordinary numpy array"},
            "gpu_launches": int(agg.get("launches", 0)),
            "roofline": roof, "kernels": kernels, "phases_ms": phases, "cpu_baseline": cpu, "parity": parity,
            "top_features": fitted.top_features_.tolist(),
            "stats": {k_: int(agg[k_] / steps) for k_ in ("n_tensor_cols", "n_general_cols", "onehot_k",
                                                           "pairs_selected", "n_chunks") if k_ in agg}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def turf_arm(args):
    """--workload c5: one step = one whole TuRF(MultiSURF) run (first fit + every pruning iteration)
    on a resident data set; e2e = TuRF(...).fit from host buffers."""
    import torch
    import torch.distributed as dist

    import fastselect_b200 as fsb

    rank, local_rank, world, barrier = init_ranks()

    t_gen = time.perf_counter()
    w = make_workload("c5", world, "strong", args.n, args.p)
    t_gen = time.perf_counter() - t_gen
    n, p = w["n"], w["p"]
    x_pinned = torch.from_numpy(w["x"]).pin_memory()
    x_in = x_pinned.numpy()
    w["x"] = x_in
    peaks, fp4 = load_peaks()

    def new_turf():
        return fsb.TuRF(fsb.MultiSURF(n_features_to_select=10, backend="gpu"), n_features_to_select=10, pct_remove=0.1)

    sizes = turf_schedule(p)
    units = float(n) * n * float(sum(sizes))

    # ---- resident run: the session stays open, every step is a whole pruning run
    base = fsb.MultiSURF(n_features_to_select=10, backend="gpu")
    sess, _ = base._open_session(x_in, w["y"])
    agg = {}

    def score(active=None):
        out = sess.score(active, want_stats=True)
        for k_, v in (sess.last_stats or {}).items():
            agg[k_] = agg.get(k_, 0) + v
        return out

    def step():
        t = new_turf()
        t.n_features_in_ = p
        t._prune(score(), score)
        return t

    for _ in range(args.warmup):
        score()                          # warm-up: full-width scoring passes (allocations, clocks)
        score(np.arange(p - p // 10))    # and one pruned pass (buffers of the incremental distance update)
    agg.clear()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        resident = step()
    barrier()
    dt = time.perf_counter() - t0
    sampler.stop_flag.set()
    tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    sess.close()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"feature_importances": resident.feature_importances_,
                                         "top_features": resident.top_features_})
    value = units * args.steps / dt

    # ---- end to end: TuRF(...).fit from host buffers (upload, column scan, every pass)
    barrier()
    t0 = time.perf_counter()
    fitted = new_turf().fit(x_in, w["y"])
    barrier()
    de = time.perf_counter() - t0
    tt = torch.tensor([de], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    de = float(tt.item())
    # parity of the run: identical selection on every rank and the two planted SNPs on top
    parity = {"ranks_identical": True}
    if world > 1:
        tf = torch.from_numpy(np.ascontiguousarray(fitted.top_features_, np.int64)).cuda()
        hi_, lo_ = tf.clone(), tf.clone()
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        parity["ranks_identical"] = bool(torch.equal(hi_, lo_))
    parity["planted_snps_selected"] = bool({25, 75} <= set(fitted.top_features_.tolist()))
    parity["note"] = "oracle parity of this shape (16 targets, first and second TuRF pass): tests/test_gpu_shapes_more.py"
    parity["ok"] = parity["ranks_identical"] and parity["planted_snps_selected"]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    steps = args.steps
    phases = {k_: agg.get(k_, 0.0) / steps for k_ in ("ms_gather", "ms_dist_tensor", "ms_select", "ms_accum_tensor",
                                                      "ms_reduce", "ms_total", "ms_host_prep")}
    fp4_peak, peak_src = fp4_denominator(peaks, fp4, burst=False)       # second-scale steps: sustained peak
    kernels = {}
    # useful accumulation work of this rank: 2 ops per (one-hot row, target, sample), rows = 2 per active SNP,
    # sharded by columns across the ranks; the distance kernel's useful work is dominated by the first pass
    useful_acc = 2.0 * 2.0 * float(sum(sizes)) / world * n * n
    useful_dist = 2.0 * 2.0 * (sizes[0] * 0.5 + float(sizes[0] - sizes[-1])) * (n / world) * n
    for ph, key, useful in (("ms_dist_tensor", "ops_dist_tensor", useful_dist), ("ms_accum_tensor", "ops_accum_tensor", useful_acc)):
        sec = phases[ph] / 1e3
        kernels[ph] = {"bound": "tensor", "achieved": useful / sec / 1e12, "peak": fp4_peak, "unit": "TOP/s fp4 (e2m1, exact integers)",
                       "frac": useful / sec / 1e12 / fp4_peak, "issued_rate": agg.get(key, 0.0) / steps / sec / 1e12, "traffic": None}
    top = max(kernels, key=lambda q: phases[q])
    roof = dict(kernels[top], kernel=top, peak_source=peak_src)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "e2m1 (FP4) one-hot / exact FP32 accum (genotype)", "data": "synthetic",
            "config": {"workload": w["desc"], "n": n, "p": p, "algo": "TuRF(MultiSURF)", "scoring_passes": len(sizes),
                       "sum_p_t": int(sum(sizes)), "sharding": f"target rows x{world}" + (", accumulation sharded by one-hot columns, exchanges through the peers' arenas over NVLink, device-side barriers" if world > 1 else ""),
                       "l2": "inputs larger than L2 (no flush needed)",
                       "step": "one whole TuRF run: first fit + every pruning iteration (encode + distances + select + accumulate each)",
                       "timing": "host wall clock around the run (barrier + synchronize both sides), max over ranks",
                       "generate_s": t_gen},
            "clocks": sampler.summary(),
            "e2e": {"value": units / de, "unit": UNIT, "h2d_bytes_per_step": int(x_in.nbytes + 4 * n + 9 * p),
                    "d2h_bytes_per_step": int(20 * p + 8 * sum(sizes)), "steps": 1, "seconds_per_fit": de,
                    "matches_resident_run": bool(np.array_equal(fitted.top_features_, resident.top_features_))},
            "parity": parity,
            "gpu_launches": int(agg.get("launches", 0)), "roofline": roof, "kernels": kernels, "phases_ms": phases,
            "cpu_baseline": None, "top_features": fitted.top_features_.tolist(), "seconds_per_turf_run": dt / steps}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()

# --------------------------------------------------------------------------- #
# joint-count path (SURVEY.md 8(f)-4): --workload j1
# --------------------------------------------------------------------------- #
J_METRIC = "mi_matrices_sample_feature_pairs_per_s"
J_UNIT = "samples*feature-pairs/s"


def make_j1(n, p):
    """J1: the matrices mRMR needs (relevance + p x p redundancy, mutual_information.py:158-196) on 0/1/2
    genotypes with a binary class; unit of work = one sample of one unordered column pair of [X | y]."""
    rs = np.random.RandomState(45)
    x = rs.randint(0, 3, (n, p)).astype(np.uint8)
    y = ((x[:, 25 % p] == 1) & (x[:, 75 % p] == 1)).astype(np.uint8) ^ (rs.random_sample(n) < 0.1).astype(np.uint8)
    return {"n": n, "p": p, "x": x, "y": y,
            "desc": f"J1: mutual-information matrices (mRMR) of {n} x {p} synthetic 0/1/2 genotypes + binary class"}


def joint_cpu(x, y, threads):
    """One timed pass of the oracle's MI matrices (the C restatement of _batch_mi_cpu, OpenMP over
    features like the reference's prange) on [x | y]; returns (seconds, (relevance, redundancy))."""
    from oracle import ref_oracle as R

    R.set_threads(threads)
    xi = np.ascontiguousarray(x, np.int32)
    yi = np.ascontiguousarray(y, np.int32)
    t0 = time.perf_counter()
    out = R.mi_matrices(xi, yi)
    return time.perf_counter() - t0, out


def joint_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_oracle as R

    R.build()
    threads = os.cpu_count() or 1
    n, p = args.n or 10_000, args.p or 10_000
    n_s, p_s = min(n, 10_000), min(p, 4000)       # ~4 s of CPU work per step on 16 threads
    w = make_j1(n_s, p_s)
    for _ in range(args.warmup):
        joint_cpu(w["x"][:200, :100], w["y"][:200], threads)
    t = 0.0
    for _ in range(args.steps):
        dt, (rel, red) = joint_cpu(w["x"], w["y"], threads)
        t += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"relevance": rel, "redundancy": red})
    units = float(n_s) * (p_s + 1) * p_s / 2
    value = args.steps * units / t
    line = {"impl": "reference", "metric": J_METRIC, "value": value, "unit": J_UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64 (CPU)",
            "data": "synthetic", "config": {"workload": make_j1(4, 4)["desc"].replace("4 x 4", f"{n} x {p}"), "n": n, "p": p},
            "cpu_baseline": {"value": value, "unit": J_UNIT, "cores": R.max_threads(), "kind": "port",
                             "sample": f"{n_s} samples x {p_s} features per step"},
            "e2e": {"value": value, "unit": J_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def joint_arm(args):
    """--workload j1: one step = fs_joint_matrix over the resident data set (encode of every column,
    marginals, the At * At^T GEMM bands, the finishing kernel; result left on the device);
    e2e = mutual_information.calculate_mi_matrices from host buffers (upload, column scan, the step,
    the p x p result copied back)."""
    import torch
    import torch.distributed as dist

    import fastselect_b200 as fsb
    from fastselect_b200 import _mi, _native
    from fastselect_b200._shard import shard_triangle

    rank, local_rank, world, barrier = init_ranks()

    w = make_j1(args.n or 10_000, args.p or 10_000)
    n, p = w["n"], w["p"]
    q = p + 1
    units = float(n) * q * (q - 1) / 2
    xa = torch.from_numpy(_mi._stack_for_upload(w["x"], w["y"])).pin_memory().numpy()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    ds = _native.Dataset(xa, np.zeros(n, np.int32), 1)
    ones8, ones32 = np.ones(q, np.uint8), np.ones(q, np.float32)
    lo, hi = shard_triangle(q, world, rank)
    buf = torch.empty((q, q), dtype=torch.float64, device="cuda")
    agg = {}

    def step():
        ds.set_features(ones8, ones32, _native.FS_ARITH_F32)       # invalidates the working set: every step re-encodes
        _, st = ds.joint_matrix(_native.FS_JOINT_MI, np.log(2.0), pos_begin=lo, pos_end=hi,
                                out_device_ptr=buf.data_ptr(), want_stats=True)
        if world > 1:
            dist.all_reduce(buf)
        for k_, v in st.items():
            agg[k_] = agg.get(k_, 0) + v

    for _ in range(args.warmup):
        step()
    agg.clear()
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    sampler.stop_flag.set()
    tt = torch.tensor([e0.elapsed_time(e1) / 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    check = buf[p, :p].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"relevance": buf[p, :p], "mi_matrix": buf})
    ds.close()

    # ---- end to end through the public API, from host buffers
    x_in, y_in = w["x"], w["y"]
    fsb.mutual_information.calculate_mi_matrices(x_in[:, :256], y_in, backend="gpu")
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rel, red = fsb.mutual_information.calculate_mi_matrices(x_in, y_in, backend="gpu")
    barrier()
    de = (time.perf_counter() - t0) / args.steps
    tt = torch.tensor([de], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    de = float(tt.item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    steps = args.steps
    phases = {k_: agg.get(k_, 0.0) / steps for k_ in ("ms_gather", "ms_dist_tensor", "ms_reduce", "ms_total")}
    ms_step = 1e3 * dt / steps
    burst = ms_step < 100.0
    bf16 = peaks.get("bf16_tflops" if burst else "bf16_tflops_sustained", 1590.0 if burst else 1400.0)
    hbm = peaks.get("hbm_gbs", 6650.0)
    gemm = agg.get("ops_dist_tensor", 0.0) / steps / max(phases["ms_dist_tensor"], 1e-9) / 1e9     # TOP/s
    # finishing kernel: reads the 4 reduced counts of every genotype pair once, writes both triangles
    my_pairs = sum(q - 1 - c for c in range(lo, hi))
    fin_bytes = my_pairs * (4.0 * 4 + 16.0)
    fin = fin_bytes / max(phases["ms_reduce"], 1e-9) / 1e6                                          # GB/s
    kernels = {
        "ms_dist_tensor": {"bound": "tensor", "achieved": gemm, "peak": 4.0 * bf16, "unit": "TOP/s fp4 (e2m1, exact integers)",
                           "frac": gemm / (4.0 * bf16), "traffic": None},
        "ms_reduce": {"bound": "hbm", "achieved": fin, "peak": hbm, "unit": "GB/s", "frac": fin / hbm, "traffic": None,
                      "note": "finishing kernel: 32 algorithmic bytes per column pair; also carries 9 float64 logarithms per pair"},
    }
    top = max(kernels, key=lambda k_: phases[k_])
    line = {"metric": J_METRIC, "value": units * steps / dt, "unit": J_UNIT, "n_gpus": world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "e2m1 (FP4) one-hot / exact FP32 counts / f64 statistic", "data": "synthetic",
            "config": {"workload": w["desc"], "n": n, "p": p, "sharding": f"row bands of the pair matrix x{world}, one allreduce",
                       "l2": "inputs and the count slab are larger than L2 (no flush needed)",
                       "timing": "CUDA events on the launching stream around the K steps, max over ranks"},
            "clocks": sampler.summary(),
            "e2e": {"value": units / de, "unit": J_UNIT, "h2d_bytes_per_step": int(xa.nbytes),
                    "d2h_bytes_per_step": int(8 * q * q), "seconds_per_call": de,
                    "matches_resident_run": bool(np.array_equal(rel, check))},
            "gpu_launches": int(agg.get("launches", 0)), "roofline": dict(kernels[top], kernel=top),
            "kernels": kernels, "phases_ms": phases, "bands": int(agg.get("n_chunks", 0) / steps),
            "cpu_baseline": None}
    n_s, p_s = min(n, 10_000), min(p, 6000)       # ~10 s of CPU work on 16 threads
    tc, _ = joint_cpu(w["x"][:n_s, :p_s], w["y"][:n_s], os.cpu_count() or 1)
    from oracle import ref_oracle as R
    line["cpu_baseline"] = {"value": float(n_s) * (p_s + 1) * p_s / 2 / tc, "unit": J_UNIT, "cores": R.max_threads(),
                            "kind": "port", "sample": f"first {n_s} samples x {p_s} features, one pass, {tc:.2f} s"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c2", "c4", "c4surf", "c5", "j1"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-parity", dest="no_parity", action="store_true", help="skip the oracle / single-GPU parity checks of the timed run")
    # (--samples / --features: torchrun's own parser treats "--n" as an ambiguous abbreviation of its options)
    ap.add_argument("--n", "--samples", dest="n", type=int, default=None)
    ap.add_argument("--p", "--features", dest="p", type=int, default=None)
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, "
                         "at most 64 MB in all: a fixed sample of the entries of a larger output)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference" and args.workload == "j1":
        joint_reference_arm(args)
    elif args.workload == "j1":
        joint_arm(args)
    elif args.impl == "reference":
        reference_arm(args)
    elif args.workload == "c5":
        turf_arm(args)
    else:
        own_arm(args)


if __name__ == "__main__":
    main()
