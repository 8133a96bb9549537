"""Round-2 diagnostic: merged-plane accumulation kernel (FS_B200_ACCUM_PAIR=3, default) against the paired
(=1) and per-row (=0) epilogues on 0/1/2 genotypes: same weights?  Prints where they differ."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import fastselect_b200 as fsb  # noqa: E402

rc = 0
for (n, p, star) in ((300, 70, False), (1000, 333, True), (2500, 1000, False), (777, 64, False)):
    rs = np.random.RandomState(n)
    y = rs.randint(0, 2, n)
    x = rs.randint(0, 3, (n, p)).astype(np.int8)
    x[:, 3] = (y + rs.randint(0, 2, n)) % 3
    w = {}
    for mode in ("3", "1", "0"):
        os.environ["FS_B200_ACCUM_PAIR"] = mode
        est = fsb.MultiSURF(n_features_to_select=5, backend="gpu", use_star=star).fit(x, y)
        w[mode] = est.feature_importances_.copy()
    d31 = np.abs(w["3"] - w["1"])
    d10 = np.abs(w["1"] - w["0"])
    scale = np.abs(w["1"]).max()
    print(f"n={n} p={p} star={star}: max|merged-paired|={d31.max():.3e} max|paired-rows|={d10.max():.3e} max|W|={scale:.3e}")
    if d31.max() > 1e-12 * max(1.0, scale):
        rc = 1
        bad = np.nonzero(d31 > 1e-12 * max(1.0, scale))[0]
        print("  differing columns:", len(bad), "of", p, "first:", bad[:24])
        print("  merged:", w["3"][bad[:6]])
        print("  paired:", w["1"][bad[:6]])
os.environ.pop("FS_B200_ACCUM_PAIR", None)
sys.exit(rc)
