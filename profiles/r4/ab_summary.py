"""Summary of profiles/r4/ab_chi2.sh: per run ms_per_step and test_chi2, the spread within A and
within B, and whether every dump of a config equals the first A dump."""
import glob
import json
import os
import sys

import numpy as np

out, dump = sys.argv[1], sys.argv[2]
for cfg in (5, 2):
    rows = {"A": [], "B": []}
    for ab in ("A", "B"):
        for i in (1, 2, 3):
            tag = f"c{cfg}_{ab}{i}"
            try:
                d = json.loads(open(os.path.join(out, tag + ".json")).read().strip().splitlines()[-1])
            except Exception as e:  # noqa: BLE001 - report and go on
                print(tag, "no result:", e)
                continue
            k = d["kernels"]
            chi2 = k.get("test_chi2") or k.get("test_chi2_w")     # config 2 is weighted
            r = (d["ms_per_step"], chi2["ms_per_step"], k["scatter1"]["ms_per_step"])
            rows[ab].append(r)
            print(f"{tag}: ms_per_step {r[0]:.2f}  test_chi2 {r[1]:.2f}  scatter1 {r[2]:.2f}  "
                  f"digest {d['config'].get('digest_check', '')[:40]}")
    for ab, rs in rows.items():
        if rs:
            a = np.array(rs)
            print(f"config {cfg} {ab}: mean ms_per_step {a[:, 0].mean():.2f} (spread {np.ptp(a[:, 0]):.2f}), "
                  f"test_chi2 {a[:, 1].mean():.2f} (spread {np.ptp(a[:, 1]):.2f}), "
                  f"scatter1 {a[:, 2].mean():.2f} (spread {np.ptp(a[:, 2]):.2f})")
    ref = os.path.join(dump, f"c{cfg}_A1")
    names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(ref, "*.npy")))
    same = bool(names)
    for other in sorted(glob.glob(os.path.join(dump, f"c{cfg}_*"))):
        for n in names:
            x, y = np.load(os.path.join(ref, n)), np.load(os.path.join(other, n))
            if x.shape != y.shape or not np.array_equal(x, y, equal_nan=True):
                same = False
                print(f"config {cfg}: {os.path.basename(other)}/{n} differs from c{cfg}_A1")
    print(f"config {cfg}: {len(names)} dumped arrays, all runs identical: {same}")
