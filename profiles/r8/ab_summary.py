"""Summary of profiles/r8/ab_retire.sh: per run ms_per_step and the kernels whose code paths the change touched, the
spread within A and within B, and whether every dump of a config equals the first A dump."""
import glob
import json
import os
import sys

import numpy as np

KERNELS = ("bucket_count", "bucket_build", "decode_write")
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
            r = (d["ms_per_step"],) + tuple(d["kernels"][k]["ms_per_step"] for k in KERNELS)
            rows[ab].append(r)
            print(f"{tag}: ms_per_step {r[0]:.2f}  " + "  ".join(f"{k} {v:.3f}" for k, v in zip(KERNELS, r[1:])) +
                  f"  digest {d['config'].get('digest_check', '')[:40]}")
    for ab, rs in rows.items():
        if rs:
            a = np.array(rs)
            print(f"config {cfg} {ab}: " + ", ".join(f"{n} {a[:, j].mean():.3f} (spread {np.ptp(a[:, j]):.3f})"
                                                      for j, n in enumerate(("ms_per_step",) + KERNELS)))
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
