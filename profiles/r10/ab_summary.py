"""Summary of profiles/r10/ab.sh: per run ms_per_step, e2e ms_per_step, device_bytes, scatter1 (ms and launches per
step), scatter2 and the page-list kernels, the spread within every arm, and whether every dump of a config equals
the first A dump."""
import glob
import json
import os
import re
import sys

import numpy as np

BOOK = ("pga_hist", "pga_scan", "pga_fill", "pgb_fill", "bucket_order", "scan_bpages", "scan_rows")
COLS = ("ms_per_step", "e2e_ms", "device_GB", "scatter1", "scatter2", "page lists")
out, dump = sys.argv[1], sys.argv[2]
for cfg in (5, 2):
    rows = {}
    for path in sorted(glob.glob(os.path.join(out, f"c{cfg}_*.json"))):
        tag = os.path.basename(path)[:-5]
        arm = re.match(rf"c{cfg}_([A-Z])\d+$", tag).group(1)
        try:
            d = json.loads(open(path).read().strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001 - report and go on
            print(tag, "no result:", e)
            continue
        k = d["kernels"]
        book = {n: k[n]["ms_per_step"] for n in BOOK if n in k}
        r = (d["ms_per_step"], d["e2e"]["ms_per_step"], d["config"]["device_bytes"] / 1e9, k["scatter1"]["ms_per_step"],
             k["scatter2"]["ms_per_step"], sum(book.values()))
        rows.setdefault(arm, []).append(r)
        print(f"{tag}: ms_per_step {r[0]:.2f}  e2e {r[1]:.2f}  device_bytes {r[2]:.2f} GB  scatter1 {r[3]:.3f} "
              f"({k['scatter1']['launches_per_step']} launches)  scatter2 {r[4]:.3f}  page lists {r[5]:.3f} (" +
              ", ".join(f"{n} {v:.3f}" for n, v in book.items()) + f")  digest {d['config'].get('digest_check', '')[:40]}")
    for arm, rs in sorted(rows.items()):
        a = np.array(rs)
        print(f"config {cfg} {arm}: " + ", ".join(f"{n} {a[:, j].mean():.3f} (range {a[:, j].min():.3f}-{a[:, j].max():.3f})"
                                                  for j, n in enumerate(COLS)))
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
