"""`-w` sample weights on the device (ps_mash_sketch, ps_mash_pairs, ps_neighbor_joining) at the sizes of bench.py's
configs 2 and 5, with subset checks against the host restatement in phenotypeseeker_b200/weights.py.

For every config: render the samples with synth_gpu.Renderer (as bench.py does), ingest them through
KmerAssociation.count (k = 16, cutoff 1), warm every kernel up once on a small subset, then run the whole device path
once with ps_profile on: kernel times from CUDA events, the wall clock of each call (each ends in a synchronise), and
the host remainder (distance table, tree replay, Newick write + parse, GSC) on a wall clock.
Config 2 also checks, on the host: 8 random samples' sketches against weights.sketch(), 2,000 random pairs against
weights.mash_distance(), and the whole NJ against weights.nj_joins() (array_equal). Config 5 checks 2 sketches and
200 pairs (the host NJ at N = 5,000 takes about 20 minutes).
usage: python profiles/r5/mash_weights.py OUT.json [config ...]   (default configs: 2 5)"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from phenotypeseeker_b200 import synth_gpu, weights as W  # noqa: E402
from phenotypeseeker_b200.pipeline import KmerAssociation  # noqa: E402

# single-threaded host path (weights.py), measured on an 8-core development machine, not on the GPU host;
# config 5 NJ extrapolated from N = 400 / 800 (x 8 per doubling)
HOST_BASELINE = {
    "note": "measured on a different CPU / extrapolated (weights.py, one thread)",
    2: {"sketch_s": "780-960", "distance_matrix_s": 6, "neighbor_joining_s": 0.1},
    5: {"sketch_s": "18000-21600", "distance_matrix_s": 2400, "neighbor_joining_s": 1200},
}
CHECKS = {2: (8, 2000, True), 5: (2, 200, False)}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [x.strip() for x in r.stdout.splitlines()[0].split(",")])) if r.returncode == 0 else {}


def kernels(ctx):
    return {k: {"launches": v["launches"], "ms": round(v["ms"], 3)} for k, v in ctx.profile_table().items()}


def device_path(ctx, names, prof):
    """the device part of weights.gsc_weights_on_device, timed -> (h, n, dm, join, branch, weights, times)"""
    t = {}
    if prof:
        ctx.profile_reset()
        ctx.profile(True)
    t0 = time.perf_counter()
    h, n = ctx.mash_sketch(0, len(names))
    t["sketch_call_s"] = time.perf_counter() - t0
    order = sorted(range(len(names)), key=lambda i: names[i] + ".msh")
    h, n = h[order], n[order]
    t0 = time.perf_counter()
    sd = ctx.mash_pairs(h, n)
    t["pairs_call_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    dm = W.printed_distances(sd)
    t["host_table_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    join, branch = ctx.neighbor_joining(dm)
    t["nj_call_s"] = time.perf_counter() - t0
    if prof:
        t["kernels"] = kernels(ctx)
        ctx.profile(False)
    t0 = time.perf_counter()
    root = W.tree_from_joins(names, join, branch)
    t["host_replay_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    tree = W.parse_newick(W.newick(root) + ";")
    t["host_newick_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    w = W.gsc_weights(tree)
    t["host_gsc_s"] = time.perf_counter() - t0
    return h, n, dm, join, branch, np.array([w[nm] for nm in names]), t


def run_config(cfg):
    plan = synth_gpu.config_plan(cfg)
    N = plan.n_samples
    rend = synth_gpu.Renderer(plan, "cuda:0")
    t0 = time.perf_counter()
    bufs, keep, batch = [], [], 50
    for b0 in range(0, N, batch):
        txt, spans = rend.render(list(range(b0, min(N, b0 + batch))))
        keep.append((txt, spans))
        bufs += [(txt.data_ptr() + spans[s][0], spans[s][1]) for s in range(b0, min(N, b0 + batch))]
    torch.cuda.synchronize()
    render_s = time.perf_counter() - t0
    ka = KmerAssociation(device=0)
    t0 = time.perf_counter()
    ka.count(bufs, 16, 1)
    ingest_s = time.perf_counter() - t0
    ctx = ka.ctx
    names = [plan.names[s] for s in range(N)]
    # warm-up: every kernel once, on a subset
    sub = min(N, 40)
    hw, nw = ctx.mash_sketch(0, sub)
    ctx.neighbor_joining(W.printed_distances(ctx.mash_pairs(hw, nw)))
    h, n, dm, join, branch, w, t = device_path(ctx, names, True)
    dev_s = sum(v["ms"] for v in t["kernels"].values()) / 1e3
    host_s = t["host_table_s"] + t["host_replay_s"] + t["host_newick_s"] + t["host_gsc_s"]
    calls_s = t["sketch_call_s"] + t["pairs_call_s"] + t["nj_call_s"]
    # checks against the host restatement
    n_sk, n_pairs, full_nj = CHECKS[cfg]
    rng = np.random.default_rng(cfg)
    order = sorted(range(N), key=lambda i: names[i] + ".msh")
    pos_of = {s: p for p, s in enumerate(order)}
    checks = {}
    bad = 0
    for s in rng.choice(N, n_sk, replace=False):
        txt, spans = keep[s // batch]
        off, ln = spans[int(s)]
        text = txt[off:off + ln].cpu().numpy().tobytes()
        p = pos_of[int(s)]
        bad += not np.array_equal(h[p, :n[p]], W.sketch(text))
    checks["sketches"] = {"checked": int(n_sk), "mismatches": int(bad)}
    bad = 0
    sd = None
    for i, j in zip(rng.integers(0, N, n_pairs), rng.integers(0, N, n_pairs)):
        d, _, _ = W.mash_distance(h[i, :n[i]], h[j, :n[j]])
        bad += (i != j) and W.printed(d) != dm[i, j]
    checks["pairs"] = {"checked": int(n_pairs), "mismatches": int(bad)}
    if full_nj:
        t0 = time.perf_counter()
        jw, bw = W.nj_joins(dm)
        checks["nj"] = {"join_equal": bool(np.array_equal(jw, join)), "branch_equal": bool(np.array_equal(bw, branch)),
                        "host_nj_joins_s": round(time.perf_counter() - t0, 3)}
    return {
        "config": cfg, "n_samples": N, "genome_len": plan.genome_len, "render_s": round(render_s, 3),
        "ingest_s": round(ingest_s, 3),
        "device_kernels_ms": t["kernels"], "device_kernels_total_s": round(dev_s, 3),
        "calls_s": {k: round(t[k], 3) for k in ("sketch_call_s", "pairs_call_s", "nj_call_s")},
        "host_s": {k: round(t[k], 3) for k in ("host_table_s", "host_replay_s", "host_newick_s", "host_gsc_s")},
        "total_s": round(calls_s + host_s, 3),
        "weights": {"mean": float(w.mean()), "min": float(w.min()), "max": float(w.max()), "finite": bool(np.isfinite(w).all())},
        "checks": checks, "host_baseline": HOST_BASELINE[cfg],
    }


def main():
    out = sys.argv[1]
    cfgs = [int(x) for x in sys.argv[2:]] or [2, 5]
    res = {"gpu": gpu_info(), "host_baseline_note": HOST_BASELINE["note"], "configs": []}
    for cfg in cfgs:
        r = run_config(cfg)
        res["configs"].append(r)
        print(json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    ok = all(c["checks"]["sketches"]["mismatches"] == 0 and c["checks"]["pairs"]["mismatches"] == 0 and
             c["checks"].get("nj", {"join_equal": True, "branch_equal": True})["join_equal"] and
             c["checks"].get("nj", {"branch_equal": True})["branch_equal"] for c in res["configs"])
    print("CHECKS", "PASSED" if ok else "FAILED")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
