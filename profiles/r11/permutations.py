"""Cost of the permutation threshold (PS_PERMUTATIONS / test(n_perm=B)) at bench.py's configs 2 and 5.

Renders a config as bench.py does (synth_gpu, device-resident text), then times on the library stream with CUDA
events: the tests without permutations, the same with B permutations (k-mer ranges where bench.py uses them), and,
from the library's own per-kernel CUDA-event profile, the min-p passes (one launch per batch of permuted columns).
Checks that the observed column's min-p (ps_minp_*) equals the smallest p ps_test_* returns at thr = 1, and records
the card's name and power limit in the same run. One JSON line per config on stdout.

usage: python profiles/r11/permutations.py [--configs 2 5] [--perms 100] [--out DIR]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def observed_minp_check(ka, pheno, binary, weights, N):
    """ps_minp_* of the observed columns against the smallest p of ps_test_* at thr = 1 (top 1 per column, selected
    on the device) in the build the context holds now (the whole union, or the first k-mer range)."""
    ctx = ka.ctx
    P = pheno.shape[1]
    w = None if weights is None or np.all(np.asarray(weights) == 1.0) else np.asarray(weights, dtype=np.float64)
    if binary:
        code = np.where(np.isnan(pheno), -1, pheno).astype(np.int8).T
        m = ctx.minp_chi2(code, w, 2, N - 2)
        ns = ctx.test_chi2(code, w, 2, N - 2, 1.0)
    else:
        m = ctx.minp_welch(pheno.T.copy(), w, 2, N - 2)
        ns = ctx.test_welch(pheno.T.copy(), w, 2, N - 2, 1.0)
    ns = ctx.select_top(P, 1) if ns else 0
    sv = ctx.fetch_survivors(ns, rowbits=False)
    best = np.ones(P)
    for j in range(P):
        p = sv["p"][sv["pheno"] == j]
        if len(p):
            best[j] = p.min()
    return bool(np.array_equal(m, best)), m.tolist()


def run_config(c, B, torch):
    import bench
    from phenotypeseeker_b200 import synth_gpu
    from phenotypeseeker_b200.pipeline import KmerAssociation
    cfg = bench.CONFIGS[c]
    device = torch.device("cuda", 0)
    plan = synth_gpu.config_plan(c)
    N = plan.n_samples
    renderer = synth_gpu.Renderer(plan, device)
    dev, spans = renderer.render(list(range(N)))
    torch.cuda.synchronize(device)
    bufs = [(dev.data_ptr() + spans[s][0], spans[s][1]) for s in range(N)]
    h2d = sum(n for _, n in spans.values())
    total_text = sum(renderer.max_text_bytes(s) for s in range(N))
    n_ranges = max(1, math.ceil(total_text / 8.5e9))            # as bench.py on one GPU
    pheno, binary = plan.pheno, cfg["binary"]
    weights = plan.weights if cfg["weighted"] else None
    ka = KmerAssociation(device=0)
    stream = torch.cuda.ExternalStream(ka.ctx.stream(), device=device)
    kw = dict(min_samples=2, max_samples=N - 2, pvalue_cutoff=cfg["pvalue"], omit_b=cfg["omit_b"], top_k=cfg["top_k"])

    def timed(n_perm):
        ka.ctx.profile_reset()
        ka.ctx.profile(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ka.count(bufs, bench.K, cfg["cutoff"])
        torch.cuda.synchronize(device)
        e0.record(stream)
        w0 = time.time()
        extra = dict(n_perm=n_perm, perm_seed=0) if n_perm else {}
        if n_ranges > 1:
            U, res = ka.test_in_ranges(pheno, binary, n_ranges, weights, n_instances=h2d, **kw, **extra)
        else:
            U = ka.build()
            res = ka.test(pheno, binary, weights, **kw, **extra)
        e1.record(stream)
        torch.cuda.synchronize(device)
        ka.ctx.profile(False)
        return U, res, e0.elapsed_time(e1), time.time() - w0, ka.ctx.profile_table()

    timed(0)                                                       # warm-up: modules, pools
    U, res0, ms0, wall0, prof0 = timed(0)
    U1, res1, ms1, wall1, prof1 = timed(B)
    assert U1 == U
    minp_k = {k: v for k, v in prof1.items() if k.startswith("minp_")}
    minp_ms = sum(v["ms"] for v in minp_k.values())
    batches = sum(v["launches"] for v in minp_k.values())
    test_k = {k: v for k, v in prof0.items() if k.startswith("test_")}
    if n_ranges > 1:          # test_in_ranges left the whole k-mer space selected, without a union: build range 0
        ka.count(bufs, bench.K, cfg["cutoff"])
        ka.build((0, ka.range_splitters[0]))
    same, m_obs = observed_minp_check(ka, pheno, binary, weights, N)
    return {
        "config": c, "workload": cfg["workload"], "card": card(), "n_samples": N, "columns": int(pheno.shape[1]),
        "U": int(U), "k_mer_ranges": n_ranges, "permutations": B,
        "build_and_test_ms_no_permutations": round(ms0, 2), "build_and_test_ms_with_permutations": round(ms1, 2),
        "wall_s_no_permutations": round(wall0, 3), "wall_s_with_permutations": round(wall1, 3),
        "test_kernel_ms": round(sum(v["ms"] for v in test_k.values()), 3),
        "minp_kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 3)} for k, v in minp_k.items()},
        "minp_ms_total": round(minp_ms, 3), "minp_batches": int(batches),
        "minp_ms_per_batch": round(minp_ms / max(batches, 1), 3), "minp_ms_per_permutation": round(minp_ms / B, 3),
        "thresholds": [r.threshold for r in res1], "bonferroni": cfg["pvalue"] / U if U else None,
        "survivors_bonferroni": [int(len(r.kmer)) for r in res0], "survivors_permutation": [int(len(r.kmer)) for r in res1],
        "observed_minp_equals_test_at_thr_1": same, "observed_minp_last_build": m_obs,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 5])
    ap.add_argument("--perms", type=int, default=100)
    ap.add_argument("--out", default=None, help="also write the lines to DIR/permutations.jsonl")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lines = []
    for c in args.configs:
        line = json.dumps(run_config(c, args.perms, torch))
        print(line, flush=True)
        lines.append(line)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "permutations.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
