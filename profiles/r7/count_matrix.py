"""Occurrence counts of K union k-mers in every sample of bench.py's configs 2 and 5: one ps_count_matrix call against
the loop of one ps_lookup per sample that the -rc path and the prediction drop-in made before.

The samples are rendered on the device by synth_gpu (as bench.py renders them) and ingested at k = 16, cutoff 1. The
queries are K distinct k-mers, ascending as the -rc path passes them, drawn from the union: from the k-mers of eight
samples spread over the cohort (every one of them is a union k-mer; building the whole config-5 union would need
k-mer ranges). One warm-up call, then one timed call over all samples with CUDA events on the library's stream (both
entry points end in a stream synchronise, so a wall clock is printed as well). With ps_count_matrix present the kernel
times of that call come from the library's per-launch events in a second, profiled call.

The tree to measure is --tree (default: this checkout); a tree without Context.count_matrix (the parent commit) runs
the lookup loop, so profiles/r7/ab_count_matrix.sh can alternate both in one job. Each run prints one JSON line with
a SHA-256 of the N x K counts, which must agree between the two sides.
usage: python profiles/r7/count_matrix.py --config {2,5} [--tree DIR] [--K 1000,100000]
       python profiles/r7/count_matrix.py --summary DIR      (the JSON files of ab_count_matrix.sh)"""
import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def measure(args):
    sys.path.insert(0, os.path.abspath(args.tree))
    import torch
    from phenotypeseeker_b200 import synth_gpu
    from phenotypeseeker_b200.pipeline import KmerAssociation
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    dev = torch.device("cuda", 0)
    plan = synth_gpu.config_plan(args.config)
    N = plan.n_samples
    text, spans = synth_gpu.Renderer(plan, dev).render(range(N))
    torch.cuda.synchronize()
    ka = KmerAssociation(device=0)
    ka.count([(text.data_ptr() + spans[s][0], spans[s][1]) for s in range(N)], 16, 1)
    torch.cuda.synchronize()
    del text
    torch.cuda.empty_cache()
    ctx = ka.ctx
    matrix = hasattr(ctx, "count_matrix")
    stream = torch.cuda.ExternalStream(ctx.stream(), device=dev)
    pool = np.unique(np.concatenate([ctx.sample_kmers(int(s))[0] for s in np.linspace(0, N - 1, 8).astype(int)]))
    rng = np.random.default_rng(args.config)
    out = []
    for K in [int(x) for x in args.K.split(",")]:
        q = np.sort(rng.choice(pool, K, replace=False))

        def call():
            if matrix:
                return ctx.count_matrix(0, N, q)
            return np.stack([ctx.lookup(s, q) for s in range(N)])
        if matrix:
            call()                                          # warm-up: one whole call
        else:
            ctx.lookup(0, q)                                # warm-up: the kernel and the buffers of one lookup
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        counts = call()
        e1.record(stream)
        e1.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        rec = dict(config=args.config, N=N, K=K, side="count_matrix" if matrix else "lookup_loop",
                   ms=e0.elapsed_time(e1), wall_ms=wall, positions=int(sum(ctx.export_stream(s)[2] for s in range(N))),
                   nonzero=float((counts > 0).mean()), sha256=hashlib.sha256(np.ascontiguousarray(counts).tobytes()).hexdigest(),
                   gpu=gpu_info())
        if matrix:
            ctx.profile(True)
            ctx.profile_reset()
            call()
            rec["kernels_ms"] = {n: round(v["ms"], 3) for n, v in ctx.profile_table().items() if v["launches"]}
            ctx.profile(False)
        print(json.dumps(rec), flush=True)
        out.append(rec)
    return out


def summary(d):
    rows = [json.loads(l) for f in sorted(glob.glob(os.path.join(d, "*.json"))) for l in open(f) if l.startswith("{")]
    print(rows[0]["gpu"] if rows else "no runs")
    for cfg in sorted({r["config"] for r in rows}):
        for K in sorted({r["K"] for r in rows if r["config"] == cfg}):
            rs = [r for r in rows if r["config"] == cfg and r["K"] == K]
            same = len({r["sha256"] for r in rs}) == 1
            for side in ("lookup_loop", "count_matrix"):
                t = [r["ms"] for r in rs if r["side"] == side]
                if t:
                    extra = next((r.get("kernels_ms") for r in rs if r["side"] == side and "kernels_ms" in r), "")
                    print(f"config {cfg} N={rs[0]['N']} K={K} {side:12s} runs={len(t)} mean={np.mean(t):10.1f} ms "
                          f"min={min(t):10.1f} max={max(t):10.1f} {extra}")
            print(f"config {cfg} K={K} counts identical across all runs: {same}")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, choices=(2, 5))
    ap.add_argument("--tree", default=HERE)
    ap.add_argument("--K", default="1000,100000")
    ap.add_argument("--summary")
    a = ap.parse_args()
    if a.summary:
        summary(a.summary)
    else:
        measure(a)
