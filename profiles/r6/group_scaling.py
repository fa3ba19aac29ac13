"""Several GPUs from one process (group.GpuGroup) against one GPU and against torchrun, at bench.py's configs 2 and 5.

For every config the samples are rendered as bench.py renders them: one synth_gpu.Renderer per rank on that rank's
device, for the rank's own block of samples, so the text is resident in HBM. A step is what bench.py times: ingest,
build, test and the gather of the survivors. The 1-GPU point is the plain KmerAssociation, in k-mer ranges when bench.py
would use them. G GPUs is GpuGroup(range(G)), for G in 2 and 4 as far as the machine has them.
Each point: one warm-up step, then STEPS timed steps, each timed on a wall clock that ends with a synchronise of every
device in use. Each result is checked against tests/golden/bench_digests.json with bench.result_digest and the test
arguments bench.py uses for that config. The card's name, power limit and SM clock come from nvidia-smi in the same
run, and `torchrun --nproc-per-node G bench.py --gpus G --config c` runs after the points for comparison.
usage: python profiles/r6/group_scaling.py OUT.json [config ...]   (default configs: 2 5)"""
import gc
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from phenotypeseeker_b200 import dist as psdist, synth_gpu  # noqa: E402
from phenotypeseeker_b200.group import GpuGroup  # noqa: E402
from phenotypeseeker_b200.pipeline import KmerAssociation  # noqa: E402

STEPS = 3
K = bench.K


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [x.strip() for x in r.stdout.splitlines()] if r.returncode == 0 else [f"nvidia-smi failed: {r.stderr.strip()}"]


def render(plan, G):
    """-> (buffers: (dev_ptr, n) per sample on its rank's device, tensors to keep alive, text bytes, bench.py's upper
    estimate of the text bytes)."""
    bufs, keep, total, est = [None] * plan.n_samples, [], 0, 0
    for r in range(G):
        dev = torch.device("cuda", r)
        block = list(psdist.sample_block(r, G, plan.n_samples))
        rend = synth_gpu.Renderer(plan, dev)
        if r == 0:
            est = sum(rend.max_text_bytes(s) for s in range(plan.n_samples))
        text, spans = rend.render(block)
        keep.append(text)
        for s, (o, n) in spans.items():
            bufs[s] = (text.data_ptr() + o, n)
            total += n
    for r in range(G):
        torch.cuda.synchronize(r)
    return bufs, keep, total, est


def timed(step, G):
    def sync():
        for r in range(G):
            torch.cuda.synchronize(r)
    U, res = step()                                         # warm-up
    sync()
    times = []
    for _ in range(STEPS):
        t0 = time.perf_counter()
        U, res = step()
        sync()
        times.append(time.perf_counter() - t0)
    return U, res, times


def point(cfg_idx, plan, G, known):
    cfg = bench.CONFIGS[cfg_idx]
    N = plan.n_samples
    weights = plan.weights if cfg["weighted"] else None
    kw = dict(min_samples=2, max_samples=N - 2, pvalue_cutoff=cfg["pvalue"], omit_b=cfg["omit_b"], top_k=cfg["top_k"])
    bufs, keep, total, est = render(plan, G)
    if G == 1:
        ka = KmerAssociation(device=0)
        n_ranges = max(1, math.ceil(est / 8.5e9))             # bench.py's one-GPU step, k-mer ranges included
        state = {"splitters": None}

        def step():
            ing = None
            if n_ranges > 1 and state["splitters"] is not None:
                ka.k = K
                ing = ka.plan_ranges(n_ranges, state["splitters"], total)["ingest"]
            ka.count(bufs, K, cfg["cutoff"], ingest_range=ing)
            if n_ranges > 1:
                U, res = ka.test_in_ranges(plan.pheno, cfg["binary"], n_ranges, weights, splitters=state["splitters"],
                                           n_instances=total, **kw)
                state["splitters"] = ka.range_splitters
                return U, res
            U = ka.build()
            return U, ka.test(plan.pheno, cfg["binary"], weights, **kw)
    else:
        g = GpuGroup(list(range(G)))

        def step():
            g.count(bufs, K, cfg["cutoff"])
            return g.test(plan.pheno, cfg["binary"], weights, **kw)
    U, res, times = timed(step, G)
    digest = bench.result_digest(U, res)
    key = f"config{cfg_idx}_n{N}_L{plan.genome_len}"
    ok = key in known and known[key]["digest"] == digest and known[key]["U"] == U
    del keep
    return {"gpus": G, "engine": "KmerAssociation" if G == 1 else "GpuGroup", "ms_per_step": [round(t * 1e3, 2) for t in times],
            "ms_median": round(float(np.median(times)) * 1e3, 2), "U": int(U), "digest": digest,
            "digest_check": "equal" if ok else f"DIFFERS from {known.get(key)}"}


def torchrun(cfg_idx, G):
    cmd = ["torchrun", "--nproc-per-node", str(G), os.path.join(ROOT, "bench.py"), "--gpus", str(G), "--config",
           str(cfg_idx), "--no-cpu-baseline"]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        return {"gpus": G, "rc": r.returncode, "error": r.stderr[-1500:]}
    line = json.loads(lines[-1])
    return {"gpus": G, "ms_per_step": line["ms_per_step"], "digest_check": line["config"]["digest_check"],
            "e2e_ms_per_step": line["e2e"]["ms_per_step"]}


def main():
    out_path = sys.argv[1]
    configs = [int(c) for c in sys.argv[2:]] or [2, 5]
    if not torch.cuda.is_available():
        raise SystemExit("needs CUDA devices (no CPU fallback)")
    ngpu = torch.cuda.device_count()
    with open(os.path.join(ROOT, "tests", "golden", "bench_digests.json")) as f:
        known = json.load(f)
    report = {"nvidia_smi name, power.limit, clocks.sm": gpu_info(), "device_count": ngpu, "steps": STEPS, "configs": {}}
    for c in configs:
        plan = synth_gpu.config_plan(c)
        pts = []
        for G in (1, 2, 4):
            if G <= ngpu:
                pts.append(point(c, plan, G, known))
                gc.collect()
                torch.cuda.empty_cache()
        tr = [torchrun(c, G) for G in (2, 4) if G <= ngpu]
        report["configs"][str(c)] = {"group": pts, "torchrun": tr}
        print(json.dumps({c: report["configs"][str(c)]}), flush=True)
    with open(out_path, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
