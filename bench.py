#!/usr/bin/env python
"""bench.py — k-mers tested/sec through count -> matrix -> chi2 / Welch -> filter (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config {1..5}] [--impl ours|reference] [--dump-outputs DIR]

--config c = BASELINE.json configs[c-1] on synthetic data of that shape (phenotypeseeker_b200/synth_gpu.py):
  1  20 x 4.3 Mbp assemblies, k=16, binary, unweighted chi2, --omit_B_correction      (the CPU-runnable case)
  2  250 x 4.3 Mbp assemblies, k=16, binary, GSC-like weights, chi2 + p<0.05 Bonferroni
  3  1,000 x 5 Mbp assemblies, continuous phenotype (2 % NA), weighted Welch t-test
  4  200 raw-read FASTQ samples (150 bp, 30x of 4.3 Mbp), k=16, min-count cutoff 3, binary
  5  5,000 x 5 Mbp assemblies x 10 binary phenotype columns                             (default: the headline)
One step = one full pass of the hot path over all samples of the config.

  value : U * P / step time (U = union k-mers = the reference's no_kmers_to_analyse, P = phenotype columns),
          FASTA/FASTQ text already resident in HBM (CUDA events on the library's stream, max over ranks)
  e2e   : the same through the public API with HOST (pinned) buffers: H2D of all text and D2H of the
          step's result inside the timed region
  N = 1 : when records + matrix exceed HBM the k-mer space is processed in ranges (KmerAssociation.test_in_ranges)
  N > 1 : strong scaling — every rank ingests its own block of samples, the k-mer space is range-sharded,
          k-mer instances travel over NVLink inside the extraction kernel (phenotypeseeker_b200/dist.py)
  result of a step: per phenotype column the survivors of the p-value filter; configs 3-5 cut them to the
          top 1000 per column on the GPU (`--n_kmers` default of the reference) before the read-back.
  --impl reference : the reference's own CPU implementation (shipped GenomeTester4 binaries + modeling.py
          stage-3 loop) on a bounded sample of the same config, all host cores.
"""
import argparse
import hashlib
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

METRIC = "k-mers tested/sec (count+matrix+test+filter)"
UNIT = "k-mers/s"
K = 16

CONFIGS = {
    1: dict(workload="BASELINE.json configs[0]: 20 synthetic 4.3 Mbp assemblies, k=16, binary phenotype, unweighted chi2, --omit_B_correction",
            binary=True, weighted=False, pvalue=0.05, omit_b=True, cutoff=1, top_k=None, ref=dict(n=20, L=200_000)),
    2: dict(workload="BASELINE.json configs[1]: 250 synthetic 4.3 Mbp assemblies, k=16, binary phenotype, GSC-like weights, chi2 + p<0.05 Bonferroni",
            binary=True, weighted=True, pvalue=0.05, omit_b=False, cutoff=1, top_k=None, ref=dict(n=250, L=60_000)),
    3: dict(workload="BASELINE.json configs[2]: 1,000 synthetic 5 Mbp assemblies, k=16, continuous phenotype (2 % NA), weighted Welch t-test, p<0.05 Bonferroni, top 1000",
            binary=False, weighted=True, pvalue=0.05, omit_b=False, cutoff=1, top_k=1000, ref=dict(n=250, L=40_000)),
    4: dict(workload="BASELINE.json configs[3]: 200 raw-read FASTQ samples (150 bp, 30x of 4.3 Mbp), k=16, min-count cutoff 3, binary phenotype, chi2 + p<0.05 Bonferroni, top 1000",
            binary=True, weighted=False, pvalue=0.05, omit_b=False, cutoff=3, top_k=1000, ref=dict(n=8, L=100_000)),
    5: dict(workload="BASELINE.json configs[4]: 5,000 synthetic 5 Mbp assemblies x 10 binary phenotype columns, k=16, chi2 + p<0.05 Bonferroni, top 1000 per column",
            binary=True, weighted=False, pvalue=0.05, omit_b=False, cutoff=1, top_k=1000, ref=dict(n=60, L=20_000)),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        busy = [x for x in sm if x > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def result_digest(U, res):
    """Size-independent fingerprint of a step's result: U and, per phenotype column, the surviving k-mers
    with their sample counts (integers only, so it does not depend on the order of floating-point sums)."""
    h = hashlib.sha256()
    h.update(np.uint64(U).tobytes())
    for r in res:
        h.update(np.ascontiguousarray(r.kmer, dtype=np.uint64).tobytes())
        h.update(np.ascontiguousarray(r.n_with, dtype=np.uint32).tobytes())
    return h.hexdigest()[:32]


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, U, res, limit=DUMP_BYTES):
    """Write what a step returned as float64 .npy files, so that two builds can be compared array by array:
    union_kmers.npy holds U; the other files have one entry per survivor, the phenotype columns of `res` one after
    the other: its column (pheno), k-mer, union row, statistic, p-value, group means, sample count and bit-packed
    matrix row (rowbits, uint32 words). Every value is exact in float64 (k-mers of k <= 26). When the survivors
    would take more than `limit` bytes, a fixed, seeded sample of them is written; survivor.npy holds the indices
    of the written survivors among all of them."""
    cols = {"pheno": np.concatenate([np.full(len(r.kmer), j) for j, r in enumerate(res)])}
    for name in ("kmer", "row", "stat", "p", "mean_x", "mean_y", "n_with", "rowbits"):
        cols[name] = np.concatenate([getattr(r, name) for r in res])
    n = len(cols["pheno"])
    per_survivor = 8 * (len(cols) + cols["rowbits"].shape[1])   # 8 one-value arrays, survivor.npy, the row words
    keep = min(n, (limit - 4096) // per_survivor)               # 4 KB for U and the .npy headers
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "union_kmers.npy"), np.array([U], dtype=np.float64))
    np.save(os.path.join(out_dir, "survivor.npy"), idx.astype(np.float64))
    for name, a in cols.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[idx].astype(np.float64))


# ---------------------------------------------------------------------------------------
def cpu_reference_run(cfg_idx, threads, steps=1, warmup=0, n_samples=None, genome_len=None):
    """The reference CPU path on a bounded sample of config cfg_idx (same generator family, fewer / shorter
    genomes): the UNMODIFIED `phenotypeseeker modeling` CLI up to the end of its hot path (oracle/ref_cli.py)
    when the reference's Python is installed under oracle/_ref, else the restated pipeline."""
    import tempfile
    import shutil
    from oracle import build as obuild, ref_pipeline, ref_cli
    from phenotypeseeker_b200 import synth
    obuild.build_all()
    cfg = CONFIGS[cfg_idx]
    n = n_samples or cfg["ref"]["n"]
    L = genome_len or cfg["ref"]["L"]
    sub = synth.config(cfg_idx - 1, n_samples=n, genome_len=L)
    real_cli = obuild.ref_python_root() is not None and obuild.ref_bin_dir() is not None
    td = tempfile.mkdtemp(prefix="psbench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        ph_file, paths = sub.write(os.path.join(td, "in"))
        P = sub.pheno.shape[1]
        times, U = [], 0
        for it in range(warmup + steps):
            if real_cli:
                extra = ["-l", str(K), "-c", str(cfg["cutoff"]), "--pvalue", str(cfg["pvalue"])] + (["--omit_B_correction"] if cfg["omit_b"] else [])
                r = ref_cli.run(ph_file, os.path.join(td, f"work{it}"), threads, extra,
                                weights=list(sub.weights) if cfg["weighted"] else None)
                dt, U = r["seconds"], r["U"]
                shutil.rmtree(os.path.join(td, f"work{it}"), ignore_errors=True)
            else:
                cols = [[None if np.isnan(v) else (int(v) if cfg["binary"] else float(v)) for v in sub.pheno[:, j]] for j in range(P)]
                t0 = time.time()
                r = ref_pipeline.run(paths, sub.names, K, cols, cfg["binary"], list(sub.weights), 2, n - 2, cfg["pvalue"],
                                     cfg["omit_b"], threads=threads, cutoff=cfg["cutoff"])
                dt, U = time.time() - t0, r["U"]
            if it >= warmup:
                times.append(dt)
    finally:
        shutil.rmtree(td, ignore_errors=True)
    sec = float(np.mean(times))
    what = "raw-read sets" if sub.meta.get("reads") else "assemblies"
    how = ("the reference's UNMODIFIED CLI (`phenotypeseeker modeling`, installed under oracle/_ref) from start to the end of its hot "
           "path (modeling.py:1644-1686: glistmaker / glistcompare / glistquery binaries + its per-k-mer Python loop)"
           + ("; sample weights injected instead of its Mash/GSC step" if cfg["weighted"] else "")
           + ("; statsmodels.ttest_ind (not installed) replaced by the restatement of oracle/stats.py" if not cfg["binary"] else "")
           ) if real_cli else ("the reference's GenomeTester4 binaries for stages 1-2 + the restated per-k-mer loop of "
                               "modeling.py:677-858 (oracle/ref_pipeline.py)")
    return {"value": U * P / sec, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": f"bounded sample of the config: {n} {what} of {L} bp genomes x {P} phenotype column(s) (U={U}); {how}, "
                      f"-nt {threads}, scratch on /dev/shm; {sec:.1f} s per run"}, sec


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    cfg = CONFIGS[args.config]
    base, sec = cpu_reference_run(args.config, threads, args.steps, args.warmup, args.ref_samples, args.ref_genome_len)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32 k-mers / f64 statistics", "data": "synthetic",
            "config": {"workload": cfg["workload"], "k": K},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    from phenotypeseeker_b200.pipeline import KmerAssociation
    from phenotypeseeker_b200 import dist as psdist, synth_gpu

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as tdist
        tdist.init_process_group("nccl", device_id=device)
    cfg = CONFIGS[args.config]
    t0 = time.time()
    plan = synth_gpu.config_plan(args.config, n_samples=args.samples, genome_len=args.genome_len)
    N = plan.n_samples
    P = plan.pheno.shape[1]
    mine = list(psdist.sample_block(rank, world, N))
    renderer = synth_gpu.Renderer(plan, device)
    dev, spans = renderer.render(mine)            # this rank's text, device-resident
    torch.cuda.synchronize(device)
    t_gen = time.time() - t0
    host = torch.empty(dev.numel(), dtype=torch.uint8).pin_memory()
    host.copy_(dev)
    hv = host.numpy()
    host_bufs = {s: hv[o:o + n] for s, (o, n) in spans.items()}
    dev_bufs = {s: (dev.data_ptr() + o, n) for s, (o, n) in spans.items()}
    h2d_bytes = sum(n for _, n in spans.values())
    total_text = sum(renderer.max_text_bytes(s) for s in range(N))     # whole job, all ranks (upper estimate)
    pheno = plan.pheno
    weights = plan.weights if cfg["weighted"] else None
    ka = KmerAssociation(device=local)
    stream = torch.cuda.ExternalStream(ka.ctx.stream(), device=device)
    kw = dict(min_samples=2, max_samples=N - 2, pvalue_cutoff=cfg["pvalue"], omit_b=cfg["omit_b"], top_k=cfg["top_k"])
    # single GPU: k-mer ranges when the instances (2 pools x 4 B) and the matrix would not fit at once
    n_ranges = args.ranges or (max(1, math.ceil(total_text / 8.5e9)) if world == 1 else 1)
    state = {"splitters": None}

    def step(bufs):
        if world == 1 and n_ranges > 1:
            # once the range boundaries of the job are known (first step), the first super-range is scattered
            # while the samples are ingested — for host buffers that is during the upload
            ing = None
            if state["splitters"] is not None:
                ka.k = K
                ing = ka.plan_ranges(n_ranges, state["splitters"], h2d_bytes)["ingest"]
            ka.count([bufs[s] for s in mine], K, cfg["cutoff"], ingest_range=ing)
            U, res = ka.test_in_ranges(pheno, cfg["binary"], n_ranges, weights, splitters=state["splitters"],
                                       n_instances=h2d_bytes, **kw)
            state["splitters"] = ka.range_splitters     # balance hint, fixed for the job
            return U, res, {}
        return psdist.run_sharded(ka, bufs, N, K, pheno, cfg["binary"], weights, rank, world, device,
                                  cutoff=cfg["cutoff"], route=args.route, **kw)

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize(device)

    def timed(bufs, steps, warmup, profile=False):
        U, res, info = 0, None, {}
        for _ in range(warmup):
            U, res, info = step(bufs)
        if profile:
            ka.ctx.profile_reset()
            ka.ctx.profile(True)
        l0 = ka.ctx.launch_count()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record(stream)
        for _ in range(steps):
            U, res, info = step(bufs)
        e1.record(stream)
        barrier()
        wall = time.time() - w0
        ms = e0.elapsed_time(e1)
        if profile:
            ka.ctx.profile(False)
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        if world > 1:
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        return float(t.item()) / steps, U, res, info, (ka.ctx.launch_count() - l0) // steps, wall / steps

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, U, res, info, launches, _ = timed(dev_bufs, args.steps, args.warmup, profile=True)
    prof = ka.ctx.profile_table()
    del dev_bufs, dev                   # the device-resident copy of the text is not part of the end-to-end run
    torch.cuda.empty_cache()
    ms_e2e, U2, res2, _, _, wall_e2e = timed(host_bufs, max(1, args.e2e_steps or args.steps), 1)
    clocks = sampler.stop() if rank == 0 else None
    assert U == U2, (U, U2)
    dev_bytes = ka.ctx.device_bytes()
    if world > 1:
        tdist.barrier()
    if rank != 0:
        if world > 1:
            tdist.destroy_process_group()
        return
    digest = result_digest(U, res)
    assert digest == result_digest(U2, res2), "device-resident and host-buffer runs disagree"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, U, res)
    n_surv = int(sum(len(r.kmer) for r in res))
    d2h_bytes = n_surv * (8 * 6 + 4 * 2 + ka.ctx.row_words() * 4) + 64
    # the same (config, size) must give the same result on any number of GPUs: compare with the committed digests
    dkey = f"config{args.config}_n{N}_L{plan.genome_len}"
    dpath = os.path.join(ROOT, "tests", "golden", "bench_digests.json")
    known = {}
    if os.path.exists(dpath):
        with open(dpath) as f:
            known = json.load(f)
    digest_check = "no committed digest for this size"
    if dkey in known:
        assert known[dkey]["digest"] == digest and known[dkey]["U"] == U, \
            f"result differs from the committed digest of {dkey}: U={U} digest={digest} expected {known[dkey]}"
        digest_check = f"equals tests/golden/bench_digests.json[{dkey}] (written by a 1-GPU run)"
    if args.write_digest and world == 1:
        known[dkey] = {"digest": digest, "U": U, "survivors": n_surv}
        outs = [dpath] + ([os.path.join(ROOT, "gpurun_out", "bench_digests.json")] if os.path.isdir(os.path.join(ROOT, "gpurun_out")) else [])
        for op in outs:       # gpurun_out/ is what comes back from the GPU box
            with open(op, "w") as f:
                json.dump(known, f, indent=1, sort_keys=True)
    peak, peak_src = peaks()
    # dominant kernel = whichever kernel name took the most time
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    dom_name = max(prof, key=lambda k_: prof[k_]["ms"])
    dom = prof[dom_name]
    per_launch_ms = dom["ms"] / max(dom["launches"], 1)
    per_launch_bytes = dom["alg_bytes"] / max(dom["launches"], 1)
    achieved = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        ent = tj.get(f"config{args.config}", {})
        if ent.get("kernel") == dom_name and world == 1 and ent.get("n_samples") == N and ent.get("dram_bytes_per_step"):
            traffic = ent["dram_bytes_per_step"] / max(dom["launches"] // args.steps, 1)     # per launch, like `achieved`
    # whole-step algorithmic bytes by SURVEY.md 8d: B1 = sum(L/4 + 4 D_s), B2 = sum(4 D_s) + U (4 + R),
    # B3 = U R + survivors (4 + 24 + R); D_s ~ positions (assemblies: nearly every k-mer is distinct)
    n_rec = float(h2d_bytes) * world if not plan.reads else 0.0
    R = 4 * ((N + 31) // 32)
    step_bytes = (n_rec / 4 + 4 * n_rec) + (4 * n_rec + U * (4 + R)) + (U * R + n_surv * (28 + R))
    line = {
        "metric": METRIC, "value": U * P / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32 k-mers / f64 statistics", "data": "synthetic",
        "config": {"workload": cfg["workload"], "k": K, "n_samples": N, "genome_len": plan.genome_len,
                   "phenotype_columns": P, "union_kmers": U, "union_kmers_per_s": U / (ms_dev * 1e-3),
                   "survivors_read_back": n_surv, "input_bytes": int(h2d_bytes * world) if world > 1 else int(h2d_bytes),
                   "kmer_ranges": n_ranges, "result_digest": digest, "digest_check": digest_check,
                   "l2": "inputs (GBs of text, GBs of k-mer instances) are far larger than the 126 MB L2",
                   "parallelism": f"kmer-range-shard x{world}" if world > 1 else f"1 GPU, {n_ranges} k-mer range(s)",
                   "device_bytes": int(dev_bytes)},
        "e2e": {"value": U * P / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes),
                "d2h_bytes_per_step": int(d2h_bytes), "ms_per_step": ms_e2e, "wall_ms_per_step": wall_e2e * 1e3},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "launches_per_step": dom["launches"] // args.steps,
                     "ms_per_launch": per_launch_ms, "alg_bytes_per_launch": per_launch_bytes,
                     "share_of_kernel_time": dom["ms"] / tot_ms,
                     "whole_step_alg_bytes": step_bytes if n_rec else None,
                     "whole_step_frac": (step_bytes / world / (ms_dev * 1e-3) / 1e9 / peak) if n_rec else None},
        "kernels": {k_: {"ms_per_step": v["ms"] / args.steps, "launches_per_step": v["launches"] // args.steps,
                         "alg_GBps": (v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else None}
                    for k_, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])},
        "clocks": clocks,
        "gen_seconds": t_gen,
    }
    if world > 1 and info.get("route") == "pages":
        # NVLink roofline of the exchange: bytes that leave this GPU inside k_scatter1 / its duration / 770 GB/s measured peer copy
        sc = prof.get("scatter1")
        if sc and sc["ms"] > 0:
            out_bytes = 4.0 * h2d_bytes * (world - 1) / world * args.steps
            gbs = out_bytes / (sc["ms"] * 1e-3) / 1e9
            line["roofline"]["nvlink"] = {"achieved": gbs, "peak": 770.0, "unit": "GB/s", "frac": gbs / 770.0,
                                          "what": "k-mer instance bytes leaving rank 0 inside k_scatter1 (4 B each) / kernel time; "
                                                  "peak = measured peer copy per direction (B200_PROFILING.md), nominal 900"}
    if world == 1 and not args.no_cpu_baseline:
        try:
            base, _ = cpu_reference_run(args.config, os.cpu_count() or 1, n_samples=args.ref_samples, genome_len=args.ref_genome_len)
            line["cpu_baseline"] = base
        except Exception as e:  # the baseline must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference",
                                    "sample": f"failed: {type(e).__name__}: {e}"}
    print(json.dumps(line))
    if world > 1:
        tdist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=5, choices=[1, 2, 3, 4, 5],
                    help="BASELINE.json configs[c-1]; default 5 = the headline shape (5,000 x 5 Mbp x 10 phenotype columns)")
    ap.add_argument("--samples", type=int, default=None, help="override the number of samples of the config")
    ap.add_argument("--genome-len", type=int, default=None, help="override the genome length of the config")
    ap.add_argument("--ranges", type=int, default=None, help="k-mer ranges on one GPU (default: from the input size)")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--ref-samples", type=int, default=None, help="samples of the bounded sample the CPU reference is timed on")
    ap.add_argument("--ref-genome-len", type=int, default=None, help="genome length of that bounded sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--write-digest", action="store_true", help="record this (1-GPU) result in tests/golden/bench_digests.json")
    ap.add_argument("--route", default="auto", choices=["auto", "pages", "streams"],
                    help="multi-GPU exchange route (phenotypeseeker_b200/dist.py)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step (device-resident run) as DIR/<name>.npy, float64, "
                         "at most 64 MB (a seeded sample of the survivors beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
