"""Row popcounts of the config-5 matrix and the walk iterations of the unweighted chi2 kernels.

Builds the config-5 job as bench.py does (same synthetic plan, k-mer ranges through KmerAssociation.test_in_ranges)
and, for every range, reads its matrix in slices before the range is tested and computes on the device:
  * the histogram of row popcounts np;
  * the rows the sample filter keeps (np >= min_samples: the parent's walk) and the rows the reachability cut keeps
    (np inside the envelope of the columns' ps_chi2_reach intervals at the range's threshold);
  * the warp iterations of the walk per row for the parent's mapping (lane l owns uint4 l and l + 32, one loop per
    32-bit word: sum over words of the max over lanes) and for k_test_chi2_sp_warp (lane l owns words l, l + 32, ...,
    one loop: max over lanes of the lane's total). The walked bits are the set ones, or the cleared valid ones when
    2 np > N.
usage: python profiles/r4/chi2_rows.py OUT.json   (needs a B200-sized device: the whole config-5 job)"""
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from bench import CONFIGS, K  # noqa: E402
from phenotypeseeker_b200 import synth_gpu  # noqa: E402
from phenotypeseeker_b200.pipeline import KmerAssociation  # noqa: E402

SLICE = 1 << 18      # rows per slice read back


def popc32(x):
    """popcount of int64 tensors holding 32-bit values"""
    x = x - ((x >> 1) & 0x55555555)
    x = (x & 0x33333333) + ((x >> 2) & 0x33333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F
    return ((x * 0x01010101) >> 24) & 0xFF


def reach_envelope(ph, N, min_s, max_s, thr):
    """ps_chi2_reach per column (phenotypeseeker_b200/csrc/ps_chi2_reach.h) and the popcount envelope of the kernel"""
    need = 0.98 * (-2.0 * math.log(thr) if thr > 0 else 1e300)
    lo_all, hi_all = None, None
    for j in range(ph.shape[1]):
        n1, n0 = int((ph[:, j] == 1).sum()), int((ph[:, j] == 0).sum())
        T = n1 + n0
        m = np.arange(max(min_s, 0), min(max_s, T - 2) + 1, dtype=np.float64)
        with np.errstate(all="ignore"):
            den = (float(n1) * n0) * (m * (T - m))
            best = np.fmax(*[T * (a * T - n1 * m) ** 2 / den for a in (np.maximum(0, m - n0), np.minimum(m, n1))])
        ok = np.flatnonzero(best >= need)
        if ok.size == 0:
            continue
        lo, hi = int(m[ok[0]]), int(m[ok[-1]]) + (N - T)
        lo_all = lo if lo_all is None else min(lo_all, lo)
        hi_all = hi if hi_all is None else max(hi_all, hi)
    return (1, 0) if lo_all is None else (lo_all, hi_all)


def walk_iterations(words, N):
    """words: R x wp int64 (32-bit values) -> (np, old iterations, new iterations) per row"""
    R, wp = words.shape
    wv = (N + 31) // 32
    pc = popc32(words)
    npop = pc.sum(1)
    valid = torch.clamp(N - 32 * torch.arange(wp, device=words.device), 0, 32)
    walked = torch.where((2 * npop > N)[:, None], valid[None, :] - pc, pc)
    walked[:, wv:] = 0
    # parent: lane l owns uint4 l and l + 32 (words 4l..4l+3 and 128+4l..); one loop per word
    old = torch.zeros(R, 256, dtype=walked.dtype, device=walked.device)
    old[:, :wp] = walked
    old_it = old.view(R, 2, 32, 4).amax(2).sum((1, 2))
    # k_test_chi2_sp_warp: lane l owns words l + 32k; one loop over all of them
    kw = (wv + 31) // 32
    new = torch.zeros(R, 32 * kw, dtype=walked.dtype, device=walked.device)
    new[:, :wv] = walked[:, :wv]
    new_it = new.view(R, kw, 32).sum(1).amax(1)
    return npop, old_it, new_it


def main():
    out = sys.argv[1]
    cfg = CONFIGS[5]
    device = torch.device("cuda", 0)
    plan = synth_gpu.config_plan(5)
    N = plan.n_samples
    renderer = synth_gpu.Renderer(plan, device)
    dev, spans = renderer.render(list(range(N)))
    torch.cuda.synchronize(device)
    bufs = [(dev.data_ptr() + spans[s][0], spans[s][1]) for s in range(N)]
    n_instances = sum(n for _, n in spans.values())
    total_text = sum(renderer.max_text_bytes(s) for s in range(N))
    n_ranges = max(1, math.ceil(total_text / 8.5e9))
    min_s, max_s = 2, N - 2
    ph = np.where(np.isnan(plan.pheno), -1, plan.pheno).astype(np.int8)
    ka = KmerAssociation(device=0)
    acc = dict(rows=0, rows_filter=0, rows_cut=0, old_it_filter=0, new_it_filter=0, new_it_cut=0)
    hist = torch.zeros(N + 1, dtype=torch.int64, device=device)
    per_range = []
    test = ka.test

    def test_and_count(pheno, binary, weights=None, pvalue_cutoff=0.05, n_union_total=None, **kw):
        U = ka.U                                   # this range's rows; n_union_total: the rows up to it (Bonferroni)
        thr = float(pvalue_cutoff) / float(n_union_total)
        lo, hi = reach_envelope(ph, N, min_s, max_s, thr)
        r = dict(U=int(U), thr=thr, np_lo=lo, np_hi=hi, rows_filter=0, rows_cut=0, old_it_filter=0, new_it_filter=0,
                 new_it_cut=0)
        for first in range(0, U, SLICE):
            cnt = min(SLICE, U - first)
            w = torch.from_numpy(ka.ctx.get_rows(first, cnt).view(np.int32)).to(device).long() & 0xFFFFFFFF
            npop, old_it, new_it = walk_iterations(w, N)
            hist.add_(torch.bincount(npop, minlength=N + 1)[:N + 1])
            f = npop >= min_s
            c = (npop >= lo) & (npop <= hi)
            r["rows_filter"] += int(f.sum())
            r["rows_cut"] += int(c.sum())
            r["old_it_filter"] += int(old_it[f].sum())
            r["new_it_filter"] += int(new_it[f].sum())
            r["new_it_cut"] += int(new_it[c].sum())
        per_range.append(r)
        acc["rows"] += int(U)
        for k in ("rows_filter", "rows_cut", "old_it_filter", "new_it_filter", "new_it_cut"):
            acc[k] += r[k]
        return test(pheno, binary, weights, pvalue_cutoff=pvalue_cutoff, n_union_total=n_union_total, **kw)

    ka.test = test_and_count
    ka.count(bufs, K, cfg["cutoff"])
    del bufs, dev                                  # the text is consumed; the slices below need the room
    torch.cuda.empty_cache()
    ka.test_in_ranges(plan.pheno, cfg["binary"], n_ranges, None, n_instances=n_instances, min_samples=min_s,
                      max_samples=max_s, pvalue_cutoff=cfg["pvalue"], omit_b=cfg["omit_b"], top_k=cfg["top_k"])
    rf, rc = max(acc["rows_filter"], 1), max(acc["rows_cut"], 1)
    summary = dict(
        n_samples=N, n_ranges=n_ranges, union_rows=acc["rows"],
        rows_passing_sample_filter=acc["rows_filter"], rows_inside_reach_envelope=acc["rows_cut"],
        walk_iterations_per_filtered_row_old_mapping=acc["old_it_filter"] / rf,
        walk_iterations_per_filtered_row_new_mapping=acc["new_it_filter"] / rf,
        walk_iterations_per_walked_row_new_kernel=acc["new_it_cut"] / rc,
        total_walk_iterations=dict(old=acc["old_it_filter"], new_mapping_no_cut=acc["new_it_filter"],
                                   new=acc["new_it_cut"]),
        per_range=per_range, popcount_hist=hist.cpu().tolist())
    with open(out, "w") as fh:
        json.dump(summary, fh)
    print(json.dumps({k: v for k, v in summary.items() if k not in ("popcount_hist", "per_range")}, indent=1))


if __name__ == "__main__":
    main()
