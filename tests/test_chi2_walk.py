"""The unweighted chi2 bit walk for rows that fill the warp (N > 2,048 samples) and the reachability cut
(phenotypeseeker_b200/csrc/ps_chi2_reach.h). On the host: the cut against every 2x2 table for random margins with
and without NA, small N, N = 5,000 and 8,190, thresholds from 1e-2 down to 1e-12 and the sample filter at its
edges. On the GPU: rows built to hit the edges of the word mapping and of the cut, against the oracle."""
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import kmers as ok
from oracle import stats as ostats


def test_reach_interval_against_every_table(tmp_path):
    exe = str(tmp_path / "chi2_reach_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "native", "chi2_reach_check.cpp")])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


def _reach(n1, n0, min_s, max_s, thr):
    """ps_chi2_reach restated: the hull of the n_with whose largest chi2 reaches 0.98 chi2_min."""
    need = 0.98 * (-2.0 * math.log(thr))
    T = n1 + n0
    hit = []
    for m in range(max(min_s, 0), min(max_s, T - 2) + 1):
        den = (n1 * n0) * (m * (T - m))
        if den == 0:
            continue
        best = max(T * (a * T - n1 * m) ** 2 / den for a in (max(0, m - n0), min(m, n1)))
        if best >= need:
            hit.append(m)
    return (hit[0], hit[-1]) if hit else (1, 0)


def _rows(rng, N, ph1, m_edges):
    """Presence rows: bits only in the words of lanes 0-7, all in one lane's words, spread evenly, at the popcounts
    in m_edges, at 2 np = N +- 1, and rows of phenotype-1 samples (survivors)."""
    W = (N + 31) // 32
    words = np.arange(W)
    samples_of = lambda wsel: np.concatenate([np.arange(w * 32, min(w * 32 + 32, N)) for w in words[wsel]])
    pools = [samples_of(words % 32 < 8), samples_of(words % 32 == 5), samples_of(words % 32 == (W - 1) % 32),
             np.arange(N)]
    rows = []
    for m in sorted(set(m_edges) | {N // 2, N // 2 + 1, (N - 1) // 2, (N + 1) // 2, 2, N - 2}):
        for pool in pools:
            for dense in (False, True):
                k = m if not dense else N - m
                if not 0 <= k <= len(pool) or not 0 < m < N:
                    continue
                r = np.zeros(N, np.uint8)
                r[rng.choice(pool, size=k, replace=False)] = 1
                rows.append(r if not dense else 1 - r)
    one = np.flatnonzero(ph1)
    for flip in (0.0, 0.01, 0.05):
        r = ph1.astype(np.uint8) ^ (rng.random(N) < flip).astype(np.uint8)
        rows.append(r)
        if len(one) > 40:                                    # a strong row with few samples
            r = np.zeros(N, np.uint8); r[one[:40 + int(flip * 100)]] = 1
            rows.append(r)
    return np.array(rows, dtype=np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("N,P,na_rate", [(2049, 3, 0.0), (3073, 5, 0.02), (4096, 12, 0.02), (4097, 12, 0.02),
                                          (5000, 10, 0.0), (5000, 13, 0.03), (6000, 4, 0.0), (7000, 11, 0.01),
                                          (8190, 11, 0.0)])
def test_full_warp_walk_and_reach_cut(N, P, na_rate, monkeypatch):
    """Every instance of k_test_chi2_sp_warp, KW = ceil(W / 32) = 3 (N = 2,049: lane 0 owns three words, the others
    two) to 8. The context is created with PSKMER_CHI2=walk so that narrow tables (W * P < 512) take the bit walk
    too, and rows of more than 16 uint4 (64 words) go to the full-warp kernel."""
    from phenotypeseeker_b200._native import Context
    rng = np.random.default_rng(N + 7 * P)
    ph = (rng.random((P, N)) < rng.uniform(0.2, 0.6, (P, 1))).astype(np.int8)
    if na_rate:
        ph[rng.random((P, N)) < na_rate] = -1
        ph[0][ph[0] < 0] = 0                                  # one complete column next to incomplete ones
    thr = 0.05 / 9e7
    edges = []
    for p in range(P):
        n1, n0 = int((ph[p] == 1).sum()), int((ph[p] == 0).sum())
        lo, hi = _reach(n1, n0, 2, N - 2, thr)
        nna = N - n1 - n0
        edges += [lo - 1, lo, hi, hi + 1, hi + nna, hi + nna + 1]
    pres = _rows(rng, N, ph[P - 1] == 1, edges)
    U = pres.shape[0]
    oracle = [ostats.chi2_rows(pres, ph[p], np.ones(N), 2, N - 2) for p in range(P)]
    monkeypatch.setenv("PSKMER_CHI2", "walk")
    ctx = Context(0)
    try:
        ctx.begin(16, N)
        assert ctx.row_words() > 64                           # one row per warp
        rows = np.zeros((U, ctx.row_words()), dtype=np.uint32)
        packed = ok.pack_rows(pres)
        rows[:, :packed.shape[1]] = packed
        ctx.load_matrix(rows, np.arange(U, dtype=np.uint64))
        for t in (2.0, thr, 1e-3):
            ns = ctx.test_chi2(ph, None, 2, N - 2, t)
            sv = ctx.fetch_survivors(ns)
            hits = 0
            for p, o in enumerate(oracle):
                keep = o["tested"] & ~np.isnan(o["p"]) & (o["p"] < t)
                sel = sv["pheno"] == p
                order = np.argsort(sv["row"][sel], kind="stable")
                assert np.array_equal(sv["row"][sel][order], np.nonzero(keep)[0]), (t, p)
                assert np.array_equal(sv["n_with"][sel][order], o["n_with"][keep])
                assert np.array_equal(sv["stat"][sel][order], o["stat"][keep])       # bit-identical
                hits += int(keep.sum())
            assert hits > 0
    finally:
        ctx.close()
