"""GPU parity tests: the CUDA path, called through the C-ABI (ctypes), against the oracle and the
golden vectors generated from the real reference. Bit-exact for k-mer sets, counts, union and
matrix; 1e-6 relative (stated by north_star) for weighted chi2 / Welch statistics and p-values;
unweighted chi2 is exact-integer arithmetic and must be bit-identical."""
import math

import numpy as np
import pytest

from conftest import stage3_inputs
from oracle import kmers as ok
from oracle import stats as ostats
from phenotypeseeker_b200 import synth
from phenotypeseeker_b200.pipeline import KmerAssociation, unpack_rows

pytestmark = pytest.mark.gpu
RTOL = 1e-6  # north_star: chi-square/t statistics and p-values within 1e-6 relative


# ---------------------------------------------------------------------------------------
# stage 1: per-sample k-mer lists == glistmaker | glistquery

def test_golden_kmer_lists(ctx, golden_kmer_lists):
    for c in golden_kmer_lists:
        ctx.begin(c["k"], 1)
        ctx.add_samples(0, [c["data"]])
        km, ct = ctx.sample_kmers(0)
        assert np.array_equal(km, c["kmers"]), (c["name"], c["k"])
        assert np.array_equal(ct, c["counts"]), (c["name"], c["k"])


@pytest.mark.parametrize("k", [1, 2, 5, 13, 15, 16, 17, 21, 31, 32])
def test_kmer_lists_vs_oracle_all_k(ctx, k):
    ds = synth.make_dataset(3, genome_len=30_000, seed=100 + k)
    ctx.begin(k, 3)
    ctx.add_samples(0, ds.files)
    for s in range(3):
        km, ct = ctx.sample_kmers(s)
        okm, oct_ = ok.count_kmers(ds.files[s], k)
        assert np.array_equal(km, okm) and np.array_equal(ct, oct_)


def test_ragged_and_empty_inputs(ctx):
    files = [b"", b">only header\n", b">h\nACG\n", b"no records at all\n", b">h\n" + b"ACGT" * 5000,
             b">a\nAC\n>b\nGT\n", b"\n\n>x\n" + b"N" * 4096 + b"ACGTACGTACGTACGTACGT\n"]
    ctx.begin(16, len(files))
    ctx.add_samples(0, files)
    for s, f in enumerate(files):
        km, ct = ctx.sample_kmers(s)
        okm, oct_ = ok.count_kmers(f, 16)
        assert np.array_equal(km, okm) and np.array_equal(ct, oct_), s
    U = ctx.build_union()
    u = ok.union([ok.count_kmers(f, 16)[0] for f in files])
    assert U == len(u) and np.array_equal(ctx.get_union(), u)


def test_tile_boundaries(ctx):
    # headers, newlines and invalid bytes right at 64-byte chunk / 16384-byte tile edges
    rng = np.random.default_rng(9)
    for shift in (0, 1, 15, 16, 17, 63, 64, 65, 4095, 4096, 4097, 16383, 16384, 16385):
        seq = rng.choice(list(b"ACGT"), size=40000).astype(np.uint8).tobytes()
        f = (b">" + b"h" * shift + b"\n" + seq[:4000] + b"\n>" + b"x" * (16384 - 7) + b"\n" + seq[4000:20000] +
             b"N\n" + b">" + b"y" * (4096 - 3) + b"\n" + seq[20000:] + b"\n")
        ctx.begin(16, 1)
        ctx.add_samples(0, [f])
        km, ct = ctx.sample_kmers(0)
        okm, oct_ = ok.count_kmers(f, 16)
        assert np.array_equal(km, okm) and np.array_equal(ct, oct_), shift


def test_fastq_reads_and_cutoff(ctx):
    ds = synth.config(3, tiny=True)          # 4 raw-read samples, 30x of 20 kbp
    for cutoff in (1, 3):
        ctx.begin(16, ds.n_samples, cutoff)
        ctx.add_samples(0, ds.files)
        lists = []
        for s in range(ds.n_samples):
            km, ct = ctx.sample_kmers(s, cutoff)
            okm, oct_ = ok.count_kmers(ds.files[s], 16, cutoff)
            assert np.array_equal(km, okm) and np.array_equal(ct, oct_)
            lists.append((okm, oct_))
        U = ctx.build_union()
        u = ok.union([l[0] for l in lists])
        assert U == len(u) and np.array_equal(ctx.get_union(), u)
        pres = ok.presence_matrix(u, lists)
        assert np.array_equal(unpack_rows(ctx.get_rows(), ds.n_samples), pres)


# ---------------------------------------------------------------------------------------
# stage 2: union + presence matrix == glistcompare -u + glistquery -l

@pytest.mark.parametrize("cfg,k", [(0, 16), (1, 13), (2, 16), (0, 21)])
def test_union_and_matrix(ctx, cfg, k):
    ds = synth.config(cfg, tiny=True)
    ctx.begin(k, ds.n_samples)
    ctx.add_samples(0, ds.files[:5])
    ctx.add_samples(5, ds.files[5:])          # two ingest batches
    lists = [ok.count_kmers(f, k) for f in ds.files]
    u = ok.union([l[0] for l in lists])
    assert ctx.build_union() == len(u)
    assert np.array_equal(ctx.get_union(), u)
    rows = ctx.get_rows()
    assert rows.shape[1] % 4 == 0
    assert np.array_equal(unpack_rows(rows, ds.n_samples), ok.presence_matrix(u, lists))
    assert not rows[:, (ds.n_samples + 31) // 32:].any()


def test_sample_groups_beyond_256(ctx):
    # N = 600 -> three sample groups of the paged partition (4-byte records carry sample & 255, the
    # page carries sample >> 8); group boundaries fall inside extraction tiles (streams are 4096
    # positions, tiles 8192)
    ds = synth.make_dataset(600, genome_len=2500, seed=78, n_clades=5, contigs=(1, 2))
    ctx.begin(13, 600)
    ctx.add_samples(0, ds.files)
    lists = [ok.count_kmers(f, 13) for f in ds.files]
    u = ok.union([l[0] for l in lists])
    assert ctx.build_union() == len(u)
    assert np.array_equal(ctx.get_union(), u)
    assert np.array_equal(unpack_rows(ctx.get_rows(), 600), ok.presence_matrix(u, lists))


def test_many_samples_wide_rows(ctx):
    # N = 300 -> 10 words/row (padded to 12): exercises multi-word rows and lane groups
    ds = synth.make_dataset(300, genome_len=3000, seed=77, n_clades=6, contigs=(1, 2))
    ctx.begin(16, 300)
    ctx.add_samples(0, ds.files)
    lists = [ok.count_kmers(f, 16) for f in ds.files]
    u = ok.union([l[0] for l in lists])
    assert ctx.build_union() == len(u)
    assert np.array_equal(unpack_rows(ctx.get_rows(), 300), ok.presence_matrix(u, lists))


@pytest.mark.parametrize("env", [{"PSKMER_ROWS": "sorted"}, {"PSKMER_BK_ROW_KB": "1"}, {"PSKMER_SC1": "regs"}])
@pytest.mark.parametrize("k", [9, 13, 16])
def test_row_builders_agree(ctx, env, k, monkeypatch):
    """Every way rows are built gives the same union and matrix as the oracle: the default (paged
    partition, bucket kernels reading their pages with 128-bit loads), a 1 KB row table (every non-trivial
    bucket goes through the big-bucket launch and several row windows), the register variant of k_scatter1
    (PSKMER_SC1=regs), and the full sort + run detection (PSKMER_ROWS=sorted)."""
    from phenotypeseeker_b200._native import Context
    rng = np.random.default_rng(5 + k)
    # low-complexity, AT-rich genomes: a few (top 16 bit) buckets hold most of the k-mers
    files = []
    for s in range(70):
        seq = rng.choice(list("ACGT"), size=6000, p=[0.47, 0.03, 0.03, 0.47])
        seq[rng.integers(0, 6000, 40)] = "N"
        files.append((">s%d\n" % s + "".join(seq) + "\n").encode())
    lists = [ok.count_kmers(f, k) for f in files]
    u = ok.union([l[0] for l in lists])
    pres = ok.presence_matrix(u, lists)
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    other = Context(0)
    try:
        for c in (ctx, other):
            c.begin(k, len(files))
            c.add_samples(0, files)
            assert c.build_union() == len(u)
            assert np.array_equal(c.get_union(), u)
            assert np.array_equal(unpack_rows(c.get_rows(), len(files)), pres)
            assert c.build_union() == len(u)                 # second build: buffers already sized
            assert np.array_equal(unpack_rows(c.get_rows(), len(files)), pres)
    finally:
        other.close()


def test_scatter1_register_variant_on_goldens_and_tile_edges(golden_kmer_lists, monkeypatch):
    """The register variant of k_scatter1 (PSKMER_SC1=regs: k-mers kept in registers between ranking and grouping;
    the default recomputes them) against the glistmaker goldens and headers / newlines / invalid bytes at chunk and
    tile edges."""
    from phenotypeseeker_b200._native import Context
    monkeypatch.setenv("PSKMER_SC1", "regs")
    c = Context(0)
    try:
        for g in golden_kmer_lists:
            c.begin(g["k"], 1)
            c.add_samples(0, [g["data"]])
            km, ct = c.sample_kmers(0)
            assert np.array_equal(km, g["kmers"]) and np.array_equal(ct, g["counts"]), (g["name"], g["k"])
        rng = np.random.default_rng(10)
        files = []
        for shift in (0, 1, 3, 4, 15, 16, 17, 59, 60, 61, 63, 64, 65, 4095, 4096, 4097, 16383, 16384, 16385):
            body = "".join(rng.choice(list("ACGT"), size=40_000))
            lines = "\n".join(body[i:i + 60] for i in range(0, len(body), 60))
            files.append((">" + "h" * shift + "\n" + lines[:20_000] + "\n>x y z\r\n" + lines[20_000:30_000].lower() +
                          "NNRY-*\n" + lines[30_000:] + ("\n" if shift % 2 else "")).encode())
        c.begin(16, len(files))
        c.add_samples(0, files)
        lists = [ok.count_kmers(f, 16) for f in files]
        for s_, l in enumerate(lists):
            km, ct = c.sample_kmers(s_)
            assert np.array_equal(km, l[0]) and np.array_equal(ct, l[1]), s_
        u = ok.union([l[0] for l in lists])
        assert c.build_union() == len(u)
        assert np.array_equal(c.get_union(), u)
        assert np.array_equal(unpack_rows(c.get_rows(), len(files)), ok.presence_matrix(u, lists))
    finally:
        c.close()


def test_kmer_range_shards_partition_the_union(ctx):
    ds = synth.config(0, tiny=True)
    ctx.begin(16, ds.n_samples)
    ctx.add_samples(0, ds.files)
    full_n = ctx.build_union()
    full_u, full_rows = ctx.get_union(), ctx.get_rows()
    cuts = [0] + [int(full_u[len(full_u) * i // 3]) for i in (1, 2)] + [0]
    got_u, got_rows = [], []
    for i in range(3):
        ctx.set_range(cuts[i], cuts[i + 1])
        ctx.build_union()
        got_u.append(ctx.get_union())
        got_rows.append(ctx.get_rows())
    assert sum(len(x) for x in got_u) == full_n
    assert np.array_equal(np.concatenate(got_u), full_u)
    assert np.array_equal(np.concatenate(got_rows), full_rows)


def test_lookup_matches_counts(ctx):
    ds = synth.config(0, tiny=True)
    ctx.begin(16, ds.n_samples)
    ctx.add_samples(0, ds.files)
    km, ct = ok.count_kmers(ds.files[2], 16)
    rng = np.random.default_rng(1)
    q = np.concatenate([rng.choice(km, 300), rng.integers(0, 1 << 32, 100).astype(np.uint64), km[:3], km[:3]])
    exp = ok.map_counts(q, km, ct)
    assert np.array_equal(ctx.lookup(2, q), exp)


# ---------------------------------------------------------------------------------------
# stage 3: chi2 / Welch == the real conduct_* methods (golden) and the oracle

def _load_presence(ctx, pres):
    ctx.begin(16, pres.shape[1])
    rows = np.zeros((pres.shape[0], ctx.row_words()), dtype=np.uint32)
    packed = ok.pack_rows(pres)
    rows[:, :packed.shape[1]] = packed
    ctx.load_matrix(rows, np.arange(pres.shape[0], dtype=np.uint64))


def test_stage3_against_golden_reference_rows(ctx, golden_stage3):
    checked = 0
    for case in golden_stage3:
        pres, ph, w = stage3_inputs(case)
        weights = None if np.all(w == 1.0) else w
        _load_presence(ctx, pres)
        U = case["U"]
        if case["kind"] == "chi2":
            thr = case["cutoff"] if case["omit_B"] else case["cutoff"] / U
            ns = ctx.test_chi2(ph, weights, case["min"], case["max"], thr)
        else:
            ns = ctx.test_welch(ph, weights, case["min"], case["max"], case["cutoff"] / U)
        sv = ctx.fetch_survivors(ns)
        got = {int(r): i for i, r in enumerate(sv["row"])}
        for r, exp in enumerate(case["rows"]):
            if exp is None:
                assert r not in got, (case["kind"], r)
                continue
            assert r in got, (case["kind"], r)
            i = got[r]
            assert exp[1] == round(float(sv["stat"][i]), 2)
            assert exp[2] == "%.2E" % sv["p"][i]
            if case["kind"] == "chi2":
                assert exp[3] == sv["n_with"][i]
                vec = exp[5:]
            else:
                assert exp[3] == round(float(sv["mean_x"][i]), 2) and exp[4] == round(float(sv["mean_y"][i]), 2)
                assert exp[5] == sv["n_with"][i]
                vec = exp[7:]
            assert list(unpack_rows(sv["rowbits"][i:i + 1], case["N"])[0]) == vec
            checked += 1
    assert checked > 100


@pytest.mark.parametrize("N,weighted,P", [(20, False, 1), (250, True, 3), (250, False, 2), (1000, True, 2),
                                          (5000, False, 10), (37, True, 1)])
def test_chi2_vs_oracle_random(ctx, N, weighted, P):
    rng = np.random.default_rng(N + P)
    U = 3000 if N <= 1000 else 600
    dens = rng.random((U, 1)) ** 2
    pres = (rng.random((U, N)) < dens).astype(np.uint8)
    ph = (rng.random((P, N)) < 0.4).astype(np.int8)
    ph[rng.random((P, N)) < 0.03] = -1
    pres[:50] = ((ph[0] == 1)[None, :] ^ (rng.random((50, N)) < 0.05)).astype(np.uint8)
    w = rng.gamma(2.0, 0.5, N) if weighted else None
    _load_presence(ctx, pres)
    ns = ctx.test_chi2(ph, w, 2, N - 2, 2.0)          # threshold 2.0: keep every tested row
    sv = ctx.fetch_survivors(ns)
    for p in range(P):
        o = ostats.chi2_rows(pres, ph[p], np.ones(N) if w is None else w, 2, N - 2)
        keep = o["tested"] & ~np.isnan(o["p"])
        sel = sv["pheno"] == p
        assert np.array_equal(sv["row"][sel], np.nonzero(keep)[0])
        assert np.array_equal(sv["n_with"][sel], o["n_with"][keep])
        if w is None:
            assert np.array_equal(sv["stat"][sel], o["stat"][keep])            # bit-identical
            np.testing.assert_allclose(sv["p"][sel], o["p"][keep], rtol=1e-13)
        else:
            np.testing.assert_allclose(sv["stat"][sel], o["stat"][keep], rtol=RTOL, atol=1e-12)
            np.testing.assert_allclose(sv["p"][sel], o["p"][keep], rtol=RTOL)
    # thresholded run keeps exactly the oracle's filtered set
    thr = 0.05 / U
    ns = ctx.test_chi2(ph, w, 2, N - 2, thr)
    sv = ctx.fetch_survivors(ns)
    for p in range(P):
        o = ostats.chi2_rows(pres, ph[p], np.ones(N) if w is None else w, 2, N - 2)
        assert np.array_equal(sv["row"][sv["pheno"] == p], np.nonzero(o["tested"] & (o["p"] < thr))[0])


@pytest.mark.parametrize("N,P,na_rate", [(5000, 13, 0.03), (8190, 3, 0.0), (9000, 2, 0.0), (250, 12, 0.0), (33, 11, 0.1),
                                          (1000, 10, 0.0)])
def test_chi2_unweighted_bit_walk_shapes(ctx, N, P, na_rate):
    """The unweighted kernel walks the row's set (or cleared) bits with packed per-sample column words, ten
    columns per walk, 12-bit fields: more than ten columns, columns with and without NA samples, rows from
    empty to full (both walk directions), the largest N it takes (8190) and one beyond (masked-popcount kernel)."""
    rng = np.random.default_rng(N * 3 + P)
    U = 400
    dens = np.concatenate([rng.random(U - 80) ** 3, 1.0 - rng.random(60) ** 3, [0.0, 1.0] * 10])[:, None]
    pres = (rng.random((U, N)) < dens).astype(np.uint8)
    ph = (rng.random((P, N)) < 0.4).astype(np.int8)
    if na_rate:
        ph[rng.random((P, N)) < na_rate] = -1
        ph[0][ph[0] < 0] = 1                                  # one complete column next to incomplete ones
    pres[:40] = ((ph[P - 1] == 1)[None, :] ^ (rng.random((40, N)) < 0.02)).astype(np.uint8)
    _load_presence(ctx, pres)
    ns = ctx.test_chi2(ph, None, 2, N - 2, 2.0)
    sv = ctx.fetch_survivors(ns)
    for p in range(P):
        o = ostats.chi2_rows(pres, ph[p], np.ones(N), 2, N - 2)
        keep = o["tested"] & ~np.isnan(o["p"])
        sel = sv["pheno"] == p
        assert np.array_equal(sv["row"][sel], np.nonzero(keep)[0]), p
        assert np.array_equal(sv["n_with"][sel], o["n_with"][keep])
        assert np.array_equal(sv["stat"][sel], o["stat"][keep])                # bit-identical
        np.testing.assert_allclose(sv["p"][sel], o["p"][keep], rtol=1e-13)


@pytest.mark.parametrize("N,weighted,P", [(12, False, 1), (100, True, 2), (1000, False, 2), (1000, True, 1),
                                          (2100, True, 1)])
def test_welch_vs_oracle_random(ctx, N, weighted, P):
    rng = np.random.default_rng(N * 7 + P)
    U = 1500
    dens = rng.random((U, 1))
    pres = (rng.random((U, N)) < dens).astype(np.uint8)
    ph = np.round(rng.normal(0, 2, (P, N)), 3)
    ph[rng.random((P, N)) < 0.02] = np.nan
    base = np.nan_to_num(ph[0])
    pres[:40] = ((base[None, :] + rng.normal(0, 1.5, (40, N))) > 0.5).astype(np.uint8)
    pres[40:60] = ((base[None, :] + rng.normal(0, 0.3, (20, N))) > 0.0).astype(np.uint8)   # tiny p-values
    w = rng.gamma(2.0, 0.5, N) + 0.05 if weighted else None
    _load_presence(ctx, pres)
    ns = ctx.test_welch(ph, w, 2, N - 2, 2.0)
    sv = ctx.fetch_survivors(ns)
    for p in range(P):
        o = ostats.welch_rows(pres, ph[p], np.ones(N) if w is None else w, 2, N - 2)
        keep = o["tested"] & ~np.isnan(o["p"])
        sel = sv["pheno"] == p
        assert np.array_equal(sv["row"][sel], np.nonzero(keep)[0])
        assert np.array_equal(sv["n_with"][sel], o["n_with"][keep])
        np.testing.assert_allclose(sv["stat"][sel], o["stat"][keep], rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(sv["p"][sel], o["p"][keep], rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(sv["mean_x"][sel], o["mean_x"][keep], rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(sv["mean_y"][sel], o["mean_y"][keep], rtol=RTOL, atol=1e-12)


@pytest.mark.parametrize("N,weighted", [(60, False), (400, True), (1000, True)])
def test_welch_discrete_phenotype_constant_groups(ctx, N, weighted):
    """Discrete phenotype values (MIC-like log2 steps, modeling.py:116-119): the LARGER group is often constant, or
    constant but for one or two samples, while the small group varies — its variance must come out as the
    reference computes it (exactly 0, or tiny), not as cancellation noise of the totals; both groups constant -> NaN -> dropped."""
    rng = np.random.default_rng(N + 3)
    U = 600
    ph = np.full((1, N), 2.0)
    odd = rng.choice(N, size=max(6, N // 10), replace=False)
    ph[0, odd] = rng.choice([-1.0, 0.0, 1.0, 3.0, 4.0, 1e3], size=len(odd))
    pres = np.zeros((U, N), dtype=np.uint8)
    for r in range(U):
        kind = r % 4
        if kind == 0:      # k-mer in most of the odd samples only: large group constant (or nearly)
            pres[r, rng.choice(odd, size=rng.integers(2, len(odd)), replace=False)] = 1
        elif kind == 1:    # k-mer in all but a few odd samples: the group WITH the k-mer is the large constant one
            pres[r] = 1
            pres[r, rng.choice(odd, size=rng.integers(2, len(odd)), replace=False)] = 0
        elif kind == 2:    # both groups constant
            pres[r, rng.choice(np.setdiff1d(np.arange(N), odd), size=rng.integers(2, 6), replace=False)] = 1
            pres[r, odd] = rng.integers(0, 2)
        else:
            pres[r] = rng.random(N) < rng.random()
    w = rng.gamma(2.0, 0.5, N) + 0.05 if weighted else None
    _load_presence(ctx, pres)
    ns = ctx.test_welch(ph, w, 2, N - 2, 2.0)
    sv = ctx.fetch_survivors(ns)
    o = ostats.welch_rows(pres, ph[0], np.ones(N) if w is None else w, 2, N - 2)
    keep = o["tested"] & ~np.isnan(o["p"])
    assert keep.sum() > U // 3
    assert np.array_equal(sv["row"], np.nonzero(keep)[0])
    np.testing.assert_allclose(sv["stat"], o["stat"][keep], rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(sv["p"], o["p"][keep], rtol=RTOL, atol=1e-300)


def test_select_top_equals_host_sort(ctx):
    """ps_select_top (radix-select on the p-value bit pattern, per phenotype column) keeps exactly what a
    host sort of ALL survivors by (p, row) would keep — including a column with fewer survivors than k."""
    rng = np.random.default_rng(123)
    N, U, P = 96, 30000, 3
    pres = (rng.random((U, N)) < rng.random(U)[:, None] * 0.9).astype(np.uint8)
    pres[:2000] = pres[0]                                   # many identical rows: ties in p
    rows = np.zeros((U, 4), dtype=np.uint32)
    packed = np.packbits(pres, axis=1, bitorder="little")
    rows.view(np.uint8).reshape(U, 16)[:, :packed.shape[1]] = packed
    pheno = (rng.random((N, P)) < 0.5).astype(np.float64)
    ka = KmerAssociation(ctx=ctx)
    ctx.begin(16, N)
    ka.k, ka.n_samples = 16, N
    ctx.load_matrix(rows, np.arange(U, dtype=np.uint64))
    ka.U = U
    full = ka.test(pheno, True, None, min_samples=2, max_samples=N - 2, pvalue_cutoff=0.3, omit_b=True)
    full[2] = full[2]
    for k in (1, 50, 700):
        cut = ka.test(pheno, True, None, min_samples=2, max_samples=N - 2, pvalue_cutoff=0.3, omit_b=True, top_k=k)
        assert ka.n_survivors == sum(len(r.kmer) for r in full)
        for f, c in zip(full, cut):
            order = np.lexsort((f.row, f.p))[:k]
            order.sort()
            assert np.array_equal(c.row, f.row[order]) and np.array_equal(c.p, f.p[order])
            assert np.array_equal(c.presence, f.presence[order])


def test_t_pvalue_far_tails(ctx):
    # strongly separated groups: p down to ~1e-200 (user_manual.md:76 shows 1e-60-scale rows)
    rng = np.random.default_rng(21)
    N, U = 600, 64
    ph = np.round(rng.normal(0, 1, N), 3)
    pres = np.zeros((U, N), dtype=np.uint8)
    for r in range(U):
        sep = 0.2 + 0.25 * r
        pres[r] = (ph + rng.normal(0, 1.0 / (1 + sep), N) > 0).astype(np.uint8)
    ph2 = ph + 3.0 * pres[-1]            # make the last rows extreme
    _load_presence(ctx, pres)
    for phv, w in ((ph, None), (ph2, rng.gamma(2.0, 0.5, N) + 0.1)):
        ns = ctx.test_welch(phv, w, 2, N - 2, 2.0)
        sv = ctx.fetch_survivors(ns)
        o = ostats.welch_rows(pres, phv, np.ones(N) if w is None else w, 2, N - 2)
        keep = o["tested"] & ~np.isnan(o["p"])
        assert np.array_equal(sv["row"], np.nonzero(keep)[0])
        assert o["p"][keep].min() < 1e-60
        np.testing.assert_allclose(sv["stat"], o["stat"][keep], rtol=RTOL)
        # below ~1e-300 the device exp() flushes to 0 where scipy still returns a denormal
        np.testing.assert_allclose(sv["p"], o["p"][keep], rtol=RTOL, atol=1e-300)


def test_t_pvalue_edges(ctx):
    # constant groups: zero variance in both -> NaN dof in the reference -> dropped
    N = 8
    pres = np.array([[1, 1, 1, 0, 0, 0, 0, 0], [1, 1, 1, 0, 0, 0, 0, 1], [0, 0, 0, 1, 1, 1, 1, 0]], np.uint8)
    ph = np.array([2.0, 2.0, 2.0, 5.0, 5.0, 5.0, 5.0, 1.0])
    _load_presence(ctx, pres)
    ns = ctx.test_welch(ph, None, 2, 6, 2.0)
    sv = ctx.fetch_survivors(ns)
    o = ostats.welch_rows(pres, ph, np.ones(N), 2, 6)
    keep = o["tested"] & ~np.isnan(o["p"])
    assert np.array_equal(sv["row"], np.nonzero(keep)[0])
    np.testing.assert_allclose(sv["p"], o["p"][keep], rtol=RTOL)


# ---------------------------------------------------------------------------------------
# whole path, every config shape at CI scale

@pytest.mark.parametrize("cfg,k", [(0, 16), (1, 16), (2, 13), (4, 16)])
def test_end_to_end_vs_oracle(ctx, cfg, k):
    ds = synth.config(cfg, tiny=True)
    ka = KmerAssociation(ctx=ctx)
    N = ds.n_samples
    omit_b = ds.binary
    pcut = 0.05 if ds.binary else 50.0
    res = ka.run(ds.files, k, ds.pheno, ds.binary, ds.weights, min_samples=2, max_samples=N - 2,
                 pvalue_cutoff=pcut, omit_b=omit_b)
    lists = [ok.count_kmers(f, k) for f in ds.files]
    u = ok.union([l[0] for l in lists])
    pres = ok.presence_matrix(u, lists)
    assert ka.U == len(u)
    total = 0
    for j, r in enumerate(res):
        if ds.binary:
            code = np.where(np.isnan(ds.pheno[:, j]), -1, ds.pheno[:, j]).astype(np.int8)
            o = ostats.chi2_rows(pres, code, ds.weights, 2, N - 2)
            thr = pcut
        else:
            o = ostats.welch_rows(pres, ds.pheno[:, j], ds.weights, 2, N - 2)
            thr = pcut / len(u)
        keep = o["tested"] & (o["p"] < thr)
        assert np.array_equal(r.row, np.nonzero(keep)[0])          # identical filtered k-mer set
        assert np.array_equal(r.kmer, u[keep])
        assert np.array_equal(r.presence, pres[keep])
        np.testing.assert_allclose(r.stat, o["stat"][keep], rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(r.p, o["p"][keep], rtol=RTOL)
        total += keep.sum()
    assert total > 0


@pytest.mark.parametrize("case", ["assemblies_k16", "groups_k13", "reads_cutoff2"])
def test_page_route_equals_single_build(ctx, case):
    """The multi-GPU exchange on one GPU: three contexts play three ranks. Each ingests its own block
    of samples, k_scatter1 appends every k-mer instance to a page of its owner's pool (here plain
    device pointers instead of CUDA IPC mappings), and every owner builds its k-mer range from its
    pool. Concatenated, the ranges must reproduce union and matrix of the single build."""
    import torch
    from phenotypeseeker_b200._native import Context
    from phenotypeseeker_b200.dist import sample_block
    G, cutoff = 3, 1
    if case == "assemblies_k16":
        ds, k = synth.config(0, tiny=True), 16
    elif case == "groups_k13":
        ds, k = synth.make_dataset(520, genome_len=2500, seed=79, n_clades=5, contigs=(1, 2)), 13    # 3 sample groups
    else:
        ds, k, cutoff = synth.config(3, tiny=True), 16, 2
    N = ds.n_samples
    ctx.begin(k, N, cutoff)
    ctx.add_samples(0, ds.files)
    full_n = ctx.build_union()
    full_u, full_rows = ctx.get_union(), ctx.get_rows()
    spl = ctx.sample_quantiles(0, G)
    assert len(spl) == G - 1 and spl == sorted(spl)
    ranks = [Context(0) for _ in range(G)]
    try:
        for r, c in enumerate(ranks):
            mine = list(sample_block(r, G, N))
            c.begin(k, N, cutoff)
            c.add_samples(mine[0], [ds.files[s] for s in mine])
        pages = max(c.route_pages_needed(G) for c in ranks)
        ptrs = [c.route_setup(G, r, spl, pages) for r, c in enumerate(ranks)]
        for c in ranks:
            c.route_peers([p[0] for p in ptrs], [p[1] for p in ptrs])
            c.route_begin()
        torch.cuda.synchronize()
        for c in ranks:
            c.route_scatter()
        torch.cuda.synchronize()
        got_u, got_rows = [], []
        for r, c in enumerate(ranks):
            U_r, ovf = c.route_build()
            assert not ovf
            got_u.append(c.get_union())
            got_rows.append(c.get_rows())
            assert len(got_u[-1]) == U_r
            if r > 0 and U_r:
                assert got_u[-1][0] >= spl[r - 1]
            if r < G - 1 and U_r:
                assert got_u[-1][-1] < spl[r]
        assert sum(len(x) for x in got_u) == full_n
        assert np.array_equal(np.concatenate(got_u), full_u)
        assert np.array_equal(np.concatenate(got_rows), full_rows)
    finally:
        for c in ranks:
            c.close()


@pytest.mark.parametrize("cfg,binary_omit", [(0, True), (1, False), (2, False)])
def test_ranged_run_equals_single_run(ctx, cfg, binary_omit):
    """Memory-bounded operation: building and testing the k-mer space in 3 ranges gives exactly the
    survivors (rows, statistics, presence) of one build, with the Bonferroni U known only at the end."""
    ds = synth.config(cfg, tiny=True)
    ka = KmerAssociation(ctx=ctx)
    N = ds.n_samples
    pcut = 0.05 if ds.binary else 200.0
    if cfg == 1:
        pcut = 500.0          # Bonferroni on: keep the test non-trivial at CI scale
    kw = dict(min_samples=2, max_samples=N - 2)
    one = ka.run(ds.files, 16, ds.pheno, ds.binary, ds.weights, pvalue_cutoff=pcut, omit_b=binary_omit, **kw)
    U1 = ka.U
    # (ranges, super-ranges): 0 = every range extracts its own k-mers; otherwise the ranges of a super-range
    # share one extraction into the level-1 page pool (ps_scatter_range) and follow top-byte boundaries
    for n_ranges, n_super in [(3, 0), (3, None), (4, 1), (5, 2)]:
        ka.count(ds.files, 16)
        U3, three = ka.test_in_ranges(ds.pheno, ds.binary, n_ranges, ds.weights, pvalue_cutoff=pcut, omit_b=binary_omit,
                                      n_super=n_super, n_instances=sum(len(f) for f in ds.files), **kw)
        assert U3 == U1, (n_ranges, n_super)
        total = 0
        for a, b in zip(one, three):
            assert np.array_equal(a.row, b.row) and np.array_equal(a.kmer, b.kmer)
            assert np.array_equal(a.stat, b.stat) and np.array_equal(a.p, b.p)
            assert np.array_equal(a.presence, b.presence) and np.array_equal(a.n_with, b.n_with)
            total += len(a.kmer)
        assert total > 0
    # the first super-range scattered while the samples are ingested (ps_ingest_scatter): same result, and
    # ps_scatter_range finds its work done (it only closes the pages: one launch)
    n_inst = sum(len(f) for f in ds.files)
    ka.count(ds.files, 16)
    plan = ka.plan_ranges(4, ctx.sample_quantiles(0, 4), n_inst, 2)
    assert plan["ingest"] is not None and plan["ingest"][0] == 0 and plan["ingest"][1] == plan["splitters"][1]
    ka.count(ds.files, 16, ingest_range=plan["ingest"])
    l0 = ctx.launch_count()
    ctx.scatter_range(*plan["ingest"][:3])
    assert ctx.launch_count() - l0 == 1
    ka.count(ds.files, 16, ingest_range=plan["ingest"])
    U4, four = ka.test_in_ranges(ds.pheno, ds.binary, 4, ds.weights, pvalue_cutoff=pcut, omit_b=binary_omit,
                                 splitters=plan["splitters"], n_super=2, n_instances=n_inst, **kw)
    assert U4 == U1
    for a, b in zip(one, four):
        assert np.array_equal(a.row, b.row) and np.array_equal(a.stat, b.stat) and np.array_equal(a.presence, b.presence)
    # announced, but another range is asked for: the pool is not used, everything is extracted again
    ka.count(ds.files, 16, ingest_range=plan["ingest"])
    U3b, three_b = ka.test_in_ranges(ds.pheno, ds.binary, 3, ds.weights, pvalue_cutoff=pcut, omit_b=binary_omit, n_super=0, **kw)
    assert U3b == U1 and all(np.array_equal(a.row, b.row) for a, b in zip(one, three_b))
    ka.count(ds.files, 16, ingest_range=plan["ingest"])          # ... also when the whole space is built at once
    assert ka.build() == U1
    # a build of some other range after a grouped run extracts again (the pool is not reused by mistake)
    q = ctx.sample_quantiles(0, 2)
    ctx.scatter_range(0, 0)
    ctx.set_range(q[0] + 12345, 0)
    u_hi = ctx.build_union()
    ctx.set_range(0, q[0] + 12345)
    assert u_hi + ctx.build_union() == U1
    ctx.set_range(0, 0)


# ---------------------------------------------------------------------------------------
# --kmerDB (modeling.py:367-372): the union cut down to a database's k-mers, on the device

@pytest.mark.parametrize("N,k", [(20, 13), (300, 16)])
def test_kmerdb_intersection_on_device(ctx, N, k):
    ds = synth.make_dataset(N, genome_len=20_000, seed=77 + N)
    lists = [ok.count_kmers(f, k) for f in ds.files]
    u = ok.union([l[0] for l in lists])
    pres = ok.presence_matrix(u, lists)
    db_text = ds.files[0][:9000] + b">extra\nACGTACGTTTGACCAGTAGGATCCAAGT\n" + ds.files[N // 2][4000:15000]
    ka = KmerAssociation(ctx=ctx)
    db = ka.kmers_of(db_text, k)                               # glistmaker on the database (GPU)
    assert np.array_equal(db, ok.count_kmers(db_text, k)[0])
    ka.count(ds.files, k)
    assert ka.build() == len(u)
    keep = np.isin(u, db)
    assert 0 < keep.sum() < len(u)
    assert ka.restrict_to(db) == int(keep.sum())               # ps_restrict_union
    assert np.array_equal(ctx.get_union(), u[keep])
    assert np.array_equal(unpack_rows(ctx.get_rows(), N), pres[keep])
    # stage 3 runs on the restricted matrix with the restricted U as the Bonferroni denominator
    res = ka.test(ds.pheno[:, :1], True, None, min_samples=2, max_samples=N - 2, pvalue_cutoff=0.05, omit_b=True)[0]
    o = ostats.chi2_rows(pres[keep], ds.pheno[:, 0].astype(np.int8), np.ones(N), 2, N - 2)
    sel = o["tested"] & (o["p"] < 0.05)
    assert np.array_equal(res.kmer, u[keep][sel]) and np.array_equal(res.stat, o["stat"][sel])
    # the host round trip (ps_get_union / ps_get_rows / ps_load_matrix) gives the same matrix
    ka.count(ds.files, k)
    ka.build()
    assert ka._restrict_to_host(db) == int(keep.sum())
    assert np.array_equal(ctx.get_union(), u[keep])
    assert np.array_equal(unpack_rows(ctx.get_rows(), N), pres[keep])
    # disjoint / empty database: empty feature vector
    ka.count(ds.files, k)
    ka.build()
    assert ka.restrict_to(np.empty(0, np.uint64)) == 0
    assert ka.test(ds.pheno[:, :1], True, None, min_samples=2, max_samples=N - 2)[0].kmer.size == 0
