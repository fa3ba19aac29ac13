"""`-w` sample weights on the device (ps_mash_sketch / ps_mash_pairs / ps_neighbor_joining, ps_mash.cuh) against the
host restatement in phenotypeseeker_b200/weights.py, bit for bit, and the host pieces the device path adds: the
(shared, denom) -> distance table, the NJ split into nj_joins + tree_from_joins, and the iterative Newick code."""
import base64
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_json
from phenotypeseeker_b200 import weights as W

sys.setrecursionlimit(max(sys.getrecursionlimit(), 1000))


# ---------------------------------------------------------------------------------------------------------------
# inputs
def _mash_gold():
    g = load_json("mash.json")
    for c in g["cases"]:
        c["data"] = base64.b64decode(c["data_b64"])
        c["h"] = np.array([int(x) for x in c["hashes"]], dtype=np.uint64)
    return g


def _random_fasta(rng, length, n_records=3, n_runs=4, lower=0.1, crlf=False, width=None):
    """Multi-record FASTA: ACGT with runs of N, some lower case, line width 1..200, LF or CRLF."""
    seq = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=length)
    for _ in range(n_runs):
        a = int(rng.integers(0, length))
        seq[a:a + int(rng.integers(1, 40))] = ord("N")
    low = rng.random(length) < lower
    seq[low] = seq[low] | 0x20
    cuts = np.sort(rng.choice(np.arange(1, length), size=n_records - 1, replace=False)) if n_records > 1 else []
    nl = b"\r\n" if crlf else b"\n"
    out = [b"junk before the first header" + nl]
    for r, (a, b) in enumerate(zip([0, *cuts], [*cuts, length])):
        w = width or int(rng.integers(1, 201))
        body = seq[a:b].tobytes()
        out.append(b">rec%d some description" % r + nl)
        out.extend(body[i:i + w] + nl for i in range(0, len(body), w))
    return b"".join(out)


def _clonal_texts(rng, n, length, n_clades=4, snp=0.002):
    """n FASTA texts from n_clades ancestors with few private SNPs; every fourth sample is an exact clone."""
    anc = [rng.choice(np.frombuffer(b"ACGT", np.uint8), size=length) for _ in range(n_clades)]
    texts = []
    for i in range(n):
        if i % 4 == 3:
            texts.append(texts[-1])
            continue
        g = anc[i % n_clades].copy()
        pos = rng.integers(0, length, size=int(length * snp))
        g[pos] = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=len(pos))
        texts.append(b">s%d\n" % i + b"\n".join(g[j:j + 80].tobytes() for j in range(0, length, 80)) + b"\n")
    return texts


def _nj_reference(names, dm):
    """neighbor_joining as it was before the split into nj_joins + tree_from_joins (the Newick text must not change)."""
    dm = [list(map(float, row)) for row in np.asarray(dm, dtype=np.float64)]
    clades = [W.Node(nm) for nm in names]
    inner, count = None, 0
    while len(dm) > 2:
        m = len(dm)
        nd = [sum(dm[i]) / (m - 2) for i in range(m)]
        min_dist = dm[1][0] - nd[1] - nd[0]
        mi, mj = 0, 1
        for i in range(1, m):
            for j in range(i):
                t = dm[i][j] - nd[i] - nd[j]
                if min_dist > t:
                    min_dist, mi, mj = t, i, j
        c1, c2 = clades[mi], clades[mj]
        count += 1
        inner = W.Node("Inner" + str(count))
        inner.add(c1); inner.add(c2)
        c1.dist = (dm[mi][mj] + nd[mi] - nd[mj]) / 2.0
        c2.dist = dm[mi][mj] - c1.dist
        clades[mj] = inner
        del clades[mi]
        for x in range(m):
            if x != mi and x != mj:
                dm[mj][x] = dm[x][mj] = (dm[mi][x] + dm[mj][x] - dm[mi][mj]) / 2.0
        del dm[mi]
        for row in dm:
            del row[mi]
    if clades[0] is inner:
        clades[0].dist = 0.0; clades[1].dist = dm[1][0]; clades[0].add(clades[1]); return clades[0]
    clades[0].dist = dm[1][0]; clades[1].dist = 0.0; clades[1].add(clades[0]); return clades[1]


def _nj_matrices():
    rng = np.random.default_rng(11)
    out = [np.array([[0, 5, 9, 9], [5, 0, 10, 10], [9, 10, 0, 8], [9, 10, 8, 0]], dtype=float)]
    for n in (3, 5, 9, 23):
        a = rng.random((n, n)); a = (a + a.T) / 2; np.fill_diagonal(a, 0); out.append(a)
    out.append(np.ones((7, 7)) - np.eye(7))                                    # all equal
    for n in (6, 17, 40):                                                      # printed distances, many ties and zeros
        v = np.array([0.0, W.printed(0.00123456789), W.printed(0.0208145), 0.05, 1.0])
        a = v[rng.integers(0, len(v), (n, n))]; a = np.triu(a, 1); a = a + a.T
        out.append(a)
    return out


def _tie_matrix(rng, n):
    v = np.array([W.printed(x) for x in (0.0, 0.000413, 0.00123456, 0.0208145, 0.0511, 0.17, 1.0)])
    a = v[rng.integers(0, len(v), (n, n))]
    clone = rng.random(n) < 0.3                     # clones of their predecessor: distance 0, identical rows
    a = np.triu(a, 1); a = a + a.T
    for i in np.flatnonzero(clone):
        if i:
            a[i] = a[i - 1]; a[:, i] = a[:, i - 1]; a[i, i - 1] = a[i - 1, i] = 0.0
    np.fill_diagonal(a, 0.0)
    return a


# ---------------------------------------------------------------------------------------------------------------
# CPU
@pytest.fixture(scope="module")
def mash_bits(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("mash") / "mash_bits_check")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "native", "mash_bits_check.cpp")])

    def run(lines, parse=True):
        r = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        return [list(map(int, ln.split())) for ln in r.stdout.splitlines()] if parse else r.stdout.splitlines()
    return run


def test_kmer_hash_equals_murmur_of_canonical_text(mash_bits):
    rng = np.random.default_rng(5)
    lines, expect = [], []
    for k in (1, 15, 16, 17, 21, 31, 32):
        for seed in (0, 42, 2 ** 32 - 1):
            words = [int(x) & ((1 << 2 * k) - 1) for x in rng.integers(0, 2 ** 63, 40, dtype=np.int64) * 2 + rng.integers(0, 2, 40)]
            words += [0, (1 << 2 * k) - 1]                               # poly-A / poly-T
            for fw in words:
                text = "".join("ACGT"[(fw >> 2 * (k - 1 - i)) & 3] for i in range(k))
                canon = min(text, text[::-1].translate(str.maketrans("ACGT", "TGCA")))
                cw = 0
                for ch in canon:
                    cw = 4 * cw + "ACGT".index(ch)
                lines.append(f"h {k} {seed} {fw}")
                expect.append([cw, int(W.murmur3_x64_128_h1(np.frombuffer(canon.encode(), np.uint8)[None, :], seed)[0])])
    assert mash_bits(lines) == expect


def test_shared_denom_rule_equals_mash_distance(mash_bits):
    rng = np.random.default_rng(6)
    pool = np.unique(rng.integers(0, 2 ** 63, 20000, dtype=np.int64).astype(np.uint64) * np.uint64(2))
    cases = []
    for _ in range(200):
        s = int(rng.choice([1, 3, 50, 1000]))
        a = np.sort(rng.choice(pool, size=int(rng.integers(0, 1200)), replace=False))[:s]
        kind = rng.integers(0, 5)
        if kind == 0:
            b = a[: int(rng.integers(0, len(a) + 1))]                      # nested
        elif kind == 1:
            b = np.setdiff1d(rng.choice(pool, 800, replace=False), a)[:s]  # disjoint
        elif kind == 2:
            b = np.empty(0, np.uint64)                                     # empty
        else:
            b = np.sort(rng.choice(pool, size=int(rng.integers(0, 1200)), replace=False))[:s]
        cases.append((s, a, b))
    lines = [f"d {s} {len(a)} " + " ".join(map(str, a.tolist())) + f" {len(b)} " + " ".join(map(str, b.tolist()))
             for s, a, b in cases]
    got = mash_bits(lines)
    for (s, a, b), (v,) in zip(cases, got):
        _, shared, denom = W.mash_distance(a, b, s=s)
        assert v == (shared << 16 | denom)


def test_nj_row_sum_equals_python_sum(mash_bits):
    """Neighbour joining's row sums go through Python's sum(), which is compensated (Neumaier) since 3.12: the
    device's psm_sum_* and the host's _row_sum must both give exactly what sum() gives there."""
    rng = np.random.default_rng(8)
    rows = []
    for t in range(3000):
        n = int(rng.integers(1, 80))
        kind = t % 4
        if kind == 0:
            x = rng.random(n)
        elif kind == 1:
            x = rng.normal(size=n) * 10.0 ** rng.integers(-8, 8, n)
        elif kind == 2:
            x = rng.choice([0.0, -0.0, W.printed(0.000413), W.printed(0.0208145), 1.0, -0.5], n)
        else:
            x = (rng.random(n) - 0.5) / 2
        rows.append([float(v) for v in x])
    rows += [[1e100, 1.0, -1e100], [-0.0], [-0.0, -0.0], [0.1] * 10]
    out = mash_bits([f"s {len(r)} " + " ".join(v.hex() for v in r) for r in rows], parse=False)
    differs = 0
    for r, line in zip(rows, out):
        got = float.fromhex(line)
        want = W._compensated_sum(r)
        assert got == want and np.signbit(got) == np.signbit(want), r
        if sys.version_info >= (3, 12):
            assert want == sum(r) and np.signbit(want) == np.signbit(sum(r))
        s = 0.0
        for v in r:
            s += v
        differs += s != want
    assert differs > 100                       # a left-to-right sum would not do


def test_distance_table_equals_printed_mash_distance():
    rng = np.random.default_rng(7)
    n = 30
    sd = np.zeros((n, n), np.uint32)
    for i in range(n):
        for j in range(i):
            denom = int(rng.choice([0, 1, 7, 150, 1000]))
            shared = int(rng.integers(0, denom + 1)) if denom else 0
            sd[i, j] = sd[j, i] = shared << 16 | denom
        sd[i, i] = 1000 << 16 | 1000
    dm = W.printed_distances(sd)
    for i in range(n):
        for j in range(n):
            want = 0.0 if i == j else W.printed(W.distance_from_counts(int(sd[i, j]) >> 16, int(sd[i, j]) & 0xFFFF))
            assert dm[i, j] == want


def test_tree_from_joins_equals_neighbor_joining():
    for dm in _nj_matrices():
        names = [f"t{i}" for i in range(len(dm))]
        want = W.newick(_nj_reference(names, dm))
        assert W.newick(W.tree_from_joins(names, *W.nj_joins(dm))) == want
        assert W.newick(W.neighbor_joining(names, dm)) == want


def test_deep_caterpillar_newick_roundtrip_and_gsc():
    n = 5000
    root = W.Node("Inner", 0.0)
    node = root
    for i in range(n - 1):                       # a ladder of depth n - 1
        node.add(W.Node(f"leaf{i}", 0.01 * (i % 7 + 1)))
        nxt = W.Node("", 0.02)
        node.add(nxt)
        node = nxt
    node.add(W.Node(f"leaf{n - 1}", 0.5))
    node.add(W.Node(f"leaf{n}", 0.25))
    text = W.newick(root) + ";"
    again = W.newick(W.parse_newick(text)) + ";"
    assert again == text
    w = W.gsc_weights(W.parse_newick(text))
    assert len(w) == n + 1 and np.isfinite(list(w.values())).all()
    assert np.mean(list(w.values())) == pytest.approx(1.0)


# ---------------------------------------------------------------------------------------------------------------
# GPU
def _device_sketch(ctx, texts, k=21, s=1000, seed=42, job_k=16, cutoff=1):
    ctx.begin(job_k, len(texts), cutoff)
    ctx.add_samples(0, list(texts))
    return ctx.mash_sketch(0, len(texts), k, s, seed)


def _rows(h, n):
    return [h[i, :n[i]] for i in range(len(n))]


@pytest.mark.gpu
def test_device_sketch_equals_mash_golden(ctx):
    g = _mash_gold()
    h, n = _device_sketch(ctx, [c["data"] for c in g["cases"]], g["k"], g["s"], g["seed"])
    for c, row in zip(g["cases"], _rows(h, n)):
        assert np.array_equal(row, c["h"]), c["name"]


@pytest.mark.gpu
def test_device_sketch_equals_host_sketch(ctx):
    rng = np.random.default_rng(21)
    texts = [_random_fasta(rng, int(rng.integers(50, 40000)), n_records=int(rng.integers(1, 6)),
                           crlf=bool(i % 2), width=(1 if i == 0 else None)) for i in range(10)]
    big = _random_fasta(rng, 3_200_000, n_records=2, width=80)                     # many chunks
    rep = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=50_000).tobytes()       # the same 50 kbp twice
    dup = b">dup\n" + rng.choice(np.frombuffer(b"ACGT", np.uint8), size=400_000).tobytes() + rep + \
          rng.choice(np.frombuffer(b"ACGT", np.uint8), size=300_000).tobytes() + rep + b"\n"
    empty = b">none\nACGTNACGTN\n>short\nACG\n"                                   # no valid 16+-window
    texts += [big, dup, empty]
    for k, s, seed in ((21, 1000, 42), (16, 100, 0), (32, 4096, 42), (21, 1, 0), (16, 1000, 42), (32, 100, 0)):
        h, n = _device_sketch(ctx, texts, k, s, seed)
        for i, (t, row) in enumerate(zip(texts, _rows(h, n))):
            assert np.array_equal(row, W.sketch(t, k, s, seed)), (k, s, seed, i)
        assert n[-1] == 0


@pytest.mark.gpu
def test_device_reader_deviations(ctx):
    """Documented: a byte 1..31 inside a sequence is skipped on the device (the host breaks the window there), and
    U / u is read as T (the host breaks the window)."""
    rng = np.random.default_rng(22)
    seq = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=20000)
    seq[rng.integers(0, len(seq), 30)] = ord("U")
    seq[rng.integers(0, len(seq), 30)] = ord("u")
    body = seq.tobytes()
    text = b">x\n" + b"\t".join(body[i:i + 500] for i in range(0, len(body), 500)) + b"\n"
    (h, n) = _device_sketch(ctx, [text])
    want = W.sketch(text.replace(b"\t", b"").replace(b"U", b"T").replace(b"u", b"T"))
    assert np.array_equal(h[0, :n[0]], want)


@pytest.mark.gpu
def test_device_sketch_does_not_depend_on_the_job(ctx):
    g = _mash_gold()
    texts = [c["data"] for c in g["cases"]]                                     # "reads" is FASTQ
    ref = None
    for job_k, cutoff in ((9, 1), (16, 1), (31, 1), (16, 2), (31, 2)):
        h, n = _device_sketch(ctx, texts, job_k=job_k, cutoff=cutoff)
        got = _rows(h, n)
        if ref is None:
            ref = got
        assert all(np.array_equal(a, b) for a, b in zip(ref, got)), (job_k, cutoff)
    assert all(np.array_equal(a, c["h"]) for a, c in zip(ref, g["cases"]))


@pytest.mark.gpu
def test_weights_calls_leave_the_job_alone(ctx):
    rng = np.random.default_rng(23)
    texts = [_random_fasta(rng, 20000, n_records=2) for _ in range(12)]
    pheno = (np.arange(12) % 2).astype(np.int8)

    def run(between):
        ctx.begin(16, len(texts), 1)
        ctx.add_samples(0, texts)
        ctx.build_union()
        if between:
            h, n = ctx.mash_sketch(0, len(texts))
            dm = W.printed_distances(ctx.mash_pairs(h, n))
            ctx.neighbor_joining(dm)
        u, rows = ctx.get_union(), ctx.get_rows()
        ns = ctx.test_chi2(pheno, None, 2, 10, 0.5)
        return u, rows, ctx.fetch_survivors(ns)

    a, b = run(False), run(True)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    for key in a[2]:
        assert np.array_equal(a[2][key], b[2][key]), key


@pytest.mark.gpu
def test_device_pairs_equal_mash_dist(ctx):
    g = _mash_gold()
    names = [c["name"] for c in g["cases"]]
    h = np.zeros((len(names), g["s"]), np.uint64)
    n = np.array([len(c["h"]) for c in g["cases"]], np.uint32)
    for i, c in enumerate(g["cases"]):
        h[i, :n[i]] = c["h"]
    sd = ctx.mash_pairs(h, n)
    for a, b, _, frac in g["dist"]:
        v = int(sd[names.index(a), names.index(b)])
        assert f"{v >> 16}/{v & 0xFFFF}" == frac, (a, b)
    # random sketches: empty, short, clones
    rng = np.random.default_rng(24)
    pool = np.unique(rng.integers(0, 2 ** 63, 60000, dtype=np.int64).astype(np.uint64) * np.uint64(2))
    N, s = 300, 1000
    sk = []
    for i in range(N):
        r = rng.random()
        if r < 0.05:
            sk.append(np.empty(0, np.uint64))
        elif r < 0.25 and sk:
            sk.append(sk[int(rng.integers(0, len(sk)))])
        else:
            m = int(rng.choice([3, 40, 700, 1000]))
            sk.append(np.sort(rng.choice(pool[: int(rng.integers(2000, len(pool)))], m, replace=False)))
    h = np.zeros((N, s), np.uint64)
    n = np.array([len(x) for x in sk], np.uint32)
    for i, x in enumerate(sk):
        h[i, :len(x)] = x
    sd = ctx.mash_pairs(h, n)
    pairs = [(i, j) for i in range(40) for j in range(40)] + list(zip(rng.integers(0, N, 4000), rng.integers(0, N, 4000)))
    for i, j in pairs:
        _, shared, denom = W.mash_distance(sk[i], sk[j], s=s)
        assert int(sd[i, j]) == (shared << 16 | denom), (i, j)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 4, 5, 37, 300, 1000])
def test_device_nj_equals_nj_joins(ctx, n):
    rng = np.random.default_rng(100 + n)
    mats = [_tie_matrix(rng, n)]
    if n <= 300:
        a = rng.random((n, n)); a = (a + a.T) / 2; np.fill_diagonal(a, 0); mats.append(a)
    if n == 37:
        texts = _clonal_texts(rng, n, 20000)
        h, c = _device_sketch(ctx, texts)
        mats.append(W.printed_distances(ctx.mash_pairs(h, c)))
    for dm in mats:
        jw, bw = W.nj_joins(dm)
        jd, bd = ctx.neighbor_joining(dm)
        assert np.array_equal(jd, jw) and np.array_equal(bd, bw)


@pytest.mark.gpu
def test_nj_rejects_bad_input(ctx):
    from phenotypeseeker_b200._native import PsError
    a = np.zeros((4, 4)); a[1, 0] = 1.0
    with pytest.raises(PsError):
        ctx.neighbor_joining(a)
    with pytest.raises(PsError):
        ctx.neighbor_joining(np.zeros((2, 2)))
    ctx.begin(16, 2, 1)
    with pytest.raises(PsError):
        ctx.mash_sketch(0, 2)                    # samples not present
    ctx.add_samples(0, [b">a\nACGTACGTACGTACGTACGTACGT\n", b">b\nACGT\n"])
    for k, s in ((0, 1000), (33, 1000), (21, 0), (21, 4097)):
        with pytest.raises(PsError):
            ctx.mash_sketch(0, 2, k, s)


@pytest.mark.gpu
def test_gsc_weights_on_device_equal_host(ctx):
    g = _mash_gold()
    names = [c["name"] for c in g["cases"]]
    texts = [c["data"] for c in g["cases"]]
    order = [4, 0, 8, 2, 6, 1, 7, 3, 5]                    # not sorted by name: the glob quirk matters
    names, texts = [names[i] for i in order], [texts[i] for i in order]
    for quirk in (False, True):
        ctx.begin(16, len(texts), 1)
        ctx.add_samples(0, texts)
        got = W.gsc_weights_on_device(ctx, names, 0, keep_glob_quirk=quirk)
        assert np.array_equal(got, W.gsc_weights_for_samples(names, texts, keep_glob_quirk=quirk)), quirk
    rng = np.random.default_rng(25)
    texts = _clonal_texts(rng, 60, 15000, n_clades=6)
    names = [f"syn{(i * 37) % 60:03d}" for i in range(60)]
    ctx.begin(16, len(texts), 1)
    ctx.add_samples(0, texts)
    for quirk in (False, True):
        got = W.gsc_weights_on_device(ctx, names, 0, keep_glob_quirk=quirk)
        assert np.array_equal(got, W.gsc_weights_for_samples(names, texts, keep_glob_quirk=quirk)), quirk


@pytest.mark.gpu
def test_install_native_weights_gpu(tmp_path, monkeypatch):
    import collections
    import types
    from phenotypeseeker_b200 import modeling_gpu
    g = _mash_gold()
    by = {c["name"]: c["data"] for c in g["cases"]}
    names = ["rel2", "other", "rel0", "rel1", "withN"]
    monkeypatch.chdir(tmp_path)

    class S:
        def __init__(self, name, address):
            self.name, self.address, self.weight = name, address, 1

    samples = collections.OrderedDict()
    for nm in names:
        p = tmp_path / (nm + ".fa")
        p.write_bytes(by[nm])
        samples[nm] = S(nm, str(p))
    m = types.SimpleNamespace(Input=type("Input", (), {"samples": samples, "num_threads": 2}),
                              Samples=type("Samples", (), {"kmer_length": 16, "cutoff": 1}),
                              phenotypes=type("phenotypes", (), {}))
    modeling_gpu.install(m, native_weights="gpu")
    m.Samples.get_feature_vector()
    m.Samples.get_weights()
    w = np.array([samples[nm].weight for nm in names])
    assert np.array_equal(w, W.gsc_weights_for_samples(names, [by[nm] for nm in names], keep_glob_quirk=True))


@pytest.mark.gpu
def test_five_thousand_samples_through_the_device_path(ctx):
    rng = np.random.default_rng(26)
    N, L = 5000, 3000
    anc = [rng.choice(np.frombuffer(b"ACGT", np.uint8), size=L) for _ in range(50)]
    texts = []
    for i in range(N):
        gnm = anc[i % 50].copy()
        pos = rng.integers(0, L, size=int(rng.integers(0, 30)))
        gnm[pos] = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=len(pos))
        texts.append(b">s\n" + gnm.tobytes() + b"\n")
    names = [f"s{i:05d}" for i in range(N)]
    ctx.begin(16, N, 1)
    ctx.add_samples(0, texts)
    w = W.gsc_weights_on_device(ctx, names, 0, keep_glob_quirk=True)
    assert w.shape == (N,) and np.isfinite(w).all() and (w > 0).all()
    assert w.mean() == pytest.approx(1.0)
