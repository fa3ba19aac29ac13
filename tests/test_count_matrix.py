"""ps_count_matrix (k_count_matrix): the N x K occurrence counts of K canonical k-mers in a block of samples, checked
against the C oracle (count_kmers + map_counts), against ps_lookup row by row, on GPU groups and in the -rc path."""
import ctypes
import gc

import numpy as np
import pytest

from oracle import kmers as ok
from phenotypeseeker_b200 import synth
from phenotypeseeker_b200 import modeling_gpu as mg
from phenotypeseeker_b200.group import GpuGroup
from phenotypeseeker_b200.pipeline import KmerAssociation

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _fresh_dropin_engine():
    yield
    mg._STATE["ka"] = None
    gc.collect()


def _canonical(x, k):
    x = np.asarray(x, dtype=np.uint64)
    rc = np.zeros_like(x)
    for i in range(k):
        rc = (rc << np.uint64(2)) | (np.uint64(3) - ((x >> np.uint64(2 * i)) & np.uint64(3)))
    return np.minimum(x, rc)


def _random_codes(rng, k, n):
    hi = 1 << (2 * k)
    return _canonical(rng.integers(0, hi, size=n, dtype=np.uint64) if hi < (1 << 63)
                      else rng.integers(0, 1 << 63, size=n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n, dtype=np.uint64), k)


def _mixed_texts(seed):
    """Multi-record FASTA with N runs, lower case and palindromes (ACGT repeats), plus FASTQ reads."""
    rng = np.random.default_rng(seed)
    out = []
    for s in range(3):
        recs = []
        for r in range(3):
            seq = "".join("ACGT"[b] for b in rng.integers(0, 4, size=1500 + 700 * r))
            seq = seq[:300] + "N" * (5 + r * 17) + seq[300:900].lower() + "ACGT" * (10 + s) + seq[900:]
            recs.append(f">s{s}_{r} contig\n" + "\n".join(seq[i:i + 70] for i in range(0, len(seq), 70)))
        out.append(("\n".join(recs) + "\n").encode())
    out += synth.config(3, tiny=True, n_samples=2, genome_len=5000).files     # FASTQ reads
    return out


def _queries(rng, lists, k, n_present, n_random):
    """Present k-mers, random canonical codes (mostly absent), duplicates, the all-A code and a repeat, shuffled."""
    union = ok.union([l[0] for l in lists])
    q = [rng.choice(union, size=n_present), _random_codes(rng, k, n_random), union[:3], union[:3],
         np.array([0], dtype=np.uint64)]
    # a k-mer of the ACGT repeats, twice: it occurs several times per sample, and for k = 4m it is its own reverse
    # complement
    q.append(_canonical([ok.str_to_kmer(("ACGT" * 8)[:k])] * 2, k))
    q = np.concatenate(q).astype(np.uint64)
    rng.shuffle(q)
    return q


def _expected(lists, q):
    return np.stack([ok.map_counts(np.asarray(q, dtype=np.uint64), *l) for l in lists])


@pytest.mark.parametrize("k", [5, 9, 13, 16, 17, 21, 31, 32])
def test_counts_equal_oracle(ctx, k):
    rng = np.random.default_rng(k)
    texts = _mixed_texts(k)
    lists = [ok.count_kmers(t, k) for t in texts]
    q = _queries(rng, lists, k, 400, 400)
    for cutoff in (1, 3):                                  # the job's cutoff does not cut the counts
        ctx.begin(k, len(texts), cutoff)
        ctx.add_samples(0, texts)
        got = ctx.count_matrix(0, len(texts), q)
        want = _expected(lists, q)
        assert np.array_equal(got, want), (k, cutoff)
        assert (want > 1).any() and ((want == 0).any() or k == 5)    # k = 5: every 5-mer occurs somewhere
        sq = np.unique(q)                                   # ascending unique queries: no expansion step
        assert np.array_equal(ctx.count_matrix(0, len(texts), sq), _expected(lists, sq))
        for s in range(len(texts)):
            assert np.array_equal(ctx.lookup(s, q), got[s]), s


@pytest.mark.parametrize("K", [1, 1000, 1 << 17, 1 << 20])
def test_query_sizes_up_to_a_saturated_filter(ctx, K):
    ds = synth.config(0, tiny=True)
    lists = [ok.count_kmers(f, 16) for f in ds.files]
    rng = np.random.default_rng(K)
    union = ok.union([l[0] for l in lists])
    q = np.concatenate([rng.choice(union, size=(K + 1) // 2), _random_codes(rng, 16, K // 2)])
    ctx.begin(16, ds.n_samples, 1)
    ctx.add_samples(0, ds.files)
    got = ctx.count_matrix(0, ds.n_samples, q)
    assert got.shape == (ds.n_samples, K)
    assert np.array_equal(got, _expected(lists, q))


def test_sub_ranges_chunks_and_job_left_intact(ctx):
    ds = synth.config(0, tiny=True, n_samples=40, genome_len=3000)
    lists = [ok.count_kmers(f, 16) for f in ds.files]
    rng = np.random.default_rng(7)
    q = np.concatenate([rng.choice(ok.union([l[0] for l in lists]), size=1 << 20), _random_codes(rng, 16, 1 << 20)])
    want = _expected(lists, q)
    ctx.begin(16, ds.n_samples, 1)
    ctx.add_samples(0, ds.files)
    U = ctx.build_union()
    u0, r0 = ctx.get_union().tobytes(), ctx.get_rows().tobytes()
    n0 = ctx.launch_count()
    # unordered queries: a sample takes 4 B per unique query plus 4 B per query on the device, and a chunk of samples
    # at most 256 MB; one filter launch, then a count and an expansion launch per chunk
    chunks = -(-ds.n_samples // ((256 << 20) // (4 * (len(np.unique(q)) + len(q)))))
    assert chunks >= 2
    assert np.array_equal(ctx.count_matrix(0, ds.n_samples, q), want)
    assert ctx.launch_count() - n0 == 1 + 2 * chunks
    for first, count in ((0, 1), (3, 4), (31, 2), (39, 1), (5, 35)):
        assert np.array_equal(ctx.count_matrix(first, count, q[:5000]), want[first:first + count, :5000]), (first, count)
    assert ctx.get_union().tobytes() == u0 and ctx.get_rows().tobytes() == r0
    assert ctx.build_union() == U


def test_bad_arguments(ctx):
    from phenotypeseeker_b200._native import PsError
    ds = synth.config(0, tiny=True, n_samples=3, genome_len=3000)
    ctx.begin(16, 4, 1)
    ctx.add_samples(0, ds.files)                           # sample 3 is never added
    q = np.arange(10, dtype=np.uint64)
    for first, count in ((0, 4), (3, 1), (-1, 2), (2, 0), (4, 1)):
        with pytest.raises(PsError):
            ctx.count_matrix(first, count, q)
    assert ctx.L.ps_count_matrix(ctx.h, 0, 1, None, 10, None) == -1
    assert ctx.count_matrix(0, 3, q[:0]).shape == (3, 0)
    qq = np.ascontiguousarray(q)
    out = np.zeros(10, dtype=np.uint32)
    assert ctx.L.ps_count_matrix(ctx.h, 0, 1, qq.ctypes.data_as(ctypes.c_void_p), (1 << 30) + 1,
                                 out.ctypes.data_as(ctypes.c_void_p)) == -1


def _devices(devs):
    import torch
    if torch.cuda.device_count() < max(devs) + 1:
        pytest.skip(f"needs {max(devs) + 1} GPUs, this machine has {torch.cuda.device_count()}")
    return devs


@pytest.mark.parametrize("devs", [[0, 0, 0], [0, 1], [0, 1, 2, 3]], ids=str)
def test_group_equals_single_context(devs):
    ds = synth.config(0, tiny=True)
    rng = np.random.default_rng(3)
    ka = KmerAssociation(device=0)
    ka.count(ds.files, 16)
    q = np.concatenate([ka.ctx.sample_kmers(0)[0][::5], _random_codes(rng, 16, 500)])
    want = ka.count_matrix(q)
    assert want.shape == (ds.n_samples, len(q)) and want.any()
    g = GpuGroup(_devices(devs))
    g.count(ds.files, 16)
    assert np.array_equal(g.count_matrix(q), want)
    assert np.array_equal(g.count_matrix(q, 3, 7), want[3:10])          # crosses rank blocks
    assert np.array_equal(g.count_matrix(q, 11), want[11:])
    assert np.array_equal(ka.count_matrix(q, 2, 5), want[2:7])


def test_real_counts_on_a_group_equal_one_gpu():
    rep = b"ACGTTGCAAGGCTTAACCGGTTAGCATCGA"
    ds = synth.config(0, tiny=True, n_samples=8, genome_len=6000)
    files = [f + b">extra\n" + rep * (s % 3 + 1) + b"\n" for s, f in enumerate(ds.files)]
    args = (files, ds.names, 16, 1, ds.pheno[:, :1], ["pheno1"], True, None, 2, 6, 1.1, True, 4)
    U1, one = mg.run_hot_path(*args, real_counts=True, device=0)
    U2, two = mg.run_hot_path(*args, real_counts=True, device=[0, 0])
    assert U1 == U2 and one["pheno1"].shape[1] > 0
    assert one["pheno1"].equals(two["pheno1"])
    assert max(int(v) for v in one["pheno1"].iloc[4:].to_numpy().ravel()) >= 2
