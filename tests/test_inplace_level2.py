"""Level-2 pages written into the level-1 pages k_scatter2 has read (ps_paged.cuh): a build consumes the level-1
pages of its bins, so a second build of them extracts again; many sample groups of small samples leave the most
partial pages per record (the level-2 reserve); and the choice of one super-range when the whole job's pool fits."""
import numpy as np
import pytest

from phenotypeseeker_b200 import synth
from phenotypeseeker_b200.pipeline import KmerAssociation, level1_pool_bytes

UNIT = 1 << 24          # k = 16: one top k-mer byte, the granularity of level-1 bins


@pytest.mark.gpu
def test_second_build_of_a_range_from_the_announced_pool(ctx):
    ds = synth.make_dataset(12, genome_len=40_000, seed=11)
    ka = KmerAssociation(ctx=ctx)
    ka.count(ds.files, 16)
    U = ka.build()
    u_all, rows_all = ctx.get_union(), ctx.get_rows()
    assert U == len(u_all) > 0
    lo, hi = 64 * UNIT, 160 * UNIT
    ka.count(ds.files, 16)
    ctx.scatter_range(0, 0)
    try:
        got = []
        for a, b in [(lo, hi), (hi, 0), (lo, hi), (0, lo)]:
            ctx.set_range(a, b)
            n = ctx.build_union()
            got.append((a, b, n, ctx.get_union(), ctx.get_rows()))
    finally:
        ctx.set_range(0, 0)
    for a, b, n, u, rows in got:
        sel = (u_all >= a) & ((u_all < b) if b else True)
        assert n == int(sel.sum()) > 0, (a, b)
        assert np.array_equal(u, u_all[sel]), (a, b)
        assert np.array_equal(rows, rows_all[sel]), (a, b)


@pytest.fixture(scope="module")
def many_groups():
    """2,000 short genomes: eight sample groups, and per record the most partial pages."""
    from oracle import kmers as ok, stats as ostats
    ds = synth.make_dataset(2000, genome_len=3_000, seed=23, contigs=(5, 10))
    lists = ok.count_many(ds.files, 16)
    u, rows = ok.union_and_rows([l[0] for l in lists])
    pres = ok.presence_matrix(u, lists)
    N = ds.n_samples
    o = ostats.chi2_rows(pres, ds.pheno[:, 0].astype(np.int8), np.ones(N), 2, N - 2)
    keep = o["tested"] & (o["p"] < 0.05)
    return ds, u, rows, pres, o, keep


def _check_survivors(res, u, pres, o, keep):
    assert keep.any()
    assert np.array_equal(res.kmer, u[keep])
    assert np.array_equal(res.stat, o["stat"][keep])
    assert np.array_equal(res.presence, pres[keep])


@pytest.mark.gpu
def test_many_sample_groups_whole_space(ctx, many_groups):
    ds, u, rows, pres, o, keep = many_groups
    N = ds.n_samples
    ka = KmerAssociation(ctx=ctx)
    ka.count(ds.files, 16)
    assert ka.build() == len(u)
    assert np.array_equal(ctx.get_union(), u)
    assert np.array_equal(ctx.get_rows(), rows)
    res = ka.test(ds.pheno, True, None, min_samples=2, max_samples=N - 2, pvalue_cutoff=0.05, omit_b=True)[0]
    _check_survivors(res, u, pres, o, keep)


@pytest.mark.parametrize("n_super", [1, 2])
@pytest.mark.gpu
def test_many_sample_groups_in_super_ranges(ctx, many_groups, n_super):
    ds, u, rows, pres, o, keep = many_groups
    N = ds.n_samples
    n_inst = sum(len(f) for f in ds.files)
    ka = KmerAssociation(ctx=ctx)
    ka.count(ds.files, 16)
    plan = ka.plan_ranges(4, ctx.sample_quantiles(0, 4), n_inst, n_super)
    assert len(plan["first_of"]) == n_super
    ka.count(ds.files, 16, ingest_range=plan["ingest"])        # the first super-range scattered during ingest
    U, res = ka.test_in_ranges(ds.pheno, True, 4, None, splitters=plan["splitters"], n_super=n_super, n_instances=n_inst,
                               min_samples=2, max_samples=N - 2, pvalue_cutoff=0.05, omit_b=True)
    assert U == len(u)
    _check_survivors(res[0], u, pres, o, keep)
    # the union and matrix of every range, built once more from the streams
    spl = plan["splitters"]
    for r in range(4):
        lo, hi = (spl[r - 1] if r else 0), (spl[r] if r < 3 else 0)
        ctx.set_range(lo, hi)
        try:
            ctx.build_union()
            sel = (u >= lo) & ((u < hi) if hi else True)
            assert np.array_equal(ctx.get_union(), u[sel])
            assert np.array_equal(ctx.get_rows(), rows[sel])
        finally:
            ctx.set_range(0, 0)


def test_one_super_range_when_the_pool_fits():
    """plan_ranges(n_super=None): one super-range when the whole job's level-1 pool, its reserve, the streams, the
    largest range's matrix and headroom fit in free plus held memory; otherwise, on a first call of a job, or with a
    context that cannot report its memory, half as many super-ranges as ranges."""

    class MemCtx:
        def __init__(self):
            self.free, self.held = 0, 0

        def mem_info(self):
            return self.free, self.held

    ka = KmerAssociation(ctx=MemCtx())
    ka.k, ka.n_samples = 16, 5000
    spl = [64 * UNIT, 128 * UNIT, 192 * UNIT]
    n = 25_000_000_000
    ka.ctx.free = 10 ** 15
    assert ka.plan_ranges(4, spl, n)["first_of"] == {0: 2, 2: 4}              # no range sizes of this job yet
    sizes = [20_000_000, 23_000_000, 21_000_000, 22_000_000]
    ka._range_sizes = {(16, 5000, tuple(spl)): sizes}
    p = ka.plan_ranges(4, spl, n)
    assert p["first_of"] == {0: 4}
    assert p["ingest"] == (0, 0, n + (1 << 20), 1.0)                          # the whole space: no slack
    # the boundary: pool + page tables + streams + the largest matrix + headroom
    m = n + (1 << 20)
    row_bytes = 160 * 4                                                        # 5,000 samples: 157 words, rounded to 160
    need = (level1_pool_bytes(m, 5000) + -(-m // 1024) * 48 + m * 3 // 8 * 9 // 8 + max(sizes) * (8 + row_bytes) * 9 // 8
            + (4 << 30))
    ka.ctx.free, ka.ctx.held = need - 100 * 10 ** 9, 100 * 10 ** 9
    assert ka.plan_ranges(4, spl, n)["first_of"] == {0: 4}
    ka.ctx.free -= 1
    assert ka.plan_ranges(4, spl, n)["first_of"] == {0: 2, 2: 4}
    ka.ctx.free = 10 ** 15
    assert ka.plan_ranges(4, [64 * UNIT, 130 * UNIT, 192 * UNIT], n)["first_of"] == {0: 2, 2: 4}   # another job
    assert ka.plan_ranges(4, spl, None)["first_of"] == {0: 2, 2: 4}           # no instance count
    assert ka.plan_ranges(4, spl, n, n_super=2)["first_of"] == {0: 2, 2: 4}   # asked for
    ka.ctx = object()                                                          # cannot report memory
    assert ka.plan_ranges(4, spl, n)["first_of"] == {0: 2, 2: 4}


def test_level1_pool_bytes_is_what_paged_begin_local_reserves():
    # config 5: 5,000 samples = 20 sample groups; 444 k_scatter1 and 444 k_scatter2 blocks on 148 SMs
    n = 25_561_787_303
    pages = -(-n // 1024) + 444 * 264 * 22
    reserve = (20 * 264 + 2 * 444) * 256
    assert level1_pool_bytes(n, 5000) == pages * 4096 + reserve * 2048
    assert 112e9 < pages * 4096 < 114e9 and 3.1e9 < reserve * 2048 < 3.3e9
