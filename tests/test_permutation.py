"""Permutation threshold (Westfall & Young's single-step min-p): the permutation generator and the threshold rule on
the host, ps_minp_chi2 / ps_minp_welch against a host min-p built from the oracle's vectorised tests, and the
threshold through every execution shape (one build, k-mer ranges, a GPU group, the drop-in)."""
import collections
import gc
import types

import numpy as np
import pytest

from oracle import kmers as ok
from oracle import stats as ostats
from phenotypeseeker_b200 import synth
from phenotypeseeker_b200.pipeline import permute_columns, permutation_thresholds

RTOL = 1e-6


# --- host: the permutation generator -------------------------------------------------------------------------------
def _table():
    rng = np.random.default_rng(3)
    ph = rng.integers(0, 2, size=(40, 3)).astype(np.float64)
    ph[rng.random(ph.shape) < 0.25] = np.nan
    ph[:, 2] = rng.normal(size=40)
    ph[[1, 7, 30], 2] = np.nan
    return ph


def test_permutations_keep_na_positions_and_permute_only_the_values():
    ph = _table()
    perm = permute_columns(ph, 25, seed=11)
    assert perm.shape == (3, 25, 40)
    for j in range(3):
        na = np.isnan(ph[:, j])
        for b in range(25):
            col = perm[j, b]
            assert np.array_equal(np.isnan(col), na)
            assert np.array_equal(np.sort(col[~na]), np.sort(ph[~na, j]))
    # the permutations differ from each other and from the observed column
    assert len({perm[2, b].tobytes() for b in range(25)}) == 25


def test_permutations_are_reproducible_and_independent_of_the_batch():
    ph = _table()
    a = permute_columns(ph, 12, seed=5)
    assert np.array_equal(a, permute_columns(ph, 12, seed=5), equal_nan=True)
    assert not np.array_equal(a, permute_columns(ph, 12, seed=6), equal_nan=True)
    batches = np.concatenate([permute_columns(ph, 5, seed=5, first=0), permute_columns(ph, 4, seed=5, first=5),
                              permute_columns(ph, 3, seed=5, first=9)], axis=1)
    assert np.array_equal(a, batches, equal_nan=True)
    # a column's permutations do not depend on the other columns drawn with it
    assert np.array_equal(a[1:2], permute_columns(ph, 12, seed=5)[1:2], equal_nan=True)
    one = permute_columns(ph[:, :2], 12, seed=5)
    assert np.array_equal(a[:2], one, equal_nan=True)


# --- host: the threshold rule --------------------------------------------------------------------------------------
def test_threshold_is_the_floor_alpha_b_plus_first_minimum():
    m = np.array([[0.3, 0.01, 0.2, 0.04, 0.5, 0.6, 0.7, 0.8, 0.9, 0.11,
                   0.12, 0.13, 0.14, 0.15, 0.16, 0.17, 0.18, 0.19, 0.21, 0.22]])
    assert permutation_thresholds(m, 0.05)[0] == 0.04          # B = 20, alpha = 0.05: q_2
    assert permutation_thresholds(m, 0.15)[0] == 0.12          # q_4
    assert permutation_thresholds(np.tile(m, (2, 5)), 0.05)[1] == 0.04    # B = 100: q_6 of five copies of each


def test_threshold_ties():
    m = np.array([[0.01, 0.01, 0.01] + [0.5] * 17])
    assert permutation_thresholds(m, 0.05)[0] == 0.01          # a k-mer needs p < 0.01: no permutation passes


def test_too_few_permutations_raise():
    with pytest.raises(ValueError):
        permutation_thresholds(np.full((2, 19), 0.5), 0.05)
    permutation_thresholds(np.full((2, 20), 0.5), 0.05)


def test_threshold_capped_at_the_cutoff():
    m = np.full((3, 40), 0.5)
    m[1, :] = 1e-4
    t = permutation_thresholds(m, 0.05)
    assert t[0] == 0.05 and t[1] == 1e-4 and t[2] == 0.05


# --- host min-p from the oracle ------------------------------------------------------------------------------------
def host_minp(pres, cols, binary, weights, min_s, max_s):
    """Smallest p over the testable rows (sample filter passed, p not NaN) of each column; 1 if none. chi2 p is
    exp(-chi2 / 2), the reference's df = 2 survival function in the form the kernels evaluate."""
    w = np.ones(pres.shape[1]) if weights is None else weights
    out = np.ones(len(cols))
    for i, col in enumerate(cols):
        if binary:
            r = ostats.chi2_rows(pres, np.where(np.isnan(col), -1, col).astype(np.int8), w, min_s, max_s)
            p = np.exp(-0.5 * r["stat"])
        else:
            r = ostats.welch_rows(pres, col, w, min_s, max_s)
            p = r["p"]
        ok_ = r["tested"] & ~np.isnan(p)
        if ok_.any():
            out[i] = min(1.0, float(p[ok_].min()))
    return out


def test_host_minp_on_a_hand_made_matrix():
    pres = np.array([[1, 1, 1, 0, 0, 0], [1, 0, 1, 0, 1, 0], [1, 1, 1, 1, 1, 0]], dtype=np.uint8)
    col = np.array([1, 1, 1, 0, 0, 0], dtype=np.float64)
    m = host_minp(pres, [col], True, None, 2, 4)
    assert m[0] == np.exp(-0.5 * 6.0)                          # row 0: the perfect split, chi2 = N = 6
    assert host_minp(pres, [col], True, None, 6, 6)[0] == 1.0  # nothing testable


# --- GPU -----------------------------------------------------------------------------------------------------------
def _job(n, seed, binary=True, na_rate=0.0, genome_len=3000, n_pheno=2, k=16):
    ds = synth.make_dataset(n, genome_len=genome_len, seed=seed, binary=binary, n_pheno=n_pheno, na_rate=na_rate,
                            n_clades=4, contigs=(1, 2), k=k)
    lists = [ok.count_kmers(f, k) for f in ds.files]
    u = ok.union([x[0] for x in lists])
    return ds, u, ok.presence_matrix(u, lists)


def _engine(ds, k=16, walk=False, monkeypatch=None):
    from phenotypeseeker_b200.pipeline import KmerAssociation
    if walk:
        monkeypatch.setenv("PSKMER_CHI2", "walk")          # read when the context is created
    ka = KmerAssociation(device=0)
    if walk:
        monkeypatch.delenv("PSKMER_CHI2")
    ka.count(ds.files, k)
    ka.build()
    return ka


CASES = {                    # name -> (samples, binary, weighted, NA rate, walk)
    "chi2": (24, True, False, 0.0, False),
    "chi2_walk": (24, True, False, 0.0, True),
    "chi2_weighted": (24, True, True, 0.0, False),
    "chi2_na": (30, True, False, 0.2, False),
    "chi2_walk_na": (30, True, False, 0.2, True),
    "chi2_wide": (1000, True, False, 0.0, False),
    "chi2_wide_walk": (1000, True, False, 0.1, True),
    "chi2_walk_warp": (2200, True, False, 0.0, True),
    "chi2_wide_weighted": (1000, True, True, 0.0, False),
    "welch": (24, False, False, 0.0, False),
    "welch_weighted": (24, False, True, 0.0, False),
    "welch_na": (30, False, True, 0.2, False),
    "welch_wide": (1000, False, False, 0.1, False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_minp_matches_the_host_reference(case, monkeypatch):
    n, binary, weighted, na, walk = CASES[case]
    ds, u, pres = _job(n, seed=41 + n, binary=binary, na_rate=na, genome_len=3000 if n < 2000 else 1200)
    ka = _engine(ds, walk=walk, monkeypatch=monkeypatch)
    assert ka.U == len(u)
    w = np.random.default_rng(n).uniform(0.2, 1.5, n) if weighted else None
    B = 6
    got = ka.permutation_minp(ds.pheno, binary, B, w, 2, n - 2, seed=9)
    assert got.shape == (ds.pheno.shape[1], B)
    cols = permute_columns(ds.pheno, B, seed=9).reshape(-1, n)
    want = host_minp(pres, cols, binary, w, 2, n - 2).reshape(got.shape)
    assert (got < 1).any()
    # unweighted chi2 is bit-identical (exact integer tables, the reference's operation order); its p = exp(-chi2/2)
    # then differs from the host's exp by at most an ulp or so (DESIGN.md §5)
    assert np.allclose(got, want, rtol=1e-13 if binary and not weighted else RTOL, atol=0), (got, want)
    # sample limits under which no k-mer is testable: min-p = 1
    assert np.array_equal(ka.permutation_minp(ds.pheno, binary, 3, w, n - 1, n, seed=9), np.ones((got.shape[0], 3)))


def _code(ph):
    return np.where(np.isnan(ph), -1, ph).astype(np.int8)


@pytest.mark.gpu
@pytest.mark.parametrize("binary", [True, False])
def test_identity_permutation_and_no_side_effects(binary):
    n = 40
    ds, _u, _pres = _job(n, seed=77, binary=binary, n_pheno=3)
    ka = _engine(ds)
    ctx = ka.ctx
    obs = ds.pheno.T.copy()

    def test_at_one():
        if binary:
            return ctx.test_chi2(_code(obs), None, 2, n - 2, 1.0)
        return ctx.test_welch(obs, None, 2, n - 2, 1.0)

    def minp():
        return ctx.minp_chi2(_code(obs), None, 2, n - 2) if binary else ctx.minp_welch(obs, None, 2, n - 2)

    ns = test_at_one()
    before = ctx.fetch_survivors(ns)
    m = minp()
    after = ctx.fetch_survivors(ns)
    for f in before:
        assert np.array_equal(before[f], after[f], equal_nan=True), f
    for j in range(obs.shape[0]):
        p = before["p"][before["pheno"] == j]
        assert len(p) and m[j] == p.min(), (j, m[j], p.min())


FIELDS = ("kmer", "row", "stat", "p", "n_with")


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.threshold == y.threshold and np.array_equal(x.minp, y.minp)
        for f in FIELDS:
            assert np.array_equal(getattr(x, f), getattr(y, f)), f


@pytest.mark.gpu
@pytest.mark.parametrize("binary", [True, False])
def test_thresholds_equal_across_execution_shapes(binary):
    from phenotypeseeker_b200.group import GpuGroup
    from phenotypeseeker_b200.pipeline import KmerAssociation
    ds = synth.config(0 if binary else 2, tiny=True)
    N = ds.n_samples
    kw = dict(min_samples=2, max_samples=N - 2, pvalue_cutoff=0.05, omit_b=False)
    ka = KmerAssociation(device=0)
    ka.count(ds.files, 16)
    ka.build()
    one = ka.test(ds.pheno, binary, None, n_perm=20, perm_seed=3, **kw)
    assert all(r.threshold is not None and r.minp.shape == (20,) for r in one)
    assert any(len(r.kmer) for r in one) or binary is False
    t = permutation_thresholds(np.stack([r.minp for r in one]), 0.05)
    assert [r.threshold for r in one] == list(t)
    # survivors under a threshold: ps_test_* at thr = threshold_j, restricted to column j
    for j, r in enumerate(one):
        if binary:
            ns = ka.ctx.test_chi2(_code(ds.pheno.T), None, 2, N - 2, r.threshold)
        else:
            ns = ka.ctx.test_welch(ds.pheno.T.copy(), None, 2, N - 2, r.threshold)
        sv = ka.ctx.fetch_survivors(ns)
        sel = sv["pheno"] == j
        assert np.array_equal(sv["kmer"][sel], r.kmer) and np.array_equal(sv["p"][sel], r.p)
    for n_super in (0, None):
        ka.count(ds.files, 16)
        U, rng = ka.test_in_ranges(ds.pheno, binary, 3, None, n_instances=ka.instances_upper(), n_super=n_super,
                                   n_perm=20, perm_seed=3, **kw)
        _same(rng, one)
    del ka
    gc.collect()
    g = GpuGroup([0, 0])
    g.count(ds.files, 16)
    _Ug, grp = g.test(ds.pheno, binary, None, n_perm=20, perm_seed=3, **kw)
    _same(grp, one)


# --- the drop-in -----------------------------------------------------------------------------------------------------
def _stand_in(ds, paths, binary):
    class Sample:
        def __init__(self, name, address, ph):
            self.name, self.address, self.weight, self.phenotypes = name, address, 1, ph

    class Pheno:
        no_results = []
        pred_scale = "binary" if binary else "continuous"
        pvalue_cutoff = 0.05
        omit_B = False
        real_counts = False
        no_kmers_to_analyse = None

        def __init__(self, name):
            self.name, self.ML_df = name, None

    samples = collections.OrderedDict()
    for i, (nm, p) in enumerate(zip(ds.names, paths)):
        samples[nm] = Sample(nm, p, {c: ("NA" if np.isnan(ds.pheno[i, j]) else
                                         (int(ds.pheno[i, j]) if binary else float(ds.pheno[i, j])))
                                     for j, c in enumerate(ds.pheno_names)})
    cols = collections.OrderedDict((c, Pheno(c)) for c in ds.pheno_names)
    Input = type("Input", (), {"samples": samples, "phenotypes_to_analyse": cols, "num_threads": 3})
    Samples = type("Samples", (), {"kmer_length": 16, "cutoff": 1, "min_samples": 2,
                                   "max_samples": ds.n_samples - 2, "kmerDB": None})
    return types.SimpleNamespace(Input=Input, Samples=Samples, phenotypes=Pheno)


@pytest.mark.gpu
@pytest.mark.parametrize("device", [0, [0, 0]], ids=["one_gpu", "group"])
def test_dropin_with_permutations(device, tmp_path, monkeypatch):
    from phenotypeseeker_b200 import modeling_gpu as mg
    from phenotypeseeker_b200.pipeline import KmerAssociation
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("PS_PERMUTATIONS", "50")
    monkeypatch.setenv("PS_PERMUTATION_SEED", "4")
    ds = synth.config(0, tiny=True)
    _ph_file, paths = ds.write(str(tmp_path / "in"))
    N = ds.n_samples
    m = _stand_in(ds, paths, True)
    mg._STATE["ka"] = None
    try:
        mg.install(m, device=device)
        m.Samples.get_feature_vector()
        m.phenotypes.kmer_testing_setup()
        for ph in m.Input.phenotypes_to_analyse.values():
            ph.test_kmers_association_with_phenotype()
    finally:
        mg._STATE["ka"] = None
        gc.collect()
    # the same job by hand: min-p of 50 permutations, each column cut at its own threshold
    ka = KmerAssociation(device=0)
    ka.count(ds.files, 16)
    ka.build()
    minp = ka.permutation_minp(ds.pheno, True, 50, None, 2, N - 2, seed=4)
    t = permutation_thresholds(minp, 0.05)
    log = (tmp_path / "log.txt").read_text()
    for j, (name, ph) in enumerate(m.Input.phenotypes_to_analyse.items()):
        r = ostats.chi2_rows(ok.presence_matrix(ka.ctx.get_union(), [ok.count_kmers(f, 16) for f in ds.files]),
                             _code(ds.pheno[:, j]), np.ones(N), 2, N - 2)
        p = np.exp(-0.5 * r["stat"])
        keep = r["tested"] & (p < t[j])
        want = sorted(ok_str for ok_str in _kmer_strings(ka.ctx.get_union()[keep]))
        got = sorted(ph.ML_df.columns) if ph.ML_df.shape[0] else []
        assert got == want, name
        assert f"Permutation threshold for {name}: p < {t[j]:.6E} (50 permutations)" in log
    assert log.count("took") == len(m.Input.phenotypes_to_analyse)


def _kmer_strings(kmers):
    from phenotypeseeker_b200.pipeline import kmers_to_str
    return kmers_to_str(kmers, 16)
