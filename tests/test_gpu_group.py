"""Several GPUs from one process (group.GpuGroup): every result equals that of a single KmerAssociation build.

On one GPU, three contexts on device 0 play three ranks (their pools are plain device pointers of one device);
the multi-device cases ([0, 1], [0, 1, 2, 3]) skip on machines with fewer GPUs."""
import collections
import gc
import types

import numpy as np
import pytest

from phenotypeseeker_b200 import synth
from phenotypeseeker_b200 import modeling_gpu as mg
from phenotypeseeker_b200 import weights as W
from phenotypeseeker_b200.group import GpuGroup
from phenotypeseeker_b200.pipeline import KmerAssociation

pytestmark = pytest.mark.gpu

FIELDS = ("kmer", "row", "stat", "p", "mean_x", "mean_y", "n_with", "rowbits")


@pytest.fixture(autouse=True)
def _fresh_dropin_engine():
    """The drop-in keeps its engine in modeling_gpu._STATE: leave none behind for the tests that follow."""
    yield
    mg._STATE["ka"] = None
    gc.collect()


def _devices(devs):
    import torch
    if torch.cuda.device_count() < max(devs) + 1:
        pytest.skip(f"needs {max(devs) + 1} GPUs, this machine has {torch.cuda.device_count()}")
    return devs


DEVICE_SETS = [[0, 0, 0], [0, 1], [0, 1, 2, 3]]


def _case(case):
    """-> (dataset, k, cutoff, test keywords, passes)."""
    kw, passes, cutoff, k = {}, None, 1, 16
    if case == "chi2_k16":
        ds = synth.config(0, tiny=True)
        kw = dict(pvalue_cutoff=0.05, omit_b=True)
    elif case == "chi2_weighted_k16":
        ds = synth.config(1, tiny=True)
        kw = dict(pvalue_cutoff=500.0, omit_b=False)           # Bonferroni on, still survivors at CI size
    elif case == "groups_k13":
        ds, k = synth.make_dataset(520, genome_len=2500, seed=79, n_clades=5, contigs=(1, 2)), 13    # 3 sample groups
        kw = dict(pvalue_cutoff=0.05, omit_b=True)
    elif case == "reads_cutoff2":
        ds, cutoff = synth.config(3, tiny=True), 2
        kw = dict(pvalue_cutoff=1.0, omit_b=True)               # 4 samples: keep every tested row
    elif case == "welch_weighted":
        ds = synth.config(2, tiny=True)
        kw = dict(pvalue_cutoff=200.0)
    elif case == "streams_k20":
        ds, k = synth.config(0, tiny=True), 20
        kw = dict(pvalue_cutoff=0.05, omit_b=True)
    else:                                                       # two passes over super-ranges, Bonferroni, top k
        assert case == "passes2"
        ds, passes = synth.config(1, tiny=True), 2
        kw = dict(pvalue_cutoff=500.0, omit_b=False, top_k=40)
    N = ds.n_samples
    kw.update(min_samples=2, max_samples=N - 2)
    return ds, k, cutoff, kw, passes


def _single(ds, k, cutoff, kw, db=None):
    ka = KmerAssociation(device=0)
    ka.count(ds.files, k, cutoff)
    ka.build()
    if db is not None:
        ka.restrict_to(db)
    res = ka.test(ds.pheno, ds.binary, ds.weights, **kw)
    U = ka.U
    ka.ctx.close()
    return U, res


def _assert_same(got, want):
    (U_g, res_g), (U_w, res_w) = got, want
    assert U_g == U_w
    assert len(res_g) == len(res_w)
    for a, b in zip(res_g, res_w):
        assert a.name == b.name
        for f in FIELDS:
            assert np.array_equal(getattr(a, f), getattr(b, f)), f


@pytest.mark.parametrize("devs", DEVICE_SETS, ids=lambda d: "dev" + "".join(map(str, d)))
@pytest.mark.parametrize("case", ["chi2_k16", "chi2_weighted_k16", "groups_k13", "reads_cutoff2", "welch_weighted",
                                  "streams_k20", "passes2"])
def test_group_equals_single_build(case, devs):
    devs = _devices(devs)
    ds, k, cutoff, kw, passes = _case(case)
    want = _single(ds, k, cutoff, kw)
    assert sum(len(r.kmer) for r in want[1]) > 0
    g = GpuGroup(devs)
    g.count(ds.files, k, cutoff)
    got = g.test(ds.pheno, ds.binary, ds.weights, passes=passes, **kw)
    _assert_same(got, want)
    assert g.U == want[0]
    got2 = g.test(ds.pheno, ds.binary, ds.weights, passes=passes, **kw)      # a second step on the same job
    _assert_same(got2, want)
    del g
    gc.collect()


@pytest.mark.parametrize("passes", [None, 2])
def test_group_restrict_equals_restrict_to(passes):
    ds, k, cutoff, kw, _ = _case("chi2_weighted_k16")
    text = ds.files[0][:len(ds.files[0]) // 3] + b"\n>x\n" + ds.files[5][-20000:]
    one = KmerAssociation(device=0)
    db = one.kmers_of(text, k)
    one.ctx.close()
    want = _single(ds, k, cutoff, kw, db=db)
    g = GpuGroup([0, 0, 0])
    assert np.array_equal(g.kmers_of(text, k), db)
    g.count(ds.files, k, cutoff)
    got = g.test(ds.pheno, ds.binary, ds.weights, restrict=db, passes=passes, **kw)
    assert 0 < want[0]
    _assert_same(got, want)


def test_group_lookup_and_weights_equal_single_context():
    ds = synth.config(0, tiny=True)
    ka = KmerAssociation(device=0)
    ka.count(ds.files, 16)
    ka.build()
    kmers = ka.ctx.get_union()[::7]
    g = GpuGroup([0, 0, 0])
    g.count(ds.files, 16)
    for s in range(ds.n_samples):
        assert np.array_equal(g.lookup(s, kmers), ka.ctx.lookup(s, kmers)), s
    for quirk in (False, True):
        want = W.gsc_weights_on_device(ka.ctx, ds.names, 0, keep_glob_quirk=quirk)
        got = W.gsc_weights_on_device(g, ds.names, 0, keep_glob_quirk=quirk)
        assert np.array_equal(got, want), quirk
    h_w, n_w = ka.ctx.mash_sketch(3, 7)
    h_g, n_g = g.mash_sketch(3, 7)                 # crosses the rank blocks [0,4) [4,8) [8,12)
    assert np.array_equal(h_g, h_w) and np.array_equal(n_g, n_w)


# --- the drop-in, driven in modeling()'s call order on stand-in reference classes -------------------------------
def _stand_in(ds, paths, binary, real_counts=False, kmer_db=None, k=16):
    class Sample:
        def __init__(self, name, address, ph):
            self.name, self.address, self.weight = name, address, 1
            self.phenotypes = ph

    class Pheno:
        no_results = []
        pred_scale = "binary" if binary else "continuous"
        pvalue_cutoff = 0.05 if binary else 200.0
        omit_B = binary
        no_kmers_to_analyse = None

        def __init__(self, name):
            self.name, self.ML_df = name, None

    Pheno.real_counts = real_counts
    samples = collections.OrderedDict()
    for i, (nm, p) in enumerate(zip(ds.names, paths)):
        ph = {c: ("NA" if np.isnan(ds.pheno[i, j]) else (int(ds.pheno[i, j]) if binary else float(ds.pheno[i, j])))
              for j, c in enumerate(ds.pheno_names)}
        samples[nm] = Sample(nm, p, ph)
    cols = collections.OrderedDict((c, Pheno(c)) for c in ds.pheno_names)
    Input = type("Input", (), {"samples": samples, "phenotypes_to_analyse": cols, "num_threads": 3})
    Samples = type("Samples", (), {"kmer_length": k, "cutoff": 1, "min_samples": 2, "max_samples": ds.n_samples - 2,
                                   "kmerDB": kmer_db})
    return types.SimpleNamespace(Input=Input, Samples=Samples, phenotypes=Pheno)


def _modeling(m, weights):
    """The stages of modeling.modeling() that install() replaces, in its order."""
    m.Samples.get_feature_vector()
    if weights:
        m.Samples.get_weights()
    m.phenotypes.kmer_testing_setup()
    for ph in m.Input.phenotypes_to_analyse.values():
        ph.test_kmers_association_with_phenotype()
    return (m.phenotypes.no_kmers_to_analyse, list(m.phenotypes.no_results),
            {n: ph.ML_df for n, ph in m.Input.phenotypes_to_analyse.items()},
            [s.weight for s in m.Input.samples.values()])


@pytest.mark.parametrize("devs", [[0, 0], [0, 1], [0, 1, 2, 3]], ids=lambda d: "dev" + "".join(map(str, d)))
@pytest.mark.parametrize("option", ["plain", "rc", "weights_gpu", "kmerdb", "welch"])
def test_install_on_a_group_equals_single_gpu(option, devs, tmp_path, monkeypatch):
    devs = _devices(devs)
    monkeypatch.chdir(tmp_path)
    binary = option != "welch"
    ds = synth.config(0 if binary else 2, tiny=True)
    ph_file, paths = ds.write(str(tmp_path / "in"))
    db = None
    if option == "kmerdb":
        db = str(tmp_path / "db.fa")
        with open(db, "wb") as f:                  # the second half of every sample: cassettes included
            f.write(b"".join(b"\n>db\n" + t[len(t) // 2:] for t in ds.files))
    out = {}
    for dev in (devs, 0):
        m = _stand_in(ds, paths, binary, real_counts=option == "rc", kmer_db=db)
        mg.install(m, device=dev, native_weights="gpu" if option == "weights_gpu" else None)
        out[str(dev)] = _modeling(m, option == "weights_gpu")
    (U_g, nr_g, df_g, w_g), (U_s, nr_s, df_s, w_s) = out[str(devs)], out["0"]
    assert U_g == U_s and U_s > 0
    assert nr_g == nr_s
    assert w_g == w_s
    assert df_g.keys() == df_s.keys()
    assert any(d.shape[1] for d in df_s.values())
    for n in df_s:
        assert df_g[n].equals(df_s[n]), n


@pytest.mark.parametrize("tag", ["chi2", "ttest"])
def test_run_hot_path_on_a_group_reproduces_reference_files(tag, tmp_path):
    from test_outputs import _case as out_case, _compare_files, _pheno_values
    gold_dir, c, ds, o = out_case(tag)
    N = ds.n_samples
    U, dfs = mg.run_hot_path(ds.files, ds.names, o["k"], 1, ds.pheno[:, :1], ["pheno1"], ds.binary, None, 2, N - 2,
                             o["pvalue"], o["omit_b"], o["T"], device=[0, 0])
    assert isinstance(mg._ka(), GpuGroup)
    mg.write_outputs(dfs["pheno1"], "pheno1", ds.names, [1] * N, _pheno_values(ds), ds.binary, o["limit"], str(tmp_path))
    _compare_files(gold_dir, c["files"], str(tmp_path))


def test_route_connect_rejects_mismatched_ranks():
    from phenotypeseeker_b200._native import Context, PsError
    ds = synth.config(0, tiny=True)
    G, N = 3, ds.n_samples
    ranks = [Context(0) for _ in range(G)]
    spare = Context(0)
    try:
        for r, c in enumerate(ranks + [spare]):
            c.begin(16, N)
            lo = N * min(r, G - 1) // G
            c.add_samples(lo, [ds.files[lo]])
        spl = ranks[0].sample_quantiles(0, G)
        pages = max(c.route_pages_needed(G) for c in ranks)
        for r, c in enumerate(ranks):
            c.route_setup(G, r, spl, pages)

        def code(c, lst):
            with pytest.raises(PsError) as e:
                c.route_connect(lst)
            return e.value.code

        assert code(ranks[0], [ranks[0], ranks[2], ranks[1]]) == -3          # wrong rank index (PS_ERR_STATE)
        assert code(ranks[0], [ranks[0], ranks[1], spare]) == -3             # a rank without a pool
        spare.route_setup(2, 1, spl[:1], pages)
        assert code(ranks[0], [ranks[0], ranks[1], spare]) == -3             # a rank of another nparts
        assert code(ranks[0], [ranks[0]] * 9) == -1                          # more than PART_MAX (PS_ERR_ARG)
        for c in ranks:
            c.route_connect(ranks)                                           # the right table is accepted
    finally:
        for c in ranks + [spare]:
            c.close()
