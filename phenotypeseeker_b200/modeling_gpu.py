"""Drop-in boundary for `phenotypeseeker modeling`: the GPU hot path behind the reference's own
method contract (SURVEY.md §8b).

`install(modeling_module)` re-wires the five methods that `modeling.modeling()` calls between
"if not Input.jump_to:" and `Input.pop_phenos_out_of_kmers()` (modeling.py:1644-1686) so that the
unmodified orchestrator, CLI, `get_ML_df` writers and sklearn stage keep working:

    Samples.get_kmer_lists            (:303-315)  -> no-op (runs inside the reference's Pool workers)
    Samples.get_feature_vector        (:351-365)  -> GPU: decode + count + union + bit matrix
    Samples.map_samples               (:317-348)  -> no-op
    phenotypes.kmer_testing_setup     (:632-657)  -> phenotypes.no_kmers_to_analyse = U
    phenotypes.test_kmers_association_with_phenotype (:659-675) -> GPU test -> self.ML_df

The contract honoured: `phenotypes.no_kmers_to_analyse`, `pheno.ML_df` (columns = surviving k-mer
strings in the reference's stripe-major order, rows positional: statistic, "%.2E" p-value, [group
means,] n_with, "| names", then N presence values), `phenotypes.no_results`, the `log.txt` timer line.

`write_outputs` restates what the unchanged `get_ML_df` (:1113-1145) then writes, so that output
files can be produced and byte-compared without the reference installed (tests/, standalone use).

The CUDA context is created lazily inside get_feature_vector — in the parent process, after the
first Pool has exited — and lives in this module, never on Samples/phenotypes instances (they are
dill-pickled into later Pools).
"""
import os
import sys
import time

import numpy as np
import pandas as pd

from .pipeline import KmerAssociation, kmers_to_str, read_sample_file

_STATE = {"ka": None, "pid": None, "devices": None, "names": None, "ranges": 1, "results": None, "db": None}


def parse_devices(spec):
    """PS_DEVICE / device= -> one device index (int: the single-GPU KmerAssociation) or a list of them (several
    entries: a GpuGroup, one rank per entry, repeats allowed). Accepts an int, "0", "0,1,2,3", "0, 0" or a sequence."""
    if isinstance(spec, str):
        parts = [p.strip() for p in spec.split(",") if p.strip()]
    elif isinstance(spec, (list, tuple, range)):
        parts = list(spec)
    else:
        return int(spec)
    if not parts:
        raise ValueError(f"no device in {spec!r}")
    devs = [int(p) for p in parts]
    return devs[0] if len(devs) == 1 else devs


def _ka(device=None):
    """The engine of this process: a KmerAssociation for one device, a GpuGroup for several. Made again when the
    process changes (fork) or an explicit `device` asks for other devices."""
    spec = None if device is None else parse_devices(device)
    if _STATE["ka"] is None or _STATE["pid"] != os.getpid() or (spec is not None and spec != _STATE["devices"]):
        devs = parse_devices(os.environ.get("PS_DEVICE", "0")) if spec is None else spec
        _STATE["ka"] = None                   # free the old engine's device memory before the new one allocates
        if isinstance(devs, int):
            _STATE["ka"] = KmerAssociation(device=devs)
        else:
            from .group import GpuGroup
            _STATE["ka"] = GpuGroup(devs)
        _STATE["pid"], _STATE["devices"] = os.getpid(), devs
    return _STATE["ka"]


def stripe_major_order(rows, n_stripes):
    """Column order of the reference's ML_df before sorting: `split -n r/T` deals union line i to
    stripe i % T (modeling.py:337-342), stripes are concatenated in order (:670-672)."""
    rows = np.asarray(rows, dtype=np.int64)
    return np.lexsort((rows, rows % int(n_stripes)))


def build_ml_df(res, k, sample_names, n_stripes, binary, counts=None):
    """PhenoResult -> the DataFrame `test_kmers_association_with_phenotype` leaves in self.ML_df."""
    order = stripe_major_order(res.row, n_stripes)
    if len(order) == 0:
        return pd.DataFrame()
    kmers = kmers_to_str(res.kmer[order], k)
    names = np.array(sample_names, dtype=object)
    pres = res.presence[order] != 0
    vals = res.presence[order] if counts is None else counts[order]
    named = pres if res.na_mask is None else pres & ~np.asarray(res.na_mask, dtype=bool)[None, :]
    nhead = 4 if binary else 6
    # one object array (rows = the positional rows of ML_df, columns = k-mers) instead of a dict of
    # Python lists: same cell types as the reference's rows (np.float64, str, int), ~4x faster to build
    cells = np.empty((nhead + len(names), len(order)), dtype=object)
    cells[0] = [np.float64(round(float(x), 2)) for x in res.stat[order]]
    cells[1] = ["%.2E" % x for x in res.p[order]]
    if not binary:
        cells[2] = [np.float64(round(float(x), 2)) for x in res.mean_x[order]]
        cells[3] = [np.float64(round(float(x), 2)) for x in res.mean_y[order]]
    cells[nhead - 2] = [int(x) for x in res.n_with[order]]
    cells[nhead - 1] = [" ".join(["|"] + list(names[m])) for m in named]
    cells[nhead:] = np.asarray(vals).T.astype(np.int64).astype(object)
    return pd.DataFrame(cells, columns=kmers)


def write_outputs(ml_df, pheno_name, sample_names, weights, pheno_values, binary, kmer_limit=None, outdir="."):
    """What the unchanged get_ML_df (modeling.py:1113-1145) does with ML_df: label, order by the
    p-value STRING (lexicographic, Appendix B3), write <stat>_results_<ph>.tsv (+ _top<N>.tsv) and
    <ph>_MLdf.csv. Returns the trimmed feature frame."""
    out_cols = (["chi2", "p-value", "num_samples_w_kmer", "samples_with_kmer"] if binary else
                ["t-test", "p-value", "+_group_mean", "-_group_mean", "num_samples_w_kmer", "samples_with_kmer"])
    df = ml_df.copy()
    df.columns.name = "k-mer"
    df.index = out_cols + list(sample_names)
    df = df.sort_values("p-value", axis=1)
    df.T[out_cols].to_csv(os.path.join(outdir, f"{out_cols[0]}_results_{pheno_name}.tsv"), sep="\t")
    if kmer_limit:
        df = df.iloc[:, :kmer_limit]
        df.T[out_cols].to_csv(os.path.join(outdir, f"{out_cols[0]}_results_{pheno_name}_top{kmer_limit}.tsv"), sep="\t")
    df = df.drop(out_cols)
    df["weights"] = list(weights)
    df["phenotype"] = list(pheno_values)
    df = df.loc[df.phenotype != "NA"]
    df.phenotype = df.phenotype.apply(pd.to_numeric)
    df.to_csv(os.path.join(outdir, pheno_name + "_MLdf.csv"))
    return df


def write_legacy_outputs(ml_df, pheno_name, binary, outdir="."):
    """The file names of PhenotypeSeeker <= 1.0 that README.md:96-105 / user_manual.md:56-88 still document
    (and BASELINE.json's north_star quotes): `chi-squared_test_results_<ph>.txt` / `t-test_results_<ph>.txt` and
    `k-mers_filtered_by_pvalue_<ph>.txt`. v1.2.4 writes neither (SURVEY.md Appendix B1); this is an optional
    extra (env PS_LEGACY_OUTPUTS=1 with install()). Layout as documented there: no header, one k-mer per
    line in test order, `kmer <tab> statistic <tab> p [<tab> mean_x <tab> mean_y] <tab> n <tab> | names`.
    Like v1.2.4 itself only the k-mers that passed the p-value filter are known, so both files hold the
    same rows. Returns the two paths."""
    nstat = 4 if binary else 6
    lines = []
    for kmer in ml_df.columns:
        head = ml_df[kmer].iloc[:nstat]
        lines.append("\t".join([str(kmer)] + [str(v) for v in head]) + "\n")
    first = ("chi-squared_test_results_" if binary else "t-test_results_") + pheno_name + ".txt"
    paths = [os.path.join(outdir, first), os.path.join(outdir, "k-mers_filtered_by_pvalue_" + pheno_name + ".txt")]
    for pth in paths:
        with open(pth, "w") as f:
            f.writelines(lines)
    return paths


def pheno_matrix(samples, pheno_names):
    """Input.samples (name -> Samples obj with .phenotypes{col -> int/float/'NA'}) -> N x P float, NaN = NA."""
    out = np.full((len(samples), len(pheno_names)), np.nan)
    for i, s in enumerate(samples):
        for j, p in enumerate(pheno_names):
            v = s.phenotypes[p]
            if not (isinstance(v, str)):
                out[i, j] = float(v)
    return out


def permutation_options():
    """PS_PERMUTATIONS=B (> 0): the permutation threshold of B phenotype permutations replaces the Bonferroni cut
    (pvalue / U) of the tests; PS_PERMUTATION_SEED (default 0) seeds them. Unset or 0: the reference's rule, and
    no keyword at all. -> keyword arguments of KmerAssociation.test / test_in_ranges / GpuGroup.test."""
    n_perm = int(os.environ.get("PS_PERMUTATIONS", "0") or 0)
    if n_perm <= 0:
        return {}
    return dict(n_perm=n_perm, perm_seed=int(os.environ.get("PS_PERMUTATION_SEED", "0") or 0))


def threshold_log_line(res):
    """The log.txt line of a column tested against a permutation threshold, None for the reference's rule."""
    if getattr(res, "threshold", None) is None:
        return None
    return f"Permutation threshold for {res.name}: p < {res.threshold:.6E} ({len(res.minp)} permutations)\n"


def run_hot_path(files, sample_names, k, cutoff, pheno, pheno_names, binary, weights, min_samples, max_samples,
                 pvalue_cutoff, omit_b, n_stripes, real_counts=False, device=None):
    """Stages 1-3 on the GPU -> (U, {pheno_name: ML_df}). Plain-data entry used by tests/standalone.
    device: as PS_DEVICE (parse_devices); several entries run on a GpuGroup. PS_PERMUTATIONS: see
    permutation_options."""
    ka = _ka(device)
    ka.count(files, k, cutoff)
    kw = dict(min_samples=min_samples, max_samples=max_samples, pvalue_cutoff=pvalue_cutoff, omit_b=omit_b,
              pheno_names=list(pheno_names), **permutation_options())
    if ka.fits_in_one_build():
        U = ka.build()
        res = ka.test(pheno, binary, weights, **kw)
    else:
        U, res = ka.test_in_ranges(pheno, binary, ka.ranges_needed(), weights, n_instances=ka.instances_upper(), **kw)
    out = {}
    for j, r in enumerate(res):
        r.na_mask = np.isnan(np.asarray(pheno, dtype=np.float64).reshape(len(sample_names), -1)[:, j])
        counts = None
        if real_counts and len(r.kmer):
            counts = ka.count_matrix(r.kmer).T
            counts = counts * (r.presence != 0)       # a count below the cutoff is 0 in the reference's list (glistmaker -c)
        out[r.name] = build_ml_df(r, k, sample_names, n_stripes, binary, counts)
    return U, out


# ---------------------------------------------------------------------------------------
def install(m, device=None, native_weights=None):
    """Re-wire the reference module `m` (PhenotypeSeeker.modeling) onto the GPU path.

    device (default: env PS_DEVICE, else 0): one device index, or several ("0,1,2,3" or a sequence) to run on a
    GpuGroup in this one process. A group builds and tests every column at once in kmer_testing_setup, as a
    single GPU does for inputs that need k-mer ranges; -rc, native_weights="gpu" and --kmerDB work on both.

    native_weights (default: env PS_NATIVE_WEIGHTS): also replace the `-w` weight computation
    (`Samples.get_mash_sketches` / `get_weights`, modeling.py:386-503: mash binary + Biopython + ete3) with
    phenotypeseeker_b200.weights — for installations without those three; see that module for what is
    pinned against the reference and what is not. True / "1": on the host, from the sample files. "gpu": sketches,
    distances and neighbour joining on the device, from the samples get_feature_vector decoded (same weights on
    well-formed FASTA / FASTQ; the text is read as the k-mer counter reads it, DESIGN.md "Reader semantics")."""
    Input, Samples, phenotypes = m.Input, m.Samples, m.phenotypes
    if native_weights is None:
        env = os.environ.get("PS_NATIVE_WEIGHTS", "0")
        native_weights = "gpu" if env == "gpu" else env == "1"
    elif native_weights != "gpu":
        native_weights = bool(native_weights)

    def get_kmer_lists(self):          # runs in Pool workers: nothing to do
        return None

    def map_samples(self):             # runs in Pool workers: nothing to do
        return None

    def get_feature_vector(cls):
        samples = list(Input.samples.values())
        ka = _ka(device)
        db = None
        if getattr(Samples, "kmerDB", None):                 # --kmerDB: glistmaker on the database, :367-372
            db = ka.kmers_of(read_sample_file(Samples.kmerDB), int(Samples.kmer_length))
        ka.count_files([s.address for s in samples], int(Samples.kmer_length), int(Samples.cutoff))   # streamed in batches
        _STATE["results"] = None
        _STATE["db"] = db
        _STATE["ranges"] = 1 if ka.fits_in_one_build() else ka.ranges_needed()
        if _STATE["ranges"] == 1:
            ka.build()
            if db is not None:
                ka.restrict_to(db)                           # glistcompare -i
        os.makedirs("K-mer_lists", exist_ok=True)   # get_mash_sketches (-w) writes its sketches there
        _STATE["names"] = [s.name for s in samples]

    def test_all_columns():
        """One pass over the matrix for ALL phenotype columns (the reference loops over them, :1680-1683);
        per-column results are cached for the per-column calls that follow. Memory-bounded jobs run in
        k-mer ranges, where build and test alternate and U is only known at the end."""
        if _STATE["results"] is not None:
            return _STATE["results"]
        ka = _ka(device)
        samples = list(Input.samples.values())
        cols = list(Input.phenotypes_to_analyse.keys())
        binary = phenotypes.pred_scale == "binary"
        ph = pheno_matrix(samples, cols)
        w = np.array([float(s.weight) for s in samples])
        kw = dict(min_samples=Samples.min_samples, max_samples=Samples.max_samples, pvalue_cutoff=phenotypes.pvalue_cutoff,
                  omit_b=bool(phenotypes.omit_B), pheno_names=cols, **permutation_options())
        if _STATE["ranges"] > 1:
            _, res = ka.test_in_ranges(ph, binary, _STATE["ranges"], w, n_instances=ka.instances_upper(),
                                       restrict=_STATE["db"], **kw)
        else:
            res = ka.test(ph, binary, w, **kw)
        for j, r in enumerate(res):
            r.na_mask = np.isnan(ph[:, j])
        _STATE["results"] = {r.name: r for r in res}
        return _STATE["results"]

    def kmer_testing_setup(cls):
        which = "Welch t-tests" if phenotypes.pred_scale == "continuous" else "chi-square tests"
        sys.stderr.write(f"\n\x1b[1;32mConducting the k-mer specific {which}:\x1b[0m\n")
        sys.stderr.flush()
        if _STATE["ranges"] > 1:
            test_all_columns()                 # U = sum of the range sizes
        phenotypes.no_kmers_to_analyse = _ka(device).U

    def test_kmers_association_with_phenotype(self):
        start = time.time()
        ka = _ka(device)
        names = _STATE["names"]
        binary = phenotypes.pred_scale == "binary"
        res = test_all_columns()[self.name]
        counts = None
        if phenotypes.real_counts and len(res.kmer):
            counts = ka.count_matrix(res.kmer).T
            counts = counts * (res.presence != 0)         # a count below the cutoff is 0 in the reference's list (glistmaker -c)
        self.ML_df = build_ml_df(res, ka.k, names, Input.num_threads, binary, counts)
        if self.ML_df.shape[0] == 0:
            self.no_results.append(self.name)
        elif os.environ.get("PS_LEGACY_OUTPUTS", "0") == "1":
            write_legacy_outputs(self.ML_df, self.name, binary)
        with open("log.txt", "a") as log:       # the reference's `timer` line (modeling.py:54-61)
            log.write(f"Func {test_kmers_association_with_phenotype} took {time.time() - start} secs\n")
            if threshold_log_line(res):
                log.write(threshold_log_line(res))

    def get_mash_sketches(self):       # runs in Pool workers: sketching happens in get_weights
        return None

    def get_weights(cls):
        from . import weights as psw
        samples = list(Input.samples.values())
        names = [s.name for s in samples]
        if native_weights == "gpu":
            # the samples get_feature_vector decoded are still on the device; ingesting them again would start a
            # new job and drop the union and matrix the tests need
            if _STATE["names"] != names or _STATE["ka"] is None or _STATE["pid"] != os.getpid():
                raise RuntimeError("native_weights='gpu' computes the weights from the samples get_feature_vector "
                                   "decoded; call it first, with the same Input.samples")
            w = psw.gsc_weights_on_device(_STATE["ka"], names, 0, keep_glob_quirk=True)
        else:
            w = psw.gsc_weights_for_samples(names, [read_sample_file(s.address) for s in samples],
                                            keep_glob_quirk=True)
        for s, wi in zip(samples, w):
            s.weight = float(wi)

    if native_weights:
        Samples.get_mash_sketches = get_mash_sketches
        Samples.get_weights = classmethod(get_weights)
    Samples.get_kmer_lists = get_kmer_lists
    Samples.map_samples = map_samples
    Samples.get_feature_vector = classmethod(get_feature_vector)
    phenotypes.kmer_testing_setup = classmethod(kmer_testing_setup)
    phenotypes.test_kmers_association_with_phenotype = test_kmers_association_with_phenotype
    return m
