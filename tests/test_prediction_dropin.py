"""CPU tests of the prediction drop-in (prediction_gpu.install): the engine behind it is an oracle-backed stand-in
with the KmerAssociation interface, so these check the wiring — when the cohort is ingested, what one
get_inp_matrix call asks of the engine, the -c threshold and the choice of engine from PS_DEVICE."""
import os
import types

import numpy as np
import pytest

from oracle import kmers as ok
from phenotypeseeker_b200 import group, synth
from phenotypeseeker_b200 import prediction_gpu as pg


class OracleEngine:
    """count_files + count_matrix from the C oracle, with a log of the calls."""

    def __init__(self, device=0):
        self.device = device
        self.calls = []

    def count_files(self, paths, k, cutoff=1):
        self.calls.append(("count_files", len(paths), k, cutoff))
        self.k = k
        self.lists = [ok.count_kmers(open(p, "rb").read(), k, cutoff) for p in paths]

    def count_matrix(self, kmers, first_idx=0, count=None):
        self.calls.append(("count_matrix", len(kmers)))
        q = np.asarray(kmers, dtype=np.uint64)
        return np.stack([ok.map_counts(q, *l) for l in self.lists])


def _module(paths, cutoff):
    """A stand-in for PhenotypeSeeker.prediction: the attributes get_inp_matrix reads."""
    samples = {f"s{i}": types.SimpleNamespace(address=p) for i, p in enumerate(paths)}

    class Phenotypes:
        pass
    Phenotypes.cutoff = cutoff

    class Samples:
        pass
    return types.SimpleNamespace(Input=types.SimpleNamespace(samples=samples), Phenotypes=Phenotypes, Samples=Samples)


def _model(p, kmers):
    m = p.Phenotypes()
    m.kmers, m.pca = list(kmers), False
    return m


@pytest.fixture
def cohort(tmp_path):
    ds = synth.config(0, tiny=True, n_samples=5, genome_len=4000)
    rep = b"ACGTTGCAAGGCTTAACCGGTTAGCATCGA"
    paths = []
    for i, f in enumerate(ds.files):
        p = tmp_path / f"s{i}.fa"
        p.write_bytes(f + b">rep\n" + rep * (i % 3 + 1) + b"\n")
        paths.append(str(p))
    return paths


@pytest.fixture
def engine(monkeypatch):
    made = []

    def make(device=0):
        made.append(OracleEngine(device))
        return made[-1]
    monkeypatch.setattr(pg, "KmerAssociation", make)
    monkeypatch.setattr(group, "GpuGroup", make)
    monkeypatch.setattr(pg, "_STATE", {"ka": None, "pid": None, "devices": None, "job": None})
    monkeypatch.delenv("PS_DEVICE", raising=False)
    return made


def _kmers(paths, k, n, seed):
    rng = np.random.default_rng(seed)
    km, _ = ok.count_kmers(open(paths[0], "rb").read(), k)
    return [ok.kmer_to_str(int(x), k) for x in rng.choice(km, n, replace=False)] + ["A" * k]


def test_one_ingest_per_k_and_matrix_equals_oracle(cohort, engine):
    p = pg.install(_module(cohort, cutoff=2))
    lists = [ok.count_kmers(open(x, "rb").read(), 16) for x in cohort]
    for seed in (1, 2):                                   # two models with k = 16
        kmers = _kmers(cohort, 16, 40, seed) + ["ACGTTGCAAGGCTTAA"]
        m = _model(p, kmers)
        m.get_inp_matrix()
        codes = np.array([pg.canonical_code(x) for x in kmers], dtype=np.uint64)
        want = np.stack([ok.map_counts(codes, *l) for l in lists]) >= 2
        assert np.array_equal(m.matrix, want.astype(np.float64))
        assert m.matrix.shape == (len(cohort), len(kmers))
    assert 0 < m.matrix[:, -1].sum() < len(cohort)     # the repeat passes -c 2 in some samples only
    ka, = engine
    assert [c[0] for c in ka.calls] == ["count_files", "count_matrix", "count_matrix"]
    assert ka.calls[0] == ("count_files", len(cohort), 16, 1)          # the job counts at cutoff 1
    m = _model(p, _kmers(cohort, 13, 20, 3))               # another k: the cohort is ingested again
    m.get_inp_matrix()
    assert [c[0] for c in ka.calls[3:]] == ["count_files", "count_matrix"] and ka.calls[3][2] == 13
    m = _model(p, [])
    m.get_inp_matrix()
    assert m.matrix.shape == (len(cohort), 0) and len(ka.calls) == 5


def test_ps_device_list_selects_a_group(cohort, engine, monkeypatch):
    monkeypatch.setenv("PS_DEVICE", "0,1")
    p = pg.install(_module(cohort, cutoff=1))
    _model(p, _kmers(cohort, 16, 5, 4)).get_inp_matrix()
    assert [e.device for e in engine] == [[0, 1]]
    monkeypatch.setenv("PS_DEVICE", "1")
    _model(p, _kmers(cohort, 16, 5, 5)).get_inp_matrix()
    assert [e.device for e in engine] == [[0, 1], 1]
    assert engine[1].calls[0][0] == "count_files"          # a new engine holds no job yet
    assert pg._engine() is engine[1] and pg._STATE["pid"] == os.getpid()
