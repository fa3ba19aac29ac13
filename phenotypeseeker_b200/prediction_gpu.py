"""k-mer lookup of `phenotypeseeker prediction` on the GPU (SURVEY.md §8f rank 1).

The reference writes the model's k-mers as a `gmer_counter` text database
(prediction.py:145-148), runs `gmer_counter -db` per sample (:72-80), thresholds the counts at
`-c` (:82-100) and zips the per-sample text files into an N x K matrix (:150-163). Here the
cohort is decoded once and one `ps_count_matrix` call (k_count_matrix: one pass over every
sample's decoded stream, a shared-memory filter in front of a search of the sorted queries)
returns the N x K occurrence counts; single-k-mer gmer_counter nodes are strand-agnostic and
equal glistmaker's canonical counts (SURVEY.md Appendix A7), so a query k-mer is canonicalised
first.

`install(prediction_module)` re-wires Samples.map_samples / Samples.kmer_counts /
Phenotypes.set_kmer_db / Phenotypes.get_inp_matrix so that the unmodified `prediction()` driver,
model loading and `predict()` keep working. The samples are read from their files in batches
(`count_files`) and stay on the device for every model of the run; they are decoded again only
when a model's k differs from the k of the job on the device.
"""
import os

import numpy as np

from .modeling_gpu import parse_devices
from .pipeline import KmerAssociation

_COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}


def canonical_code(kmer: str) -> int:
    """k-mer string -> canonical 2-bit code (A0 C1 G2 T3, first base most significant)."""
    s = kmer.upper().replace("U", "T")
    rc = "".join(_COMP[c] for c in reversed(s))
    v = lambda t: int("".join(str("ACGT".index(c)) for c in t), 4)
    return min(v(s), v(rc))


def _codes(kmers):
    return np.array([canonical_code(x) for x in kmers], dtype=np.uint64)


def _threshold(counts, cutoff):
    return (counts >= int(cutoff)).astype(np.float64)


def presence_matrix(buffers, kmers, cutoff=1, device=0, ka=None):
    """N x K float matrix of (count >= cutoff) for N samples (raw FASTA/FASTQ bytes) and K
    k-mer strings — the matrix Phenotypes.get_inp_matrix builds (prediction.py:150-159).
    Returns (matrix, counts)."""
    kmers = list(kmers)
    if not kmers:
        return np.zeros((len(buffers), 0)), np.zeros((len(buffers), 0), dtype=np.uint32)
    ka = ka or KmerAssociation(device=device)
    ka.count(list(buffers), len(kmers[0]), 1)
    counts = ka.count_matrix(_codes(kmers))
    return _threshold(counts, cutoff), counts


_STATE = {"ka": None, "pid": None, "devices": None, "job": None}


def _engine(device=None):
    """The engine of this process (as modeling_gpu._ka): a KmerAssociation for one device, a GpuGroup for several
    (PS_DEVICE or device=, modeling_gpu.parse_devices). Made again after a fork or for other devices."""
    spec = parse_devices(os.environ.get("PS_DEVICE", "0") if device is None else device)
    if _STATE["ka"] is None or _STATE["pid"] != os.getpid() or spec != _STATE["devices"]:
        _STATE["ka"] = None                   # free the old engine's device memory before the new one allocates
        if isinstance(spec, int):
            _STATE["ka"] = KmerAssociation(device=spec)
        else:
            from . import group
            _STATE["ka"] = group.GpuGroup(spec)
        _STATE.update(pid=os.getpid(), devices=spec, job=None)
    return _STATE["ka"]


def install(p, device=None):
    """Re-wire the reference module `p` (PhenotypeSeeker.prediction). device: as PS_DEVICE (default: env PS_DEVICE,
    else 0); several entries count on a GpuGroup."""

    def map_samples(self, pheno):          # Pool worker: nothing to do
        return None

    def kmer_counts(self, pheno):          # Pool worker: nothing to do
        return None

    def set_kmer_db(self):
        return None

    def get_inp_matrix(self):
        kmers = [str(x) for x in self.kmers]
        samples = list(p.Input.samples.values())
        if kmers:
            ka = _engine(device)
            job = (len(kmers[0]), tuple(s.address for s in samples))
            if _STATE["job"] != job:       # the cohort at this model's k is not on the device yet
                _STATE["job"] = None
                ka.count_files(list(job[1]), job[0], 1)
                _STATE["job"] = job
            self.matrix = _threshold(ka.count_matrix(_codes(kmers)), p.Phenotypes.cutoff)
        else:
            self.matrix = np.zeros((len(samples), 0))
        if self.pca:
            self.scaled_matrix = self.scaler.transform(self.matrix)
            self.matrix = self.pca_model.transform(self.scaled_matrix)
            self.matrix = self.matrix[:, self.PCs_to_keep]

    p.Samples.map_samples = map_samples
    p.Samples.kmer_counts = kmer_counts
    p.Phenotypes.set_kmer_db = set_kmer_db
    p.Phenotypes.get_inp_matrix = get_inp_matrix
    return p
