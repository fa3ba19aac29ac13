"""Several GPUs from one process: one libpskmer context per device, one thread per rank.

`GpuGroup(devices)` runs the sharded hot path of dist.py (dist.ingest, dist.build_and_test) with a
dist.ThreadGroup for the collectives instead of torch.distributed: no torchrun, no NCCL, no CUDA IPC. Rank r
ingests the samples dist.sample_block(r, G, N) and owns one contiguous k-mer range per pass; k_scatter1 stores
each k-mer instance straight into the owner's receive pool, over peer access that ps_route_connect enables.
Results, U and the k-mer order are those of a single build (merge_results on rank 0).

Every call starts one thread per rank and joins them all before it returns: no thread outlives a call (the
reference's modeling() forks Pools after the tests). ctypes releases the GIL during every library call, so the
ranks' host work runs in parallel.

Besides build and test, a group offers the per-sample device work of the drop-in, each on the context that holds
the sample: lookup and count_matrix (-rc counts) and mash_sketch, with mash_pairs and neighbor_joining on the first context, so
that weights.gsc_weights_on_device takes a group as it takes a context.
"""
import numpy as np

from . import dist as psdist
from .pipeline import KmerAssociation

PART_MAX = 8          # ranks of one route (PART_MAX of csrc/ps_extract.cuh)


class GpuGroup:
    """count -> build and test on several GPUs of one process. devices: one entry per rank (repeats allowed: several
    ranks may share a GPU)."""

    def __init__(self, devices):
        devices = [int(d) for d in devices]
        if not 1 <= len(devices) <= PART_MAX:
            raise ValueError(f"a GPU group has 1..{PART_MAX} ranks, got {len(devices)}")
        self.devices = devices
        self.world = len(devices)
        self.group = psdist.ThreadGroup(self.world)
        self.engines = [KmerAssociation(device=d) for d in devices]
        self.k = None
        self.n_samples = 0
        self.U = 0

    def _run(self, fn):
        """fn(rank) on one thread per rank, with that rank's device current. A failed call leaves the ranks' page
        routes in different states, so they are dropped: the next call plans them again, together."""
        import torch

        def body(r):
            torch.cuda.set_device(self.devices[r])
            return fn(r)
        try:
            return self.group.run(body)
        except BaseException:
            for ka in self.engines:
                ka._page_route = None
            raise

    def _owner(self, sample):
        for r in range(self.world):
            if sample in psdist.sample_block(r, self.world, self.n_samples):
                return r
        raise IndexError(f"no sample {sample} in a job of {self.n_samples}")

    # --kmerDB (modeling.py:361-372)
    def kmers_of(self, buffer, k):
        """Database k-mers of one FASTA/FASTQ text, on the first context (KmerAssociation.kmers_of): call BEFORE
        count()."""
        return self.engines[0].kmers_of(buffer, k)

    # stage 1 (modeling.py:1649-1652)
    def count(self, buffers, k, cutoff=1):
        """buffers: per-sample raw FASTA/FASTQ bytes (host) or (device_ptr, nbytes) tuples on the owning rank's
        device."""
        self.k, self.n_samples = int(k), len(buffers)

        def one(r):
            block = psdist.sample_block(r, self.world, self.n_samples)
            psdist.ingest(self.engines[r], {s: buffers[s] for s in block}, self.n_samples, k, r, self.world, cutoff)
        self._run(one)

    def count_files(self, paths, k, cutoff=1, batch_bytes=2 << 30):
        """Stage 1 from files: each rank reads its block in batches on its own thread (KmerAssociation.count_files)."""
        self.k, self.n_samples = int(k), len(paths)

        def one(r):
            mine = psdist.begin_block(self.engines[r], self.n_samples, k, r, self.world, cutoff)
            if mine:
                self.engines[r].add_files(mine[0], [paths[s] for s in mine], batch_bytes)
        self._run(one)

    def instances_upper(self):
        return sum(ka.instances_upper() for ka in self.engines)

    # stages 2-3
    def test(self, pheno, binary, weights=None, min_samples=2, max_samples=None, pvalue_cutoff=0.05, omit_b=False,
             pheno_names=None, top_k=None, restrict=None, passes=None, n_perm=0, perm_seed=0):
        """Build and test on every rank (dist.build_and_test) -> (U, [PhenoResult per phenotype column]), merged
        on rank 0: global rows and ascending k-mer order as in a single build. restrict: ascending database k-mers
        (--kmerDB), any number of passes. passes: super-ranges of the k-mer space (None: as the pool budget needs).
        n_perm, perm_seed: permutation thresholds as KmerAssociation.test; each rank computes the min-p over its own
        k-mers and the ranks' minima are min-reduced, so thresholds and survivors equal one GPU's.
        A page-pool overflow is retried once with the doubled pools; the samples are not ingested again."""
        import torch
        ph = np.asarray(pheno, dtype=np.float64)
        if ph.ndim == 1:
            ph = ph[:, None]
        kw = dict(min_samples=min_samples, max_samples=max_samples, pvalue_cutoff=pvalue_cutoff, omit_b=omit_b,
                  pheno_names=pheno_names, top_k=top_k, n_perm=n_perm, perm_seed=perm_seed)

        def one(r):
            try:
                return psdist.build_and_test(self.engines[r], self.n_samples, self.k, ph, binary, weights, r,
                                             self.world, torch.device("cuda", self.devices[r]), group=self.group,
                                             restrict=restrict, passes=passes, **kw)
            except psdist.PoolOverflow:
                return None       # every rank sees the same overflow flag, and has doubled its pools

        for _attempt in range(2):
            out = self._run(one)
            if all(o is not None for o in out):
                self.U = int(out[0][0])
                return self.U, out[0][1]
        raise psdist.PoolOverflow("a page pool overflowed twice while routing k-mers, also with pools twice as large")

    def fits_in_one_build(self):
        """False: a group builds each rank's k-mer ranges on that rank's GPU, never the whole space in one build
        (the drop-in therefore tests every column at once, as for a run in k-mer ranges)."""
        return False

    def ranges_needed(self):
        """One k-mer range per rank; build and test add passes over super-ranges when the pools need them."""
        return self.world

    def test_in_ranges(self, pheno, binary, n_ranges, weights=None, n_instances=None, restrict=None, **kw):
        """KmerAssociation.test_in_ranges on the group: n_ranges beyond one per rank asks for that many passes
        (rounded up); the page pools are sized from the ranks' own instance counts, n_instances is not needed."""
        passes = -(-int(n_ranges) // self.world) if n_ranges > self.world else None
        return self.test(pheno, binary, weights, restrict=restrict, passes=passes, **kw)

    # per-sample device work (-rc counts, -w weights), on the context that holds the sample
    def lookup(self, sample, kmers):
        return self.engines[self._owner(sample)].lookup(sample, kmers)

    def count_matrix(self, kmers, first_idx=0, count=None):
        """(count, K) uint32 occurrences of `kmers` in samples first_idx .. first_idx + count - 1 (all from first_idx
        by default): each rank counts its share on its own context, parts in sample order (Context.count_matrix)."""
        first_idx = int(first_idx)
        count = self.n_samples - first_idx if count is None else int(count)
        q = np.ascontiguousarray(kmers, dtype=np.uint64)
        wanted = range(first_idx, first_idx + count)

        def one(r):
            block = psdist.sample_block(r, self.world, self.n_samples)
            lo, hi = max(block.start, wanted.start), min(block.stop, wanted.stop)
            return self.engines[r].count_matrix(q, lo, hi - lo) if hi > lo else None
        parts = [p for p in self._run(one) if p is not None]
        if not parts:
            return np.zeros((0, len(q)), dtype=np.uint32)
        return np.concatenate(parts)

    def mash_sketch(self, first_idx, count, k=21, s=1000, seed=42):
        """Sketches of samples first_idx .. first_idx + count - 1, each rank's share on its own context, in sample
        order (Context.mash_sketch)."""
        first_idx, count = int(first_idx), int(count)
        wanted = range(first_idx, first_idx + count)

        def one(r):
            block = psdist.sample_block(r, self.world, self.n_samples)
            lo, hi = max(block.start, wanted.start), min(block.stop, wanted.stop)
            return self.engines[r].mash_sketch(lo, hi - lo, k, s, seed) if hi > lo else None
        parts = [p for p in self._run(one) if p is not None]
        if not parts:
            return np.empty((0, int(s)), dtype=np.uint64), np.empty(0, dtype=np.uint32)
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    def mash_pairs(self, hashes, n_hashes):
        return self.engines[0].mash_pairs(hashes, n_hashes)

    def neighbor_joining(self, dm):
        return self.engines[0].neighbor_joining(dm)
