"""Host-side driver of the hot path: count -> union/matrix -> chi2 / Welch -> filter.

Mirrors the stage order and the keep rules of `modeling.modeling()` lines 1644-1686 and
`phenotypes.get_kmers_tested` (modeling.py:677-858) on top of the C-ABI (`_native.Context`).
Everything numeric happens on the GPU; this module only shapes inputs and outputs.
"""
import gzip
import math
import os
from fractions import Fraction

import numpy as np

from ._native import Context, PsError  # noqa: F401


def kmer_to_str(x, k):
    x = int(x)
    return "".join("ACGT"[(x >> (2 * (k - 1 - i))) & 3] for i in range(k))


def kmers_to_str(arr, k):
    """Vectorised u64 -> k-mer strings."""
    arr = np.asarray(arr, dtype=np.uint64)
    if len(arr) == 0:
        return []
    shifts = (2 * (k - 1 - np.arange(k))).astype(np.uint64)
    codes = ((arr[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)
    letters = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    return [row.tobytes().decode() for row in letters]


def read_sample_file(path):
    """Raw bytes of a FASTA/FASTQ file; .gz is inflated on the host (glistmaker accepts .gz)."""
    with open(path, "rb") as f:
        head = f.read(2)
    if head == b"\x1f\x8b":
        with gzip.open(path, "rb") as f:
            return f.read()
    with open(path, "rb") as f:
        return f.read()


PS_SMS = 148                # B200
PAGE_TABLE_BYTES = 48       # per level-1 page: its meta, two level-2 metas and page-list entries, a share of a tile
HEADROOM_BYTES = 4 << 30    # union, sort and test buffers of a range, the runtime's own


def level1_pool_bytes(n_instances, n_samples):
    """Device bytes of the level-1 page pool for n_instances records of n_samples samples, as ps_api.cu's
    paged_begin_local reserves it: 4 KB pages for the records, the pages every k_scatter1 block (3 per SM) may hold
    open per bin (264) and sample group (+2), then the level-2 reserve of 2 KB pages (256 per level-1 stream and two
    per k_scatter2 block). The level-2 pages proper are written into the level-1 pages k_scatter2 has read."""
    groups = (int(n_samples) + 255) // 256
    pages = -(-int(n_instances) // 1024) + 3 * PS_SMS * 264 * (groups + 2)
    reserve = (groups * 264 + 2 * 3 * PS_SMS) * 256
    return pages * 4096 + reserve * 2048


def unpack_rows(rowbits, n_samples):
    """S x W uint32 -> S x N uint8 presence (sample s = bit s%32 of word s//32)."""
    rb = np.ascontiguousarray(rowbits, dtype=np.uint32)
    if rb.size == 0:
        return np.zeros((rb.shape[0], n_samples), dtype=np.uint8)
    bits = np.unpackbits(rb.view(np.uint8).reshape(rb.shape[0], -1), axis=1, bitorder="little")
    return bits[:, :n_samples]


class PhenoResult:
    """Survivors of one phenotype column. The matrix rows travel bit-packed (`rowbits`, S x W uint32, sample
    s = bit s % 32 of word s // 32); `presence` (S x N uint8) is unpacked on first use only — with 5,000
    samples a survivor's row is 640 bytes packed and 5,000 unpacked."""

    def __init__(self, name, kmer, row, stat, p, mean_x, mean_y, n_with, presence=None, na_mask=None, rowbits=None,
                 n_samples=None):
        self.name = name
        self.kmer = kmer          # u64 canonical k-mers of the survivors, ascending
        self.row = row            # rank of each survivor in the sorted union
        self.stat = stat          # chi2 or t
        self.p = p
        self.mean_x = mean_x      # Welch only
        self.mean_y = mean_y
        self.n_with = n_with
        self.na_mask = na_mask    # N bool, samples whose phenotype is NA (set by the boundary shim)
        self._presence = None if presence is None else np.ascontiguousarray(presence, dtype=np.uint8)
        if rowbits is None:
            assert presence is not None
            n_samples = self._presence.shape[1]
            W = (((n_samples + 31) // 32) + 3) // 4 * 4
            rowbits = np.zeros((self._presence.shape[0], W), dtype=np.uint32)
            if self._presence.size:
                pk = np.packbits(self._presence, axis=1, bitorder="little")
                rowbits.view(np.uint8).reshape(rowbits.shape[0], -1)[:, :pk.shape[1]] = pk
        self.rowbits = np.ascontiguousarray(rowbits, dtype=np.uint32)
        self.n_samples = int(n_samples)
        self.threshold = None     # permutation threshold of the column (test(n_perm=...)), else None
        self.minp = None          # its B permutation minima

    @property
    def presence(self):
        if self._presence is None:
            self._presence = unpack_rows(self.rowbits, self.n_samples)
        return self._presence

    def take(self, idx):
        """Rows idx (index array or boolean mask) as a new PhenoResult."""
        return PhenoResult(self.name, self.kmer[idx], self.row[idx], self.stat[idx], self.p[idx], self.mean_x[idx],
                           self.mean_y[idx], self.n_with[idx], na_mask=self.na_mask, rowbits=self.rowbits[idx],
                           n_samples=self.n_samples)


def trim_top(res, top_k):
    """The top_k survivors of one PhenoResult by (p, row) — the numeric `--n_kmers` cut of
    modeling.py:1128-1131 — back in ascending k-mer (row) order."""
    if top_k is None or len(res.kmer) <= top_k:
        return res
    order = np.lexsort((res.row, res.p))[:top_k]
    order.sort()
    return res.take(order)


def permute_columns(pheno, n_perm, seed=0, first=0):
    """Permutations first .. first + n_perm - 1 of every column of an N x P phenotype table (NaN = NA) -> P x n_perm x N.
    A permutation shuffles the column's non-NA values among its non-NA samples: NA positions stay, and so do the
    samples' weights, so the sample filter (n_with / n_without) of every k-mer is that of the observed column.
    Permutation b of column j is drawn from numpy.random.default_rng((seed, j, b)) alone: it does not depend on which
    other permutations or columns are drawn with it (any batching gives the same columns)."""
    ph = np.asarray(pheno, dtype=np.float64)
    if ph.ndim == 1:
        ph = ph[:, None]
    N, P = ph.shape
    out = np.empty((P, int(n_perm), N))
    for j in range(P):
        col = ph[:, j]
        idx = np.flatnonzero(~np.isnan(col))
        vals = col[idx]
        out[j] = col
        for b in range(int(n_perm)):
            out[j, b, idx] = vals[np.random.default_rng((int(seed), j, int(first) + b)).permutation(len(idx))]
    return out


def permutation_thresholds(minp, alpha):
    """Westfall & Young's single-step min-p threshold per column: minp is P x B (the smallest p of each permuted column
    over all testable k-mers), alpha the family-wise error rate (the p-value cut-off). With q_1 <= ... <= q_B the sorted
    minima of a column, t = q_{floor(alpha B) + 1}; at most floor(alpha B) permutations have a k-mer below it. Returns
    min(t, alpha) per column: a k-mer survives iff p < that. B < 1/alpha permutations cannot give a threshold."""
    m = np.atleast_2d(np.asarray(minp, dtype=np.float64))
    B = m.shape[1]
    k = math.floor(Fraction(repr(float(alpha))) * B)     # exact: 0.05 * 20 is 1, not 0.999...
    if k < 1:
        raise ValueError(f"{B} permutations cannot give a threshold at alpha = {alpha}: at least "
                         f"{math.ceil(1 / Fraction(repr(float(alpha))))} are needed")
    if k >= B:
        return np.full(m.shape[0], float(alpha))
    return np.minimum(np.sort(m, axis=1)[:, k], float(alpha))


def _unit_weights_as_none(weights):
    """The reference's default weight is the int 1: all-ones weights run the exact integer tables."""
    if weights is None:
        return None
    w = np.asarray(weights, dtype=np.float64)
    return None if np.all(w == 1.0) else w


PERM_BATCH_BYTES = 256 << 20        # host bytes of permuted columns handed to ps_minp_* at once


class KmerAssociation:
    """count -> matrix -> test on one GPU (or one k-mer-range shard of a multi-GPU job)."""

    def __init__(self, device=0, ctx=None):
        self.ctx = ctx or Context(device)
        self.k = None
        self.n_samples = 0
        self.U = 0

    # stage 1 (modeling.py:1649-1652)
    def count(self, buffers, k, cutoff=1, batch_bytes=2 << 30, ingest_range=None):
        """buffers: per-sample raw FASTA/FASTQ bytes (host) or (device_ptr, nbytes) tuples.
        ingest_range: (lo, hi, n_instances, share) from plan_ranges()["ingest"] — the first super-range of a
        run in k-mer ranges is scattered while the samples are ingested (ps_ingest_scatter), i.e. during
        the upload of host buffers."""
        self.k = int(k)
        self.n_samples = len(buffers)
        self.ctx.begin(self.k, self.n_samples, int(cutoff))
        if ingest_range is not None and int(cutoff) == 1 and 9 <= self.k <= 16:
            self.ctx.ingest_scatter(*ingest_range)
        i = 0
        while i < len(buffers):
            j, tot = i, 0
            while j < len(buffers):
                nb = buffers[j][1] if isinstance(buffers[j], tuple) else len(buffers[j])
                if j > i and tot + nb > batch_bytes:
                    break
                tot += nb
                j += 1
            self.ctx.add_samples(i, buffers[i:j])
            i = j

    def count_files(self, paths, k, cutoff=1, batch_bytes=2 << 30):
        """Stage 1 from files, streamed: a batch of files is read (and .gz inflated), handed to the GPU and
        dropped before the next one is read, so host memory holds one batch instead of every sample
        (raw-read sets are GBs each; the reference, too, touches one sample per worker at a time)."""
        self.k = int(k)
        self.n_samples = len(paths)
        self.ctx.begin(self.k, self.n_samples, int(cutoff))
        self.add_files(0, paths, batch_bytes)

    def add_files(self, first_idx, paths, batch_bytes=2 << 30):
        """Samples first_idx, first_idx + 1, ... of the job begun from files, read in batches as count_files does."""
        i = 0
        while i < len(paths):
            batch, tot, j = [], 0, i
            while j < len(paths):
                nb = os.path.getsize(paths[j])
                if j > i and tot + nb > batch_bytes:
                    break
                batch.append(read_sample_file(paths[j]))
                tot += len(batch[-1])
                j += 1
            self.ctx.add_samples(first_idx + i, batch)
            del batch
            i = j

    def fits_in_one_build(self, headroom=0.8):
        """Whether union + matrix of the whole k-mer space fit in this GPU's memory at once: the page pool
        (4 B per k-mer instance, + 10 %, and its level-2 reserve) plus a matrix with one row per (pessimistically)
        every fourth instance. When not, the job runs in k-mer ranges (test_in_ranges)."""
        import torch
        n = self.ctx.instances_upper()
        row_bytes = self.ctx.row_words() * 4
        need = level1_pool_bytes(n * 1.1, self.n_samples) + (n / 4) * (8 + row_bytes) + (1 << 30)
        free, _total = torch.cuda.mem_get_info(self.ctx.device)
        return need <= (free + self.ctx.device_bytes()) * headroom

    def ranges_needed(self, headroom=0.8):
        import torch
        n = self.ctx.instances_upper()
        row_bytes = self.ctx.row_words() * 4
        free, _total = torch.cuda.mem_get_info(self.ctx.device)
        have = (free + self.ctx.device_bytes()) * headroom - (1 << 30) - level1_pool_bytes(0, self.n_samples)
        need = n * 4 * 1.3 + (n / 4) * (8 + row_bytes)
        return max(1, int(np.ceil(need / max(have, 1))))

    def instances_upper(self):
        return self.ctx.instances_upper()

    # stage 2 (modeling.py:1656-1663, 641-644)
    def build(self, kmer_range=None):
        if kmer_range is not None:
            self.ctx.set_range(*kmer_range)
        self.U = self.ctx.build_union()
        return self.U

    # --kmerDB (modeling.py:361-372): feature vector = union AND the k-mers of a database FASTA
    def kmers_of(self, buffer, k):
        """Sorted distinct canonical k-mers of one FASTA/FASTQ text (`glistmaker <kmerDB> -w k`,
        modeling.py:370). Uses the context as a one-sample job: call BEFORE count()."""
        self.ctx.begin(int(k), 1, 1)
        self.ctx.add_samples(0, [buffer])
        return self.ctx.sample_kmers(0)[0]

    def restrict_to(self, db_kmers, chunk=1 << 22):
        """`glistcompare -i db union` (modeling.py:371): keep the union k-mers that are in db_kmers
        (ascending u64) and their matrix rows; U becomes the size of the intersection — the number
        `kmer_testing_setup` then counts with `wc -l` (:641-644). Call after build(). Runs on the device
        (ps_restrict_union: binary search per union k-mer, scan, compaction of union and matrix); returns
        the new U."""
        db = np.ascontiguousarray(db_kmers, dtype=np.uint64)
        if hasattr(self.ctx, "restrict_union"):
            self.U = self.ctx.restrict_union(db)
            return self.U
        return self._restrict_to_host(db, chunk)

    def _restrict_to_host(self, db, chunk=1 << 22):
        """The same through ps_get_union / ps_get_rows / ps_load_matrix (contexts without ps_restrict_union:
        the stand-in of tests/test_kmerdb_host.py)."""
        u = self.ctx.get_union()
        pos = np.searchsorted(db, u)
        keep = (pos < len(db)) & (db[np.minimum(pos, max(len(db) - 1, 0))] == u) if len(db) else np.zeros(len(u), bool)
        idx = np.nonzero(keep)[0]
        rows = np.empty((len(idx), self.ctx.row_words()), dtype=np.uint32)
        done = 0
        for a in range(0, len(u), chunk):                      # bounded host memory
            part = self.ctx.get_rows(a, min(chunk, len(u) - a))
            sel = keep[a:a + chunk]
            n = int(sel.sum())
            rows[done:done + n] = part[sel]
            done += n
        self.ctx.load_matrix(rows, u[idx])
        self.U = len(idx)
        return self.U

    # per-sample device work of the drop-in (-rc counts, -w weights); GpuGroup has the same methods
    def lookup(self, sample, kmers):
        """Counts of `kmers` in one sample (ps_lookup)."""
        return self.ctx.lookup(sample, kmers)

    def count_matrix(self, kmers, first_idx=0, count=None):
        """(count, K) uint32 occurrences of `kmers` in samples first_idx .. first_idx + count - 1 (all samples from
        first_idx by default): one device pass (ps_count_matrix)."""
        count = self.n_samples - int(first_idx) if count is None else int(count)
        return self.ctx.count_matrix(first_idx, count, kmers)

    def mash_sketch(self, first_idx, count, k=21, s=1000, seed=42):
        return self.ctx.mash_sketch(first_idx, count, k, s, seed)

    def mash_pairs(self, hashes, n_hashes):
        return self.ctx.mash_pairs(hashes, n_hashes)

    def neighbor_joining(self, dm):
        return self.ctx.neighbor_joining(dm)

    # stage 3 (modeling.py:1679-1683)
    def test(self, pheno, binary, weights=None, min_samples=2, max_samples=None, pvalue_cutoff=0.05,
             omit_b=False, n_union_total=None, pheno_names=None, top_k=None, n_perm=0, perm_seed=0, minp=None):
        """pheno: N x P float array, NaN = NA (binary columns hold 0/1).

        Keep rule (modeling.py:738, 795): chi2 keeps p < cutoff (omit_B) or p < cutoff/U;
        the t-test always uses cutoff/U. U defaults to this context's union size;
        pass n_union_total when this context holds only a shard of the k-mer space.
        top_k: keep only the top_k survivors per column by p-value, selected on the GPU before anything
        is copied to the host (`--n_kmers`, modeling.py:1128-1131); self.n_survivors is the count before the cut.
        n_perm > 0: the permutation threshold replaces cutoff/U (not the uncorrected omit_B rule): column j keeps
        p < permutation_thresholds(minp, cutoff)[j], minp from permutation_minp(..., n_perm, seed=perm_seed), or
        the P x B `minp` given (minima already combined over k-mer ranges or shards). The results then carry
        `threshold` and `minp` of their column.
        """
        ph = np.asarray(pheno, dtype=np.float64)
        if ph.ndim == 1:
            ph = ph[:, None]
        N, P = ph.shape
        assert N == self.n_samples
        if max_samples is None:
            max_samples = N - 2
        U = self.U if n_union_total is None else n_union_total
        names = pheno_names or [f"pheno{j + 1}" for j in range(P)]
        w = _unit_weights_as_none(weights)
        perm = (n_perm > 0 or minp is not None) and not (binary and omit_b)
        if perm:
            if minp is None:
                permutation_thresholds(np.ones((1, int(n_perm))), pvalue_cutoff)     # too few permutations: raise now
                minp = self.permutation_minp(ph, binary, n_perm, w, min_samples, max_samples, perm_seed)
            cut = permutation_thresholds(minp, pvalue_cutoff)
            thr = float(cut.max())
        elif U == 0:
            thr = 0.0
        elif binary and omit_b:
            thr = float(pvalue_cutoff)
        else:
            thr = float(pvalue_cutoff) / float(U)
        if binary:
            code = np.where(np.isnan(ph), -1, ph).astype(np.int8).T
            ns = self.ctx.test_chi2(code, w, min_samples, max_samples, thr)
        else:
            ns = self.ctx.test_welch(ph.T.copy(), w, min_samples, max_samples, thr)
        self.n_survivors = ns
        if top_k is not None:
            ns = self.ctx.select_top(P, int(top_k))
        sv = self.ctx.fetch_survivors(ns)
        out = []
        for j in range(P):
            sel = sv["pheno"] == j
            if perm:
                sel &= sv["p"] < cut[j]     # one pass at the largest threshold, each column cut to its own
            out.append(trim_top(PhenoResult(
                name=names[j], kmer=sv["kmer"][sel], row=sv["row"][sel], stat=sv["stat"][sel],
                p=sv["p"][sel], mean_x=sv["mean_x"][sel], mean_y=sv["mean_y"][sel],
                n_with=sv["n_with"][sel], rowbits=sv["rowbits"][sel], n_samples=N), top_k))
            if perm:
                out[-1].threshold, out[-1].minp = float(cut[j]), np.asarray(minp[j], dtype=np.float64)
        return out

    def permutation_minp(self, pheno, binary, n_perm, weights=None, min_samples=2, max_samples=None, seed=0):
        """Min-p of n_perm permutations of every phenotype column (permute_columns) over this build's union: P x n_perm,
        entry [j, b] = the smallest p (chi2 or Welch, as test() computes it) over the k-mers that pass the sample
        filter in permutation b of column j, 1.0 if none. Union, matrix and the survivors of the last test stay."""
        ph = np.asarray(pheno, dtype=np.float64)
        if ph.ndim == 1:
            ph = ph[:, None]
        N, P = ph.shape
        assert N == self.n_samples
        n_perm = int(n_perm)
        if max_samples is None:
            max_samples = N - 2
        w = _unit_weights_as_none(weights)
        out = np.empty((P, n_perm))
        step = max(1, PERM_BATCH_BYTES // max(1, 8 * P * N))
        for b0 in range(0, n_perm, step):
            nb = min(step, n_perm - b0)
            cols = permute_columns(ph, nb, seed, first=b0).reshape(P * nb, N)
            if binary:
                m = self.ctx.minp_chi2(np.where(np.isnan(cols), -1, cols).astype(np.int8), w, min_samples, max_samples)
            else:
                m = self.ctx.minp_welch(cols, w, min_samples, max_samples)
            out[:, b0:b0 + nb] = m.reshape(P, nb)
        return out

    def run(self, buffers, k, pheno, binary, weights=None, cutoff=1, **kw):
        self.count(buffers, k, cutoff)
        self.build()
        return self.test(pheno, binary, weights, **kw)

    def _one_super_range(self, n_ranges, spl, n_instances):
        """Whether the level-1 pool of the whole job fits beside everything else the context holds: the pool and its
        reserve (level1_pool_bytes, as ps_scatter_range will size it), its page tables, the 2-bit streams, the
        matrix of the largest range and some headroom, against the device's free memory plus what the context holds
        now. The range sizes come from the previous test_in_ranges of the same job; without them, or with a context
        that cannot report its memory, the answer is no."""
        sizes = getattr(self, "_range_sizes", {}).get((self.k, self.n_samples, tuple(spl)))
        mem_info = getattr(self.ctx, "mem_info", None)
        if not n_instances or not sizes or mem_info is None:
            return False
        free, held = mem_info()
        n = int(n_instances) + (1 << 20)
        row_bytes = ((((self.n_samples + 31) // 32) + 3) // 4 * 4) * 4
        need = (level1_pool_bytes(n, self.n_samples) + -(-n // 1024) * PAGE_TABLE_BYTES + n * 3 // 8 * 9 // 8
                + max(sizes) * (8 + row_bytes) * 9 // 8 + HEADROOM_BYTES)
        return need <= free + held

    def plan_ranges(self, n_ranges, splitters, n_instances=None, n_super=None):
        """Range boundaries, super-range grouping and pool capacities of a run in k-mer ranges (test_in_ranges).
        n_super None: one super-range when its pool fits (_one_super_range), else half as many as ranges.
        -> dict(splitters, grouped, slack, first_of {first range of a super-range: one past its last},
        ingest (lo, hi, n_instances, share) of the FIRST super-range for count(ingest_range=...) or None)."""
        spl = [int(x) for x in splitters]
        assert len(spl) == n_ranges - 1
        grouped = bool(n_ranges > 1 and (n_super is None or n_super) and 9 <= self.k <= 16)
        if grouped:
            unit = 1 << (2 * self.k - 8)
            spl = [max(unit, (x + unit // 2) // unit * unit) for x in spl]
            for i in range(1, len(spl)):                       # keep them strictly ascending
                spl[i] = max(spl[i], spl[i - 1] + unit)
            grouped = spl[-1] < (1 << (2 * self.k))
        if n_super is None:
            n_super = 1 if grouped and self._one_super_range(n_ranges, spl, n_instances) else (n_ranges + 1) // 2
        slack = 1.15 if grouped else 1.3
        first_of, ingest = {}, None
        if grouped:
            n_super = min(int(n_super), n_ranges)
            for s_ in range(n_super):
                a, b = s_ * n_ranges // n_super, (s_ + 1) * n_ranges // n_super
                first_of[a] = b
            if n_instances:
                b = first_of[0]
                ingest = (0, 0 if b == n_ranges else spl[b - 1], self._super_capacity(n_instances, slack, 0, b, n_ranges),
                          b / n_ranges)
        return {"splitters": spl, "grouped": grouped, "slack": slack, "first_of": first_of, "ingest": ingest}

    @staticmethod
    def _super_capacity(n_instances, slack, a, b, n_ranges):
        """Level-1 pool capacity (records) of the super-range of ranges [a, b): its share of the job's instances with
        slack; the whole space takes n_instances itself, the text bytes, which already bound the positions."""
        if b - a == n_ranges:
            return int(n_instances) + (1 << 20)
        return int(n_instances * slack * (b - a) / n_ranges) + (1 << 20)

    def test_in_ranges(self, pheno, binary, n_ranges, weights=None, pvalue_cutoff=0.05, omit_b=False,
                       splitters=None, n_instances=None, top_k=None, n_super=None, restrict=None, n_perm=0,
                       perm_seed=0, **kw):
        """Stages 2-3 when records or matrix do not fit in HBM at once (SURVEY.md §7 "memory at
        config 5"): the k-mer space is cut into n_ranges contiguous ranges (quantiles of sample 0,
        or `splitters` from an earlier call on the same job), each range is built and tested on its
        own, and the survivors are concatenated — ranges are ascending, so k-mer order and global
        ranks are those of a single build.

        n_super (k = 9..16; default: one when the whole job's level-1 pool fits, else half as many as ranges;
        0 = off): the ranges are grouped into n_super
        super-ranges whose k-mer instances are extracted ONCE into the level-1 page pool
        (ps_scatter_range); the ranges of a super-range then start from that pool. Their boundaries are
        moved to the nearest multiple of 4^(k-4) (a top-k-mer-byte boundary) for that.

        The Bonferroni threshold needs U = sum of all range sizes, known only at the end. Range r is
        therefore tested against the provable bound U >= U_0 + ... + U_r (the union sizes seen so
        far), i.e. a laxer threshold, and the exact pvalue/U filter is applied afterwards.
        n_instances: k-mer instances of the whole job (positions); sizes the page pools of a range
        (ps_set_capacity_hint) instead of reserving for every position of the input.
        restrict (--kmerDB database k-mers): only with n_ranges == 1, which restricts the one build.
        n_perm > 0 (test()): each range's pass also gives that range's min-p of the permuted columns; the minima
        are combined over the ranges (element-wise minimum) and the range is tested against the thresholds of the
        minima seen so far, which can only fall as ranges follow: again a laxer cut, the exact one at the end.
        Call after count(). Returns (U, [PhenoResult per phenotype column])."""
        if restrict is not None and n_ranges > 1:
            raise RuntimeError("--kmerDB needs union and matrix in GPU memory at once; this input needs "
                               f"{n_ranges} k-mer ranges")
        ph = np.asarray(pheno, dtype=np.float64)
        if ph.ndim == 1:
            ph = ph[:, None]
        if splitters is None:
            splitters = self.ctx.sample_quantiles(0, n_ranges) if n_ranges > 1 else []
        spl = [int(x) for x in splitters]
        assert len(spl) == n_ranges - 1
        plan = self.plan_ranges(n_ranges, spl, n_instances, n_super)
        spl, grouped, slack, first_of = plan["splitters"], plan["grouped"], plan["slack"], plan["first_of"]
        self.range_splitters = spl
        perm = n_perm > 0 and not (binary and omit_b)
        minp = np.ones((ph.shape[1], int(n_perm))) if perm else None
        if perm:
            permutation_thresholds(minp, pvalue_cutoff)      # too few permutations: raise before any build
        parts, U, sizes = [], 0, []
        for r in range(n_ranges):
            lo = 0 if r == 0 else spl[r - 1]
            hi = 0 if r == n_ranges - 1 else spl[r]
            if r in first_of:
                b = first_of[r]
                self.ctx.scatter_range(lo, 0 if b == n_ranges else spl[b - 1],
                                       self._super_capacity(n_instances, slack, r, b, n_ranges) if n_instances else 0)
            if n_ranges > 1:
                self.ctx.set_range(lo, hi)
                if n_instances:
                    self.ctx.set_capacity_hint(int(n_instances * slack / n_ranges) + (1 << 20))
            u_r = self.build()
            if restrict is not None:
                u_r = self.restrict_to(restrict)
            if perm and u_r:
                minp = np.minimum(minp, self.permutation_minp(ph, binary, n_perm, weights, kw.get("min_samples", 2),
                                                              kw.get("max_samples"), perm_seed))
            res = self.test(ph, binary, weights, pvalue_cutoff=pvalue_cutoff, omit_b=omit_b, top_k=top_k,
                            n_union_total=(U + u_r) if not (binary and omit_b) else None, minp=minp,
                            **kw) if u_r else None
            parts.append((U, res))
            U += u_r
            sizes.append(u_r)
        if n_ranges > 1:
            self.ctx.set_range(0, 0)      # back to the whole k-mer space
            self._range_sizes = {(self.k, self.n_samples, tuple(spl)): sizes}   # the next call's super-range choice
        self.U = U
        exact = float(pvalue_cutoff) if (binary and omit_b) else (float(pvalue_cutoff) / U if U else 0.0)
        cut = permutation_thresholds(minp, pvalue_cutoff) if perm else np.full(ph.shape[1], exact)
        out = []
        W = self.ctx.row_words()
        for j in range(ph.shape[1]):
            cols = {f: [] for f in ("kmer", "row", "stat", "p", "mean_x", "mean_y", "n_with", "rowbits")}
            name = None
            for base, res in parts:
                if res is None:
                    continue
                r = res[j]
                name = r.name
                keep = r.p < cut[j]
                cols["kmer"].append(r.kmer[keep]); cols["row"].append(r.row[keep] + np.uint64(base))
                for f in ("stat", "p", "mean_x", "mean_y", "n_with", "rowbits"):
                    cols[f].append(getattr(r, f)[keep])
            cat = lambda f, dt: (np.concatenate(cols[f]) if cols[f] else np.empty(0, dt))
            out.append(trim_top(PhenoResult(
                name=name or f"pheno{j + 1}", kmer=cat("kmer", np.uint64), row=cat("row", np.uint64),
                stat=cat("stat", np.float64), p=cat("p", np.float64),
                mean_x=cat("mean_x", np.float64), mean_y=cat("mean_y", np.float64), n_with=cat("n_with", np.uint32),
                rowbits=(np.concatenate(cols["rowbits"]) if cols["rowbits"] else np.zeros((0, W), np.uint32)),
                n_samples=self.n_samples), top_k))
            if perm:
                out[-1].threshold, out[-1].minp = float(cut[j]), minp[j]
        return U, out
