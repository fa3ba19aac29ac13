"""ctypes binding of libpskmer.so (include/pskmer.h). No CPU fallback: if the library or a
CUDA device is missing, every entry point raises."""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PSKMER_LIB") or os.path.join(HERE, "libpskmer.so")

c_void_pp = ctypes.POINTER(ctypes.c_void_p)
c_u64_p = ctypes.POINTER(ctypes.c_uint64)

# name -> (restype, argtypes); also the list of symbols include/pskmer.h declares
SIGNATURES = {
    "ps_version": (ctypes.c_int, []),
    "ps_ctx_create": (ctypes.c_int, [ctypes.c_int, c_void_pp]),
    "ps_ctx_destroy": (None, [ctypes.c_void_p]),
    "ps_last_error": (ctypes.c_char_p, [ctypes.c_void_p]),
    "ps_begin": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint32]),
    "ps_set_range": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64]),
    "ps_set_capacity_hint": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64]),
    "ps_scatter_range": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64]),
    "ps_ingest_scatter": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_double]),
    "ps_add_samples": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_void_pp,
                                      ctypes.POINTER(ctypes.c_size_t)]),
    "ps_sample_kmers": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)]),
    "ps_build_union": (ctypes.c_int, [ctypes.c_void_p, c_u64_p]),
    "ps_row_words": (ctypes.c_int, [ctypes.c_void_p]),
    "ps_get_union": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p]),
    "ps_get_rows": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p]),
    "ps_load_matrix": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]),
    "ps_restrict_union": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, c_u64_p]),
    "ps_test_chi2": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                    ctypes.c_int, ctypes.c_int, ctypes.c_double, c_u64_p]),
    "ps_test_welch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_double, c_u64_p]),
    "ps_minp_chi2": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                    ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "ps_minp_welch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "ps_select_top": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, c_u64_p]),
    "ps_fetch_survivors": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t] + [ctypes.c_void_p] * 9),
    "ps_lookup": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t,
                                 ctypes.c_void_p]),
    "ps_count_matrix": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t,
                                       ctypes.c_void_p]),
    "ps_export_stream": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_void_pp, c_void_pp, c_u64_p]),
    "ps_import_stream": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                        ctypes.c_uint64]),
    "ps_import_streams": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                         ctypes.c_void_p, c_u64_p]),
    "ps_route_pages_needed": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_u64_p]),
    "ps_instances_upper": (ctypes.c_uint64, [ctypes.c_void_p]),
    "ps_route_setup": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_u64_p, ctypes.c_uint64, c_void_pp,
                                      c_void_pp]),
    "ps_route_peers": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_void_pp, c_void_pp]),
    "ps_route_connect": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, c_void_pp]),
    "ps_route_begin": (ctypes.c_int, [ctypes.c_void_p]),
    "ps_route_scatter": (ctypes.c_int, [ctypes.c_void_p]),
    "ps_route_build": (ctypes.c_int, [ctypes.c_void_p, c_u64_p, ctypes.POINTER(ctypes.c_int)]),
    "ps_ipc_export": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_char_p]),
    "ps_ipc_open": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, c_void_pp]),
    "ps_ipc_close_all": (ctypes.c_int, [ctypes.c_void_p]),
    "ps_sample_quantiles": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_u64_p]),
    "ps_mash_sketch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p]),
    "ps_mash_pairs": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_void_p]),
    "ps_neighbor_joining": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_void_p]),
    "ps_stream": (ctypes.c_void_p, [ctypes.c_void_p]),
    "ps_launch_count": (ctypes.c_uint64, [ctypes.c_void_p]),
    "ps_profile_enable": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "ps_profile_count": (ctypes.c_int, [ctypes.c_void_p]),
    "ps_profile_get": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_char_p),
                                      c_u64_p, ctypes.POINTER(ctypes.c_double),
                                      ctypes.POINTER(ctypes.c_double)]),
    "ps_profile_reset": (ctypes.c_int, [ctypes.c_void_p]),
    "ps_device_bytes": (ctypes.c_uint64, [ctypes.c_void_p]),
}


class PsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libpskmer error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Load libpskmer.so (building it is __graft_entry__.build()'s / build.py's job)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PsError(-100, f"{LIB_PATH} is missing: run `python -m phenotypeseeker_b200.build` "
                            "(there is no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError if the ABI drifted
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class Context:
    """One GPU's worth of the hot path. Thin, 1:1 with the C-ABI; raises on every error."""

    def __init__(self, device=0):
        self.L = load()
        h = ctypes.c_void_p()
        rc = self.L.ps_ctx_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise PsError(rc, (self.L.ps_last_error(None) or b"").decode())
        self.h = h
        self.device = device
        self.k = 0
        self.n_samples = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.ps_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise PsError(rc, (self.L.ps_last_error(self.h) or b"").decode())

    # -- job ---------------------------------------------------------------------------
    def begin(self, k, n_samples, cutoff=1):
        self._ck(self.L.ps_begin(self.h, int(k), int(n_samples), int(cutoff)))
        self.k, self.n_samples = int(k), int(n_samples)

    def set_range(self, lo, hi):
        self._ck(self.L.ps_set_range(self.h, int(lo), int(hi)))

    def set_capacity_hint(self, n_instances):
        self._ck(self.L.ps_set_capacity_hint(self.h, int(n_instances)))

    def scatter_range(self, lo, hi, n_instances=0):
        """Extract the instances of the k-mers in [lo, hi) once into the level-1 page pool; builds of
        top-byte-aligned sub-ranges then start from it (ps_scatter_range)."""
        self._ck(self.L.ps_scatter_range(self.h, int(lo), int(hi), int(n_instances)))

    def ingest_scatter(self, lo, hi, n_instances, share=1.0):
        """Scatter every sample for the k-mer range [lo, hi) while it is ingested (ps_ingest_scatter); call between
        begin() and the first add_samples()."""
        self._ck(self.L.ps_ingest_scatter(self.h, int(lo), int(hi), int(n_instances), float(share)))

    def add_samples(self, first_idx, buffers):
        """buffers: list of bytes / bytearray / numpy uint8 arrays (host), or (device_ptr, nbytes)
        tuples for text already resident on the GPU."""
        n = len(buffers)
        ptrs = (ctypes.c_void_p * n)()
        lens = (ctypes.c_size_t * n)()
        keep = []
        for i, b in enumerate(buffers):
            if isinstance(b, tuple):
                ptrs[i], lens[i] = int(b[0]), int(b[1])
            elif isinstance(b, np.ndarray):
                a = np.ascontiguousarray(b.view(np.uint8))
                keep.append(a)
                ptrs[i], lens[i] = a.ctypes.data, a.nbytes
            else:
                a = np.frombuffer(b, dtype=np.uint8)
                keep.append(a)
                ptrs[i], lens[i] = (a.ctypes.data if len(a) else 0), len(a)
        self._ck(self.L.ps_add_samples(self.h, int(first_idx), n, ptrs, lens))

    def sample_kmers(self, idx, cutoff=1):
        n = ctypes.c_size_t()
        self._ck(self.L.ps_sample_kmers(self.h, int(idx), int(cutoff), None, None, 0, ctypes.byref(n)))
        km = np.empty(n.value, dtype=np.uint64)
        ct = np.empty(n.value, dtype=np.uint32)
        if n.value:
            self._ck(self.L.ps_sample_kmers(self.h, int(idx), int(cutoff), _ptr(km), _ptr(ct), n.value,
                                            ctypes.byref(n)))
        return km, ct

    def build_union(self):
        u = ctypes.c_uint64()
        self._ck(self.L.ps_build_union(self.h, ctypes.byref(u)))
        self.U = u.value
        return u.value

    def row_words(self):
        return self.L.ps_row_words(self.h)

    def get_union(self, first=0, count=None):
        count = self.U - first if count is None else count
        out = np.empty(count, dtype=np.uint64)
        self._ck(self.L.ps_get_union(self.h, int(first), int(count), _ptr(out)))
        return out

    def get_rows(self, first=0, count=None):
        count = self.U - first if count is None else count
        out = np.empty((count, self.row_words()), dtype=np.uint32)
        self._ck(self.L.ps_get_rows(self.h, int(first), int(count), _ptr(out)))
        return out

    def load_matrix(self, rows, kmers=None):
        """rows: U x row_words uint32 (host); kmers: U uint64 or None."""
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        assert rows.ndim == 2 and rows.shape[1] == self.row_words()
        km = None if kmers is None else np.ascontiguousarray(kmers, dtype=np.uint64)
        self._ck(self.L.ps_load_matrix(self.h, rows.shape[0], _ptr(km), _ptr(rows)))
        self.U = rows.shape[0]

    def restrict_union(self, db_kmers):
        """--kmerDB: keep the union k-mers that are in db_kmers (ascending distinct u64) and their rows, on the
        device; returns the new U."""
        db = np.ascontiguousarray(db_kmers, dtype=np.uint64)
        u = ctypes.c_uint64()
        self._ck(self.L.ps_restrict_union(self.h, _ptr(db) if len(db) else None, len(db), ctypes.byref(u)))
        self.U = u.value
        return u.value

    # -- tests -------------------------------------------------------------------------
    def test_chi2(self, pheno, weights, min_samples, max_samples, p_threshold):
        """pheno: P x N int8 (1/0/-1=NA); weights: N float64 or None."""
        ph = np.ascontiguousarray(pheno, dtype=np.int8)
        if ph.ndim == 1:
            ph = ph[None, :]
        assert ph.shape[1] == self.n_samples
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        ns = ctypes.c_uint64()
        self._ck(self.L.ps_test_chi2(self.h, ph.shape[0], _ptr(ph), _ptr(w), int(min_samples),
                                     int(max_samples), float(p_threshold), ctypes.byref(ns)))
        return ns.value

    def test_welch(self, pheno, weights, min_samples, max_samples, p_threshold):
        """pheno: P x N float64, NaN = NA."""
        ph = np.ascontiguousarray(pheno, dtype=np.float64)
        if ph.ndim == 1:
            ph = ph[None, :]
        assert ph.shape[1] == self.n_samples
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        ns = ctypes.c_uint64()
        self._ck(self.L.ps_test_welch(self.h, ph.shape[0], _ptr(ph), _ptr(w), int(min_samples),
                                      int(max_samples), float(p_threshold), ctypes.byref(ns)))
        return ns.value

    def minp_chi2(self, pheno, weights, min_samples, max_samples):
        """Smallest p per column over the union k-mers that pass the sample filter (1.0 if none).
        pheno: C x N int8 (1/0/-1=NA), typically permuted columns; weights: N float64 or None. -> C float64."""
        ph = np.ascontiguousarray(pheno, dtype=np.int8)
        if ph.ndim == 1:
            ph = ph[None, :]
        assert ph.shape[1] == self.n_samples
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        out = np.empty(ph.shape[0], dtype=np.float64)
        self._ck(self.L.ps_minp_chi2(self.h, ph.shape[0], _ptr(ph), _ptr(w), int(min_samples), int(max_samples),
                                     _ptr(out)))
        return out

    def minp_welch(self, pheno, weights, min_samples, max_samples):
        """As minp_chi2 for the Welch test. pheno: C x N float64, NaN = NA."""
        ph = np.ascontiguousarray(pheno, dtype=np.float64)
        if ph.ndim == 1:
            ph = ph[None, :]
        assert ph.shape[1] == self.n_samples
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        out = np.empty(ph.shape[0], dtype=np.float64)
        self._ck(self.L.ps_minp_welch(self.h, ph.shape[0], _ptr(ph), _ptr(w), int(min_samples), int(max_samples),
                                      _ptr(out)))
        return out

    def select_top(self, n_pheno, n_top):
        n = ctypes.c_uint64()
        self._ck(self.L.ps_select_top(self.h, int(n_pheno), int(n_top), ctypes.byref(n)))
        return n.value

    def fetch_survivors(self, n, rowbits=True):
        wp = self.row_words()
        out = {
            "pheno": np.empty(n, np.int32), "row": np.empty(n, np.uint64), "kmer": np.empty(n, np.uint64),
            "stat": np.empty(n, np.float64), "p": np.empty(n, np.float64),
            "mean_x": np.empty(n, np.float64), "mean_y": np.empty(n, np.float64),
            "n_with": np.empty(n, np.uint32),
            "rowbits": np.empty((n, wp), np.uint32) if rowbits else None,
        }
        self._ck(self.L.ps_fetch_survivors(self.h, n, _ptr(out["pheno"]), _ptr(out["row"]), _ptr(out["kmer"]),
                                           _ptr(out["stat"]), _ptr(out["p"]), _ptr(out["mean_x"]),
                                           _ptr(out["mean_y"]), _ptr(out["n_with"]), _ptr(out["rowbits"])))
        return out

    def lookup(self, idx, kmers):
        q = np.ascontiguousarray(kmers, dtype=np.uint64)
        out = np.zeros(len(q), dtype=np.uint32)
        self._ck(self.L.ps_lookup(self.h, int(idx), _ptr(q), len(q), _ptr(out)))
        return out

    def count_matrix(self, first_idx, count, kmers):
        """(count, K) uint32: occurrences of every k-mer in samples first_idx .. first_idx + count - 1."""
        q = np.ascontiguousarray(kmers, dtype=np.uint64)
        out = np.zeros((int(count), len(q)), dtype=np.uint32)
        self._ck(self.L.ps_count_matrix(self.h, int(first_idx), int(count), _ptr(q), len(q), _ptr(out)))
        return out

    # -- exchange ----------------------------------------------------------------------
    def export_stream(self, idx):
        seq, bad, n = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_uint64()
        self._ck(self.L.ps_export_stream(self.h, int(idx), ctypes.byref(seq), ctypes.byref(bad),
                                         ctypes.byref(n)))
        return seq.value, bad.value, n.value

    def import_stream(self, idx, seq_ptr, bad_ptr, n_pos):
        self._ck(self.L.ps_import_stream(self.h, int(idx), ctypes.c_void_p(seq_ptr),
                                         ctypes.c_void_p(bad_ptr), int(n_pos)))

    def import_streams(self, first_idx, seq_ptr, bad_ptr, n_pos_list):
        n = len(n_pos_list)
        arr = (ctypes.c_uint64 * n)(*[int(x) for x in n_pos_list])
        self._ck(self.L.ps_import_streams(self.h, int(first_idx), n, ctypes.c_void_p(seq_ptr),
                                          ctypes.c_void_p(bad_ptr), arr))

    def route_pages_needed(self, nparts, passes=1):
        n = ctypes.c_uint64()
        self._ck(self.L.ps_route_pages_needed(self.h, int(nparts), int(passes), ctypes.byref(n)))
        return n.value

    def instances_upper(self):
        return self.L.ps_instances_upper(self.h)

    def route_setup(self, nparts, my_rank, splitters, pages_per_sender):
        """-> (pool device pointer, meta device pointer) of this GPU's receive pool."""
        spl = (ctypes.c_uint64 * max(len(splitters), 1))(*[int(x) for x in splitters])
        pool, meta = ctypes.c_void_p(), ctypes.c_void_p()
        self._ck(self.L.ps_route_setup(self.h, int(nparts), int(my_rank), spl, int(pages_per_sender),
                                       ctypes.byref(pool), ctypes.byref(meta)))
        return pool.value, meta.value

    def route_clear(self):
        self._ck(self.L.ps_route_setup(self.h, 0, 0, None, 0, None, None))

    def route_peers(self, pool_ptrs, meta_ptrs):
        n = len(pool_ptrs)
        pp = (ctypes.c_void_p * n)(*[int(x) for x in pool_ptrs])
        mp = (ctypes.c_void_p * n)(*[int(x) for x in meta_ptrs])
        self._ck(self.L.ps_route_peers(self.h, n, pp, mp))

    def route_connect(self, contexts):
        """Pools of every rank of one process (contexts[r] is rank r, this context among them), with peer access
        from this context's device to the others' (ps_route_connect)."""
        n = len(contexts)
        hs = (ctypes.c_void_p * n)(*[c.h.value if c.h else None for c in contexts])
        self._ck(self.L.ps_route_connect(self.h, n, hs))

    def route_begin(self):
        self._ck(self.L.ps_route_begin(self.h))

    def route_scatter(self):
        self._ck(self.L.ps_route_scatter(self.h))

    def route_build(self):
        """-> (U of this GPU's range, overflow flag)."""
        u, ovf = ctypes.c_uint64(), ctypes.c_int()
        self._ck(self.L.ps_route_build(self.h, ctypes.byref(u), ctypes.byref(ovf)))
        self.U = u.value
        return u.value, bool(ovf.value)

    def ipc_export(self, dev_ptr):
        buf = ctypes.create_string_buffer(64)
        self._ck(self.L.ps_ipc_export(self.h, ctypes.c_void_p(dev_ptr), buf))
        return buf.raw

    def ipc_open(self, handle: bytes):
        p = ctypes.c_void_p()
        self._ck(self.L.ps_ipc_open(self.h, handle, ctypes.byref(p)))
        return p.value

    def ipc_close_all(self):
        self._ck(self.L.ps_ipc_close_all(self.h))

    def sample_quantiles(self, idx, nq):
        out = (ctypes.c_uint64 * max(nq - 1, 1))()
        self._ck(self.L.ps_sample_quantiles(self.h, int(idx), int(nq), out))
        return [int(out[i]) for i in range(nq - 1)]

    # -- -w sample weights --------------------------------------------------------------
    def mash_sketch(self, first_idx, count, k=21, s=1000, seed=42):
        """MinHash sketches of samples first_idx..first_idx+count-1 -> (count x s uint64, count uint32 lengths);
        row i holds its n[i] ascending hashes first, zeros after them."""
        h = np.empty((int(count), int(s)), dtype=np.uint64)
        n = np.empty(int(count), dtype=np.uint32)
        self._ck(self.L.ps_mash_sketch(self.h, int(first_idx), int(count), int(k), int(s), int(seed), _ptr(h), _ptr(n)))
        return h, n

    def mash_pairs(self, hashes, n_hashes):
        """hashes: n x s uint64 (as mash_sketch returns them), n_hashes: n -> n x n uint32, shared << 16 | denom."""
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        nh = np.ascontiguousarray(n_hashes, dtype=np.uint32)
        n, s = h.shape
        out = np.empty((n, n), dtype=np.uint32)
        self._ck(self.L.ps_mash_pairs(self.h, n, s, _ptr(h), _ptr(nh), _ptr(out)))
        return out

    def neighbor_joining(self, dm):
        """dm: n x n symmetric float64, n >= 3 -> (join: (n-2) x 2 int32 list positions (mi, mj) per step,
        branch: 2(n-2)+1 float64, the two branch lengths of every step and the last remaining distance)."""
        d = np.ascontiguousarray(dm, dtype=np.float64)
        n = d.shape[0]
        join = np.empty((max(n - 2, 0), 2), dtype=np.int32)
        branch = np.empty(2 * max(n - 2, 0) + 1, dtype=np.float64)
        self._ck(self.L.ps_neighbor_joining(self.h, n, _ptr(d), _ptr(join), _ptr(branch)))
        return join, branch

    # -- instrumentation ---------------------------------------------------------------
    def stream(self):
        return self.L.ps_stream(self.h)

    def launch_count(self):
        return self.L.ps_launch_count(self.h)

    def device_bytes(self):
        return self.L.ps_device_bytes(self.h)

    def mem_info(self):
        """(free bytes of the device, bytes this context holds): what a build could take."""
        import torch
        free, _total = torch.cuda.mem_get_info(self.device)
        return int(free), int(self.device_bytes())

    def profile(self, on):
        self._ck(self.L.ps_profile_enable(self.h, 1 if on else 0))

    def profile_reset(self):
        self._ck(self.L.ps_profile_reset(self.h))

    def profile_table(self):
        n = self.L.ps_profile_count(self.h)
        rows = {}
        for i in range(n):
            name = ctypes.c_char_p()
            l = ctypes.c_uint64()
            ms = ctypes.c_double()
            ab = ctypes.c_double()
            self._ck(self.L.ps_profile_get(self.h, i, ctypes.byref(name), ctypes.byref(l), ctypes.byref(ms),
                                           ctypes.byref(ab)))
            rows[name.value.decode()] = {"launches": l.value, "ms": ms.value, "alg_bytes": ab.value}
        return rows
