"""Multi-GPU sharding of the hot path: one process per GPU (torch.distributed, NCCL).

Counting is independent per sample and testing is independent per k-mer; the one coupling
is regrouping sample-major data into k-mer-major rows (SURVEY.md §8e). Rank r ingests the
contiguous block of samples [N*r/G, N*(r+1)/G) and owns one contiguous k-mer RANGE (not a
hash bucket): contiguous ranges keep the global sorted order — a survivor's global rank is
range base + row — which the reference's output column order depends on. Ranges are balanced
with splitters taken once per job from the quantiles of sample 0's sorted k-mer list (same species).

Exchange routes:
  * "pages" (k = 9..16, assemblies and raw reads alike; the default): every GPU owns a receive
    pool of 4 KB pages, mapped into its peers with CUDA IPC once per job. The extraction kernel of
    a sender (k_scatter1) groups its k-mer instances by (owner, top k-mer byte) and appends each
    group straight to pages of the owner's pool — 4-byte records, ~128-byte runs, plain stores over
    NVLink. No counts are exchanged, nothing is extracted twice, there is no send buffer and no
    copy on the receiver: the all-to-all IS the write-out of the extraction kernel, and what the
    receiver finds is already the level-1 partition of its own range. Two stream-ordered barriers
    (tiny all-reduces) fence the exchange; the host is not involved.
  * "streams" (k > 16): the 2-bit packed streams (3 bits per base) are all-gathered and each
    rank extracts its own range from all of them; extraction is then replicated on every rank.

Collectives per step: all_gather (pool sizes; sticky, so IPC handles move only when a pool grows),
2 x all_reduce (barriers), all_reduce (U, the Bonferroni denominator, modeling.py:641-644, plus
the pool-overflow flag), one all_gather of the packed survivors.

The collectives go through a group object with torch.distributed's calls (all_reduce,
all_gather_into_tensor, broadcast) plus the exchange of the receive pools:
  * TorchGroup: one process per GPU (torchrun, NCCL); pools are mapped with CUDA IPC.
  * ThreadGroup: one thread per rank inside one process (group.GpuGroup); pools are plain device
    pointers of the other contexts, connected by ps_route_connect, which also enables peer access.
"""
import threading

import numpy as np

from .pipeline import KmerAssociation, PhenoResult


def sample_block(rank, world, n_samples):
    """Samples owned (ingested) by `rank`: a contiguous block."""
    return range(n_samples * rank // world, n_samples * (rank + 1) // world)


def range_of(rank, splitters):
    """k-mer range [lo, hi) of `rank` given world-1 ascending splitters; None = whole space."""
    if not splitters:
        return None
    lo = 0 if rank == 0 else splitters[rank - 1]
    hi = 0 if rank == len(splitters) else splitters[rank]     # 0 = unbounded
    return lo, hi


def stream_layout(lens, world):
    """Per-rank byte layout of the padded all-gather. lens[s] = padded positions of sample s.
    -> (per_rank sample lists, per-rank total positions, max positions)."""
    n = len(lens)
    per_rank = [list(sample_block(r, world, n)) for r in range(world)]
    rank_pos = [int(sum(int(lens[s]) for s in per_rank[r])) for r in range(world)]
    return per_rank, rank_pos, max(rank_pos) if rank_pos else 0


def merge_results(gathered, bases):
    """Rank-0 merge of per-range survivor lists. gathered[r] = list over phenotypes of tuples
    (name, kmer, row, stat, p, mean_x, mean_y, n_with, rowbits, n_samples); bases[r] = global rank of
    range r's first union k-mer. Ranges are ascending, so concatenation keeps k-mer order."""
    out = []
    for j in range(len(gathered[0])):
        parts = [g[j] for g in gathered]
        rows = [np.asarray(p[2], dtype=np.uint64) + np.uint64(bases[r]) for r, p in enumerate(parts)]
        out.append(PhenoResult(
            name=parts[0][0], kmer=np.concatenate([p[1] for p in parts]), row=np.concatenate(rows),
            stat=np.concatenate([p[3] for p in parts]), p=np.concatenate([p[4] for p in parts]),
            mean_x=np.concatenate([p[5] for p in parts]), mean_y=np.concatenate([p[6] for p in parts]),
            n_with=np.concatenate([p[7] for p in parts]), rowbits=np.concatenate([p[8] for p in parts]),
            n_samples=parts[0][9]))
    return out


_FIELDS = (("kmer", np.uint64), ("row", np.uint64), ("stat", np.float64), ("p", np.float64),
           ("mean_x", np.float64), ("mean_y", np.float64), ("n_with", np.uint32))


def pack_results(res):
    """Survivors of all phenotypes -> (counts per phenotype, one flat uint8 buffer); matrix rows travel
    bit-packed as they left the GPU (row_words x 4 bytes per survivor)."""
    counts = [len(r.kmer) for r in res]
    parts = []
    for r in res:
        for name, dt in _FIELDS:
            parts.append(np.ascontiguousarray(getattr(r, name), dtype=dt).view(np.uint8).reshape(-1))
        parts.append(np.ascontiguousarray(r.rowbits, dtype=np.uint32).view(np.uint8).reshape(-1))
    buf = np.concatenate(parts) if parts else np.empty(0, np.uint8)
    return counts, buf


def unpack_results(names, counts, buf, n_samples):
    """Inverse of pack_results -> list of tuples in merge_results' layout."""
    out, off = [], 0
    W = (((n_samples + 31) // 32) + 3) // 4 * 4
    for name, n in zip(names, counts):
        vals = []
        for _, dt in _FIELDS:
            nb = n * np.dtype(dt).itemsize
            vals.append(buf[off:off + nb].view(dt).copy())
            off += nb
        rb = buf[off:off + n * W * 4].view(np.uint32).reshape(n, W).copy()
        off += n * W * 4
        out.append((name, vals[0], vals[1], vals[2], vals[3], vals[4], vals[5], vals[6], rb, n_samples))
    return out


class PoolOverflow(RuntimeError):
    """A receive page pool overflowed while routing k-mers. Every rank raises it at the same point and has doubled
    its pools for the next step, which can simply be run again."""


class TorchGroup:
    """Collectives of one process per GPU: torch.distributed (NCCL), receive pools mapped with CUDA IPC. Lives for
    the process (TORCH_GROUP), so the survivor all-gather keeps its sticky capacity from step to step."""

    def __init__(self):
        self.gather_cap = 1 << 16       # bytes per rank of the survivor all-gather (grows when a rank needs more)

    def all_reduce(self, t):
        import torch.distributed as dist
        dist.all_reduce(t)

    def all_gather_into_tensor(self, out, t):
        import torch.distributed as dist
        dist.all_gather_into_tensor(out, t)

    def broadcast(self, t, src):
        import torch.distributed as dist
        dist.broadcast(t, src=src)

    def connect_pools(self, ctx, rank, world, device, pool, meta):
        """Every rank's receive pool into ctx's route (ps_route_peers), through CUDA IPC handles."""
        import torch
        h = np.frombuffer(ctx.ipc_export(pool) + ctx.ipc_export(meta), dtype=np.uint8).copy()
        allh = torch.empty(world * 128, dtype=torch.uint8, device=device)
        self.all_gather_into_tensor(allh, torch.from_numpy(h).to(device))
        allh = allh.cpu().numpy().reshape(world, 128)
        pools = [pool if d == rank else ctx.ipc_open(allh[d, :64].tobytes()) for d in range(world)]
        metas = [meta if d == rank else ctx.ipc_open(allh[d, 64:].tobytes()) for d in range(world)]
        ctx.route_peers(pools, metas)


TORCH_GROUP = TorchGroup()


class ThreadGroup:
    """The collectives of TorchGroup for `world` threads of one process; rank r is the thread that run() started
    for it. Data moves device to device (Tensor.copy_), never through the host.

    Like NCCL's, a collective is ordered after the work queued on the caller's current stream: it synchronises that
    stream (the library stream inside build_and_test) BEFORE it meets the other ranks, so that, used as a barrier,
    no rank scatters into a pool whose ps_route_begin memset is still queued. It synchronises again after reading the
    other ranks' tensors and meets them once more, so no rank reuses a tensor another one is still reading.

    When a rank raises, run() aborts the barrier: the other ranks get BrokenBarrierError instead of waiting forever,
    and run() re-raises the first error in the caller."""

    def __init__(self, world):
        self.world = int(world)
        self.gather_cap = 1 << 16
        self._slots = [None] * self.world
        self._local = threading.local()
        self._bar = threading.Barrier(self.world)

    def run(self, fn):
        """fn(rank) on one thread per rank; every thread is joined before this returns. -> [result per rank]."""
        self._bar = threading.Barrier(self.world)
        out, errs, lock = [None] * self.world, [], threading.Lock()

        def body(r):
            self._local.rank = r
            try:
                out[r] = fn(r)
            except BaseException as e:       # noqa: B902 - handed to the caller below
                with lock:
                    errs.append(e)
                self._bar.abort()

        threads = [threading.Thread(target=body, args=(r,), name=f"ps-rank{r}") for r in range(self.world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errs:
            first = next((e for e in errs if not isinstance(e, threading.BrokenBarrierError)), errs[0])
            raise first
        return out

    def _sync(self, t):
        import torch
        if t.is_cuda:
            torch.cuda.current_stream(t.device).synchronize()

    def _collective(self, t, combine):
        """Meet the other ranks with t, return combine(every rank's t) once every rank has read what it needs."""
        self._sync(t)
        self._slots[self._local.rank] = t
        self._bar.wait()
        res = combine(list(self._slots))
        self._sync(res)
        self._bar.wait()
        return res

    def all_reduce(self, t):
        def total(ts):
            acc = ts[0].to(t.device, copy=True)
            for x in ts[1:]:
                acc += x.to(t.device)
            return acc
        t.copy_(self._collective(t, total))

    def all_gather_into_tensor(self, out, t):
        n = t.numel()
        assert out.numel() == self.world * n, "every rank gathers equal parts"

        def gather(ts):
            for r, x in enumerate(ts):
                assert x.numel() == n, "every rank gathers equal parts"
                out[r * n:(r + 1) * n].copy_(x.reshape(-1))
            return out
        self._collective(t, gather)

    def broadcast(self, t, src):
        t.copy_(self._collective(t, lambda ts: ts[src].to(t.device, copy=True)))

    def connect_pools(self, ctx, rank, world, device, pool, meta):
        """Every rank's receive pool into ctx's route: the contexts meet here after their ps_route_setup, and
        ps_route_connect reads the pools from them (and enables peer access). Nobody changes a route before every
        rank has read all of them."""
        self._slots[rank] = ctx
        self._bar.wait()
        ctx.route_connect(list(self._slots))
        self._bar.wait()


def _cap_owner(group):
    """The object that carries the survivor all-gather's capacity: the group, or the process-wide TorchGroup when
    the caller hands torch.distributed itself."""
    return group if hasattr(group, "gather_cap") else TORCH_GROUP


def gather_results(parts, rank, world, device, dist, top_k=None, p_exact=None):
    """Per-range U + survivors of every rank with ONE collective: an all-gather of fixed-capacity
    buffers [header | payload]. parts = this rank's passes, each (U_local, [PhenoResult per column]);
    header = passes x (U_local, payload bytes, survivors per column). Every rank sees every header, so
    all ranks agree when the capacity has to grow (then, and only then, a second round). Ranges ascend
    pass-major, then by rank: that is the order of the merge and of the global row numbers.
    p_exact: final threshold, one for all columns or one per column (passes test against a laxer one while U is
    still growing).
    -> merged list on rank 0, None elsewhere."""
    import torch
    from .pipeline import trim_top
    res0 = parts[0][1]
    n_samples = res0[0].n_samples if res0 else 0
    P = len(res0)
    hdr_rows, bufs = [], []
    for U_local, res in parts:
        counts, buf = pack_results(res)
        hdr_rows.append([U_local, len(buf)] + counts)
        bufs.append(buf)
    buf = np.concatenate(bufs) if bufs else np.empty(0, np.uint8)
    hdr = np.array(hdr_rows, dtype=np.int64).reshape(-1).view(np.uint8)
    owner = _cap_owner(dist)
    while True:
        cap = owner.gather_cap
        mine = np.zeros(len(hdr) + cap, dtype=np.uint8)
        mine[:len(hdr)] = hdr
        if len(buf) <= cap:
            mine[len(hdr):len(hdr) + len(buf)] = buf
        t = torch.from_numpy(mine).to(device)
        allt = torch.empty(world * len(mine), dtype=torch.uint8, device=device)
        dist.all_gather_into_tensor(allt, t)
        allh = allt.cpu().numpy().reshape(world, -1)
        metas = allh[:, :len(hdr)].copy().view(np.int64).reshape(world, len(parts), -1)
        need = int(metas[:, :, 1].sum(axis=1).max())
        if need <= cap:
            break
        owner.gather_cap = 2 * need
    if rank != 0:
        return None
    names = [r.name for r in res0]
    gathered, bases, base = [], [], 0
    offs = [0] * world
    for j in range(len(parts)):
        for r in range(world):
            nb = int(metas[r, j, 1])
            payload = allh[r, len(hdr) + offs[r]:len(hdr) + offs[r] + nb]
            offs[r] += nb
            gathered.append(unpack_results(names, [int(x) for x in metas[r, j, 2:2 + P]], payload, n_samples))
            bases.append(base)
            base += int(metas[r, j, 0])
    out = []
    for j, r in enumerate(merge_results(gathered, bases)):
        if p_exact is not None:
            r = r.take(r.p < (p_exact[j] if np.ndim(p_exact) else p_exact))
        out.append(trim_top(r, top_k))
    return out


class _DevView:
    """Expose a raw device pointer to torch through __cuda_array_interface__."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def exchange_streams(ka: KmerAssociation, n_samples, rank, world, device, dist=TORCH_GROUP):
    """All-gather every rank's packed stream block; import the blocks this rank does not own.
    Returns the bytes received over NVLink by this rank."""
    import torch

    ctx = ka.ctx
    mine = list(sample_block(rank, world, n_samples))
    lens = torch.zeros(n_samples, dtype=torch.int64, device=device)
    first = None
    if mine:
        exported = [ctx.export_stream(s) for s in mine]       # consecutive in this rank's pool
        first = exported[0]
        lens[mine[0]:mine[-1] + 1] = torch.tensor([e[2] for e in exported], dtype=torch.int64, device=device)
    dist.all_reduce(lens)
    lens_h = lens.cpu().numpy()
    per_rank, rank_pos, max_pos = stream_layout(lens_h, world)
    seq_all = torch.empty(world * (max_pos // 4), dtype=torch.uint8, device=device)
    bad_all = torch.empty(world * (max_pos // 8), dtype=torch.uint8, device=device)
    seq_mine = seq_all[rank * (max_pos // 4):(rank + 1) * (max_pos // 4)]
    bad_mine = bad_all[rank * (max_pos // 8):(rank + 1) * (max_pos // 8)]
    my_pos = rank_pos[rank]
    if mine:
        seq_mine[:my_pos // 4] = torch.as_tensor(_DevView(first[0], my_pos // 4), device=device)
        bad_mine[:my_pos // 8] = torch.as_tensor(_DevView(first[1], my_pos // 8), device=device)
    dist.all_gather_into_tensor(seq_all, seq_mine.clone())
    dist.all_gather_into_tensor(bad_all, bad_mine.clone())
    torch.cuda.synchronize(device)
    for r in range(world):
        if r == rank or not per_rank[r]:
            continue
        ctx.import_streams(per_rank[r][0], seq_all.data_ptr() + r * (max_pos // 4),
                           bad_all.data_ptr() + r * (max_pos // 8), [int(lens_h[s]) for s in per_rank[r]])
    return int((max_pos // 4 + max_pos // 8) * (world - 1))


POOL_BUDGET_BYTES = 38e9      # one level-1 pool per GPU; level 2 writes into its read pages (and a small reserve)


class PageRoute:
    """Per-job state of the "pages" exchange on one rank: pass count, splitters, the agreed sub-pool size
    and the CUDA IPC mappings of the peers' pools. Everything here is set up once per job and reused by
    every step (a step only all-gathers the per-rank instance counts to see that the job is the same);
    it is redone, collectively, when the job changes or a pool has to grow."""

    def __init__(self, ka, rank, world, device):
        self.ka, self.rank, self.world, self.device = ka, rank, world, device
        self.key = None            # (k, n_samples, per-rank instance counts) the plan was made for
        self.passes = 1            # super-ranges of the k-mer space, one exchange each
        self.splitters = None      # world * passes - 1 ascending k-mer boundaries
        self.pages = 0             # pages per sender in every receive pool: agreed target (sticky maximum)
        self.live_pages = 0        # ... and what the pools are set up for right now
        self.bar = None

    def barrier(self, dist):
        """Stream-ordered barrier: an all-reduce of one word on the library's stream (no host sync)."""
        dist.all_reduce(self.bar)

    def pass_range(self, j):
        """(lo, hi) of super-range j (0 = unbounded) and the world - 1 splitters inside it."""
        W, S = self.world, self.splitters
        lo = 0 if j == 0 else S[j * W - 1]
        hi = 0 if j == self.passes - 1 else S[(j + 1) * W - 1]
        return lo, hi, S[j * W:j * W + W - 1]

    def prepare(self, k, n_samples, dist, torch, passes=None):
        """passes: number of super-ranges; None = as many as the pool budget needs."""
        ctx = self.ka.ctx
        if self.bar is None:
            self.bar = torch.zeros(1, dtype=torch.int32, device=self.device)
        mine = torch.tensor([ctx.instances_upper()], dtype=torch.int64, device=self.device)
        allc = torch.empty(self.world, dtype=torch.int64, device=self.device)
        dist.all_gather_into_tensor(allc, mine)
        counts = tuple(int(x) for x in allc.cpu().tolist())
        key = (k, n_samples, counts, passes)
        if key != self.key:
            # a new job: passes so that a pool fits the budget, then quantile splitters of sample 0 (held by rank 0)
            total = sum(counts)
            self.passes = int(passes) if passes else max(1, int(np.ceil(total * 1.5 * 4 / (self.world * POOL_BUDGET_BYTES))))
            nq = self.world * self.passes
            spl_t = torch.zeros(max(nq - 1, 1), dtype=torch.int64, device=self.device)
            if self.rank == 0:
                q = ctx.sample_quantiles(0, nq)
                spl_t[:len(q)] = torch.tensor(np.array(q, dtype=np.uint64).view(np.int64), dtype=torch.int64,
                                              device=self.device)
            dist.broadcast(spl_t, src=0)
            self.splitters = [int(x) for x in spl_t.cpu().numpy().view(np.uint64)][:nq - 1]
            need = torch.tensor([ctx.route_pages_needed(self.world, self.passes)], dtype=torch.int64, device=self.device)
            allneed = torch.empty(self.world, dtype=torch.int64, device=self.device)
            dist.all_gather_into_tensor(allneed, need)
            self.pages = max(self.pages, int(allneed.max().item()))
            self.key = key
        if self.pages != self.live_pages:
            # pools (re)allocated on every rank: unmap the old ones first (CUDA IPC; threads map nothing), then
            # exchange the new ones
            ctx.ipc_close_all()
            self.barrier(dist)
            torch.cuda.synchronize(self.device)
            pool, meta = ctx.route_setup(self.world, self.rank, self.pass_range(0)[2], self.pages)
            dist.connect_pools(ctx, self.rank, self.world, self.device, pool, meta)
            self.live_pages = self.pages


class _Marks:
    """PS_DIST_TIMING=1: device-synchronised wall-clock marks of rank 0, written to stderr."""

    def __init__(self, rank, device):
        import os
        self.on = bool(os.environ.get("PS_DIST_TIMING")) and rank == 0
        self.device, self.marks = device, []

    def __call__(self, name):
        if self.on:
            import time
            import torch
            torch.cuda.synchronize(self.device)
            self.marks.append((name, time.time()))

    def report(self):
        if self.on:
            import sys
            sys.stderr.write("[dist timing ms] " + " ".join(
                f"{b[0]}={1e3 * (b[1] - a[1]):.1f}" for a, b in zip(self.marks, self.marks[1:])) + "\n")


def begin_block(ka: KmerAssociation, n_samples, k, rank, world, cutoff=1):
    """Start the job on this rank's context (all n_samples, global indices) -> the samples this rank ingests."""
    ka.k, ka.n_samples = int(k), int(n_samples)
    ka.ctx.begin(int(k), int(n_samples), int(cutoff))
    ka._streams_imported = False
    if world == 1:
        ka.ctx.route_clear()
    return list(sample_block(rank, world, n_samples))


def ingest(ka: KmerAssociation, buffers_by_sample, n_samples, k, rank, world, cutoff=1):
    """Ingest step of run_sharded: begin + add_samples of this rank's block. buffers_by_sample: {sample_idx: bytes
    or (dev_ptr, n)} for exactly sample_block(rank, world, n_samples)."""
    mine = begin_block(ka, n_samples, k, rank, world, cutoff)
    assert sorted(buffers_by_sample) == mine, "this rank must hold exactly its own block of samples"
    if mine:
        ka.ctx.add_samples(mine[0], [buffers_by_sample[s] for s in mine])


def build_and_test(ka: KmerAssociation, n_samples, k, pheno, binary, weights, rank, world, device, route="auto",
                   group=None, restrict=None, passes=None, marks=None, **test_kw):
    """Build-and-test step of run_sharded, after ingest() on every rank: the exchange, each rank's union and matrix
    of its k-mer ranges, the tests, the exact filter and the gather of the survivors on rank 0.
    group: TorchGroup (default, torch.distributed) or ThreadGroup. restrict: ascending distinct database k-mers
    (--kmerDB): each range keeps only those (ps_restrict_union) and U counts what is left. passes: number of
    super-ranges of the "pages" route (None: as many as the pool budget needs). A page-pool overflow raises
    PoolOverflow after every rank has doubled its pools: running this step again (without a new ingest) retries.
    n_perm > 0 (test_kw, with perm_seed): permutation thresholds (KmerAssociation.test); every pass min-reduces the
    ranks' min-p of the permuted columns over their own k-mers, so thresholds and survivors are those of one build.
    Returns (U_total, results on rank 0 / None elsewhere, info)."""
    ctx = ka.ctx
    dist = TORCH_GROUP if group is None else group
    mark = marks or _Marks(rank, device)
    if world == 1:
        U = ka.build()
        if restrict is not None:
            U = ka.restrict_to(restrict)
        res = ka.test(pheno, binary, weights, **test_kw)
        return U, res, {"U_local": U, "nvlink_bytes": 0, "splitters": []}
    import torch
    from .pipeline import permutation_thresholds

    n_perm, perm_seed = int(test_kw.pop("n_perm", 0)), test_kw.pop("perm_seed", 0)
    perm = n_perm > 0 and not (binary and test_kw.get("omit_b"))
    P = np.asarray(pheno).reshape(n_samples, -1).shape[1]
    minp = np.ones((P, n_perm)) if perm else None
    alpha = float(test_kw.get("pvalue_cutoff", 0.05))
    if perm:
        permutation_thresholds(minp, alpha)          # too few permutations: raise before any build

    def combine_minp(m_local):
        """Element-wise minimum of every rank's min-p (an all-gather: the collectives have no min-reduce)."""
        t = torch.from_numpy(np.ascontiguousarray(m_local, dtype=np.float64).reshape(-1)).to(device)
        allt = torch.empty(world * t.numel(), dtype=torch.float64, device=device)
        dist.all_gather_into_tensor(allt, t)
        return np.minimum(minp, allt.cpu().numpy().reshape(world, P, n_perm).min(axis=0))

    def test_pass(n_union_total):
        nonlocal minp
        if not perm:
            return ka.test(pheno, binary, weights, n_union_total=n_union_total, **test_kw)
        minp = combine_minp(ka.permutation_minp(pheno, binary, n_perm, weights, test_kw.get("min_samples", 2),
                                                test_kw.get("max_samples"), perm_seed))
        return ka.test(pheno, binary, weights, minp=minp, **test_kw)

    if route == "auto":
        route = "pages" if 9 <= int(k) <= 16 else "streams"
    if route == "pages" and not 9 <= int(k) <= 16:
        raise ValueError("route='pages' handles k = 9..16")
    stream = torch.cuda.ExternalStream(ctx.stream(), device=device)
    with torch.cuda.stream(stream):
        parts = []            # per pass: (U_local, [PhenoResult])
        if route == "pages":
            pr = getattr(ka, "_page_route", None)
            if pr is None or (pr.rank, pr.world) != (rank, world):
                pr = ka._page_route = PageRoute(ka, rank, world, device)
            pr.prepare(int(k), int(n_samples), dist, torch, passes)
            spl = pr.splitters
            mark("prepare")
            U_seen = 0
            exact = not (binary and test_kw.get("omit_b"))
            for j in range(pr.passes):
                lo, hi, spl_j = pr.pass_range(j)
                if pr.passes > 1:
                    ctx.set_range(lo, hi)
                ctx.route_setup(world, rank, spl_j, pr.pages)      # same sizes: nothing moves, new splitters
                ctx.route_begin()
                pr.barrier(dist)            # every pool is clean before anybody writes into it
                ctx.route_scatter()
                pr.barrier(dist)            # every sender's stores have landed
                U_local, ovf = ctx.route_build()
                if restrict is not None and not ovf:
                    U_local = ctx.restrict_union(restrict)
                ka.U = U_local
                u = torch.tensor([U_local, 1 if ovf else 0], dtype=torch.int64, device=device)
                dist.all_reduce(u)
                U_seen += int(u[0].item())
                if int(u[1].item()):
                    pr.pages *= 2          # same decision on every rank: larger pools from the next step on
                    if pr.passes > 1:
                        ctx.set_range(0, 0)
                    raise PoolOverflow("a page pool overflowed while routing k-mers (skewed k-mer ranges); "
                                       "the next step will use pools twice as large")
                # Bonferroni needs the total U: a pass tests against the union seen so far (a laxer threshold),
                # the exact filter follows when every pass is done
                parts.append((U_local, test_pass(U_seen if exact else None)))
                mark(f"pass{j}")
            if pr.passes > 1:
                ctx.set_range(0, 0)
            U_total = U_seen
            nvl_bytes = None
        else:
            ctx.route_clear()
            nvl_bytes = 0
            if not getattr(ka, "_streams_imported", False):      # imported streams stay until the next ingest
                nvl_bytes = exchange_streams(ka, n_samples, rank, world, device, dist)
                ka._streams_imported = True
            mark("exchange")
            spl = ctx.sample_quantiles(0, world)          # identical on every rank: all hold sample 0
            U_local = ka.build(range_of(rank, spl))
            if restrict is not None:
                U_local = ka.restrict_to(restrict)
            mark("build")
            u = torch.tensor([U_local], dtype=torch.int64, device=device)
            dist.all_reduce(u)
            U_total = int(u[0].item())
            parts.append((U_local, test_pass(U_total)))
            mark("test")
        if perm:
            p_exact = permutation_thresholds(minp, alpha)
        elif binary and test_kw.get("omit_b"):
            p_exact = None
        else:
            p_exact = alpha / U_total if U_total else 0.0
        merged = gather_results(parts, rank, world, device, dist, top_k=test_kw.get("top_k"), p_exact=p_exact)
        if perm and merged is not None:
            for j, r in enumerate(merged):
                r.threshold, r.minp = float(p_exact[j]), minp[j]
        mark("gather")
    mark.report()
    return U_total, merged, {"U_local": sum(p[0] for p in parts), "nvlink_bytes": nvl_bytes, "splitters": spl, "route": route,
                             "passes": len(parts)}


def run_sharded(ka: KmerAssociation, buffers_by_sample, n_samples, k, pheno, binary, weights,
                rank, world, device, cutoff=1, route="auto", group=None, **test_kw):
    """Whole hot path on `world` GPUs: ingest() then build_and_test(). buffers_by_sample: {sample_idx: bytes or
    (dev_ptr, n)} for the samples this rank owns (sample_block(rank, world, n_samples)). group: see build_and_test.
    Returns (U_total, results on rank 0 / None elsewhere, info)."""
    marks = _Marks(rank, device)
    marks("start")
    ingest(ka, buffers_by_sample, n_samples, k, rank, world, cutoff)
    if world > 1:
        marks("ingest")
    return build_and_test(ka, n_samples, k, pheno, binary, weights, rank, world, device, route=route, group=group,
                          marks=marks, **test_kw)
