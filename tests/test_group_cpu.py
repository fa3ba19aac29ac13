"""Host side of several GPUs in one process, on the CPU: the thread collectives (dist.ThreadGroup), the runner of
group.GpuGroup (errors, no thread left behind, the page-pool overflow retry) with stand-in engines, the gather
capacity per group, and PS_DEVICE parsing. The device side is covered by tests/test_gpu_group.py."""
import threading
import time

import numpy as np
import pytest
import torch

from phenotypeseeker_b200 import dist as psdist
from phenotypeseeker_b200 import group as psgroup
from phenotypeseeker_b200.modeling_gpu import parse_devices
from phenotypeseeker_b200.pipeline import PhenoResult


def test_thread_collectives_match_torch_distributed_semantics():
    G = 3
    tg = psdist.ThreadGroup(G)
    base = [torch.arange(5, dtype=torch.int64) * (r + 1) + r for r in range(G)]

    def one(r):
        red = base[r].clone()
        tg.all_reduce(red)
        gat = torch.empty(G * 5, dtype=torch.int64)
        tg.all_gather_into_tensor(gat, base[r].clone())
        bc = base[r].clone()
        tg.broadcast(bc, src=2)
        fl = torch.tensor([0.5 * (r + 1)], dtype=torch.float64)
        tg.all_reduce(fl)
        return red, gat, bc, fl

    out = tg.run(one)
    want_sum = base[0] + base[1] + base[2]
    for red, gat, bc, fl in out:
        assert torch.equal(red, want_sum)                        # all_reduce (SUM), in place on every rank
        assert torch.equal(gat, torch.cat(base))                 # all_gather_into_tensor: rank-major
        assert torch.equal(bc, base[2])                          # broadcast from src
        assert fl.item() == 3.0


class _FakeCtx:
    def __init__(self, log):
        self.log = log

    def begin(self, k, n, cutoff=1):
        self.log.append(("begin", k, n))

    def route_clear(self):
        pass

    def add_samples(self, first, bufs):
        self.log.append(("add", first, len(bufs)))


class _FakeEngine:
    """Stands in for KmerAssociation: records what the group ingests."""
    log = []

    def __init__(self, device=0):
        self.ctx = _FakeCtx(_FakeEngine.log)
        self.k = None
        self.n_samples = 0


@pytest.fixture
def cpu_group(monkeypatch):
    _FakeEngine.log = []
    monkeypatch.setattr(psgroup, "KmerAssociation", _FakeEngine)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    return psgroup.GpuGroup([0, 0, 0])


def test_rank_error_reaches_the_caller_and_no_thread_survives(cpu_group):
    before = threading.active_count()

    def one(r):
        if r == 1:
            raise ValueError("rank 1 failed before the collective")
        t = torch.ones(3)
        cpu_group.group.all_reduce(t)           # ranks 0 and 2 would wait here forever without the abort
        return t

    t0 = time.time()
    with pytest.raises(ValueError, match="rank 1 failed"):
        cpu_group._run(one)
    assert time.time() - t0 < 5
    assert threading.active_count() == before

    def again(r):                               # the group is usable again afterwards
        t = torch.ones(2)
        cpu_group.group.all_reduce(t)
        return int(t.sum())
    assert cpu_group._run(again) == [6] * 3


def _big_result(j, n):
    rng = np.random.default_rng(j)
    return PhenoResult(name="ph", kmer=np.arange(n, dtype=np.uint64), row=np.arange(n, dtype=np.uint64),
                       stat=rng.random(n), p=rng.random(n), mean_x=rng.random(n), mean_y=rng.random(n),
                       n_with=np.full(n, 2, np.uint32), presence=np.ones((n, 6), np.uint8))


def test_gather_capacity_lives_on_the_group():
    a, b = psdist.ThreadGroup(2), psdist.ThreadGroup(2)
    cap0 = a.gather_cap
    assert b.gather_cap == cap0

    def gather(tg, n):
        return tg.run(lambda r: psdist.gather_results([(n, [_big_result(r, n)])], r, 2, torch.device("cpu"), tg))

    out = gather(a, 4000)                      # 4,000 survivors x ~70 bytes > the initial 64 KB
    assert a.gather_cap > cap0 and b.gather_cap == cap0
    assert out[1] is None and len(out[0][0].kmer) == 8000
    assert np.array_equal(out[0][0].row, np.arange(8000, dtype=np.uint64))     # rank 1's rows follow rank 0's
    grown = a.gather_cap
    gather(b, 10)
    assert b.gather_cap == cap0 and a.gather_cap == grown


def test_ps_device_parsing():
    assert parse_devices("0") == 0 and parse_devices(0) == 0 and parse_devices("3") == 3
    assert parse_devices("0,1") == [0, 1]
    assert parse_devices("0, 0") == [0, 0]
    assert parse_devices("0,1,2,3") == [0, 1, 2, 3]
    assert parse_devices([0, 0, 0]) == [0, 0, 0]
    assert parse_devices([2]) == 2
    with pytest.raises(ValueError):
        parse_devices("")


def test_pool_overflow_is_retried_once_without_a_new_ingest(cpu_group, monkeypatch):
    N = 7
    cpu_group.count([b">s\nACGT\n"] * N, 16, 1)
    ingested = list(_FakeEngine.log)
    assert sorted(e[1] for e in ingested if e[0] == "add") == [0, 2, 4]       # blocks [0,2) [2,4) [4,7)
    calls = []

    def build_and_test(ka, n, k, pheno, binary, weights, rank, world, device, group=None, **kw):
        calls.append(rank)
        t = torch.tensor([1])
        group.all_reduce(t)               # every rank has counted its call before any rank decides
        if len(calls) <= world:
            raise psdist.PoolOverflow("a page pool overflowed while routing k-mers")
        return 42, ([PhenoResult("p", np.zeros(0, np.uint64), np.zeros(0, np.uint64), np.zeros(0), np.zeros(0),
                                 np.zeros(0), np.zeros(0), np.zeros(0, np.uint32), np.zeros((0, N), np.uint8))]
                    if rank == 0 else None), {}

    monkeypatch.setattr(psdist, "build_and_test", build_and_test)
    U, res = cpu_group.test(np.zeros((N, 1)), True)
    assert U == 42 and cpu_group.U == 42 and res[0].name == "p"
    assert len(calls) == 6                               # 3 ranks x (first attempt + one retry)
    assert _FakeEngine.log == ingested                   # nothing was ingested again

    calls.clear()

    def always(ka, n, k, pheno, binary, weights, rank, world, device, group=None, **kw):
        calls.append(rank)
        raise psdist.PoolOverflow("a page pool overflowed while routing k-mers")

    monkeypatch.setattr(psdist, "build_and_test", always)
    with pytest.raises(psdist.PoolOverflow):
        cpu_group.test(np.zeros((N, 1)), True)
    assert len(calls) == 6                               # retried exactly once
    assert _FakeEngine.log == ingested
