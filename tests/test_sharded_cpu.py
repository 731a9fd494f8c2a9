"""CPU suite for the multi-rank host logic: row partition, all-gather layout and global reduce over a
world_size-2 (and 3) gloo group.  Local search and merge are oracle stand-ins (no GPU here)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ragfin_oracle as O
from ragfin_b200.sharded import ShardedSearcher, shard_bounds


def test_shard_bounds_cover_rows_exactly():
    for n, w in ((10, 3), (16, 8), (7, 8), (0, 2), (10_000_000, 8), (100_000_001, 4)):
        spans = [shard_bounds(n, w, r) for r in range(w)]
        assert sum(c for _, c in spans) == n
        pos = 0
        for row0, cnt in spans:
            assert row0 == min(pos, n) and cnt >= 0
            pos += cnt
    with pytest.raises(ValueError):
        shard_bounds(10, 2, 2)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n, k, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x = O.normalize_rows(O.synth_rows(21, 0, n, 64, dup_every=5), "bf16")
        q = O.synth_rows(22, 0, 3, 64)
        row0, cnt = shard_bounds(n, world, rank)

        def local_search(queries, kk):
            ids, sc = O.cosine_topk(queries.numpy(), x[row0:row0 + cnt], kk, id_base=row0)
            return torch.from_numpy(ids), torch.from_numpy(sc)

        def merge(ids, sc, parts, kk):            # all-gather layout [parts, nq, k]
            assert ids.shape == (parts, 3, kk)
            mi, ms = O.merge_topk([ids[p].numpy() for p in range(parts)], [sc[p].numpy() for p in range(parts)], kk)
            return torch.from_numpy(mi), torch.from_numpy(ms)

        s = ShardedSearcher(local_search, merge)
        assert s.world == world and s.rank == rank
        for _ in range(2):                        # second call reuses the gather buffers
            ids, sc = s.search(torch.from_numpy(q), k)
        want_i, want_s = O.cosine_topk(q, x, k)
        ok = np.array_equal(ids.numpy(), want_i) and np.array_equal(sc.numpy().view(np.uint32), want_s.view(np.uint32))
        out[rank] = int(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n,k", [(2, 101, 10), (3, 50, 20), (2, 5, 10)])
def test_sharded_search_over_gloo(world, n, k):
    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), n, k, out), nprocs=world, join=True)
    assert dict(out) == {r: 1 for r in range(world)}


class _GlooExchange:
    """Stand-in for engine.PeerExchange (peer-memory stores need GPUs): same interface, the records travel through a
    gloo all-gather.  Exercises ShardedSearcher's exchange branch: local hits written into per-(nq, k) buffers, one
    collective call per step, fallback to the packed path when a record exceeds the exchange's capacity."""

    def __init__(self, world, max_record_bytes):
        self.world, self.max_record_bytes, self.steps = world, max_record_bytes, 0

    def allgather_merge(self, ids, scores):
        self.steps += 1
        gi = [torch.empty_like(ids) for _ in range(self.world)]
        gs = [torch.empty_like(scores) for _ in range(self.world)]
        dist.all_gather(gi, ids)
        dist.all_gather(gs, scores)
        mi, ms = O.merge_topk([t.numpy() for t in gi], [t.numpy() for t in gs], ids.shape[1])
        return torch.from_numpy(mi), torch.from_numpy(ms)


def _worker_exchange(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n, dim = 300, 32
        x = O.normalize_rows(O.synth_rows(31, 0, n, dim, dup_every=7), "f16")
        row0, cnt = shard_bounds(n, world, rank)
        calls = []

        def local_search(queries, kk, out_ids=None, out_scores=None):
            ids, sc = O.cosine_topk(queries.numpy(), x[row0:row0 + cnt], kk, id_base=row0)
            calls.append((out_ids is not None, queries.shape[0], kk))
            if out_ids is not None:                      # the exchange branch hands in its per-(nq, k) buffers
                out_ids.copy_(torch.from_numpy(ids)); out_scores.copy_(torch.from_numpy(sc))
                return out_ids, out_scores
            return torch.from_numpy(ids), torch.from_numpy(sc)

        def merge(ids, sc, parts, kk):
            mi, ms = O.merge_topk([ids[p].numpy() for p in range(parts)], [sc[p].numpy() for p in range(parts)], kk)
            return torch.from_numpy(mi), torch.from_numpy(ms)

        ex = _GlooExchange(world, max_record_bytes=4 * 10 * 12)      # fits 4 queries x k = 10, not 9 x 10
        s = ShardedSearcher(local_search, merge, exchange=ex)
        ok = True
        for nq in (4, 4, 9, 1):
            q = O.synth_rows(40 + nq, 0, nq, dim)
            ids, sc = s.search(torch.from_numpy(q), 10)
            wi, ws = O.cosine_topk(q, x, 10)
            ok &= np.array_equal(ids.numpy(), wi) and np.array_equal(sc.numpy().view(np.uint32), ws.view(np.uint32))
        ok &= ex.steps == 3                                           # the 9-query batch took the all-gather path
        ok &= [c[0] for c in calls] == [True, True, False, True]
        out[rank] = int(ok)
    finally:
        dist.destroy_process_group()


def test_exchange_branch_and_its_fallback_over_gloo():
    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker_exchange, args=(2, _free_port(), out), nprocs=2, join=True)
    assert dict(out) == {0: 1, 1: 1}


class _FakeIndex:
    """Stand-in with the two members ShardedSearcher reads for the one-kernel decision."""
    device = 0

    def __init__(self, eligible):
        self.eligible = eligible

    def fused_eligible(self, nq, k):
        return self.eligible(nq, k)


class _FakeExchange:
    """Stand-in for PeerExchange: records which entry point a search took; `search_sharded*` answer from the full matrix
    (what the real kernel's exchange + reduce produces on every rank)."""
    max_record_bytes = 1 << 20

    def __init__(self, x, log):
        self.x, self.log = x, log

    def search_sharded(self, index, queries, k, out_ids=None, out_scores=None, stream=None):
        self.log.append("one-kernel")
        ids, sc = O.cosine_topk(queries.numpy(), self.x, k)
        return torch.from_numpy(ids), torch.from_numpy(sc)

    def search_sharded_host(self, index, q, k, out_ids=None, out_scores=None):
        self.log.append("one-kernel-host")
        ids, sc = O.cosine_topk(np.asarray(q), self.x, k)          # numpy or torch CPU buffers, as the real one
        if out_ids is not None:
            np.asarray(out_ids)[...] = ids
            np.asarray(out_scores)[...] = sc
            return out_ids, out_scores
        return ids, sc

    def allgather_merge(self, ids, scores, stream=None):
        self.log.append("push-merge")
        parts = [torch.empty_like(ids) for _ in range(dist.get_world_size())]
        sparts = [torch.empty_like(scores) for _ in range(dist.get_world_size())]
        dist.all_gather(parts, ids.contiguous())
        dist.all_gather(sparts, scores.contiguous())
        mi, ms = O.merge_topk([p.numpy() for p in parts], [p.numpy() for p in sparts], ids.shape[1])
        return torch.from_numpy(mi), torch.from_numpy(ms)


def _worker_fused_agreement(rank, world, port, out):
    """Rank 1's shard is 'too small' for the one-kernel search at k = 5: NO rank may take it for that shape (a rank on another
    path would leave its peers waiting inside the kernel); at k = 3 every rank is eligible and all of them take it."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n, dim = 300, 32
        x = O.normalize_rows(O.synth_rows(31, 0, n, dim), "f32")
        q = O.synth_rows(32, 0, 2, dim)
        row0, cnt = shard_bounds(n, world, rank)
        log = []

        def local_search(queries, kk, out_ids=None, out_scores=None):
            ids, sc = O.cosine_topk(queries.numpy(), x[row0:row0 + cnt], kk, id_base=row0)
            if out_ids is not None:
                out_ids.copy_(torch.from_numpy(ids)); out_scores.copy_(torch.from_numpy(sc))
                return out_ids, out_scores
            return torch.from_numpy(ids), torch.from_numpy(sc)

        idx = _FakeIndex(lambda nq, k: not (rank == 1 and k == 5))
        s = ShardedSearcher(local_search, None, exchange=_FakeExchange(x, log), index=idx)
        ok = True
        for k, want_path in ((3, "one-kernel"), (5, "push-merge"), (3, "one-kernel")):
            ids, sc = s.search(torch.from_numpy(q), k)
            wi, ws = O.cosine_topk(q, x, k)
            ok &= np.array_equal(ids.numpy(), wi) and np.array_equal(sc.numpy().view(np.uint32), ws.view(np.uint32))
            ok &= log[-1] == want_path
        hi, hs = s.search_host(q, 3)
        ok &= log[-1] == "one-kernel-host" and np.array_equal(hi, O.cosine_topk(q, x, 3)[0])
        hi, hs = s.search_host(q, 5)               # not eligible everywhere: device staging around search()
        ok &= log[-1] == "push-merge" and np.array_equal(hi, O.cosine_topk(q, x, 5)[0])
        # the caller's own torch CPU buffers (what bench.py's e2e leg passes), both branches: results land in them
        for k, want_path in ((3, "one-kernel-host"), (5, "push-merge")):
            oi, osc = torch.full((2, k), -9, dtype=torch.int64), torch.zeros((2, k), dtype=torch.float32)
            ri, rs = s.search_host(torch.from_numpy(q), k, out_ids=oi, out_scores=osc)
            wi, ws = O.cosine_topk(q, x, k)
            ok &= log[-1] == want_path and np.array_equal(oi.numpy(), wi) and np.array_equal(osc.numpy().view(np.uint32), ws.view(np.uint32))
            ok &= np.array_equal(np.asarray(ri), wi) and np.array_equal(np.asarray(rs).view(np.uint32), ws.view(np.uint32))
        one = s.search_host(q[0], 3)                 # a single query as a 1-D array ...
        ok &= np.array_equal(np.asarray(one[0]), O.cosine_topk(q[:1], x, 3)[0])
        one = s.search_host(q[0].tolist(), 5)        # ... and as a plain list, on the staging branch
        ok &= one[0].shape == (1, 5) and np.array_equal(one[0], O.cosine_topk(q[:1], x, 5)[0])
        ok &= s._fused == {(2, 3): True, (2, 5): False, (1, 3): True, (1, 5): False}
        out[rank] = int(ok)
    finally:
        dist.destroy_process_group()


def test_one_kernel_path_is_taken_only_when_every_rank_can(monkeypatch):
    # the stand-ins are host code: a rank that saw a GPU would stage its queries there (search_host, fused_ok)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    world = 2
    ctx = mp.get_context("spawn")
    out = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker_fused_agreement, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
    assert all(p.exitcode == 0 for p in procs)
    assert dict(out) == {0: 1, 1: 1}
