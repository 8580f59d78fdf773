"""GPU: incremental adds and deletes on the one-process-per-GPU deployment (include/svsb200.h svsb_shard_mutations_*,
svsb_compact).  Virtual ranks: 2, 3, 4 and 8 single-device shard engines in one process, on distinct GPUs when visible,
otherwise all on device 0, driven through the C ABI rank by rank with the collectives replaced by concatenations.  A
random walk of adds and deletes (ids ascending, some deletes hitting appended rows) runs against a host mirror of the live
rows; every tenth step every rank's answers must equal, bit for bit (scores as uint32, ids, order), both a fresh load of
the mirror over the same ranks and Engine([0]) over it.  ShardedRetriever.apply_mutations runs once on a real
world-size-1 NCCL group, and over CUDA IPC in two processes when two GPUs are visible."""
import os
import socket
import threading

import numpy as np
import pytest

from _util import oracle

pytestmark = pytest.mark.gpu

D = 96
KS = (7, 100, 2048, 2300, 10 ** 9)


def _devices(count):
    import torch
    have = max(torch.cuda.device_count(), 1)
    return [i % have for i in range(count)]


def _unit(rng, n):
    m = rng.standard_normal((n, D)).astype(np.float32)
    return m / np.sqrt((m * m).sum(axis=1))[:, None]


class Ranks:
    """world shard backends with the query exchange connected; `live[r]` / `rows[r]`: live / physical rows of rank r."""

    def __init__(self, world):
        from svs_b200.sharded import CudaShardBackend
        os.environ["SVSB_XCHG_TIMEOUT_MS"] = "10000"            # a protocol bug must fail the test, not hang the GPU
        self.backs = [CudaShardBackend(d) for d in _devices(world)]
        self.world = world
        self.connected = False

    def load(self, m, ids):
        from svs_b200.sharded import partition
        self.live = []
        for r, b in enumerate(self.backs):
            row0, cnt = partition(len(m), self.world, r)
            b.set_shard(row0)
            b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
            self.live.append(cnt)
        self.rows = list(self.live)
        if not self.connected:                                    # windows outlive loads and updates
            for r, b in enumerate(self.backs):
                b.exchange_handle(self.world, r)
            for b in self.backs:
                b.exchange_connect_local(self.backs)
            self.connected = True

    def apply(self, dels, aids, rows):
        """The protocol of ShardedRetriever.apply_mutations."""
        last = self.world - 1
        got = [b.mutations_prepare(dels, aids, rows, r == last) for r, b in enumerate(self.backs)]
        ok = sum(f for f, _ in got) == len(dels) and (len(aids) == 0 or aids[0] > max(x for _, x in got))
        for b in self.backs:
            b.mutations_commit(ok)
        if ok:
            self.live = [lv - f for lv, (f, _) in zip(self.live, got)]
            self.live[last] += len(aids)
            self.rows[last] += len(aids)
        return ok

    def compact(self):
        row0 = 0
        for b, lv in zip(self.backs, self.live):
            b.compact(row0)
            row0 += lv
        self.rows = list(self.live)

    def peer(self, qs, k):
        """Pipelined single queries through the peer exchange: every rank's (scores, ids) per query."""
        import torch
        outs = [b.new_outputs(len(qs), k) for b in self.backs]
        dqs = [b.device_queries(qs) for b in self.backs]
        for j in range(len(qs)):
            for b, dq, (o_s, o_i, o_c) in zip(self.backs, dqs, outs):
                b.enqueue_query_peer(dq[j], k, o_s[j], o_i[j], o_c[j], pipelined=True)
        for b in self.backs:
            b.join()
        torch.cuda.synchronize()
        res = []
        for o_s, o_i, o_c in outs:
            s, i, c = o_s.cpu().numpy(), o_i.cpu().numpy(), o_c.cpu().numpy()
            res.append([(s[j, :c[j]], i[j, :c[j]]) for j in range(len(qs))])
        return res

    def peer_sync(self, qs, k):
        """svsb_query_peer called SPMD from one thread per rank."""
        res = [[None] * len(qs) for _ in self.backs]
        errors = []

        def work(r):
            try:
                for j, q in enumerate(qs):
                    res[r][j] = self.backs[r].query_peer(q, k)
            except Exception as ex:                               # pragma: no cover - reported below
                errors.append(ex)
        threads = [threading.Thread(target=work, args=(r,)) for r in range(self.world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(timeout=120)
        assert not errors, errors
        return res

    def collective(self, qs, k):
        """The collective path: local records (k <= 2048) or sorted records of cap = largest live shard (k > 2048)."""
        import torch
        n = sum(self.live)
        k = min(k, n)
        big = k > 2048
        cap = min(k, max(self.live)) if big else k
        recs = [b.new_records(len(qs), cap) for b in self.backs]
        for b, rec in zip(self.backs, recs):
            dq = b.device_queries(qs)
            for j in range(len(qs)):
                b.enqueue_local(dq[j], cap, rec[j], seq=j)
            b.join()
        torch.cuda.synchronize()
        res = []
        for b in self.backs:
            out = []
            for j in range(len(qs)):
                g = torch.stack([rec[j].to(b.device) for rec in recs]).contiguous()
                o_s, o_i, o_c = b.new_outputs(1, k if not big else self.world * cap)
                if big:
                    b.enqueue_merge_sorted(g, self.world, cap, k, o_s[0], o_i[0], o_c[0])
                else:
                    b.enqueue_merge(g, self.world, 1, k, o_s, o_i, o_c)
                c = int(o_c[0].item())
                out.append((o_s[0, :c].cpu().numpy(), o_i[0, :c].cpu().numpy()))
            res.append(out)
        return res

    def batch_local(self, qs, k):
        import torch
        recs = []
        for b in self.backs:
            rec = b.new_records(len(qs), k)
            assert b.batch_local(b.device_queries(qs), k, rec) >= 0
            recs.append(rec)
        torch.cuda.synchronize()
        return self._merge(recs, qs, k)

    def _merge(self, recs, qs, k):
        res = []
        for b in self.backs:
            g = torch_cat([rec.to(b.device) for rec in recs])
            o_s, o_i, o_c = b.new_outputs(len(qs), k)
            b.enqueue_merge(g, self.world, len(qs), k, o_s, o_i, o_c)
            s, i, c = o_s.cpu().numpy(), o_i.cpu().numpy(), o_c.cpu().numpy()
            res.append([(s[j, :c[j]], i[j, :c[j]]) for j in range(len(qs))])
        return res

    def batch_global(self, qs, k):
        """The global-threshold plan (ShardedRetriever._global_plan / _batch) with cap = k; None if a rank declines."""
        import torch
        probes = [b.batch_global_probe(k) for b in self.backs]
        if not all(p[0] for p in probes):
            return None
        n = sum(self.live)
        f = max(min(1.0, p[1] / max(1, p[2])) for p in probes)
        lam = min(k, n) * f
        rank = int(np.ceil(lam + 6.0 * np.sqrt(lam) + 4.0))
        if rank > 32:
            return None
        norm = max(p[3] for p in probes)
        dqs = [b.device_queries(qs) for b in self.backs]
        tops = [b.new_tops(len(qs)) for b in self.backs]
        for b, dq, t in zip(self.backs, dqs, tops):
            b.batch_sample_tops(dq, k, norm, t)
        torch.cuda.synchronize()
        recs = []
        for b, dq in zip(self.backs, dqs):
            tops_all = torch.stack([t.to(b.device) for t in tops]).contiguous()
            rec = b.new_records(len(qs), k)
            b.batch_global_records(dq, k, tops_all, self.world, rank, k, rec)
            recs.append(rec)
        torch.cuda.synchronize()
        res = []
        for b in self.backs:
            g = torch.stack([rec.to(b.device) for rec in recs]).contiguous()
            o_s, o_i, o_c = b.new_outputs(len(qs), k)
            b.enqueue_merge_verified(g, self.world, len(qs), k, k, min(k, n), o_s, o_i, o_c)
            s, i, c = o_s.cpu().numpy(), o_i.cpu().numpy(), o_c.cpu().numpy()
            assert (c == min(k, n)).all(), c
            res.append([(s[j, :c[j]], i[j, :c[j]]) for j in range(len(qs))])
        return res

    def close(self):
        for b in self.backs:
            b.close()


def torch_cat(ts):
    import torch
    return torch.cat(ts).contiguous()


def _same(got, want, what):
    s, i = got
    ws, wi = want
    assert len(s) == len(ws), what
    assert np.array_equal(np.asarray(s, np.float32).view(np.uint32), np.asarray(ws, np.float32).view(np.uint32)), what
    assert np.array_equal(i, wi), what


def _check(ranks, fresh, one, mirror_m, mirror_ids, qs, step):
    """Every rank's answers on every path against a fresh load over the same ranks and against Engine([0])."""
    fresh.load(mirror_m, mirror_ids)
    one.load(mirror_m, mirror_ids)
    assert sum(ranks.live) == len(mirror_ids)
    for k in KS:
        want = [one.query(q, k) for q in qs]
        paths = [("collective", ranks.collective(qs, k), fresh.collective(qs, k))]
        if k <= 2048:
            paths.append(("peer", ranks.peer(qs, k), fresh.peer(qs, k)))
            paths.append(("batch", ranks.batch_local(qs, k), fresh.batch_local(qs, k)))
        if k == 100:
            paths.append(("peer_sync", ranks.peer_sync(qs, k), fresh.peer_sync(qs, k)))
        for name, got, ref in paths:
            for r in range(ranks.world):
                for j in range(len(qs)):
                    what = (step, name, k, r, j)
                    _same(got[r][j], want[j], what)
                    _same(ref[r][j], want[j], what)


@pytest.fixture(scope="module")
def one():
    import svs_b200
    e = svs_b200.Engine([0])
    yield e
    e.close()


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_random_updates_answer_as_a_fresh_load_on_every_rank(world, one, monkeypatch):
    pytest.importorskip("torch")
    monkeypatch.setenv("SVSB_BATCH_MIN_ROWS", "64")             # the batched coarse pass on shards of a few hundred rows
    rng = np.random.default_rng(500 + world)
    n0 = 3000
    m = _unit(rng, n0)
    m[9] = m[n0 - 4]                                             # an exact tie across shards
    ids = np.cumsum(rng.integers(1, 4, size=n0)).astype(np.int64)
    qs = np.concatenate([oracle.synth_queries(2, D, world, "normal"), m[[9]]])
    ranks, fresh = Ranks(world), Ranks(world)
    try:
        ranks.load(m, ids)
        mm, mi = m.copy(), ids.copy()
        appended = []
        steps = 300
        for step in range(1, steps + 1):
            n_del = int(rng.integers(0, 12))
            pool = mi if not appended or rng.random() < 0.5 else np.intersect1d(mi, np.array(appended))
            dels = rng.choice(pool, size=min(n_del, len(pool)), replace=False).astype(np.int64) if len(pool) else np.zeros(0, np.int64)
            n_add = int(rng.integers(0, 25))
            aids = (int(mi.max()) if len(mi) else 0) + np.cumsum(rng.integers(1, 3, size=n_add)).astype(np.int64)
            if n_add and rng.random() < 0.1 and len(dels) == 0 and len(mi):
                top = int(mi.max())                              # delete and re-insert the largest id
                dels, aids = np.array([top], np.int64), np.concatenate([[top], aids[:-1]]).astype(np.int64)
            rows = _unit(rng, n_add)
            assert ranks.apply(dels, aids, rows)
            keep = ~np.isin(mi, dels)
            mm, mi = np.concatenate([mm[keep], rows]), np.concatenate([mi[keep], aids])
            appended += aids.tolist()
            if step % 10 == 0:
                _check(ranks, fresh, one, mm, mi, qs, step)
        assert ranks.live[-1] > -(-n0 // world)                 # the last shard outgrew the size its workspaces began at
        # refusals leave every rank's state unchanged: an unknown delete id, an id not above the live maximum
        assert not ranks.apply(np.array([10 ** 12], np.int64), np.zeros(0, np.int64), np.zeros((0, D), np.float32))
        assert not ranks.apply(np.zeros(0, np.int64), np.array([int(mi.max())], np.int64), _unit(rng, 1))
        # batches decline the global-threshold plan on tombstoned shards; compaction makes them eligible
        tomb = sum(ranks.rows) != sum(ranks.live)
        if tomb:
            assert ranks.batch_global(qs, 7) is None
        ranks.compact()
        _check(ranks, fresh, one, mm, mi, qs, "compacted")
        for k in (7,):
            got = ranks.batch_global(qs, k)
            assert got is not None
            want = [one.query(q, k) for q in qs]
            for r in range(world):
                for j in range(len(qs)):
                    _same(got[r][j], want[j], ("global", k, r, j))
        # top_pairs after compaction: the pair export accepts the compacted shards, contiguous in rank order
        from test_gpu_pairs_sharded import _assert_same, _top_pairs
        got_desc = [b.pairs_export() for b in ranks.backs]
        assert all(g[1] == 0 for g in got_desc), [g[2] for g in got_desc]
        for r, b in enumerate(ranks.backs):
            b.pairs_connect_local(world, r, ranks.backs)
        norm = max(1.0 + g[3] for g in got_desc)
        one.load(mm, mi)
        want = one.top_pairs(200)
        for r, got in enumerate(_top_pairs(ranks.backs, len(mi), 200, norm)):
            _assert_same(got, want, ("pairs", r))
        for b in ranks.backs:
            b.pairs_disconnect()
    finally:
        ranks.close()
        fresh.close()


def _fresh_equal(e, ref, qs, what):
    assert e.shape == ref.shape, what
    n = e.shape[0]
    r1, i1 = e.read_rows(0, n)
    r2, i2 = ref.read_rows(0, n)
    assert np.array_equal(r1.view(np.uint32), r2.view(np.uint32)) and np.array_equal(i1, i2), what
    assert e.generation_rows() == ref.generation_rows() == (n, n), what
    for k in (1, 10, 100, 3000):
        for q in qs:
            a, b = e.query(q, k), ref.query(q, k)
            assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32)) and np.array_equal(a[1], b[1]), (what, k)


@pytest.mark.parametrize("d", [1536, 190])
def test_compact_equals_a_fresh_load_on_one_device(d, monkeypatch):
    """svsb_compact: rows, ids, shape, norm statistics in check mode, the filter route the bench loop takes, answers."""
    import svs_b200
    monkeypatch.setenv("SVSB_FILTER_MIN_MB", "1")                # the filters' shadows at a test size
    rng = np.random.default_rng(d)
    n = 40_000
    m = rng.standard_normal((n, d)).astype(np.float32)
    m /= np.sqrt((m * m).sum(axis=1))[:, None]
    m[::97] *= np.float32(1.01)                                  # rows outside the norm tolerance
    ids = np.arange(3, 3 + 2 * n, 2, dtype=np.int64)
    qs = oracle.synth_queries(3, d, 11, "normal")
    dels = np.concatenate([ids[:500], ids[7000:7040], ids[::13], ids[-3:]])
    dels = np.unique(dels)
    add = rng.standard_normal((700, d)).astype(np.float32) / np.float32(np.sqrt(d))
    add_ids = ids[-1] + 1 + np.arange(700, dtype=np.int64)
    keep = ~np.isin(ids, dels)
    lm, li = np.concatenate([m[keep], add]), np.concatenate([ids[keep], add_ids])
    with svs_b200.Engine([0]) as e, svs_b200.Engine([0]) as ref:
        e.load(m, ids)
        e.apply_mutations(dels, add_ids, add)
        e.apply_mutations(add_ids[5:9], [], None)
        keep2 = ~np.isin(li, add_ids[5:9])
        lm, li = lm[keep2], li[keep2]
        snap = e.snapshot()                                      # a pinned generation keeps reading its rows
        before = snap.query(qs[0], 50)
        e.compact()
        ref.load(lm, li)
        _fresh_equal(e, ref, qs, d)
        assert e.norm_stats() == ref.norm_stats() and e.norm_stats()[1] > 0
        routes = []
        for x in (e, ref):
            x.bench_set_queries(qs)
            x.bench_run(10, 3)
            routes.append((x.bench_filter_route(), x.bench_last_result(10)))
        assert routes[0] == routes[1]
        assert routes[0][0] == (8 if d <= 1536 else routes[0][0])
        after = snap.query(qs[0], 50)
        assert np.array_equal(before[0].view(np.uint32), after[0].view(np.uint32)) and np.array_equal(before[1], after[1])
        snap.release()
        # compaction at another global row offset: answers unchanged, a reload-free no-tombstone compaction too
        e.compact(1000)
        _fresh_equal(e, ref, qs, (d, "offset"))
        e.apply_mutations(li[:5], [], None)
        e.compact(0)
        ref.load(lm[5:], li[5:])
        _fresh_equal(e, ref, qs, (d, "again"))
    with svs_b200.Engine([0]) as e:                              # every row deleted: a load of no rows
        e.load(m[:10], ids[:10])
        e.apply_mutations(ids[:10], [], None)
        e.compact()
        assert e.shape[0] == 0 and e.generation_rows() == (0, 0)


def test_compact_refuses_a_multi_device_engine_and_a_pending_update_blocks_loads(monkeypatch):
    import svs_b200
    from svs_b200._lib import SVSB_E_INVALID, SVSB_E_STATE
    from svs_b200.sharded import CudaShardBackend
    rng = np.random.default_rng(3)
    m = _unit(rng, 100)
    ids = np.arange(100, dtype=np.int64)
    monkeypatch.setenv("SVSB_ALLOW_DUP_DEVICES", "1")            # two shard engines on device 0 where one GPU is visible
    with svs_b200.Engine([0, 0]) as multi:
        multi.load(m, ids)
        with pytest.raises(svs_b200.EngineError) as ex:
            multi.compact()
        assert ex.value.code == SVSB_E_INVALID
    b = CudaShardBackend(0)
    try:
        b.load_rows(m, ids)
        assert b.mutations_prepare(np.array([3, 1000], np.int64), np.array([200], np.int64), _unit(rng, 1), True) == (1, 99)
        for call in (lambda: b.engine.load(m, ids), lambda: b.engine.apply_mutations([4], [], None), lambda: b.compact(0),
                     lambda: b.mutations_prepare(np.array([5], np.int64), np.zeros(0, np.int64), np.zeros((0, D), np.float32), True)):
            with pytest.raises(svs_b200.EngineError) as ex:
                call()
            assert ex.value.code == SVSB_E_STATE
        assert b.engine.generation_rows() == (100, 100)          # nothing published yet
        b.mutations_commit(False)
        assert b.engine.generation_rows() == (100, 100)
        b.mutations_commit(False)                                # nothing pending: a no-op
        with pytest.raises(svs_b200.EngineError):
            b.mutations_commit(True)
        b.mutations_prepare(np.array([3], np.int64), np.array([200], np.int64), _unit(rng, 1), True)
        b.mutations_commit(True)
        assert b.engine.generation_rows() == (101, 100)
    finally:
        b.close()


def test_world_size_one_process_group_applies_mutations():
    torch = pytest.importorskip("torch")
    import torch.distributed as dist
    from svs_b200.sharded import ShardedRetriever
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ["MASTER_PORT"] = "29591"
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        _sharded_session(ShardedRetriever(0, 1, 0, exchange="peer"))
    finally:
        dist.destroy_process_group()


def _sharded_session(sr):
    """Load, add, delete, refuse, compact through ShardedRetriever; returns the answers."""
    from svs_b200 import EngineError
    rng = np.random.default_rng(42)
    m = _unit(rng, 5000)
    ids = np.arange(1, 5001, dtype=np.int64) * 3
    qs = oracle.synth_queries(4, D, 43, "normal")
    sr.load_global(m, ids)
    add = _unit(rng, 40)
    add_ids = np.arange(20_000, 20_040, dtype=np.int64)
    sr.apply_mutations(ids[100:160], add_ids, add)
    keep = ~np.isin(ids, ids[100:160])
    lm, li = np.concatenate([m[keep], add]), np.concatenate([ids[keep], add_ids])
    with pytest.raises(EngineError):
        sr.apply_mutations([7], [], None)                          # not an id
    out = []
    for k in (10, 100, 3000):
        for q in qs:
            got = sr.retrieve(q, k)
            oracle.compare_retrieval(got, oracle.superheavy(lm, li, q, k), oracle.scores_of(lm, q), li)
            out.append(got)
    many = sr.retrieve_many(qs, 50)
    assert many == [sr.retrieve(q, 50) for q in qs]
    pairs = sr.top_pairs(20)                                       # compacts first
    assert sr._shard_rows == sr._shard_live
    oracle.compare_pairs(pairs, oracle.top_pairwise(lm, li, 20), np.dot(lm, lm.T), li)
    out += [many, pairs, [sr.retrieve(q, 100) for q in qs]]
    sr.close()
    return out


def _ipc_worker(rank, world, port, ret):
    import torch
    import torch.distributed as dist
    from svs_b200.sharded import ShardedRetriever
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["SVSB_XCHG_TIMEOUT_MS"] = "10000"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        ret[rank] = _sharded_session(ShardedRetriever(rank, world, rank, exchange="peer"))
    finally:
        dist.destroy_process_group()


def test_apply_mutations_over_cuda_ipc_in_two_processes():
    torch = pytest.importorskip("torch")
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (NCCL runs one rank per GPU)")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_ipc_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret[0] == ret[1]
