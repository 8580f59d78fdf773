"""GPU: the one-process-per-GPU shard path (svsb_set_shard / svsb_enqueue_local_topk /
svsb_enqueue_merge_records) on ONE device: two shard engines stand in for two ranks and the all-gather is
a concatenation.  The collective itself is covered on CPU with gloo (tests/test_sharded_gloo.py) and on
N GPUs by bench.py under torchrun; the peer windows over CUDA IPC by two processes on two GPUs."""
import os
import socket

import numpy as np
import pytest

from _util import oracle

pytestmark = pytest.mark.gpu


def test_two_shard_engines_and_merge_records_match_the_oracle():
    torch = pytest.importorskip("torch")
    from svs_b200.sharded import CudaShardBackend, partition
    n, d = 30_001, 256
    m = oracle.synth_matrix_uniform(n, d, 5)
    m[7] = m[n - 3]                                            # exact tie across shards
    ids = np.cumsum(np.random.default_rng(2).integers(1, 4, size=n)).astype(np.int64)
    world = 2
    backs = []
    for r in range(world):
        b = CudaShardBackend(0)
        row0, cnt = partition(n, world, r)
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
        backs.append(b)
    qs = oracle.synth_queries(5, d, 6)
    qs[1] = m[7]
    try:
        for k in (1, 100, 1000, 2048):
            batch = len(qs)
            dq = backs[0].device_queries(qs)
            recs = [b.new_records(batch, k) for b in backs]
            for r, b in enumerate(backs):
                for j in range(batch):
                    b.enqueue_local(dq[j], k, recs[r][j], time_kernel=(k == 100))
            torch.cuda.synchronize()
            gathered = torch.stack(recs, dim=0).contiguous()   # [world, batch, 2k+1]: what all_gather yields
            o_s, o_i, o_c = backs[0].new_outputs(batch, k)
            backs[0].enqueue_merge(gathered, world, batch, k, o_s, o_i, o_c)
            torch.cuda.synchronize()
            for j in range(batch):
                c = int(o_c[j])
                got = list(zip(o_s[j, :c].cpu().numpy().tolist(), o_i[j, :c].cpu().numpy().tolist()))
                oracle.compare_retrieval(got, oracle.superheavy(m, ids, qs[j], k), oracle.scores_of(m, qs[j]), ids)
            if k >= 2:
                c = int(o_c[1])
                assert o_i[1, :2].cpu().numpy().tolist() == [int(ids[7]), int(ids[n - 3])]   # tie: ascending id
            if k == 100:
                assert backs[0].collect_kernel_ms() > 0 and backs[1].collect_kernel_ms() > 0
    finally:
        for b in backs:
            b.close()


def test_two_shard_engines_batched_records_equal_the_single_query_records():
    """svsb_batch_local_records (tensor-core coarse pass + exact refine per shard) must give the same merged
    answer, bit for bit, as the per-query records, and match the oracle."""
    torch = pytest.importorskip("torch")
    from svs_b200.sharded import CudaShardBackend, partition
    n, d, k, batch = 24_001, 256, 50, 40
    m = oracle.synth_matrix_uniform(n, d, 8)
    m[11] = m[n - 5]                                           # exact tie across shards
    ids = np.cumsum(np.random.default_rng(3).integers(1, 4, size=n)).astype(np.int64)
    world = 2
    backs = []
    for r in range(world):
        b = CudaShardBackend(0)
        row0, cnt = partition(n, world, r)
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
        backs.append(b)
    qs = oracle.synth_queries(batch, d, 9)
    qs[2] = m[11]
    try:
        dq = backs[0].device_queries(qs)
        outs = []
        for mode in ("batch", "single"):
            recs = [b.new_records(batch, k) for b in backs]
            for r, b in enumerate(backs):
                if mode == "batch":
                    assert b.batch_local(dq, k, recs[r]) == 0            # nobody needed the fallback
                else:
                    for j in range(batch):
                        b.enqueue_local(dq[j], k, recs[r][j])
            torch.cuda.synchronize()
            gathered = torch.stack(recs, dim=0).contiguous()
            o_s, o_i, o_c = backs[0].new_outputs(batch, k)
            backs[0].enqueue_merge(gathered, world, batch, k, o_s, o_i, o_c)
            torch.cuda.synchronize()
            outs.append((o_s.cpu().numpy().copy(), o_i.cpu().numpy().copy(), o_c.cpu().numpy().copy()))
        assert np.array_equal(outs[0][0].view(np.uint32), outs[1][0].view(np.uint32))
        assert np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[0][2], outs[1][2])
        s, i, c = outs[0]
        for j in range(0, batch, 5):
            got = list(zip(s[j, :c[j]].tolist(), i[j, :c[j]].tolist()))
            oracle.compare_retrieval(got, oracle.superheavy(m, ids, qs[j], k), oracle.scores_of(m, qs[j]), ids)
        assert i[2, :2].tolist() == [int(ids[11]), int(ids[n - 5])]     # tie: ascending id, across shards
    finally:
        for b in backs:
            b.close()


def _global_batch(backs, world, n, qs, k, sample_rank=None, cap=None):
    """The global-threshold batch protocol of ShardedRetriever._batch with the all-gathers done by torch.stack."""
    import torch
    batch = len(qs)
    probes = [b.batch_global_probe(k) for b in backs]
    assert all(p[0] for p in probes), probes
    f = max(min(1.0, p[1] / p[2]) for p in probes)
    lam = min(k, n) * f
    rank = int(np.ceil(lam + 6.0 * np.sqrt(lam) + 4.0)) if sample_rank is None else sample_rank
    assert rank <= 32
    norm = max(p[3] for p in probes)
    dq = backs[0].device_queries(qs)
    tops = [b.new_tops(batch) for b in backs]
    for r, b in enumerate(backs):
        b.batch_sample_tops(dq, k, norm, tops[r])
    tops_all = torch.stack(tops, dim=0).contiguous()
    cap = k if cap is None else cap
    recs = [b.new_records(batch, cap) for b in backs]
    for r, b in enumerate(backs):
        b.batch_global_records(dq, k, tops_all, world, rank, cap, recs[r])
    gathered = torch.stack(recs, dim=0).contiguous()
    o_s, o_i, o_c = backs[0].new_outputs(batch, k)
    backs[0].enqueue_merge_verified(gathered, world, batch, cap, k, min(k, n), o_s, o_i, o_c)
    torch.cuda.synchronize()
    per_rank_counts = [rec[:, 2 * cap].cpu().numpy().view(np.int32).reshape(batch, 2) for rec in recs]
    return o_s.cpu().numpy(), o_i.cpu().numpy(), o_c.cpu().numpy(), dq, per_rank_counts


@pytest.mark.parametrize("world,n,d,k", [(2, 24_001, 256, 50), (3, 40_000, 128, 100), (3, 30_000, 64, 7)])
def test_global_threshold_batch_records_equal_the_single_query_records(world, n, d, k):
    """svsb_batch_sample_tops -> (all-gather) -> svsb_batch_global_records -> (all-gather) ->
    svsb_enqueue_merge_batch_records: ONE filter threshold per query for all ranks, every rank re-scores only what can
    reach the global top k.  Verified answers must equal the per-query records' merge bit for bit and match the oracle."""
    torch = pytest.importorskip("torch")
    from svs_b200.sharded import CudaShardBackend, partition
    batch = 300
    m = oracle.synth_matrix_uniform(n, d, 8)
    m[11] = m[n - 5]                                           # exact tie across shards
    ids = np.cumsum(np.random.default_rng(3).integers(1, 4, size=n)).astype(np.int64)
    backs = []
    for r in range(world):
        b = CudaShardBackend(0)
        row0, cnt = partition(n, world, r)
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
        backs.append(b)
    qs = oracle.synth_queries(batch, d, 9)
    qs[2] = m[11]
    try:
        s, i, c, dq, prc = _global_batch(backs, world, n, qs, k)
        assert (c == k).all(), np.nonzero(c != k)[0][:10]       # random rows, random queries: every query verified
        recs = [b.new_records(batch, k) for b in backs]
        for r, b in enumerate(backs):
            for j in range(batch):
                b.enqueue_local(dq[j], k, recs[r][j])
            b.join()
        torch.cuda.synchronize()
        o_s, o_i, o_c = backs[0].new_outputs(batch, k)
        backs[0].enqueue_merge(torch.stack(recs, dim=0).contiguous(), world, batch, k, o_s, o_i, o_c)
        torch.cuda.synchronize()
        assert np.array_equal(s.view(np.uint32), o_s.cpu().numpy().view(np.uint32))
        assert np.array_equal(i, o_i.cpu().numpy()) and np.array_equal(c, o_c.cpu().numpy())
        for j in range(0, batch, 37):
            got = list(zip(s[j, :c[j]].tolist(), i[j, :c[j]].tolist()))
            oracle.compare_retrieval(got, oracle.superheavy(m, ids, qs[j], k), oracle.scores_of(m, qs[j]), ids)
        assert i[2, :2].tolist() == [int(ids[11]), int(ids[n - 5])]     # tie: ascending id, across shards
        assert (sum(p[:, 1].astype(np.int64) for p in prc) >= k).all()     # the ranks' verification counts add up to >= k
        assert all((p[:, 0] >= 0).all() and (p[:, 0] <= k).all() for p in prc)
        # truncated records: each rank ships at most `cap` entries.  A generous cap changes nothing; a cap below a
        # shard's share of the top k must be refused (-1) for exactly the queries where it mattered, never answered wrong.
        share = k / world
        for cap in (min(k, int(np.ceil(share + 6.0 * np.sqrt(share) + 4.0))), max(1, int(share))):
            if world * cap > 2048:
                continue
            s2, i2, c2, _, prc2 = _global_batch(backs, world, n, qs, k, cap=cap)
            ok = c2 == k
            assert set(np.unique(c2)) <= {-1, k}
            assert np.array_equal(s2[ok].view(np.uint32), s[ok].view(np.uint32)) and np.array_equal(i2[ok], i[ok])
            if cap > share + 1:
                assert ok.mean() > 0.95, (cap, ok.mean())
            else:
                assert (~ok).any()                          # some shard held more than k / world of some query's top k
            need = np.zeros(batch, dtype=bool)              # would the full answer have needed an entry a rank did not ship?
            top_rows = [set(i[j, :k].tolist()) for j in range(batch)]
            for r in range(world):
                row0, cnt = partition(n, world, r)
                mine = set(ids[row0:row0 + cnt].tolist())
                for j in range(batch):
                    need[j] |= len(top_rows[j] & mine) > cap
            assert not (ok & need).any()
    finally:
        for b in backs:
            b.close()


@pytest.mark.parametrize("world,n,d,k", [(2, 24_001, 256, 50), (4, 60_000, 128, 100)])
def test_batch_peer_exchange_virtual_ranks_equal_the_collective_form(world, n, d, k):
    """svsb_batch_peer: the whole batch with BOTH exchanges fused into the kernels (sample maxima and candidate records
    stored straight into every rank's batch window, consumers behind flag waits) -- `world` shard engines of this process,
    one stream each, stand in for the ranks.  Every rank must hold the answer of the collective form (stacked
    all-gathers), bit for bit; several batches in a row exercise the two window slots."""
    torch = pytest.importorskip("torch")
    from svs_b200.sharded import CudaShardBackend, partition
    batch = 260
    m = oracle.synth_matrix_uniform(n, d, 18)
    ids = np.cumsum(np.random.default_rng(4).integers(1, 4, size=n)).astype(np.int64)
    backs = []
    for r in range(world):
        b = CudaShardBackend(0)
        row0, cnt = partition(n, world, r)
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
        backs.append(b)
    try:
        probes = [b.batch_global_probe(k) for b in backs]
        assert all(p[0] for p in probes)
        f = max(min(1.0, p[1] / p[2]) for p in probes)
        lam = k * f
        rank = int(np.ceil(lam + 6.0 * np.sqrt(lam) + 4.0))
        norm = max(p[3] for p in probes)
        share = k / world
        cap = min(k, int(np.ceil(share + 6.0 * np.sqrt(share) + 4.0)))
        for r, b in enumerate(backs):
            b.batch_exchange_handle(world, r, 128)
        for b in backs:
            b.batch_exchange_connect_local(backs)
            b.batch_peer_prepare(batch, k)
        streams = [torch.cuda.Stream() for _ in range(world)]
        outs = [b.new_outputs(batch, k) for b in backs]
        for rep in range(5):
            qs = oracle.synth_queries(batch, d, 40 + rep)
            ref_s, ref_i, ref_c, dq, _ = _global_batch(backs, world, n, qs, k, cap=cap)
            torch.cuda.synchronize()
            for r, b in enumerate(backs):                      # every rank's whole batch is enqueued before any is awaited
                with torch.cuda.stream(streams[r]):
                    b.batch_peer(dq, k, norm, rank, cap, *outs[r], defer_merge=(rep % 2 == 1))
            if rep % 2 == 1:                                   # pipelined form: the merges are enqueued by the flush
                for r, b in enumerate(backs):
                    with torch.cuda.stream(streams[r]):
                        b.batch_peer_flush()
            torch.cuda.synchronize()
            for r in range(world):
                o_s, o_i, o_c = (t.cpu().numpy() for t in outs[r])
                assert np.array_equal(o_c, ref_c), (rep, r, np.nonzero(o_c != ref_c)[0][:8], o_c[:8])
                ok = ref_c == k
                assert ok.mean() > 0.9
                assert np.array_equal(o_s[ok].view(np.uint32), ref_s[ok].view(np.uint32)) and np.array_equal(o_i[ok], ref_i[ok])
            for j in range(0, batch, 61):
                if ref_c[j] == k:
                    got = list(zip(ref_s[j, :k].tolist(), ref_i[j, :k].tolist()))
                    oracle.compare_retrieval(got, oracle.superheavy(m, ids, qs[j], k), oracle.scores_of(m, qs[j]), ids)
        # a stream of three pipelined batches: the merge of each is enqueued behind the first phase of the next
        refs, dqs = [], []
        for rep in range(3):
            qs = oracle.synth_queries(batch, d, 60 + rep)
            ref_s, ref_i, ref_c, dq, _ = _global_batch(backs, world, n, qs, k, cap=cap)
            refs.append((ref_s, ref_i, ref_c)); dqs.append(dq.clone())
        torch.cuda.synchronize()
        outs3 = [[b.new_outputs(batch, k) for _ in range(3)] for b in backs]
        for rep in range(3):
            for r, b in enumerate(backs):
                with torch.cuda.stream(streams[r]):
                    b.batch_peer(dqs[rep], k, norm, rank, cap, *outs3[r][rep], defer_merge=True)
        for r, b in enumerate(backs):
            with torch.cuda.stream(streams[r]):
                b.batch_peer_flush()
        torch.cuda.synchronize()
        for rep in range(3):
            ref_s, ref_i, ref_c = refs[rep]
            ok = ref_c == k
            for r in range(world):
                o_s, o_i, o_c = (t.cpu().numpy() for t in outs3[r][rep])
                assert np.array_equal(o_c, ref_c), (rep, r)
                assert np.array_equal(o_s[ok].view(np.uint32), ref_s[ok].view(np.uint32)) and np.array_equal(o_i[ok], ref_i[ok])
    finally:
        for b in backs:
            b.batch_exchange_disconnect()
        for b in backs:
            b.close()


def test_global_threshold_batch_refuses_what_it_cannot_verify():
    """Rows stored in an order correlated with the queries (every shard's strided sample then over-represents the top) and
    a sample_rank far too small: the thresholds come out too high, the ranks' verification counts do not add up to k,
    and the merge reports count -1 for such queries -- on the verified ones the answer is still exact."""
    torch = pytest.importorskip("torch")
    from svs_b200.sharded import CudaShardBackend, partition
    world, n, d, k, batch = 2, 20_000, 64, 100, 32
    m = oracle.synth_matrix_uniform(n, d, 21)
    ids = np.arange(1, n + 1, dtype=np.int64)
    qs = oracle.synth_queries(batch, d, 22)
    backs = []
    for r in range(world):
        b = CudaShardBackend(0)
        row0, cnt = partition(n, world, r)
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
        backs.append(b)
    try:
        import os
        os.environ["SVSB_BATCH_GLOBAL_ANY_RANK"] = "1"         # let the test pass a rank below the statistical bound
        try:
            s, i, c, dq, prc = _global_batch(backs, world, n, qs, k, sample_rank=1)
        finally:
            del os.environ["SVSB_BATCH_GLOBAL_ANY_RANK"]
        # threshold = (largest sample value of all) - 2 eps: almost never k rows above it
        assert (c < 0).sum() >= batch // 2
        assert set(np.unique(c)) <= {-1, k}
        for j in np.nonzero(c == k)[0]:
            got = list(zip(s[j, :k].tolist(), i[j, :k].tolist()))
            oracle.compare_retrieval(got, oracle.superheavy(m, ids, qs[j], k), oracle.scores_of(m, qs[j]), ids)
    finally:
        for b in backs:
            b.close()


def test_merge_records_rank_merge_and_unsorted_fallback():
    """svsb_enqueue_merge_records on crafted records: lists sorted descending take the rank merge (one binary search per
    other list, no sort); a list that is NOT sorted makes the kernel fall back to the bitonic sort.  Both must return
    the k largest keys in order, with ragged counts and an empty list."""
    torch = pytest.importorskip("torch")
    from svs_b200.sharded import CudaShardBackend
    rng = np.random.default_rng(77)
    b = CudaShardBackend(0)
    b.load_rows(np.ones((4, 4), np.float32), np.arange(4, dtype=np.int64))      # the merge only needs an engine
    try:
        for world, batch, k, shuffle in ((3, 2, 50, False), (3, 2, 50, True), (8, 5, 100, False), (16, 1, 128, False), (2, 3, 1, True),
                                         (8, 9, 100, False), (3, 12, 50, True), (2, 8, 1, False)):   # batch >= 8: the small-record kernel
            rec = np.zeros((world, batch, 2 * k + 1), dtype=np.int64)
            want = []
            for q in range(batch):
                pool = []
                for l in range(world):
                    c = 0 if (l == 1 and world > 2) else int(rng.integers(1, k + 1))
                    keys = np.unique(rng.integers(1, 2 ** 62, size=c, dtype=np.int64))[::-1].copy()   # unique, descending
                    c = len(keys)
                    if shuffle:
                        rng.shuffle(keys)
                    ids = rng.integers(0, 2 ** 40, size=c, dtype=np.int64)
                    rec[l, q, :c] = keys
                    rec[l, q, k:k + c] = ids
                    rec[l, q, 2 * k] = c
                    pool += list(zip(keys.tolist(), ids.tolist()))
                pool.sort(reverse=True)
                want.append(pool[:k])
            o_s, o_i, o_c = b.new_outputs(batch, k)
            b.enqueue_merge(torch.from_numpy(rec).cuda(), world, batch, k, o_s, o_i, o_c)
            torch.cuda.synchronize()
            for q in range(batch):
                c = int(o_c[q])
                assert c == len(want[q])
                assert o_i[q, :c].cpu().numpy().tolist() == [i for _, i in want[q]], (world, batch, k, shuffle, q)
    finally:
        b.close()


def _two_backends(m, ids, world=2, timeout_ms=5000):
    import os
    from svs_b200.sharded import CudaShardBackend, partition
    os.environ["SVSB_XCHG_TIMEOUT_MS"] = str(timeout_ms)        # a protocol bug must fail the test, not hang the GPU
    backs = []
    for r in range(world):
        b = CudaShardBackend(0)
        row0, cnt = partition(len(m), world, r)
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
        backs.append(b)
    for r, b in enumerate(backs):
        assert len(b.exchange_handle(world, r)) == 64
    for b in backs:
        b.exchange_connect_local(backs)
    return backs


def test_peer_exchange_pipelined_two_virtual_ranks_match_the_oracle():
    """The fused exchange (selection epilogue pushes the record into every rank's window; the merge kernel waits
    for the flags) with two shard engines on ONE device: windows connected by plain pointers, similarity passes on
    the shared stream, selection + push + waiting merge on each engine's side stream.  40 queries per k cycle
    through the 4 window slots ten times; every rank must hold the identical, oracle-matching answer."""
    torch = pytest.importorskip("torch")
    n, d = 30_001, 256
    m = oracle.synth_matrix_uniform(n, d, 15)
    m[7] = m[n - 3]                                            # exact tie across shards
    ids = np.cumsum(np.random.default_rng(12).integers(1, 4, size=n)).astype(np.int64)
    backs = _two_backends(m, ids)
    qs = oracle.synth_queries(40, d, 16)
    qs[1] = m[7]
    try:
        dq = backs[0].device_queries(qs)
        for k in (1, 100, 1500, 2048):                         # 2 * 1500 > 2048: the merge's scratch path
            outs = [b.new_outputs(len(qs), k) for b in backs]
            for j in range(len(qs)):
                for b, (o_s, o_i, o_c) in zip(backs, outs):
                    b.enqueue_query_peer(dq[j], k, o_s[j], o_i[j], o_c[j], time_kernel=(k == 100), pipelined=True)
            for b in backs:
                b.join()
            torch.cuda.synchronize()
            res = [(o_s.cpu().numpy(), o_i.cpu().numpy(), o_c.cpu().numpy()) for o_s, o_i, o_c in outs]
            assert np.array_equal(res[0][0].view(np.uint32), res[1][0].view(np.uint32))      # same bits on both ranks
            assert np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[0][2], res[1][2])
            s, i, c = res[0]
            assert (c == min(k, n)).all()
            for j in range(0, len(qs), 3):
                got = list(zip(s[j, :c[j]].tolist(), i[j, :c[j]].tolist()))
                oracle.compare_retrieval(got, oracle.superheavy(m, ids, qs[j], k), oracle.scores_of(m, qs[j]), ids)
            if k >= 2:
                assert i[1, :2].tolist() == [int(ids[7]), int(ids[n - 3])]                   # tie: ascending id
            if k == 100:
                assert backs[0].collect_kernel_ms() > 0 and backs[1].collect_kernel_ms() > 0
    finally:
        for b in backs:
            b.close()


def test_peer_exchange_synchronous_query_from_two_threads_and_an_empty_shard():
    """svsb_query_peer (host buffers, result written into pinned host memory by the merge kernel) called SPMD from
    one thread per virtual rank; 3 ranks over 2 rows leave the last shard empty (count-0 record)."""
    pytest.importorskip("torch")
    import threading
    n, d, k = 20_000, 128, 50
    m = oracle.synth_matrix_uniform(n, d, 25)
    ids = np.arange(10, 10 + n, dtype=np.int64)
    qs = oracle.synth_queries(12, d, 26)
    for rows, world in ((n, 2), (2, 3)):
        backs = _two_backends(m[:rows], ids[:rows], world)
        results = [[None] * len(qs) for _ in range(world)]
        errors = []

        def work(r):
            try:
                for j, q in enumerate(qs):
                    results[r][j] = backs[r].query_peer(q, k)
            except Exception as ex:                            # pragma: no cover - reported below
                errors.append(ex)

        try:
            threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
            for t in threads:
                t.start()
            for t in threads:
                t.join(timeout=120)
            assert not errors, errors
            assert all(not t.is_alive() for t in threads), "a rank is stuck waiting for a peer's record"
            for j, q in enumerate(qs):
                s0, i0 = results[0][j]
                for r in range(1, world):
                    assert np.array_equal(s0.view(np.uint32), results[r][j][0].view(np.uint32))
                    assert np.array_equal(i0, results[r][j][1])
                got = list(zip(s0.tolist(), i0.tolist()))
                oracle.compare_retrieval(got, oracle.superheavy(m[:rows], ids[:rows], q, k), oracle.scores_of(m[:rows], q), ids[:rows])
        finally:
            for b in backs:
                b.close()


def test_peer_exchange_submit_wait_keeps_three_queries_in_flight():
    """svsb_query_peer_submit / _wait: host buffers in and out with up to 3 queries pending per rank.  Submits are
    non-blocking, so one host thread drives all virtual ranks SPMD; every rank must get the bits the single-device
    engine computes for the whole matrix."""
    pytest.importorskip("torch")
    import svs_b200
    n, d = 25_000, 192
    m = oracle.synth_matrix_uniform(n, d, 45)
    ids = np.arange(7, 7 + n, dtype=np.int64)
    qs = oracle.synth_queries(30, d, 46)
    with svs_b200.Engine([0]) as one:
        one.load(m, ids)
        want = {k: [one.query(q, k) for q in qs] for k in (10, 100, 1200)}
    oracle.compare_retrieval(list(zip(*[x.tolist() for x in want[100][0]])), oracle.superheavy(m, ids, qs[0], 100),
                             oracle.scores_of(m, qs[0]), ids)
    for world in (2, 3):
        backs = _two_backends(m, ids, world)
        try:
            for k in (10, 100, 1200):
                pend, got = [], [[] for _ in backs]
                for q in qs:
                    pend.append([b.query_peer_submit(q, k) for b in backs])
                    if len(pend) == 3:
                        with pytest.raises(svs_b200.EngineError, match="pending already"):
                            backs[0].query_peer_submit(q, k)                 # a 4th is refused (nothing enqueued), not queued
                        for r, b in enumerate(backs):
                            got[r].append(b.query_peer_wait(pend[0][r], k))
                        pend.pop(0)
                for p in pend:
                    for r, b in enumerate(backs):
                        got[r].append(b.query_peer_wait(p[r], k))
                for r in range(world):
                    assert len(got[r]) == len(qs)
                    for a, w in zip(got[r], want[k]):
                        assert np.array_equal(a[0].view(np.uint32), w[0].view(np.uint32)) and np.array_equal(a[1], w[1])
        finally:
            for b in backs:
                b.close()


def test_peer_exchange_missing_peer_times_out_instead_of_hanging():
    """A rank whose peer never issues the query must get an error after SVSB_XCHG_TIMEOUT_MS, not a hung GPU."""
    pytest.importorskip("torch")
    import time
    import svs_b200
    n, d = 4_000, 64
    m = oracle.synth_matrix_uniform(n, d, 35)
    ids = np.arange(n, dtype=np.int64)
    backs = _two_backends(m, ids, timeout_ms=300)
    try:
        t0 = time.time()
        with pytest.raises(svs_b200.EngineError, match="did not arrive"):
            backs[0].query_peer(oracle.synth_queries(1, d, 36)[0], 10)      # rank 1 never calls
        assert 0.25 < time.time() - t0 < 5.0
    finally:
        for b in backs:
            b.close()


@pytest.mark.parametrize("exchange", ["peer", "collective"])
def test_world_size_one_process_group_runs_the_real_collective(exchange):
    torch = pytest.importorskip("torch")
    import os
    import torch.distributed as dist
    from svs_b200.sharded import ShardedRetriever
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ["MASTER_PORT"] = "29581" if exchange == "peer" else "29582"
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        sr = ShardedRetriever(0, 1, 0, exchange=exchange)
        assert sr.exchange == exchange
        sr.load_synthetic(50_000, 1536, seed=3, id0=1, id_step=1)
        rows, ids = sr.backend.engine.read_rows(0, 50_000)
        qs = oracle.synth_queries(11, 1536, 7)
        for q in qs[:3]:
            oracle.compare_retrieval(sr.retrieve(q, 100), oracle.superheavy(rows, ids, q, 100), oracle.scores_of(rows, q), ids)
        sr.set_queries(qs)
        ms = sr.run_queries(100, 11, time_gemv=True)
        assert ms > 0
        many = sr.retrieve_many(qs, 100)                        # batched: coarse pass + refine, all-gather, merge
        assert sr.last_fallbacks == 0
        for j in (0, 5, 10):
            assert many[j] == sr.retrieve(qs[j], 100)
        # page-locked tensor in, page-locked buffers out: the same bits as the pageable form
        ps, pi, pc = sr.retrieve_many_pinned(torch.from_numpy(qs).pin_memory(), 100)
        as_, ai, ac = sr.retrieve_many_arrays(qs, 100)
        assert np.array_equal(ps.view(np.uint32), as_.view(np.uint32)) and np.array_equal(pi, ai) and np.array_equal(pc, ac)
        with pytest.raises(ValueError):
            sr.retrieve_many_pinned(torch.from_numpy(qs), 100)  # not pinned
        sr.close()
    finally:
        dist.destroy_process_group()


def _peer_worker(rank, world, port, mats, ids, qs, k, ret):
    import torch
    import torch.distributed as dist
    from svs_b200.sharded import ShardedRetriever
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["SVSB_XCHG_TIMEOUT_MS"] = "10000"               # a protocol bug must fail the test, not hang the GPU
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sr = ShardedRetriever(rank, world, rank, exchange="peer")
        out = []
        for m in mats:                                          # the second matrix is a reload over the same windows
            sr.load_global(m, ids)
            single = [sr.retrieve(q, k) for q in qs[:3]]
            s, i = sr.wait(sr.submit(qs[3], k))
            many = sr.retrieve_many(qs, k)
            out.append((single, [(float(a), int(b)) for a, b in zip(s, i)], many, sr._batch_peer_ready))
        sr.close()
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def test_peer_windows_over_cuda_ipc_in_two_processes():
    """Both peer windows opened over real CUDA IPC: two processes, one GPU each, the query exchange for retrieve and
    submit / wait, the batch window for retrieve_many.  Every rank must hold the oracle's answer, before and after a
    reload."""
    torch = pytest.importorskip("torch")
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (NCCL runs one rank per GPU)")
    n, d, k = 60_000, 128, 100
    mats = [oracle.synth_matrix_uniform(n, d, seed) for seed in (71, 72)]
    ids = np.cumsum(np.random.default_rng(73).integers(1, 4, size=n)).astype(np.int64)
    qs = oracle.synth_queries(64, d, 74)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_peer_worker, args=(2, port, mats, ids, qs, k, ret), nprocs=2, join=True)
    assert ret[0] == ret[1]                                     # every rank holds the same answers
    for m, (single, waited, many, batch_peer) in zip(mats, ret[0]):
        assert batch_peer                                       # the batch went through the batch window
        for q, got in zip(qs[:3], single):
            oracle.compare_retrieval(got, oracle.superheavy(m, ids, q, k), oracle.scores_of(m, q), ids)
        oracle.compare_retrieval(waited, oracle.superheavy(m, ids, qs[3], k), oracle.scores_of(m, qs[3]), ids)
        assert len(many) == len(qs)
        for q, got in zip(qs, many):
            oracle.compare_retrieval(got, oracle.superheavy(m, ids, q, k), oracle.scores_of(m, q), ids)
