"""GPU: the one-process-per-GPU deployment above 2048 results per query.  svsb_enqueue_local_topk fully sorts a shard's
keys into one record, svsb_enqueue_merge_sorted_records rank-merges the gathered records, and ShardedRetriever routes
retrieve, submit / wait, retrieve_many and retrieve_many_pinned through them.  The answer must be what one
single-device engine over the whole matrix returns, bit for bit, as tests/test_gpu_multi.py checks for the in-process
multi-device engine."""
import os
import socket

import numpy as np
import pytest

from _util import oracle

pytestmark = pytest.mark.gpu


def _backends(m, ids, world):
    from svs_b200.sharded import CudaShardBackend, partition
    backs = []
    for r in range(world):
        b = CudaShardBackend(0)
        row0, cnt = partition(len(m), world, r)
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + cnt]), np.ascontiguousarray(ids[row0:row0 + cnt]))
        backs.append(b)
    return backs


def _same(got, want):
    assert len(got[0]) == len(want[0])
    assert np.array_equal(np.asarray(got[0], np.float32).view(np.uint32), np.asarray(want[0], np.float32).view(np.uint32))
    assert np.array_equal(np.asarray(got[1]), np.asarray(want[1]))


@pytest.mark.parametrize("world,n,d", [(2, 50_000, 192), (3, 50_001, 190)])
def test_virtual_ranks_large_k_records_merge_to_the_single_device_answer(world, n, d):
    """`world` shard engines on one device stand in for the ranks; the all-gather is a torch.stack."""
    torch = pytest.importorskip("torch")
    import svs_b200
    m = oracle.synth_matrix_uniform(n, d, 81)
    m[9] = m[n - 4]                                            # an exact tie across shards
    ids = np.cumsum(np.random.default_rng(82).integers(1, 4, size=n)).astype(np.int64)
    qs = oracle.synth_queries(3, d, 83)
    qs[1] = m[9]
    ks = (2049, 5000, n, 10 ** 9)
    with svs_b200.Engine([0]) as one:
        one.load(m, ids)
        want = {k: [one.query(q, k) for q in qs] for k in ks}
    backs = _backends(m, ids, world)
    try:
        dq = backs[0].device_queries(qs)
        for k in ks:
            kk = min(k, n)
            cap = min(kk, -(-n // world))
            for j in range(len(qs)):
                recs = [b.new_records(1, cap) for b in backs]
                for b, rec in zip(backs, recs):
                    b.enqueue_local(dq[j], cap, rec[0], time_kernel=(k == 5000))
                    b.join()
                torch.cuda.synchronize()
                gathered = torch.stack(recs, dim=0).contiguous()  # [world, 1, 2 cap + 1]: what all_gather yields
                o_s, o_i, o_c = backs[0].new_outputs(1, kk)
                backs[0].enqueue_merge_sorted(gathered, world, cap, kk, o_s[0], o_i[0], o_c[0])
                torch.cuda.synchronize()
                assert int(o_c[0]) == kk
                _same((o_s[0].cpu().numpy(), o_i[0].cpu().numpy()), want[k][j])
            if k == 5000:
                assert backs[0].collect_kernel_ms() > 0
        s, i = want[2049][1]
        assert i[:2].tolist() == [int(ids[9]), int(ids[n - 4])]           # tie: ascending id, across shards
        oracle.compare_retrieval(list(zip(s.tolist(), i.tolist())), oracle.superheavy(m, ids, qs[1], 2049),
                                 oracle.scores_of(m, qs[1]), ids)
        # a k <= 2048 record on the same slot afterwards is unchanged by the large-k calls before it
        rec_small = [b.new_records(1, 100) for b in backs]
        for b, rec in zip(backs, rec_small):
            b.enqueue_local(dq[0], 100, rec[0])
            b.join()
        o_s, o_i, o_c = backs[0].new_outputs(1, 100)
        backs[0].enqueue_merge(torch.stack(rec_small, dim=0).contiguous(), world, 1, 100, o_s, o_i, o_c)
        torch.cuda.synchronize()
        _same((o_s[0].cpu().numpy(), o_i[0].cpu().numpy()), (want[2049][0][0][:100], want[2049][0][1][:100]))
    finally:
        for b in backs:
            b.close()


def test_merge_sorted_records_refuses_a_truncated_record():
    """A record whose count says it lost entries (bit 30, or above cap) cannot be merged exactly: count -1."""
    torch = pytest.importorskip("torch")
    from svs_b200._lib import EngineError
    from svs_b200.sharded import CudaShardBackend
    b = CudaShardBackend(0)
    b.load_rows(np.ones((4, 4), np.float32), np.arange(4, dtype=np.int64))      # the merge only needs an engine
    try:
        cap, k = 3000, 5000
        rng = np.random.default_rng(5)
        rec = np.zeros((2, 2 * cap + 1), dtype=np.int64)
        pool = []
        for l, c in enumerate((cap, 1234)):
            keys = np.unique(rng.integers(1, 2 ** 62, size=c, dtype=np.int64))[::-1].copy()
            c = len(keys)
            rec[l, :c] = keys
            rec[l, cap:cap + c] = np.arange(c) + 10_000 * l
            rec[l, 2 * cap] = c
            pool += list(zip(keys.tolist(), (np.arange(c) + 10_000 * l).tolist()))
        pool.sort(reverse=True)
        o_s, o_i, o_c = b.new_outputs(1, k)
        b.enqueue_merge_sorted(torch.from_numpy(rec).cuda(), 2, cap, k, o_s[0], o_i[0], o_c[0])
        torch.cuda.synchronize()
        assert int(o_c[0]) == min(k, len(pool))
        assert o_i[0, :int(o_c[0])].cpu().numpy().tolist() == [i for _, i in pool[:k]]
        for bad in (rec[1, 2 * cap] | (1 << 30), cap + 1, -1):
            r2 = rec.copy()
            r2[1, 2 * cap] = bad
            b.enqueue_merge_sorted(torch.from_numpy(r2).cuda(), 2, cap, k, o_s[0], o_i[0], o_c[0])
            torch.cuda.synchronize()
            assert int(o_c[0]) == -1
        with pytest.raises(EngineError):
            b.enqueue_merge_sorted(torch.from_numpy(rec).cuda(), 2, 0, k, o_s[0], o_i[0], o_c[0])
    finally:
        b.close()


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


@pytest.mark.parametrize("exchange", ["peer", "collective"])
def test_world_size_one_process_group_answers_full_rankings(exchange):
    torch = pytest.importorskip("torch")
    import torch.distributed as dist
    import svs_b200
    from svs_b200.sharded import ShardedRetriever
    n, d = 30_000, 192
    m = oracle.synth_matrix_uniform(n, d, 91)
    ids = np.arange(3, 3 + n, dtype=np.int64)
    qs = oracle.synth_queries(4, d, 92)
    with svs_b200.Engine([0]) as one:
        one.load(m, ids)
        want = [one.query(q, n) for q in qs]
        want5k = one.query(qs[0], 5000)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ["MASTER_PORT"] = str(_free_port())
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        sr = ShardedRetriever(0, 1, 0, exchange=exchange)
        assert sr.exchange == exchange
        sr.load_global(m, ids)
        _same(sr.retrieve_arrays(qs[0], n), want[0])
        _same(sr.retrieve_arrays(qs[0], 5000), want5k)
        _same(sr.retrieve_arrays(qs[1], 10 ** 9), want[1])
        got = sr.retrieve(qs[2], n)
        _same(([s for s, _ in got], [i for _, i in got]), want[2])
        h = sr.submit(qs[3], n)
        assert h[0] == "done"
        _same(sr.wait(h), want[3])
        s, i, c = sr.retrieve_many_arrays(qs, n)
        assert (c == n).all()
        for j in range(len(qs)):
            _same((s[j], i[j]), want[j])
        ps, pi, pc = sr.retrieve_many_pinned(torch.from_numpy(qs).pin_memory(), n)
        assert np.array_equal(ps.view(np.uint32), s.view(np.uint32)) and np.array_equal(pi, i) and np.array_equal(pc, c)
        many = sr.retrieve_many(qs[:2], n)
        assert many[1] == [(float(a), int(b)) for a, b in zip(*want[1])]
        assert sr.retrieve(qs[0], 100) == sr.retrieve(qs[0], n)[:100]       # the k <= 2048 path agrees
        sr.close()
    finally:
        dist.destroy_process_group()


def _two_gpu_worker(rank, world, port, mats, ids, qs, ret):
    import torch
    import torch.distributed as dist
    from svs_b200.sharded import ShardedRetriever
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sr = ShardedRetriever(rank, world, rank, exchange="peer")
        out = []
        for m in mats:                                          # the second matrix is a reload with another N
            sr.load_global(m, ids[:len(m)])
            out.append([sr.retrieve(q, len(m)) for q in qs])
        sr.close()
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def test_full_ranking_in_two_processes_before_and_after_a_reload():
    torch = pytest.importorskip("torch")
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (NCCL runs one rank per GPU)")
    d = 128
    mats = [oracle.synth_matrix_uniform(n, d, seed) for n, seed in ((40_000, 95), (25_001, 96))]
    ids = np.cumsum(np.random.default_rng(97).integers(1, 4, size=40_000)).astype(np.int64)
    qs = oracle.synth_queries(2, d, 98)
    ret = mp.Manager().dict()
    mp.spawn(_two_gpu_worker, args=(2, _free_port(), mats, ids, qs, ret), nprocs=2, join=True)
    assert ret[0] == ret[1]                                     # every rank holds the same answers
    for m, lists in zip(mats, ret[0]):
        for q, got in zip(qs, lists):
            assert len(got) == len(m)
            oracle.compare_retrieval(got, oracle.superheavy(m, ids[:len(m)], q, len(m)), oracle.scores_of(m, q), ids[:len(m)])
