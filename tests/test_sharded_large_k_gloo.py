"""ShardedRetriever above 2048 results per query on CPU: world-size 2 and 3 `gloo` runs with NumPy stand-ins for the
shard compute.  Covers the host logic of the large-k path: the record capacity every rank derives from `partition`, the
agreement on the local phase before the collective, the all-gather of the sorted records, the rank merge, the one buffer
set keyed by that capacity, and every public entry point (retrieve, submit / wait, retrieve_many) under both exchanges."""
import os
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from _util import oracle
from test_sharded_gloo import NumpyPeerBackend, NumpyShardBackend, _free_port, key_score

from svs_b200._lib import SVSB_E_NOMEM, EngineError
from svs_b200.sharded import ShardedRetriever


class SortedMergeMixin:
    """svsb_enqueue_merge_sorted_records restated in NumPy: records [n_lists][2 * cap + 1], counts in the low 32 bits
    of the last word; a count outside [0, cap] makes the merge answer -1."""

    def enqueue_merge_sorted(self, gathered, n_lists, cap, k, out_scores, out_ids, out_count):
        g = gathered.numpy().reshape(n_lists, 2 * cap + 1)
        keys, ids = [], []
        for l in range(n_lists):
            c = int(np.int32(np.uint32(int(g[l, 2 * cap]) & 0xFFFFFFFF)))
            if c < 0 or c > cap:
                out_count.numpy()[...] = -1
                return
            kl = g[l, :c].view(np.uint64)
            assert (np.diff(kl.astype(object)) < 0).all() if c > 1 else True     # the local phase wrote it sorted
            keys.append(kl); ids.append(g[l, cap:cap + c])
        keys, ids = np.concatenate(keys), np.concatenate(ids)
        order = np.argsort(keys)[::-1][:k]
        out_scores.numpy()[:len(order)] = key_score(keys[order])
        out_ids.numpy()[:len(order)] = ids[order]
        out_count.numpy()[...] = len(order)


class LargeKBackend(SortedMergeMixin, NumpyShardBackend):
    fail_above = None                          # k above which enqueue_local refuses, as a failed sort-buffer allocation

    def enqueue_local(self, q, k, record_row, time_kernel=False, seq=0):
        if self.fail_above is not None and k > self.fail_above:
            raise EngineError(SVSB_E_NOMEM, "cudaMalloc(&sortbuf, (size_t)need * 8): out of memory")
        super().enqueue_local(q, k, record_row, time_kernel, seq)


class LargeKPeerBackend(SortedMergeMixin, NumpyPeerBackend):
    pass


def _run(fn, world, args, timeout=180):
    """Spawn `world` ranks; a rank blocked in a collective fails the test instead of hanging it."""
    ctx = mp.start_processes(fn, args=(world, _free_port(), *args), nprocs=world, join=False, start_method="spawn")
    deadline = time.time() + timeout
    while not ctx.join(timeout=max(0.1, deadline - time.time())):
        if time.time() > deadline:
            for p in ctx.processes:
                p.terminate()
            pytest.fail("a rank did not finish: blocked in a collective?")


def _init(rank, world, port):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _data(n, d, seed):
    m = oracle.synth_matrix_normal(n, d, seed)
    m[5] = m[n - 2]                                            # an exact tie across the two ends (different shards)
    ids = np.cumsum(np.random.default_rng(seed + 1).integers(1, 4, size=n)).astype(np.int64)
    return m, ids


def _check(got, m, ids, q, n):
    want = oracle.superheavy(m, ids, q, n)
    assert len(got) == len(want) == min(n, len(m))
    oracle.compare_retrieval(got, want, oracle.scores_of(m, q), ids)


def _worker(rank, world, port, exchange, ret):
    _init(rank, world, port)
    try:
        d = 16
        n1, n2 = 5003, 4100
        m, ids = _data(n1, d, 3)
        be = LargeKPeerBackend() if exchange == "peer" else LargeKBackend()
        sr = ShardedRetriever(rank, world, backend=be)
        assert sr.exchange == exchange
        sr.load_global(m, ids)
        qs = oracle.synth_queries(5, d, 4, "normal")
        qs[1] = m[5]                                           # rows 5 and n - 2 tie at the top
        out = []
        per = -(-n1 // world)
        for n in (2049, 5000, n1, 10 ** 9):
            for q in qs[:2]:
                got = sr.retrieve(q, n)
                _check(got, m, ids, q, n)
                out.append(got)
            assert sr._big[0] == min(n, per)                   # one buffer set, keyed by the record capacity
        assert [i for _, i in sr.retrieve(qs[1], 2049)[:2]] == [int(ids[5]), int(ids[n1 - 2])]   # tie: ascending id
        assert sr.retrieve(qs[0], 10) == sr.retrieve(qs[0], 3000)[:10]      # the k <= 2048 path agrees
        # submit / wait: answered synchronously
        h = sr.submit(qs[2], 3000)
        assert h[0] == "done"
        s, i = sr.wait(h)
        got = [(float(a), int(b)) for a, b in zip(s, i)]
        _check(got, m, ids, qs[2], 3000)
        out.append(got)
        # retrieve_many: one large-k query at a time into (b, k) outputs
        s, i, c = sr.retrieve_many_arrays(qs[:3], 2500)
        assert s.shape == (3, 2500) and i.shape == (3, 2500) and (c == 2500).all()
        many = sr.retrieve_many(qs[:3], 10 ** 9)
        for j in range(3):
            assert [(float(a), int(b)) for a, b in zip(s[j], i[j])] == sr.retrieve(qs[j], 2500)
            _check(many[j], m, ids, qs[j], n1)
        out.append(many)
        # a reload that changes N, and with it the record capacity
        m2, ids2 = _data(n2, d, 7)
        sr.load_global(m2, ids2)
        assert sr._big is None                                 # dropped on reload
        for n in (2049, 10 ** 9):
            got = sr.retrieve(qs[3], n)
            _check(got, m2, ids2, qs[3], n)
            out.append(got)
        assert sr._big[0] == min(n2, -(-n2 // world))
        # N < world: some shards are empty; the clipped k is small and takes the ordinary path
        sr.load_global(m2[:world - 1], ids2[:world - 1])
        got = sr.retrieve(m2[0], 10 ** 9)
        _check(got, m2[:world - 1], ids2[:world - 1], m2[0], 10 ** 9)
        out.append(got)
        ret[rank] = out
        dist.barrier()
        sr.close()
        assert sr._big is None
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("exchange", ["collective", "peer"])
@pytest.mark.parametrize("world", [2, 3])
def test_large_k_retrieve_matches_the_oracle_on_every_rank(world, exchange):
    ret = mp.Manager().dict()
    _run(_worker, world, (exchange, ret))
    assert len(ret) == world
    for r in range(1, world):
        assert ret[r] == ret[0]                                # every rank holds the identical answer


def _failing_worker(rank, world, port, ret):
    _init(rank, world, port)
    try:
        d = 8
        m, ids = _data(9000, d, 11)                         # records of 3000 or more entries: the full sort
        be = LargeKBackend()
        if rank == world - 1:
            be.fail_above = 2048                               # this rank cannot allocate its sort buffer
        sr = ShardedRetriever(rank, world, backend=be)
        sr.load_global(m, ids)
        q = oracle.synth_queries(1, d, 12, "normal")[0]
        with pytest.raises(EngineError, match="out of memory") as info:
            sr.retrieve(q, 3000)
        assert info.value.code == SVSB_E_NOMEM
        with pytest.raises(EngineError, match="out of memory"):
            sr.retrieve_many(q[None, :], 10 ** 9)
        got = sr.retrieve(q, 100)                              # the ranks are still in step
        _check(got, m, ids, q, 100)
        ret[rank] = (str(info.value), got)
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_a_refused_local_phase_raises_the_same_error_on_every_rank(world):
    ret = mp.Manager().dict()
    _run(_failing_worker, world, (ret,))
    assert len(ret) == world
    for r in range(1, world):
        assert ret[r] == ret[0]
