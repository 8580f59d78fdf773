"""GPU: pairwise top pairs of the one-process-per-GPU deployment (include/svsb200.h svsb_pairs_*).  Virtual ranks: 2, 3, 4
and 8 single-device shard engines in one process, on distinct GPUs when visible, otherwise all on device 0, connected
with svsb_pairs_connect_local and driven through the C ABI rank by rank (no rank waits on another, so one thread does);
the all-gather is a concatenation.  Every rank's merged answer must equal Engine([0]).top_pairs over the global matrix
bit for bit (scores as uint32, ids, order).  ShardedRetriever.top_pairs runs through a real NCCL collective on a
world-size-1 group, and over real CUDA IPC handles in a 2-process group when two GPUs are visible."""
import os
import socket

import numpy as np
import pytest

from _util import oracle

pytestmark = pytest.mark.gpu

WORLDS = (2, 3, 4, 8)


def _devices(count):
    import torch
    have = max(torch.cuda.device_count(), 1)
    return [i % have for i in range(count)]


@pytest.fixture(scope="module")
def ranks():
    import svs_b200
    from svs_b200.sharded import CudaShardBackend
    one = svs_b200.Engine([0])
    backs = {w: [CudaShardBackend(d) for d in _devices(w)] for w in WORLDS}
    yield one, backs
    one.close()
    for bs in backs.values():
        for b in bs:
            b.pairs_disconnect()
    for bs in backs.values():
        for b in bs:
            b.close()


def _unit(rng, shape, dist):
    m = rng.random(shape, dtype=np.float32) if dist == "uniform" else rng.standard_normal(shape).astype(np.float32)
    m /= np.maximum(np.sqrt((m * m).sum(axis=1)), 1e-12)[:, None]
    return m


def _split(n_rows, world):
    from svs_b200.sharded import partition
    return [partition(n_rows, world, r)[1] for r in range(world)]


def _load(backs, m, ids, rows=None):
    """Disconnect, load each rank's slice (rows[r] rows, default: the sharded partition), export, connect.
    Returns the agreed max_row_norm."""
    from svs_b200 import EngineError
    rows = rows or _split(len(m), len(backs))
    for b in backs:
        b.pairs_disconnect()
    row0 = 0
    for b, c in zip(backs, rows):
        b.set_shard(row0)
        b.load_rows(np.ascontiguousarray(m[row0:row0 + c]), np.ascontiguousarray(ids[row0:row0 + c]))
        row0 += c
    got = [b.pairs_export() for b in backs]
    for _desc, status, message, _dev in got:
        if status:
            raise EngineError(status, message)
    for r, b in enumerate(backs):
        b.pairs_connect_local(len(backs), r, backs)
    return max(1.0 + g[3] for g in got)


def _top_pairs(backs, n_rows, n, norm):
    """The protocol of ShardedRetriever.top_pairs with the collectives replaced by concatenations: every rank's answer."""
    import torch
    from svs_b200 import EngineError
    n = min(n, n_rows * (n_rows - 1) // 2)
    if n <= 0:
        return [[] for _ in backs]
    owns, counts = [], []
    for b in backs:
        own = b.new_pair_lists(n)
        status, message, count = b.pairs_local(n, norm, own)
        if status:
            raise EngineError(status, message)
        owns.append(own)
        counts.append(count)
    stride = max(1, max(counts))
    answers = []
    for b in backs:
        lists = tuple(torch.cat([o[i][:, :stride].to(b.device) for o in owns]).contiguous() for i in range(3))
        out = b.new_pair_lists(n)
        assert b.pairs_merge(lists, counts, n, out) == n
        s, a, c = (x[0].cpu().numpy() for x in out)
        answers.append([(float(x), int(y), int(z)) for x, y, z in zip(s, a, c)])
    return answers


def _assert_same(got, want, what):
    assert len(got) == len(want), what
    gs = np.array([s for s, _, _ in got], np.float32)
    ws = np.array([s for s, _, _ in want], np.float32)
    assert np.array_equal(gs.view(np.uint32), ws.view(np.uint32)), what
    assert [(a, b) for _, a, b in got] == [(a, b) for _, a, b in want], what


def _check_all(backs, m, ids, n, want, what, rows=None):
    norm = _load(backs, m, ids, rows)
    for r, got in enumerate(_top_pairs(backs, len(m), n, norm)):
        _assert_same(got, want, (what, r))


@pytest.mark.parametrize("n_rows,d,n,dist", [
    (4, 3, 10, "normal"),               # the shapes of test_gpu_pairs_multi.py
    (300, 64, 50, "normal"),
    (1500, 96, 1000, "uniform"),
    (4875, 1536, 10000, "uniform"),
    (5000, 256, 100, "normal"),
    (3001, 100, 1, "normal"),
    (1001, 64, 300, "normal"),
    (20_011, 96, 5000, "uniform"),
    (5, 16, 10, "normal"),
])
def test_sharded_top_pairs_equal_the_single_device_engine(ranks, n_rows, d, n, dist):
    one, backs = ranks
    rng = np.random.default_rng(n_rows + d)
    m = _unit(rng, (n_rows, d), dist)
    ids = np.cumsum(rng.integers(1, 4, size=n_rows)).astype(np.int64)
    one.load(m, ids)
    want = one.top_pairs(n)
    oracle.compare_pairs(want, oracle.top_pairwise(m, ids, n), np.dot(m, m.T), ids)
    for w, bs in backs.items():
        _check_all(bs, m, ids, n, want, (w, n_rows, d, n))


def test_one_row_and_empty_shards(ranks):
    one, backs = ranks
    rng = np.random.default_rng(11)
    m = _unit(rng, (1400, 32), "normal")
    ids = np.arange(3, 1403, dtype=np.int64)
    one.load(m, ids)
    want = one.top_pairs(700)
    splits = {2: [0, 1400], 3: [1, 0, 1399], 4: [700, 0, 1, 699], 8: [0, 1, 1300, 0, 1, 0, 97, 1]}
    for w, bs in backs.items():
        _check_all(bs, m, ids, 700, want, w, rows=splits[w])


def test_identical_rows_in_different_shards_come_out_in_row_order(ranks):
    one, backs = ranks
    rng = np.random.default_rng(3)
    n_rows = 2500
    m = _unit(rng, (n_rows, 48), "normal")
    dup = [10, 11, 1300, 2490]
    for r in dup[:-1]:
        m[r] = m[dup[-1]]
    ids = np.arange(100, 100 + n_rows, dtype=np.int64)
    one.load(m, ids)
    want = one.top_pairs(8)
    assert [(a - 100, b - 100) for _, a, b in want[:6]] == [(dup[a], dup[b]) for a in range(4) for b in range(a + 1, 4)]
    for w, bs in backs.items():
        _check_all(bs, m, ids, 8, want, w)


def test_edge_cases_and_a_reload_between_calls(ranks):
    import ctypes as C
    one, backs = ranks
    rng = np.random.default_rng(4)
    m = _unit(rng, (50, 16), "normal")
    ids = np.arange(50, dtype=np.int64)
    one.load(m, ids)
    everything = one.top_pairs(10 ** 6)
    assert len(everything) == 50 * 49 // 2
    m2 = _unit(rng, (3000, 64), "uniform")
    ids2 = np.arange(7, 3007, dtype=np.int64)
    one.load(m2, ids2)
    want2 = one.top_pairs(400)
    for w, bs in backs.items():
        norm = _load(bs, m, ids)
        for r, got in enumerate(_top_pairs(bs, 50, 10 ** 6, norm)):   # n above all pairs: clipped to the global count
            _assert_same(got, everything, (w, r))
        cnt = C.c_int64(-1)
        assert bs[0]._lib.svsb_pairs_local(bs[0].engine._h, None, 0, C.c_float(norm), None, None, None, C.byref(cnt)) == 0
        assert cnt.value == 0                                            # n = 0: nothing
        _check_all(bs, m2, ids2, 400, want2, w)                          # a reload re-exports
        norm = _load(bs, m[:1], ids[:1])
        assert _top_pairs(bs, 1, 5, norm) == [[] for _ in bs]
        for b in bs:                                                     # one global row: no pairs on any rank
            own = b.new_pair_lists(1)
            assert b.pairs_local(5, norm, own)[::2] == (0, 0)


def test_refusals(ranks):
    import ctypes
    import svs_b200
    from svs_b200 import _lib
    one, backs = ranks
    rng = np.random.default_rng(6)
    d = 32
    m = _unit(rng, (400, d), "normal")
    ids = np.arange(1, 401, dtype=np.int64)
    dups = np.repeat(_unit(rng, (1, d), "normal"), 3000, axis=0)
    big = np.concatenate([dups, _unit(rng, (100, d), "normal")])
    big_ids = np.arange(1, len(big) + 1, dtype=np.int64)
    want_big = oracle.top_pairwise(big, big_ids, 25)
    for w, bs in backs.items():
        _load(bs, m, ids)
        for b in bs:
            b.pairs_disconnect()
        bs[-1].engine.apply_mutations([int(ids[-1])], [], None)         # tombstones on the last rank: it refuses to export
        _desc, status, message, _dev = bs[-1].pairs_export()
        assert status == _lib.SVSB_E_INVALID and "tombstoned" in message, (w, status, message)
        for b in bs[:-1]:
            assert b.pairs_export()[1] == 0
        with pytest.raises(svs_b200.EngineError) as ex:                # the refusing rank has nothing to connect to
            bs[0].pairs_connect_local(w, 0, bs)
        assert ex.value.code == _lib.SVSB_E_INVALID
        try:                                                            # thousands of identical rows: answer or SVSB_E_NOMEM
            norm = _load(bs, big, big_ids)
            answers = _top_pairs(bs, len(big), 25, norm)
        except svs_b200.EngineError as err:
            assert err.code == _lib.SVSB_E_NOMEM, (w, str(err))
        else:
            for got in answers:
                oracle.compare_pairs(got, want_big, np.dot(big, big.T), big_ids)
                assert got == answers[0]
    os.environ["SVSB_ALLOW_DUP_DEVICES"] = "1"
    with svs_b200.Engine([0, 0]) as e:                                  # a multi-device engine is not a shard
        e.load(m, ids)
        rc = e._lib.svsb_pairs_export(e._h, None, None, ctypes.create_string_buffer(_lib.PAIRS_DESC_BYTES))
        assert rc == _lib.SVSB_E_INVALID
    from svs_b200.sharded import CudaShardBackend
    fresh = CudaShardBackend(0)
    try:
        assert fresh.pairs_export()[1] == _lib.SVSB_E_NOT_LOADED
    finally:
        fresh.close()


def test_world_size_one_process_group_runs_the_real_collective():
    torch = pytest.importorskip("torch")
    import torch.distributed as dist
    import svs_b200
    from svs_b200.sharded import ShardedRetriever
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ["MASTER_PORT"] = str(_free_port())
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        rng = np.random.default_rng(21)
        m1 = _unit(rng, (6000, 128), "normal")
        m2 = _unit(rng, (2000, 128), "uniform")
        ids1 = np.arange(1, 6001, dtype=np.int64)
        ids2 = np.arange(9, 2009, dtype=np.int64)
        with svs_b200.Engine([0]) as one:
            one.load(m1, ids1)
            want1 = one.top_pairs(2000)
            one.load(m2, ids2)
            want2 = one.top_pairs(300)
        sr = ShardedRetriever(0, 1, 0)
        sr.load_global(m1, ids1)
        _assert_same(sr.top_pairs(2000), want1, "first load")
        _assert_same(sr.top_pairs(2000), want1, "second call, same export")
        assert sr.top_pairs(0) == []
        sr.load_global(m2, ids2)
        _assert_same(sr.top_pairs(300), want2, "after a reload")
        sr.close()
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _two_process_worker(rank, world, port, m, ids, n, ret):
    import torch
    import torch.distributed as dist
    from svs_b200.sharded import ShardedRetriever
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sr = ShardedRetriever(rank, world, rank)
        sr.load_global(m, ids)
        first = sr.top_pairs(n)
        sr.load_global(m[::-1].copy(), ids[::-1].copy())                # a reload: the shards are exported again
        second = sr.top_pairs(n)
        ret[rank] = (first, second)
        sr.close()
    finally:
        dist.destroy_process_group()


def test_two_processes_over_cuda_ipc():
    torch = pytest.importorskip("torch")
    import torch.multiprocessing as mp
    import svs_b200
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (NCCL runs one rank per GPU)")
    rng = np.random.default_rng(31)
    m = _unit(rng, (9001, 96), "normal")
    m[17] = m[8990]                                                     # an exact tie across the two shards
    ids = np.cumsum(rng.integers(1, 4, size=len(m))).astype(np.int64)
    with svs_b200.Engine([0]) as one:
        one.load(m, ids)
        want1 = one.top_pairs(3000)
        one.load(m[::-1].copy(), ids[::-1].copy())
        want2 = one.top_pairs(3000)
    ret = mp.Manager().dict()
    mp.spawn(_two_process_worker, args=(2, _free_port(), m, ids, 3000, ret), nprocs=2, join=True)
    for r in range(2):
        _assert_same(ret[r][0], want1, r)
        _assert_same(ret[r][1], want2, r)
