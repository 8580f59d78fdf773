"""GPU: svsb_top_pairs on multi-device engines (multi.cu: multi_top_pairs).  Every device runs its share of the static
plan (engine.cu: pairs_plan) with its own running threshold, re-scores its survivors exactly and device 0 rank-merges
the lists.  The answer must equal the single-device engine's bit for bit (scores as uint32, ids, order) and pass the
oracle's restatement of document_top_pairwise_scores.  On a one-GPU box the devices are virtual shards of device 0
(SVSB_ALLOW_DUP_DEVICES=1); with more GPUs visible the same tests use them."""
import os
import threading

import numpy as np
import pytest

from _util import oracle

pytestmark = pytest.mark.gpu


def _devices(count):
    try:
        import torch
        have = torch.cuda.device_count()
    except Exception:
        have = 1
    return [i % max(have, 1) for i in range(count)]


@pytest.fixture(scope="module")
def engines():
    import svs_b200
    os.environ["SVSB_ALLOW_DUP_DEVICES"] = "1"
    one = svs_b200.Engine([0])
    multi = {n: svs_b200.Engine(_devices(n)) for n in (2, 3, 8)}
    yield one, multi
    one.close()
    for e in multi.values():
        e.close()


def _unit(rng, shape, dist):
    m = rng.random(shape, dtype=np.float32) if dist == "uniform" else rng.standard_normal(shape).astype(np.float32)
    m /= np.maximum(np.sqrt((m * m).sum(axis=1)), 1e-12)[:, None]
    return m


def _assert_same(got, want, what):
    assert len(got) == len(want), what
    gs = np.array([s for s, _, _ in got], np.float32)
    ws = np.array([s for s, _, _ in want], np.float32)
    assert np.array_equal(gs.view(np.uint32), ws.view(np.uint32)), what
    assert [(a, b) for _, a, b in got] == [(a, b) for _, a, b in want], what


@pytest.mark.parametrize("n_rows,d,n,dist", [
    (4, 3, 10, "normal"),               # the shapes of test_gpu_pairs.py ...
    (300, 64, 50, "normal"),
    (1500, 96, 1000, "uniform"),
    (4875, 1536, 10000, "uniform"),
    (5000, 256, 100, "normal"),
    (3001, 100, 1, "normal"),
    (1001, 64, 300, "normal"),          # ... rows not divisible by 2, 3 or 8
    (20_011, 96, 5000, "uniform"),      # several 1024-row blocks per rectangle, a bootstrap sample on every device
    (5, 16, 10, "normal"),              # fewer rows than devices: empty and one-row shards
])
def test_multi_device_top_pairs_equal_the_single_device_engine(engines, n_rows, d, n, dist):
    one, multi = engines
    rng = np.random.default_rng(n_rows + d)
    m = _unit(rng, (n_rows, d), dist)
    ids = np.cumsum(rng.integers(1, 4, size=n_rows)).astype(np.int64)
    one.load(m, ids)
    want = one.top_pairs(n)
    assert len(want) == min(n, n_rows * (n_rows - 1) // 2)
    oracle.compare_pairs(want, oracle.top_pairwise(m, ids, n), np.dot(m, m.T), ids)
    for nd, e in multi.items():
        e.load(m, ids)
        _assert_same(e.top_pairs(n), want, (nd, n_rows, d, n))


def test_identical_rows_in_the_first_a_middle_and_the_last_shard_come_out_in_row_order(engines):
    one, multi = engines
    rng = np.random.default_rng(3)
    n_rows = 2500
    m = _unit(rng, (n_rows, 48), "normal")
    dup = [10, 11, 1300, 2490]                                     # shards 0, 0, middle, last for 2, 3 and 8 devices
    for r in dup[:-1]:
        m[r] = m[dup[-1]]
    ids = np.arange(100, 100 + n_rows, dtype=np.int64)
    one.load(m, ids)
    want = one.top_pairs(8)
    expect = [(dup[a], dup[b]) for a in range(4) for b in range(a + 1, 4)]
    assert [(a - 100, b - 100) for _, a, b in want[:6]] == expect
    for nd, e in multi.items():
        e.load(m, ids)
        got = e.top_pairs(8)
        _assert_same(got, want, nd)
        assert all(abs(s - 1.0) < 1e-5 for s, _, _ in got[:6])


def test_edge_cases_give_the_single_device_results(engines):
    one, multi = engines
    rng = np.random.default_rng(4)
    m = _unit(rng, (50, 16), "normal")
    ids = np.arange(50, dtype=np.int64)
    one.load(m, ids)
    everything = one.top_pairs(10 ** 6)
    assert len(everything) == 50 * 49 // 2
    for nd, e in multi.items():
        e.load(m, ids)
        assert e.top_pairs(0) == []
        _assert_same(e.top_pairs(10 ** 6), everything, nd)
        e.load(m[:1], ids[:1])
        assert e.top_pairs(5) == []


def test_a_snapshot_answers_from_its_generation_after_a_reload(engines):
    one, multi = engines
    rng = np.random.default_rng(5)
    m1 = _unit(rng, (3000, 64), "normal")
    m2 = _unit(rng, (2200, 64), "uniform")
    ids1 = np.arange(1, 3001, dtype=np.int64)
    ids2 = np.arange(7, 2207, dtype=np.int64)
    one.load(m1, ids1)
    want1 = one.top_pairs(400)
    one.load(m2, ids2)
    want2 = one.top_pairs(400)
    for nd, e in multi.items():
        e.load(m1, ids1)
        snap = e.snapshot()
        e.load(m2, ids2)
        _assert_same(snap.top_pairs(400), want1, nd)
        _assert_same(e.top_pairs(400), want2, nd)
        snap.release()


def test_refusals(engines):
    import svs_b200
    one, multi = engines
    rng = np.random.default_rng(6)
    d = 32
    m = _unit(rng, (400, d), "normal")
    ids = np.arange(1, 401, dtype=np.int64)
    # thousands of identical rows: millions of pairs at the same score, more than a candidate list holds
    dups = np.repeat(_unit(rng, (1, d), "normal"), 3000, axis=0)
    big = np.concatenate([dups, _unit(rng, (100, d), "normal")])
    big_ids = np.arange(1, len(big) + 1, dtype=np.int64)
    want_big = oracle.top_pairwise(big, big_ids, 25)
    for nd, e in multi.items():
        e.load(m, ids)
        e.apply_mutations([5, 200], [], None)                      # tombstones: the pair path asks for a reload
        with pytest.raises(svs_b200.EngineError) as ex:
            e.top_pairs(10)
        assert ex.value.code == svs_b200._lib.SVSB_E_INVALID
        e.load(big, big_ids)
        try:
            got = e.top_pairs(25)
        except svs_b200.EngineError as err:
            assert err.code == svs_b200._lib.SVSB_E_NOMEM, (nd, str(err))
        else:
            oracle.compare_pairs(got, want_big, np.dot(big, big.T), big_ids)


def test_top_pairs_while_another_thread_keeps_queries_in_flight(engines):
    one, multi = engines
    n_rows, d = 30_000, 128
    m = oracle.synth_matrix_normal(n_rows, d, 71)
    ids = np.arange(1, n_rows + 1, dtype=np.int64)
    qs = oracle.synth_queries(12, d, 72, dist="normal")
    one.load(m, ids)
    want_q = [one.query(q, 20) for q in qs]
    want_p = one.top_pairs(3000)
    for nd, e in multi.items():
        e.load(m, ids)
        stop = threading.Event()
        errors = []
        done = [0]

        def worker():
            try:
                j = 0
                while not stop.is_set() or done[0] < 6:
                    pend = [e.submit(qs[(j + t) % len(qs)], 20) for t in range(3)]
                    for t, p in enumerate(pend):
                        s, i = p.result()
                        w = want_q[(j + t) % len(qs)]
                        assert np.array_equal(s.view(np.uint32), w[0].view(np.uint32)) and np.array_equal(i, w[1])
                    j += 3
                    done[0] += 1
            except Exception as ex:                                # noqa: BLE001
                errors.append(repr(ex))
        th = threading.Thread(target=worker)
        th.start()
        try:
            for _ in range(3):
                _assert_same(e.top_pairs(3000), want_p, nd)
        finally:
            stop.set()
            th.join()
        assert errors == [], errors
        assert done[0] >= 6
