"""GPU: the single-query int8 filter (DESIGN.md section 4, K1f8) returns exactly what the fp32 similarity kernel K1 returns.

Every case answers the same query with SVSB_FILTER=0 (K1) and SVSB_FILTER=1 (pass over the int8 shadow, exact re-score of
the candidates) and compares scores as uint32, ids and order.  SVSB_FILTER_MIN_MB=0 lets small matrices take the filter;
`bench_filter_route` and `bench_filter_stats` confirm which route the device-resident loop took.  The helpers serve
test_gpu_filter8.py and test_gpu_filter8_edges.py as well."""
import numpy as np
import pytest

import svs_b200
from _util import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _filter_on_small_matrices(monkeypatch):
    monkeypatch.setenv("SVSB_FILTER_MIN_MB", "0")
    monkeypatch.delenv("SVSB_FILTER", raising=False)


def _same(a, b):
    return (len(a[0]) == len(b[0]) and np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))
            and np.array_equal(a[1], b[1]))


def _both(monkeypatch, fn):
    monkeypatch.setenv("SVSB_FILTER", "0")
    ref = fn()
    monkeypatch.setenv("SVSB_FILTER", "1")
    got = fn()
    monkeypatch.delenv("SVSB_FILTER")
    return ref, got


def _check_query(monkeypatch, e, q, k):
    ref, got = _both(monkeypatch, lambda: e.query(q, k))
    assert _same(ref, got), (k, ref[0][:5], got[0][:5])
    return got


def _bits(res):
    return [np.float32(s).view(np.uint32) for s, _ in res]


def _check_bench(monkeypatch, e, qs, k, expect_filter=True):
    """The device-resident loop (pipelined and serial): last answer and the route it took."""
    e.bench_set_queries(qs)
    for pipe in ("1", "0"):
        monkeypatch.setenv("SVSB_PIPELINE", pipe)
        res = []
        for f in ("0", "1"):
            monkeypatch.setenv("SVSB_FILTER", f)
            e.bench_run(k, len(qs) + 1)
            res.append(e.bench_last_result(k))
            filtered = f == "1" and expect_filter
            assert e.bench_filter_route() == (8 if filtered else 0)
            took, rescored = e.bench_filter_stats()
            assert took == filtered
            if took:
                assert rescored >= min(k, e.generation_rows()[1])
        assert res[0] == res[1] and _bits(res[0]) == _bits(res[1])
    monkeypatch.delenv("SVSB_PIPELINE")
    monkeypatch.delenv("SVSB_FILTER")


def _gaussian(n, d, seed):
    return oracle.synth_matrix_normal(n, d, seed)


@pytest.mark.parametrize("d", [64, 100, 762, 1536, 3072])
@pytest.mark.parametrize("dist", ["uniform", "normal"])
def test_filter_matches_k1_over_d(monkeypatch, d, dist):
    n = 30_000
    m = oracle.synth_matrix_uniform(n, d, 3) if dist == "uniform" else _gaussian(n, d, 3)
    ids = np.arange(10, 10 + n, dtype=np.int64)
    qs = oracle.synth_queries(3, d, 4, dist="uniform" if dist == "uniform" else "normal")
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for q in qs:
            got = _check_query(monkeypatch, e, q, 100)
            ora = oracle.superheavy(m, ids, q, 100)
            oracle.compare_retrieval(list(zip(got[0].tolist(), got[1].tolist())), ora, oracle.scores_of(m, q), ids)
        _check_bench(monkeypatch, e, qs, 100)


@pytest.mark.parametrize("k", [1, 10, 100, 1000, 2048])
def test_filter_matches_k1_over_k(monkeypatch, k):
    n, d = 50_000, 256
    m = oracle.synth_matrix_uniform(n, d, 5)
    ids = np.arange(n, dtype=np.int64) * 3 + 1
    qs = oracle.synth_queries(2, d, 6)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for q in qs:
            _check_query(monkeypatch, e, q, k)
        _check_bench(monkeypatch, e, qs, k)


@pytest.mark.parametrize("n", [1, 5, 63, 64, 65, 700])
def test_filter_small_n(monkeypatch, n):
    d = 1536                                   # 32 rows per TMA tile of the int8 ring
    m = oracle.synth_matrix_uniform(n, d, 7)
    ids = np.arange(n, dtype=np.int64) + 100
    q = oracle.synth_queries(1, d, 8)[0]
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for k in sorted({1, 3, n, 100}):
            _check_query(monkeypatch, e, q, k)
        _check_bench(monkeypatch, e, q[None, :], min(n, 10))


def test_filter_identical_rows(monkeypatch):
    n, d = 40_000, 128
    row = oracle.synth_matrix_uniform(1, d, 9)
    m = np.repeat(row, n, axis=0)
    ids = np.arange(n, dtype=np.int64)
    q = oracle.synth_queries(1, d, 10)[0]
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for k in (1, 100, 2048):
            got = _check_query(monkeypatch, e, q, k)
            assert got[1].tolist() == list(range(k))        # ties: ascending row
        _check_bench(monkeypatch, e, q[None, :], 100)


def test_filter_rows_sorted_by_similarity(monkeypatch):
    n, d = 30_000, 512
    m = oracle.synth_matrix_uniform(n, d, 11)
    q = oracle.synth_queries(1, d, 12)[0]
    m = m[np.argsort(m @ q)]                   # ascending: the best rows are the last group
    ids = np.arange(n, dtype=np.int64)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for k in (1, 100, 1000):
            _check_query(monkeypatch, e, q, k)


def test_filter_non_finite_query(monkeypatch):
    n, d = 20_000, 256
    m = oracle.synth_matrix_uniform(n, d, 13)
    ids = np.arange(n, dtype=np.int64)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for bad in (np.nan, np.inf, -np.inf):
            q = oracle.synth_queries(1, d, 14)[0].copy()
            q[17] = bad
            for k in (1, 100):
                _check_query(monkeypatch, e, q, k)
        huge = oracle.synth_queries(1, d, 15)[0] * np.float32(1e30)
        _check_query(monkeypatch, e, huge, 100)


def test_filter_tombstones_and_appends(monkeypatch):
    n, d = 30_000, 384
    m = oracle.synth_matrix_uniform(n, d, 16)
    ids = np.arange(1, n + 1, dtype=np.int64)
    qs = oracle.synth_queries(2, d, 17)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        snap = e.snapshot()
        before = [snap.query(q, 100) for q in qs]
        # delete the current winners of both queries, so every answer changes
        dels = np.unique(np.concatenate([e.query(q, 50)[1] for q in qs]))
        e.apply_mutations(dels, [], None)
        for q in qs:
            _check_query(monkeypatch, e, q, 100)
        _check_bench(monkeypatch, e, qs, 100)
        # appended rows after the shadow exists: rows close to the queries, which must be found
        add = np.concatenate([qs, oracle.synth_matrix_uniform(2000, d, 18)]).astype(np.float32)
        add /= np.linalg.norm(add, axis=1, keepdims=True)
        add_ids = np.arange(n + 1, n + 1 + len(add), dtype=np.int64)
        e.apply_mutations([], add_ids, add)
        for i, q in enumerate(qs):
            got = _check_query(monkeypatch, e, q, 100)
            assert got[1][0] == add_ids[i]
        _check_bench(monkeypatch, e, qs, 100)
        # enough appends to re-allocate the shard (and its shadow)
        big = oracle.synth_matrix_uniform(n // 4, d, 19)
        e.apply_mutations([], np.arange(n + 10_000, n + 10_000 + len(big), dtype=np.int64), big)
        for q in qs:
            _check_query(monkeypatch, e, q, 100)
        _check_bench(monkeypatch, e, qs, 100)
        # the snapshot still answers from the generation it pinned
        for q, b in zip(qs, before):
            assert _same(b, _both(monkeypatch, lambda: snap.query(q, 100))[1])
        snap.release()


def test_filter_rows_beyond_fp16_range_take_k1(monkeypatch):
    n, d = 20_000, 256
    m = oracle.synth_matrix_uniform(n, d, 20)
    m[123] *= 20.0                             # one row of norm 20 > 8
    ids = np.arange(n, dtype=np.int64)
    q = oracle.synth_queries(1, d, 21)[0]
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        got = _check_query(monkeypatch, e, q, 100)
        assert got[1][0] == 123
        _check_bench(monkeypatch, e, q[None, :], 100, expect_filter=False)


def test_filter_submit_wait_three_in_flight(monkeypatch):
    n, d = 40_000, 1536
    m = oracle.synth_matrix_uniform(n, d, 22)
    ids = np.arange(n, dtype=np.int64)
    qs = oracle.synth_queries(9, d, 23)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)

        def run():
            out, pend = [], []
            for q in qs:
                pend.append(e.submit(q, 100))
                if len(pend) == 3:
                    out.append(pend.pop(0).result())
            out += [p.result() for p in pend]
            return out
        ref, got = _both(monkeypatch, run)
        assert all(_same(a, b) for a, b in zip(ref, got))
