"""GPU: more cases of the single-query int8 filter (DESIGN.md section 4, K1f8) against K1, next to test_gpu_filter.py's.

d = 2000, small n around the int8 ring's 32-row tiles, signed and adversarial rows, tiny-scale queries, an append that
raises the shadow's error word E, and the automatic route on a C2-like shape, besides the kinds of case both modules
run.  Every case compares SVSB_FILTER=0 (K1) with the filter as uint32 scores, ids and order, through
test_gpu_filter.py's helpers."""
import numpy as np
import pytest

import svs_b200
from _util import oracle
from test_gpu_filter import _bits, _both, _check_bench, _check_query, _filter_on_small_matrices, _same  # noqa: F401

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("d", [64, 100, 762, 1536, 2000, 3072])
@pytest.mark.parametrize("dist", ["uniform", "normal"])
def test_filter8_matches_k1_over_d(monkeypatch, d, dist):
    n = 30_000
    m = oracle.synth_matrix_uniform(n, d, 3) if dist == "uniform" else oracle.synth_matrix_normal(n, d, 3)
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
def test_filter8_matches_k1_over_k(monkeypatch, k):
    n, d = 50_000, 256
    m = oracle.synth_matrix_uniform(n, d, 5)
    ids = np.arange(n, dtype=np.int64) * 3 + 1
    qs = oracle.synth_queries(2, d, 6)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for q in qs:
            _check_query(monkeypatch, e, q, k)
        _check_bench(monkeypatch, e, qs, k)


@pytest.mark.parametrize("n", [1, 5, 31, 32, 33, 700])
def test_filter8_small_n(monkeypatch, n):
    d = 1536                                   # 32 rows per TMA tile of the int8 ring
    m = oracle.synth_matrix_uniform(n, d, 7)
    ids = np.arange(n, dtype=np.int64) + 100
    q = oracle.synth_queries(1, d, 8)[0]
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for k in sorted({1, 3, n, 100}):
            _check_query(monkeypatch, e, q, k)
        _check_bench(monkeypatch, e, q[None, :], min(n, 10))


def test_filter8_adversarial_rows(monkeypatch):
    """Signed rows, rows with one large component, all-zero rows and identical rows in one matrix."""
    n, d = 40_000, 512
    rng = np.random.default_rng(30)
    m = rng.standard_normal((n, d)).astype(np.float32)
    m[::7, rng.integers(0, d)] *= 200.0                        # one dominant component: a coarse scale for the rest
    m /= np.linalg.norm(m, axis=1, keepdims=True)
    m[100:300] = 0.0
    m[5000:9000] = m[5000]
    ids = np.arange(n, dtype=np.int64)
    qs = [oracle.synth_queries(1, d, 31, dist="normal")[0], m[5000].copy(), np.zeros(d, np.float32)]
    one_big = np.full(d, 1e-4, np.float32)
    one_big[3] = 1.0
    qs.append(one_big)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for q in qs:
            for k in (1, 100, 2048):
                _check_query(monkeypatch, e, q, k)
        _check_bench(monkeypatch, e, np.stack(qs), 100)


def test_filter8_non_finite_query(monkeypatch):
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
        for scale in (1e30, 1e-30):
            _check_query(monkeypatch, e, oracle.synth_queries(1, d, 15)[0] * np.float32(scale), 100)


def test_filter8_tombstones_appends_snapshot(monkeypatch):
    n, d = 30_000, 384
    m = oracle.synth_matrix_uniform(n, d, 16)
    ids = np.arange(1, n + 1, dtype=np.int64)
    qs = oracle.synth_queries(2, d, 17)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        snap = e.snapshot()
        before = [snap.query(q, 100) for q in qs]
        dels = np.unique(np.concatenate([e.query(q, 50)[1] for q in qs]))
        e.apply_mutations(dels, [], None)
        for q in qs:
            _check_query(monkeypatch, e, q, 100)
        _check_bench(monkeypatch, e, qs, 100)
        # appended rows after the shadow exists, one of them with a large component (E grows): they must be found
        add = np.concatenate([qs, oracle.synth_matrix_uniform(2000, d, 18)]).astype(np.float32)
        add[5, 0] = 50.0
        add /= np.linalg.norm(add, axis=1, keepdims=True)
        add_ids = np.arange(n + 1, n + 1 + len(add), dtype=np.int64)
        e.apply_mutations([], add_ids, add)
        for i, q in enumerate(qs):
            got = _check_query(monkeypatch, e, q, 100)
            assert got[1][0] == add_ids[i]
        _check_bench(monkeypatch, e, qs, 100)
        # enough appends to re-allocate the shard (and its shadows)
        big = oracle.synth_matrix_uniform(n // 4, d, 19)
        e.apply_mutations([], np.arange(n + 10_000, n + 10_000 + len(big), dtype=np.int64), big)
        for q in qs:
            _check_query(monkeypatch, e, q, 100)
        _check_bench(monkeypatch, e, qs, 100)
        for q, b in zip(qs, before):
            assert _same(b, _both(monkeypatch, lambda: snap.query(q, 100))[1])
        snap.release()


def test_filter8_submit_wait_three_in_flight(monkeypatch):
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


def test_automatic_route_takes_int8_and_matches_k1_on_c2_like_shape(monkeypatch):
    n, d, k = 200_000, 1536, 100
    qs = oracle.synth_queries(4, d, 24)
    with svs_b200.Engine([0]) as e:
        e.load_synthetic(n, d, seed=0, id0=1, id_step=1)
        e.bench_set_queries(qs)
        e.bench_run(k, 8)
        assert e.bench_filter_route() == 8
        took, rescored = e.bench_filter_stats()
        assert took and k <= rescored < n // 10
        auto = e.bench_last_result(k)
        monkeypatch.setenv("SVSB_FILTER", "0")
        e.bench_run(k, 8)
        assert e.bench_filter_route() == 0
        k1 = e.bench_last_result(k)
        assert k1 == auto and _bits(k1) == _bits(auto)
