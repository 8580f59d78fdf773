"""GPU: svsb_query (GEMV + exact top-k) against the oracle's superheavy() -- reference
src/svs/kb.py:1622-1627 -- through the C ABI.  fp32 scores: <= 1e-5 relative (BASELINE.json);
ids and ranks exact except across near-ties (oracle.compare_retrieval)."""
import os
import threading

import numpy as np
import pytest

from _util import golden_npz, oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    import svs_b200
    e = svs_b200.Engine()
    yield e
    e.close()


def _check(engine, m, ids, q, k):
    got = engine.retrieve(q, k)
    x = oracle.scores_of(m, q)
    want = oracle.superheavy(m, ids, q, k)
    rep = oracle.compare_retrieval(got, want, x, ids)
    assert rep["max_rel_score_err"] <= 1e-5
    return rep


@pytest.mark.parametrize("name", ["superheavy_d96.npz", "superheavy_d1536.npz"])
@pytest.mark.parametrize("variant", ["1", "2"])
def test_golden_vectors_from_the_reference(engine, name, variant, monkeypatch):
    monkeypatch.setenv("SVSB_GEMV_VARIANT", variant)
    g = golden_npz(name)
    m, ids, qs = g["matrix"], g["emb_ids"], g["queries"]
    engine.load(m, ids)
    assert engine.shape == m.shape
    for qi in range(len(qs)):
        for k in g["ks"]:
            got = engine.retrieve(qs[qi], int(k))
            want = list(zip(g[f"top_q{qi}_k{k}_scores"].tolist(), g[f"top_q{qi}_k{k}_ids"].tolist()))
            oracle.compare_retrieval(got, want, g[f"scores_q{qi}"], ids)


@pytest.mark.parametrize("variant", ["1", "2"])
@pytest.mark.parametrize("n,d,k", [(1, 4, 1), (5, 3, 3), (4, 2, 10), (100, 1, 5), (1000, 7, 50), (777, 33, 100),
                                   (4096, 768, 100), (10_548, 1536, 10), (20_000, 3072, 1000), (50_000, 128, 100),
                                   (3001, 1537, 17), (2000, 6000, 10)])
def test_shapes_including_d_not_multiple_of_four(engine, n, d, k, variant, monkeypatch):
    monkeypatch.setenv("SVSB_GEMV_VARIANT", variant)
    rng = np.random.default_rng(n + d)
    m = rng.standard_normal((n, d)).astype(np.float32)
    m /= np.maximum(np.sqrt((m * m).sum(axis=1)), 1e-12)[:, None]
    ids = np.cumsum(rng.integers(1, 5, size=n)).astype(np.int64)
    engine.load(m, ids)
    back, back_ids = engine.read_rows(0, n)
    assert back.tobytes() == m.tobytes() and (back_ids == ids).all()         # stored verbatim
    for s in range(3):
        q = rng.standard_normal(d).astype(np.float32)
        q /= np.sqrt((q * q).sum())
        _check(engine, m, ids, q, k)


def test_the_plain_c_oracle_accepts_the_engine_too(engine):
    """Second checker: oracle/svs_oracle_c.c (its own dot product, its own selection) judges the CUDA path through the
    same tolerance-aware comparator as the NumPy oracle does."""
    import shutil
    import sys
    if shutil.which("gcc") is None and shutil.which("cc") is None and not os.path.exists(
            os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libsvs_oracle_c.so")):
        pytest.skip("no C compiler and no prebuilt C oracle")
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import build_oracle_c
    oc = build_oracle_c.OracleC()
    rng = np.random.default_rng(123)
    for n, d, k in ((3000, 96, 10), (20_000, 1536, 100), (5000, 257, 1000)):
        m = rng.standard_normal((n, d)).astype(np.float32)
        m /= np.sqrt((m * m).sum(axis=1))[:, None]
        ids = np.cumsum(rng.integers(1, 4, size=n)).astype(np.int64)
        engine.load(m, ids)
        for _ in range(2):
            q = rng.standard_normal(d).astype(np.float32)
            q /= np.sqrt((q * q).sum())
            want = oc.superheavy(m, ids, q, k)
            rep = oracle.compare_retrieval(engine.retrieve(q, k), want, oc.scores(m, q), ids)
            assert rep["max_rel_score_err"] <= 1e-5


@pytest.mark.parametrize("tune_a", ["1", "2", "3", "4", "5", "6", "7", "8", "9"])
def test_every_ldg_instantiation_is_correct(engine, tune_a, monkeypatch):
    """Every LDG instantiation returns K1's bits (oracle/k1_exact.py), not just scores within the oracle's tolerance."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import k1_exact
    monkeypatch.setenv("SVSB_GEMV_VARIANT", "1")
    monkeypatch.setenv("SVSB_GEMV_TUNE_A", tune_a)
    m = oracle.synth_matrix_uniform(30_011, 1536, 3)
    ids = np.arange(1, len(m) + 1, dtype=np.int64)
    engine.load(m, ids)
    q = oracle.synth_queries(1, 1536, 4)[0]
    _check(engine, m, ids, q, 100)
    s, i = engine.query(q, 100)
    want_bits, want_ids = k1_exact.k1_topk_exact(m, ids, q, 100)
    assert np.array_equal(s.view(np.uint32), want_bits) and np.array_equal(i, want_ids)


def test_reference_unit_test_matrix_and_uninormalised_rows(engine):
    # reference tests/test_kb.py:761-796 loads rows that are NOT unit vectors; scores are raw dot products
    m = np.array([[1.0, 3.5], [2.0, 3.5], [2.0, 1.0], [3.5, 4.0]], dtype=np.float32)
    ids = np.array([1, 2, 3, 4], dtype=np.int64)
    engine.load(m, ids)
    got = engine.retrieve(np.array([1.0, 0.0], dtype=np.float32), 4)
    assert got == [(3.5, 4), (2.0, 2), (2.0, 3), (1.0, 1)]         # tie 2.0: ascending id
    dev, bad = engine.norm_stats()
    assert bad == 4 and dev == pytest.approx(np.sqrt(3.5 ** 2 + 16) - 1, rel=1e-6)


def test_retrieve_ranks_of_the_reference_integration_test(engine):
    # reference tests/test_kb.py:1739-1781: stub vectors for "third/first/second/forth doc"
    m = np.array([[0.01, 0.0, 1.0], [1.0, 0.001, 0.0], [0.0, 1.0, 0.0001]], dtype=np.float32)
    ids = np.array([1, 2, 3], dtype=np.int64)
    engine.load(m, ids)
    rank = lambda q: [i for _, i in engine.retrieve(np.array(q, dtype=np.float32), 3)]
    assert rank([1.0, 0.001, 0.0]) == [2, 1, 3]       # first, third, second
    assert rank([0.0, 1.0, 0.0001]) == [3, 2, 1]      # second, first, third
    assert rank([0.01, 0.0, 1.0]) == [1, 2, 3]        # third, first, second
    assert [i for _, i in engine.retrieve(np.array([0.707, 0.707, 0.0], dtype=np.float32), 1)] == [2]


def test_edge_behaviour_matches_numpy(engine):
    m = oracle.synth_matrix_normal(50, 8, 1)
    engine.load(m, np.arange(50, dtype=np.int64))
    q = m[3].copy()
    assert engine.retrieve(q, 0) == [] and engine.retrieve(q, -3) == []       # util.py:200-201
    assert len(engine.retrieve(q, 500)) == 50                                  # util.py:198-199
    assert engine.retrieve(q, 1)[0][1] == 3
    with pytest.raises(ValueError):                                             # np.dot shape error
        engine.retrieve(np.zeros(9, dtype=np.float32), 5)
    engine.load(np.zeros((0, 0), dtype=np.float32), np.zeros(0, dtype=np.int64))
    assert engine.shape == (0, 0)
    with pytest.raises(ValueError):                                             # empty KB (SURVEY 8a)
        engine.retrieve(np.zeros(8, dtype=np.float32), 5)
    engine.invalidate()
    assert not engine.is_loaded()
    import svs_b200
    with pytest.raises(svs_b200.EngineError):
        engine.retrieve(q, 1)


def test_all_tied_scores_mock_embedder(engine):
    # svs.embeddings.mock returns [1,0,0] for everything: every score ties (SURVEY 8a)
    m = np.tile(np.array([[1.0, 0.0, 0.0]], dtype=np.float32), (5, 1))
    engine.load(m, np.array([1, 2, 3, 4, 5], dtype=np.int64))
    assert engine.retrieve(np.array([1.0, 0.0, 0.0], dtype=np.float32), 3) == [(1.0, 1), (1.0, 2), (1.0, 3)]


def test_full_ranking_n_equals_len(engine):
    # n = len(kb) is a real use (examples/dad_jokes notebook): large-k path
    m = oracle.synth_matrix_normal(10_548, 64, 2)
    ids = np.arange(1, 10_549, dtype=np.int64)
    engine.load(m, ids)
    q = oracle.synth_queries(1, 64, 3, "normal")[0]
    rep = _check(engine, m, ids, q, 10_548)
    assert rep["n"] == 10_548


def test_normalize_mode_divides_rows_by_their_norm(engine):
    rng = np.random.default_rng(0)
    m = rng.random((1000, 96), dtype=np.float32) + 0.5
    engine.load(m, np.arange(1000, dtype=np.int64), normalize=True)
    back, _ = engine.read_rows(0, 1000)
    want = m / np.sqrt((m.astype(np.float64) ** 2).sum(axis=1))[:, None]
    np.testing.assert_allclose(back, want, rtol=3e-7)
    dev, bad = engine.norm_stats()
    assert bad == 1000 and dev > 1.0          # statistics describe the rows as supplied


def test_snapshot_survives_invalidate_and_reload(engine):
    a = oracle.synth_matrix_normal(300, 32, 5)
    b = oracle.synth_matrix_normal(200, 32, 6)
    engine.load(a, np.arange(300, dtype=np.int64))
    snap = engine.snapshot()
    q = a[17].copy()
    assert snap.retrieve(q, 1)[0][1] == 17
    engine.invalidate()
    assert snap.retrieve(q, 1)[0][1] == 17                         # still the old arrays
    engine.load(b, np.arange(1000, 1200, dtype=np.int64))
    assert snap.retrieve(q, 1)[0][1] == 17 and snap.shape == (300, 32)
    assert engine.retrieve(b[5], 1)[0][1] == 1005
    snap.release()


def test_concurrent_queries_from_threads_with_reloads(engine):
    m = oracle.synth_matrix_normal(20_000, 256, 11)
    ids = np.arange(20_000, dtype=np.int64)
    engine.load(m, ids)
    qs = oracle.synth_queries(16, 256, 12, "normal")
    expect = [[i for _, i in engine.retrieve(q, 20)] for q in qs]
    errors = []

    def worker(t):
        try:
            for it in range(20):
                j = (t * 7 + it) % len(qs)
                got = [i for _, i in engine.retrieve(qs[j], 20)]
                if got != expect[j]:
                    errors.append((t, it, j))
        except Exception as ex:  # noqa
            errors.append(repr(ex))
    threads = [threading.Thread(target=worker, args=(t,)) for t in range(8)]
    for t in threads:
        t.start()
    for _ in range(3):
        engine.load(m, ids)                                        # same data: results must not change
    for t in threads:
        t.join()
    assert errors == []


def test_virtual_shards_match_single_device(monkeypatch):
    """The multi-device path (row shards + candidate gather + merge kernel) on one GPU."""
    import svs_b200
    monkeypatch.setenv("SVSB_ALLOW_DUP_DEVICES", "1")
    m = oracle.synth_matrix_uniform(40_003, 192, 21)
    ids = np.cumsum(np.random.default_rng(1).integers(1, 3, size=len(m))).astype(np.int64)
    qs = oracle.synth_queries(4, 192, 22)
    for shards in (2, 3, 8):
        e = svs_b200.Engine([0] * shards)
        try:
            e.load(m, ids)
            back, bid = e.read_rows(0, len(m))
            assert back.tobytes() == m.tobytes() and (bid == ids).all()
            for q in qs:
                for k in (1, 100, 300, 2048):
                    _check(e, m, ids, q, k)
            # ties across shard boundaries resolve by ascending id
            e.load(np.ones((1000, 4), dtype=np.float32), np.arange(1000, dtype=np.int64))
            assert [i for _, i in e.retrieve(np.ones(4, dtype=np.float32), 7)] == list(range(7))
            # fewer rows than shards
            e.load(m[:2], ids[:2])
            _check(e, m[:2], ids[:2], qs[0], 5)
        finally:
            e.close()


def test_bench_path_computes_the_same_result(engine):
    m = oracle.synth_matrix_uniform(60_000, 1536, 31)
    ids = np.arange(5, 60_005, dtype=np.int64)
    engine.load(m, ids)
    qs = oracle.synth_queries(5, 1536, 32)
    engine.bench_set_queries(qs)
    r = engine.bench_run(100, 5, with_gemv=True)
    assert r["total_ms"] > 0 and r["gemv_ms"] > 0 and r["launches"] == 10
    got = engine.bench_last_result(100)                            # the 5th query (index 4)
    oracle.compare_retrieval(got, oracle.superheavy(m, ids, qs[4], 100), oracle.scores_of(m, qs[4]), ids)
    assert engine.retrieve(qs[4], 100) == got


def test_oversized_n_returns_the_full_ranking(engine):
    """get_top_k clips n to the row count (src/svs/util.py:198-199): n = 2**31, 2**32 + 3 or 10**12 must neither wrap
    around in a 32-bit argument nor size a buffer -- every one of them is the full ranking."""
    m = oracle.synth_matrix_normal(777, 48, 5)
    ids = np.arange(10, 10 + 777, dtype=np.int64)
    engine.load(m, ids)
    q = oracle.synth_queries(1, 48, 6, dist="normal")[0]
    full = engine.retrieve(q, 777)
    oracle.compare_retrieval(full, oracle.superheavy(m, ids, q, 777), oracle.scores_of(m, q), ids)
    for n in (778, 2**31 - 1, 2**31, 2**31 + 3, 2**32, 2**32 + 3, 10**12):
        assert engine.retrieve(q, n) == full
    snap = engine.snapshot()
    assert snap.retrieve(q, 10**12) == full
    s, i, c = engine.query_batch(np.stack([q, q]), 10**12)
    assert s.shape == (2, 777) and c.tolist() == [777, 777] and [(float(a), int(b)) for a, b in zip(s[1], i[1])] == full
    s, i, c = snap.query_batch(np.stack([q, q]), 2**31)
    assert s.shape == (2, 777) and c.tolist() == [777, 777]
    assert engine.retrieve(q, -(2**40)) == [] and engine.retrieve(q, 0) == []
    snap.release()
