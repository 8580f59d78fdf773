"""GPU: every exact path against the bit-exact CPU restatement of K1 (oracle/k1_exact.py).

Each path promises svsb_query's bits, and svsb_query's bits are K1's summation order (gemv_tma_kernel).  Here they are
compared with that order computed on the CPU, as uint32 score bits plus ids, nothing else allowed: the single-query
kernels (TMA and LDG variants, every instantiation), the batched paths (tensor-core coarse pass + exact refine, the
multi-query passes), the int8 filter, the in-process multi-device merge, the bench loop, a generation with
tombstones and appended rows, and the pair search.  d covers one chunk per lane and less (d <= 128), ragged ld, the
multi-query limits, and both sides of the TMA kernel's row limit (d = 12 800) where K1 hands over to the LDG kernel."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import k1_exact as kx  # noqa: E402

pytestmark = pytest.mark.gpu

D_ALL = [1, 3, 4, 5, 127, 128, 129, 190, 1536, 1537, 3072, 3073, 12800, 12801, 13000, 16384]
D_LONG = [129, 190, 1537, 3073, 12801, 16384]


@pytest.fixture(scope="module")
def engine():
    import svs_b200
    e = svs_b200.Engine()
    yield e
    e.close()


def _rows_for(d):
    return 4099 if d <= 4096 else 4097                             # ragged: not a multiple of any tile; coarse path needs 4096


def _data(d, seed, n=None, b=4):
    rng = np.random.default_rng(seed * 100_003 + d)
    n = n or _rows_for(d)
    m = rng.standard_normal((n, d)).astype(np.float32)
    m /= np.maximum(np.sqrt((m.astype(np.float64) ** 2).sum(axis=1)), 1e-30).astype(np.float32)[:, None]
    ids = np.cumsum(rng.integers(1, 5, n)).astype(np.int64) + 7   # not contiguous
    q = rng.standard_normal((b, d)).astype(np.float32)
    q /= np.sqrt((q.astype(np.float64) ** 2).sum(axis=1)).astype(np.float32)[:, None]
    return m, ids, q


def _assert_bits(got_scores, got_ids, m, ids, q, k, live=None, what=""):
    want_b, want_i = kx.k1_topk_exact(m, ids, q, k, live)
    got_b = np.asarray(got_scores, np.float32).view(np.uint32)
    assert len(got_b) == len(want_b), f"{what}: {len(got_b)} results, expected {len(want_b)}"
    bad = np.nonzero((got_b != want_b) | (np.asarray(got_ids) != want_i))[0]
    assert len(bad) == 0, (f"{what}: rank {bad[0]}: got ({got_b[bad[0]]:#010x}, {got_ids[bad[0]]}) "
                           f"expected ({want_b[bad[0]]:#010x}, {want_i[bad[0]]}); {len(bad)} ranks differ")


def _list_bits(lst):
    return np.array([s for s, _ in lst], np.float32), np.array([i for _, i in lst], np.int64)


@pytest.mark.parametrize("d", D_ALL)
def test_query_auto_variant(engine, d):
    m, ids, q = _data(d, 1)
    engine.load(m, ids)
    for j, k in enumerate((1, 50, 2100)):
        s, i = engine.query(q[j], k)
        _assert_bits(s, i, m, ids, q[j], k, what=f"k={k}")


@pytest.mark.parametrize("tune_b", ["800", "1600"])
@pytest.mark.parametrize("d", [d for d in D_ALL if d <= 12800])
def test_query_every_tma_instantiation(engine, d, tune_b, monkeypatch):
    monkeypatch.setenv("SVSB_GEMV_VARIANT", "2")
    monkeypatch.setenv("SVSB_GEMV_TUNE_B", tune_b)                 # 8 or 16 consumer warps, default ring
    m, ids, q = _data(d, 2)
    engine.load(m, ids)
    s, i = engine.query(q[0], 64)
    _assert_bits(s, i, m, ids, q[0], 64)


@pytest.mark.parametrize("tune_a", [str(a) for a in range(1, 10)])
@pytest.mark.parametrize("d", D_LONG)
def test_query_every_ldg_instantiation(engine, d, tune_a, monkeypatch):
    """The LDG kernel unrolls U chunks per step (U odd for 1, 2, 3, 7, 9) and has a tail loop: a lane's chunks must
    still alternate between the two accumulators exactly as in K1."""
    monkeypatch.setenv("SVSB_GEMV_VARIANT", "1")
    monkeypatch.setenv("SVSB_GEMV_TUNE_A", tune_a)
    m, ids, q = _data(d, 3, n=1031)
    engine.load(m, ids)
    s, i = engine.query(q[0], 40)
    _assert_bits(s, i, m, ids, q[0], 40)


@pytest.mark.parametrize("d", D_ALL)
def test_query_batch_coarse_path(engine, d, monkeypatch):
    monkeypatch.setenv("SVSB_MQ_MAX", "1")
    m, ids, q = _data(d, 4, b=24)
    engine.load(m, ids)
    k = 30
    s, i, c = engine.query_batch(q, k)
    if d >= 16:                                                    # below 16 the tensor-core path does not apply
        cand, resc, flags = engine.batch_stats(len(q))
        assert (flags == 0).all(), flags
    for j in range(len(q)):
        _assert_bits(s[j, :c[j]], i[j, :c[j]], m, ids, q[j], k, what=f"query {j}")


@pytest.mark.parametrize("d", D_ALL)
def test_query_batch_multi_query_path(engine, d, monkeypatch):
    monkeypatch.setenv("SVSB_MQ_MAX", "64")
    m, ids, q = _data(d, 5, b=9)
    engine.load(m, ids)
    s, i, c = engine.query_batch(q, 17)
    for j in range(len(q)):
        _assert_bits(s[j, :c[j]], i[j, :c[j]], m, ids, q[j], 17, what=f"query {j}")


@pytest.mark.parametrize("route", ["1", "8"])
@pytest.mark.parametrize("d", D_ALL)
def test_filters(d, route, monkeypatch):
    """The int8 filter, switched on by SVSB_FILTER=1 and by =8 (any value but 0), on a matrix of any size: the
    re-scored candidates must carry K1's bits.  d above the filter's row limit takes K1 itself."""
    import svs_b200
    monkeypatch.setenv("SVSB_FILTER", route)
    monkeypatch.setenv("SVSB_FILTER_MIN_MB", "0")
    m, ids, q = _data(d, 6)
    with svs_b200.Engine() as e:                                    # a fresh engine: the shadows are built at load
        e.load(m, ids)
        for j, k in enumerate((1, 100)):
            s, i = e.query(q[j], k)
            _assert_bits(s, i, m, ids, q[j], k, what=f"k={k}")


@pytest.mark.parametrize("d", [5, 129, 1537, 12801])
def test_three_virtual_devices(d, monkeypatch):
    import svs_b200
    monkeypatch.setenv("SVSB_ALLOW_DUP_DEVICES", "1")
    m, ids, q = _data(d, 7)
    with svs_b200.Engine([0, 0, 0]) as e:
        e.load(m, ids)
        for j, k in enumerate((1, 77, 2500)):
            s, i = e.query(q[j], k)
            _assert_bits(s, i, m, ids, q[j], k, what=f"k={k}")
        s, i, c = e.query_batch(q, 20)
        for j in range(len(q)):
            _assert_bits(s[j, :c[j]], i[j, :c[j]], m, ids, q[j], 20, what=f"batch query {j}")


@pytest.mark.parametrize("d", [3, 190, 1536, 12801])
def test_bench_loop(engine, d):
    m, ids, q = _data(d, 8)
    engine.load(m, ids)
    engine.bench_set_queries(q)
    k = 25
    engine.bench_run(k, 2)
    s, i = _list_bits(engine.bench_last_result(k))
    # the loop cycles through the uploaded queries: the last of 2 iterations answered query 1
    _assert_bits(s, i, m, ids, q[1], k)


@pytest.mark.parametrize("d", [5, 190, 1537, 12801])
def test_generation_with_tombstones_and_appends(engine, d):
    m, ids, q = _data(d, 9)
    n0 = len(m) - 300
    engine.load(m[:n0], ids[:n0])
    rng = np.random.default_rng(d)
    dels = rng.choice(ids[:n0], 500, replace=False)
    engine.apply_mutations(dels, ids[n0:], m[n0:])
    live = ~np.isin(ids, dels)
    phys, nlive = engine.generation_rows()
    assert phys == len(m) and nlive == live.sum()
    for j, k in enumerate((1, 60, 2100)):
        s, i = engine.query(q[j], k)
        _assert_bits(s, i, m[live], ids[live], q[j], k, what=f"k={k}")
    s, i, c = engine.query_batch(q, 60)
    for j in range(len(q)):
        _assert_bits(s[j, :c[j]], i[j, :c[j]], m[live], ids[live], q[j], 60, what=f"batch query {j}")


def _assert_pairs(got, m, ids, n):
    want = kx.top_pairs_exact(m, ids, n)
    assert len(got) == len(want)
    row_of = {int(x): r for r, x in enumerate(ids)}
    for r, ((s, a, b), (wb, wa, wbb)) in enumerate(zip(got, want)):
        gb = int(np.array([s], np.float32).view(np.uint32)[0])
        # every reported score is the pair re-score's bits of that very pair
        assert gb == int(np.array([kx.pair_exact(m, row_of[a], row_of[b])]).view(np.uint32)[0]), f"rank {r}: pair ({a}, {b})"
        assert (gb, a, b) == (wb, wa, wbb), f"rank {r}: got ({gb:#010x}, {a}, {b}) expected ({wb:#010x}, {wa}, {wbb})"


@pytest.mark.parametrize("d", [16, 129, 1537, 12801])
def test_top_pairs(engine, d):
    m, ids, _ = _data(d, 10, n=1500 if d < 10_000 else 700)
    m[100] = m[7]                                                   # an exact duplicate: the best pair, ties ordered by rows
    m[300] = m[7]
    engine.load(m, ids)
    for n in (1, 100, 1000):
        _assert_pairs(engine.top_pairs(n), m, ids, n)
