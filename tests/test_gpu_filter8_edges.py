"""GPU: edges of the int8 filter pass's staged side data (DESIGN.md section 4, K1f8).

The pass copies each tile's row scales (and tombstone bytes) into shared memory with the rows, in 16-byte units, and a
consumer warp scores two rows of a tile at once.  These cases put the last tile's row count off every multiple of 2, 4
and 16, place tombstones in the partial last tile and on tile boundaries (32-row tiles at d = 1536, 16-row tiles at
d = 3072), and append rows in place after the shadow exists, so their scales come in through the staged copy.  Each
case compares SVSB_FILTER=0 (K1) with =8 as uint32 scores, ids and order, through `query` and the bench loop."""
import numpy as np
import pytest

import svs_b200
from _util import oracle
from test_gpu_filter8 import _check_bench, _check_query, _filter_on_small_matrices  # noqa: F401  (autouse fixture)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("d,n", [(1536, n) for n in (3, 4, 15, 16, 17, 63, 64, 65, 100_003)]
                         + [(3072, n) for n in (15, 16, 17, 33, 100_003)])
def test_filter8_partial_last_tile(monkeypatch, d, n):
    m = oracle.synth_matrix_uniform(n, d, 40)
    ids = np.arange(n, dtype=np.int64) + 7
    qs = np.concatenate([oracle.synth_queries(1, d, 41), m[n - 1:n]])      # the last row is the second query's top-1
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        for q in qs:
            for k in sorted({1, min(n, 10), n, 100}):
                _check_query(monkeypatch, e, q, k)
        assert _check_query(monkeypatch, e, qs[1], 1)[1][0] == ids[n - 1]
        _check_bench(monkeypatch, e, qs, min(n, 100))


@pytest.mark.parametrize("d,tile", [(1536, 32), (3072, 16)])
def test_filter8_tombstones_on_tile_edges(monkeypatch, d, tile):
    n = 40 * tile + 7                                            # a partial last tile of 7 rows
    m = oracle.synth_matrix_uniform(n, d, 42)
    ids = np.arange(1, n + 1, dtype=np.int64)
    q = oracle.synth_queries(1, d, 43)[0]
    top = oracle.superheavy(m, ids, q, 5)
    rows = {0, tile - 1, tile, 2 * tile - 1, 2 * tile, 17 * tile, n - 7, n - 5, n - 2, n - 1}
    dels = np.unique(np.array(sorted(rows), dtype=np.int64) + 1)
    dels = np.unique(np.concatenate([dels, np.array([i for _, i in top[:3]], dtype=np.int64)]))
    qs = np.stack([q, m[n - 1], m[tile]])                       # two queries whose top-1 rows are deleted
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        e.apply_mutations(dels, [], None)
        for qq in qs:
            for k in (1, 10, 100, n - len(dels)):
                got = _check_query(monkeypatch, e, qq, k)
                assert not np.isin(got[1], dels).any()
        _check_bench(monkeypatch, e, qs, 100)


@pytest.mark.parametrize("d", [1536, 3072])
def test_filter8_appends_in_place(monkeypatch, d):
    n = 5_000 + 3
    m = oracle.synth_matrix_uniform(n, d, 44)
    ids = np.arange(1, n + 1, dtype=np.int64)
    with svs_b200.Engine([0]) as e:
        e.load(m, ids)
        _check_query(monkeypatch, e, oracle.synth_queries(1, d, 45)[0], 10)       # builds the shadow
        nxt = n + 1
        for count, seed in ((1, 46), (6, 47), (29, 48)):          # in place: the load leaves room for 1024 rows
            add = oracle.synth_matrix_uniform(count, d, seed)
            add_ids = np.arange(nxt, nxt + count, dtype=np.int64)
            nxt += count
            e.apply_mutations([], add_ids, add)
            for i in range(count):
                got = _check_query(monkeypatch, e, add[i], 3)
                assert got[1][0] == add_ids[i]
            _check_bench(monkeypatch, e, add[:4], 50)
        e.apply_mutations(np.array([n, nxt - 1], dtype=np.int64), [], None)      # tombstones over the appended tail
        for q in (m[n - 1], add[-1]):
            got = _check_query(monkeypatch, e, q, 20)
            assert n not in got[1] and nxt - 1 not in got[1]
        _check_bench(monkeypatch, e, np.stack([m[n - 1], add[-1]]), 20)
