"""ShardedRetriever.apply_mutations and compact on CPU: 2, 3 and 4 `gloo` ranks with a NumPy backend that restates
svsb_shard_mutations_prepare / _commit and svsb_compact (tombstones, appends on the last rank, compaction at the prefix
sum of the live counts).  Exercises the collective protocol -- prepare on every rank, one object all-gather of the
outcomes, publish everywhere or drop everywhere -- and the state that follows an update (row count, record capacity of
the large-k path, epochs, the pair path's compaction) against the oracle over a mirror of the live rows, on every rank."""
import numpy as np
import pytest

from _util import oracle
from test_sharded_gloo import np_keys
from test_sharded_large_k_gloo import SortedMergeMixin, _init, _run
from test_sharded_pairs_gloo import NumpyPairsBackend

from svs_b200._lib import SVSB_E_NOMEM, SVSB_E_STATE, EngineError
from svs_b200.sharded import ShardedRetriever

D = 16


class MutatingBackend(SortedMergeMixin, NumpyPairsBackend):
    """Physical rows, ids and a live mask per shard; an update is built off to the side and published or dropped."""
    refuse_prepare = 0                    # SVSB_E_* this rank's prepare raises (0: none)

    def load_rows(self, rows, ids):
        super().load_rows(rows, ids)
        self.live = np.ones(len(ids), bool)
        self.pending = None

    def enqueue_local(self, q, k, record_row, time_kernel=False, seq=0):
        rows = np.nonzero(self.live)[0]
        x = oracle.scores_of(self.m, q.numpy())[rows] if len(self.m) else np.zeros(0, np.float32)
        keys = np_keys(x, self.row0 + rows)                  # tombstoned rows keep their place in the global row order
        order = np.argsort(keys)[::-1][:k]
        rec = record_row.numpy()
        rec[:len(order)] = keys[order].view(np.int64)
        rec[k:k + len(order)] = self.ids[rows[order]]
        rec[2 * k] = len(order)

    def mutations_prepare(self, dels, aids, rows, append_here):
        if self.refuse_prepare:
            raise EngineError(self.refuse_prepare, "prepare refused on purpose")
        if self.pending is not None:
            raise EngineError(SVSB_E_STATE, "an update is pending")
        if len(np.unique(dels)) != len(dels) or (len(aids) > 1 and (np.diff(aids) <= 0).any()):
            raise EngineError(SVSB_E_STATE, "duplicate delete id or inserted ids not ascending")
        hit = self.live & np.isin(self.ids, dels)
        live = self.live & ~hit
        max_live = int(self.ids[live].max()) if live.any() else -2 ** 63
        m, ids = self.m, self.ids
        if append_here and len(aids):
            m, ids = np.concatenate([m.reshape(-1, D), rows]), np.concatenate([ids, aids])
            live = np.concatenate([live, np.ones(len(aids), bool)])
        self.pending = (m, ids, live)
        return int(hit.sum()), max_live

    def mutations_commit(self, publish):
        p, self.pending = self.pending, None
        if publish:
            self.m, self.ids, self.live = p

    def compact(self, global_row0):
        self.m, self.ids = np.ascontiguousarray(self.m[self.live]), self.ids[self.live]
        self.live = np.ones(len(self.ids), bool)
        self.row0 = global_row0

    def pairs_export(self):
        assert self.live.all(), "the pair search was asked for on a tombstoned shard"
        return super().pairs_export()


class Mirror:
    """The live rows in global row order, as a fresh load would hold them."""

    def __init__(self, m, ids):
        self.m, self.ids = m.copy(), ids.copy()

    def apply(self, dels, aids, rows):
        keep = ~np.isin(self.ids, dels)
        self.m, self.ids = self.m[keep], self.ids[keep]
        if len(aids):
            self.m, self.ids = np.concatenate([self.m, rows]), np.concatenate([self.ids, aids])


def _rows(rng, n):
    m = rng.standard_normal((n, D)).astype(np.float32)
    return (m / np.sqrt((m * m).sum(axis=1))[:, None]).astype(np.float32)


def _check(sr, mirror, qs, ks=(1, 10, 64)):
    out = []
    for k in ks:
        for q in qs:
            got = sr.retrieve(q, k)
            want = oracle.superheavy(mirror.m, mirror.ids, q, k)
            assert len(got) == len(want) == min(k, len(mirror.ids))
            oracle.compare_retrieval(got, want, oracle.scores_of(mirror.m, q), mirror.ids)
            out.append(got)
    many = sr.retrieve_many(qs, 10)
    assert many == [sr.retrieve(q, 10) for q in qs]
    assert sr.n == len(mirror.ids) and sum(sr._shard_live) == sr.n
    return out + [many]


def _update(sr, mirror, dels, aids, rows):
    sr.apply_mutations(dels, aids, rows)
    mirror.apply(np.asarray(dels, np.int64), np.asarray(aids, np.int64), rows)


def _refused(sr, code, dels, aids, rows):
    with pytest.raises(EngineError) as ex:
        sr.apply_mutations(dels, aids, rows)
    assert ex.value.code == code
    return ex.value.message


def _worker(rank, world, port, ret):
    _init(rank, world, port)
    try:
        rng = np.random.default_rng(1000 + world)               # every rank draws the same data
        out = []
        sr = ShardedRetriever(rank, world, backend=MutatingBackend())
        n = 300
        m = _rows(rng, n)
        ids = np.cumsum(rng.integers(1, 4, size=n)).astype(np.int64)
        mirror = Mirror(m, ids)
        sr.load_global(m, ids)
        qs = np.concatenate([oracle.synth_queries(3, D, 5, "normal"), m[[7, n - 3]]])
        out += _check(sr, mirror, qs)
        # deletes spread over every rank (fewer than the compaction fraction: tombstones stay)
        per = -(-n // world)
        dels = [int(ids[r * per + 3]) for r in range(world)] + [int(ids[n - 1])]
        _update(sr, mirror, dels, [], None)
        assert sum(sr._shard_rows) == n and sr.n == n - len(dels)
        out += _check(sr, mirror, qs)
        # delete and re-insert the largest id in one update, with two more appends behind it
        top = int(mirror.ids.max())
        add = _rows(rng, 3)
        _update(sr, mirror, [top], [top, top + 1, top + 5], add)
        out += _check(sr, mirror, qs)
        # refusals: every rank raises the same error and the next call answers from the unchanged state
        msgs = [_refused(sr, SVSB_E_STATE, [int(ids[0]), 10 ** 9], [], None),                 # an unknown delete id
                _refused(sr, SVSB_E_STATE, [], [top + 5], _rows(rng, 1)),                    # not above the global maximum
                _refused(sr, SVSB_E_STATE, [], [int(ids[0]) + 0], _rows(rng, 1))]
        sr.backend.refuse_prepare = SVSB_E_NOMEM if rank == world // 2 else 0             # one rank's prepare refuses
        msgs.append(_refused(sr, SVSB_E_NOMEM, [int(mirror.ids[0])], [top + 9], _rows(rng, 1)))
        sr.backend.refuse_prepare = 0
        out += [msgs] + _check(sr, mirror, qs)
        # every row of rank 0 deleted: past the drop-in's dead-row fraction the shards are compacted
        own0 = [int(i) for i in ids[:per] if i in set(mirror.ids.tolist())]
        _update(sr, mirror, own0, [], None)
        assert sr._shard_rows == sr._shard_live and sr._shard_live[0] == 0
        assert sr.row0 == sum(sr._shard_live[:rank])
        out += _check(sr, mirror, qs)
        # the last shard grows past every other: the large-k path's record capacity follows it
        big = mirror.ids.max() + 1 + np.arange(2600, dtype=np.int64) * 2
        _update(sr, mirror, [], big, _rows(rng, len(big)))
        assert max(sr._shard_live) == sr._shard_live[-1] > -(-sr.n // world)
        for k in (2049, 2500, 10 ** 9):
            for q in qs[:2]:
                got = sr.retrieve(q, k)
                want = oracle.superheavy(mirror.m, mirror.ids, q, k)
                assert len(got) == min(k, sr.n)
                oracle.compare_retrieval(got, want, oracle.scores_of(mirror.m, q), mirror.ids)
                out.append(got)
        assert sr._big[0] == min(10 ** 9, sr._shard_live[-1])
        # deletes that hit appended rows, then top_pairs: it compacts first (the export asserts no tombstones)
        _update(sr, mirror, [int(big[0]), int(big[7]), int(mirror.ids[1])], [], None)
        assert sum(sr._shard_rows) > sr.n
        got = sr.top_pairs(25)
        oracle.compare_pairs(got, oracle.top_pairwise(mirror.m, mirror.ids, 25), np.dot(mirror.m, mirror.m.T), mirror.ids)
        assert sr._shard_rows == sr._shard_live
        out += [got] + _check(sr, mirror, qs)
        # compact on demand of an already compact matrix changes nothing
        sr.compact()
        out += _check(sr, mirror, qs[:2])
        ret[rank] = out
    finally:
        import torch.distributed as dist
        dist.destroy_process_group()


def _tiny_worker(rank, world, port, ret):
    """n < world: the last shard starts empty and takes every append."""
    _init(rank, world, port)
    try:
        rng = np.random.default_rng(77)
        m = _rows(rng, 2)
        ids = np.array([4, 9], np.int64)
        mirror = Mirror(m, ids)
        sr = ShardedRetriever(rank, world, backend=MutatingBackend())
        sr.load_global(m, ids)
        assert sr._shard_live[-1] == 0
        qs = oracle.synth_queries(3, D, 8, "normal")
        out = _check(sr, mirror, qs, ks=(1, 5))
        add = _rows(rng, 5)
        _update(sr, mirror, [], [10, 11, 15, 16, 20], add)
        assert sr._shard_live[-1] == 5
        out += _check(sr, mirror, qs, ks=(1, 3, 100))
        _update(sr, mirror, [4, 9, 15], [21], _rows(rng, 1))
        out += _check(sr, mirror, qs, ks=(1, 3, 100))
        ret[rank] = out
    finally:
        import torch.distributed as dist
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_sharded_mutations_match_the_oracle_on_every_rank(world):
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    _run(_worker, world, (ret,))
    assert len(ret) == world
    for r in range(1, world):
        assert ret[r] == ret[0]                                 # every rank holds the identical answers


def test_appends_onto_an_empty_last_shard():
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    _run(_tiny_worker, 4, (ret,))
    assert len(ret) == 4 and all(ret[r] == ret[0] for r in range(4))
