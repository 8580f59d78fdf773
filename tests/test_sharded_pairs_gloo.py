"""ShardedRetriever.top_pairs on CPU: 2, 3 and 5 `gloo` ranks with a NumPy backend that restates svsb_pairs_local /
svsb_pairs_merge through the plan, per-device threshold and rank-merge restatement of tests/test_pairs_multi_logic.py.
Exercises the SPMD protocol -- export, descriptor all-gather, connect, one agreed row-norm bound, the status all-gather
that makes every rank refuse alike, the padded list all-gather, the merge, the re-export after a reload -- against the
oracle's top_pairwise on the global matrix, on every rank."""
import os
import pickle
import zlib

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from _util import oracle
from test_pairs_multi_logic import device_list, eps_of, plan, rank_merge, reference
from test_sharded_gloo import NumpyShardBackend, _free_port

from svs_b200 import EngineError
from svs_b200._lib import SVSB_E_INVALID, SVSB_E_NOMEM


class NumpyPairsBackend(NumpyShardBackend):
    """CPU stand-in for CudaShardBackend's svsb_pairs_* wrappers (test infrastructure).  The descriptor carries the
    shard itself (what the peers map over CUDA IPC on the GPU); a rank's pass is test_pairs_multi_logic.device_list over
    its tasks of plan(shard rows), in 16-row blocks."""
    refuse_export = 0                     # SVSB_E_* this rank's export returns (0: none)
    refuse_local = 0                      # ... and its local pass

    def pairs_export(self):
        if self.refuse_export:
            return b"", self.refuse_export, "export refused on purpose", 0.0
        dev = np.abs(np.sqrt((self.m.astype(np.float64) ** 2).sum(axis=1)) - 1.0).max() if len(self.m) else 0.0
        self.exported = (self.row0, self.m.copy(), self.ids.copy())
        return pickle.dumps(self.exported), 0, "", float(np.float32(dev))

    def pairs_connect(self, world, rank, descs):
        shards = [self.exported if r == rank else pickle.loads(d) for r, d in enumerate(descs)]
        for (r0, m, _), (r1, _, _) in zip(shards, shards[1:]):
            assert r1 == r0 + len(m), "row ranges not contiguous in rank order"
        self.world, self.rank = world, rank
        self.shard_rows = [len(m) for _, m, _ in shards]
        self.gm = np.concatenate([m for _, m, _ in shards]).astype(np.float32)
        self.gids = np.concatenate([i for _, _, i in shards]).astype(np.int64)

    def pairs_disconnect(self):
        self.gm = self.gids = None

    def new_pair_lists(self, count, lists=1):
        return (torch.zeros((lists, count), dtype=torch.float32), torch.zeros((lists, count), dtype=torch.int64),
                torch.zeros((lists, count), dtype=torch.int64))

    def pairs_local(self, n, max_row_norm, out):
        if self.refuse_local:
            return self.refuse_local, "local pass refused on purpose", 0
        m = self.gm
        exact = np.dot(m, m.T)
        m16 = (m * np.float32(4096)).astype(np.float16).astype(np.float32)
        coarse = (m16 @ m16.T) / np.float32(4096.0 * 4096.0)
        # the agreed bound is the global one: the margin of the restated pass over the whole matrix
        assert abs(max_row_norm - (1.0 + np.abs(np.sqrt((m.astype(np.float64) ** 2).sum(axis=1)) - 1.0).max())) < 1e-6
        row0 = list(np.cumsum([0] + self.shard_rows[:-1]))
        s, a, b = device_list(m, exact, coarse, row0, self.rank, plan(self.shard_rows)[self.rank], n, 2 * eps_of(m), 16)
        out[0].numpy()[0, :len(s)] = s
        out[1].numpy()[0, :len(s)] = a
        out[2].numpy()[0, :len(s)] = b
        return 0, "", len(s)

    def pairs_merge(self, lists, counts, n, out):
        merged = rank_merge([(lists[0].numpy()[l, :c], lists[1].numpy()[l, :c], lists[2].numpy()[l, :c])
                             for l, c in enumerate(counts)], n)
        for k, (s, a, b) in enumerate(merged):
            out[0].numpy()[0, k] = s
            out[1].numpy()[0, k] = self.gids[a]
            out[2].numpy()[0, k] = self.gids[b]
        return len(merged)


def _unit(rng, n, d):
    m = rng.standard_normal((n, d)).astype(np.float32)
    return (m / np.sqrt((m * m).sum(axis=1))[:, None]).astype(np.float32)


def _case(name, world):
    """(matrix, ids) of a named case; every rank builds the same from the seed."""
    rng = np.random.default_rng(zlib.crc32(f"{name}/{world}".encode()))
    n_rows = {"uneven": 211, "empty_shards": 3, "one_row_shards": 2 * world - 1, "duplicates": 157, "reload": 120}[name]
    m = _unit(rng, n_rows, 16)
    if name == "duplicates":                       # copies of one row on both sides of every rank boundary
        per = -(-n_rows // world)
        src = m[5].copy()
        for r0 in range(per, n_rows, per):
            m[r0 - 1] = src
            m[r0] = src
        m[n_rows - 1] = src
    ids = np.cumsum(rng.integers(1, 4, size=n_rows)).astype(np.int64)
    return np.ascontiguousarray(m), ids


def _check(sr, m, ids, n):
    got = sr.top_pairs(n)
    total = len(m) * (len(m) - 1) // 2
    assert got == reference(m, ids, min(n, total))
    oracle.compare_pairs(got, oracle.top_pairwise(m, ids, n), np.dot(m, m.T), ids)
    return got


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from svs_b200.sharded import ShardedRetriever
        out = []
        sr = ShardedRetriever(rank, world, backend=NumpyPairsBackend())
        for name in ("uneven", "empty_shards", "one_row_shards", "duplicates"):
            m, ids = _case(name, world)
            sr.load_global(m, ids)
            for n in (1, 37, 10 ** 6):                      # 10**6: more than all pairs
                out.append(_check(sr, m, ids, n))
            assert sr.top_pairs(0) == [] and sr.top_pairs(-3) == []
            if name == "duplicates":                       # exact ties across shards come out in row order
                top = sr.top_pairs(3)
                row = {int(x): r for r, x in enumerate(ids)}
                assert [(row[a], row[b]) for _, a, b in top] == sorted((row[a], row[b]) for _, a, b in top)
                assert all(abs(s - 1.0) < 1e-5 for s, _, _ in top)
        # a reload between calls: the next call re-exports and answers from the new rows
        m1, ids1 = _case("reload", world)
        sr.load_global(m1, ids1)
        out.append(_check(sr, m1, ids1, 50))
        m2, ids2 = _case("uneven", world)
        sr.load_global(m2[:150], ids2[:150] + 7)
        out.append(_check(sr, m2[:150], ids2[:150] + 7, 50))
        sr.load_global(m1[:1], ids1[:1])                   # one global row: no pairs
        assert sr.top_pairs(5) == []
        # refusals: one rank refuses, every rank raises the same code, and the next call answers again
        sr.load_global(m1, ids1)
        last = world - 1
        sr.backend.refuse_export = SVSB_E_INVALID if rank == last else 0
        with pytest.raises(EngineError) as ex:
            sr.top_pairs(10)
        assert ex.value.code == SVSB_E_INVALID
        sr.backend.refuse_export = 0
        sr.backend.refuse_local = SVSB_E_NOMEM if rank == 1 else 0
        with pytest.raises(EngineError) as ex:
            sr.top_pairs(10)
        assert ex.value.code == SVSB_E_NOMEM
        sr.backend.refuse_local = 0
        out.append(_check(sr, m1, ids1, 10))
        ret[rank] = out
        sr.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 5])
def test_sharded_top_pairs_match_the_oracle_on_every_rank(world):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    assert len(ret) == world
    for r in range(1, world):
        assert ret[r] == ret[0]                            # every rank holds the identical answer
