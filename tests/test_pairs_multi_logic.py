"""The LOGIC of the multi-device pair search (multi.cu: multi_top_pairs), restated in NumPy and driven on adversarial data:
the static plan over shard pairs (engine.cu: pairs_plan), each device's pass over its tasks in 1024-row blocks (smaller
here) with its OWN running threshold on fp16-rounded coarse scores, the exact re-score, each device's top min(n, count)
list, and device 0's rank merge.  Whatever the data -- every top pair inside one shard or in one cross block, duplicate
rows across shard boundaries, more pairs asked than exist -- the result must equal the exact top n of np.dot(M, M.T) under
the engine's order (score desc, first row asc, second row asc), and pass oracle.compare_pairs against oracle.top_pairwise."""
import bisect
import zlib

import numpy as np
import pytest

from _util import oracle


def plan(shard_rows):
    """engine.cu: pairs_plan.  Task = (peer, m0, m1, q0, q1): own rows [m0, m1) x peer rows [q0, q1); peer == self is the
    upper triangle of the own shard."""
    G = len(shard_rows)
    tasks = [[] for _ in range(G)]

    def add(dev, peer, m0, m1, q0, q1):
        if m1 > m0 and q1 > q0 and (peer != dev or m1 - m0 >= 2):
            tasks[dev].append((peer, m0, m1, q0, q1))
    for a in range(G):
        add(a, a, 0, shard_rows[a], 0, shard_rows[a])
        for t in range(1, (G + 1) // 2):
            b = (a + t) % G
            add(a, b, 0, shard_rows[a], 0, shard_rows[b])
    if G % 2 == 0:
        for a in range(G // 2):
            b = a + G // 2
            h = shard_rows[b] // 2
            add(a, b, 0, shard_rows[a], 0, h)
            add(b, a, h, shard_rows[b], 0, shard_rows[a])
    return tasks


def shards(n, G):
    """engine.cu: alloc_generation -- ceil(n / G) rows per device in scan order, the last devices may get fewer or none."""
    per = -(-n // G)
    row0 = [min(n, i * per) for i in range(G)]
    return row0, [min(n, (i + 1) * per) - row0[i] for i in range(G)]


def task_pairs(row0, dev, task):
    """The (global row, global row) pairs a task covers, as (smaller, larger)."""
    peer, m0, m1, q0, q1 = task
    if peer == dev:
        r = np.arange(row0[dev], row0[dev] + m1)
        i, j = np.triu_indices(len(r), k=1)
        return r[i], r[j]
    a = np.repeat(np.arange(row0[dev] + m0, row0[dev] + m1), q1 - q0)
    b = np.tile(np.arange(row0[peer] + q0, row0[peer] + q1), m1 - m0)
    return np.minimum(a, b), np.maximum(a, b)


def task_work(task, dev):
    peer, m0, m1, q0, q1 = task
    return (m1 - m0) * (m1 - m0 - 1) // 2 if peer == dev else (m1 - m0) * (q1 - q0)


SHARD_SETS = {
    "equal": lambda G: [60] * G,
    "unequal": lambda G: [7 + 13 * i for i in range(G)],
    "empty_and_one_row": lambda G: [0 if i % 3 == 1 else (1 if i % 3 == 2 else 25) for i in range(G)],
}


@pytest.mark.parametrize("kind", list(SHARD_SETS))
@pytest.mark.parametrize("G", range(1, 9))
def test_the_plan_covers_every_pair_exactly_once(G, kind):
    rows = SHARD_SETS[kind](G)
    N = sum(rows)
    row0 = list(np.cumsum([0] + rows[:-1]))
    cover = np.zeros((N, N), np.int64)
    tasks = plan(rows)
    for dev in range(G):
        for t in tasks[dev]:
            i, j = task_pairs(row0, dev, t)
            np.add.at(cover, (i, j), 1)
    iu = np.triu_indices(N, k=1)
    assert (cover[iu] == 1).all()
    assert cover.sum() == N * (N - 1) // 2                        # nothing on or below the diagonal
    if kind == "equal":
        work = [sum(task_work(t, dev) for t in tasks[dev]) for dev in range(G)]
        assert max(work) <= 1.05 * (N * (N - 1) / 2) / G


def test_the_plan_balances_large_equal_shards():
    for G in range(1, 9):
        s = 125_000
        tasks = plan([s] * G)
        work = [sum(task_work(t, dev) for t in tasks[dev]) for dev in range(G)]
        total = G * s * (G * s - 1) // 2
        assert sum(work) == total
        assert max(work) <= 1.0001 * total / G


# ---- the pass, per device --------------------------------------------------------------------------------------------
def ordered(scores):
    """common.cuh: f32_to_ordered -- the engine's total order on fp32 scores as uint32."""
    b = np.asarray(scores, np.float32).view(np.uint32).astype(np.uint64)
    return np.where(b & 0x80000000, ~b & 0xffffffff, b | 0x80000000).astype(np.uint64)


def eps_of(m):
    """engine.cu: top_pairs_gen's error bound of the fp16 coarse score."""
    d = m.shape[1]
    R = np.float32(1.0) + np.float32(np.abs(np.sqrt((m.astype(np.float64) ** 2).sum(axis=1)) - 1.0).max())
    coef = np.float32(9.765625e-4 + 2.384185791015625e-7 + d * (2.384185791015625e-7 + 1.1920928955078125e-7))
    return float(coef * (R * np.float32(1.000001)) ** 2 + np.float32(1e-8))


def engine_order(s, i, j):
    """indices sorting (score desc, i asc, j asc)"""
    return np.lexsort((j, i, -ordered(s).astype(np.int64)))


def device_list(m, exact, coarse, row0, dev, tasks, n, eps2, block):
    """One device: blocks of `block` query rows, running threshold = (n-th largest coarse seen) - 2 eps, compaction; then
    the exact re-score of the survivors and their top min(n, count) in the engine's order."""
    thr = -np.inf
    li = np.zeros(0, np.int64); lj = np.zeros(0, np.int64); lo = np.zeros(0, np.float32)
    for peer, m0, m1, q0, q1 in tasks:
        if peer == dev:
            blocks = [(q, min(q + block, m1)) for q in range(0, m1 - 1, block)]
        else:
            blocks = [(q, min(q + block, q1)) for q in range(q0, q1, block)]
        for b0, b1 in blocks:
            if peer == dev:          # queries b0..b1 of the own shard against every later row of it
                qi = np.repeat(np.arange(b0, b1), m1); mj = np.tile(np.arange(m1), b1 - b0)
                keep = mj > qi
                gi, gj = row0[dev] + qi[keep], row0[dev] + mj[keep]
            else:
                qi = np.repeat(np.arange(b0, b1), m1 - m0); mj = np.tile(np.arange(m0, m1), b1 - b0)
                a, b = row0[peer] + qi, row0[dev] + mj
                gi, gj = np.minimum(a, b), np.maximum(a, b)
            c = coarse[gi, gj]
            sel = c >= thr
            li = np.concatenate([li, gi[sel]]); lj = np.concatenate([lj, gj[sel]]); lo = np.concatenate([lo, c[sel]])
            if len(lo) >= n:
                thr = max(thr, float(np.sort(lo)[-n]) - eps2)
                keep = lo >= thr
                li, lj, lo = li[keep], lj[keep], lo[keep]
    s = exact[li, lj]
    o = engine_order(s, li, lj)[:min(n, len(li))]
    return s[o], li[o], lj[o]


def rank_merge(lists, n):
    """select.cu: merge_sorted_pairs_kernel -- an entry's rank is its index in its own list plus, per other list, the
    number of entries ahead of it (binary search under the 96-bit key)."""
    total = sum(len(s) for s, _, _ in lists)
    kk = min(n, total)
    out = [None] * kk
    keyed = [[((-int(o), int(a), int(b))) for o, a, b in zip(ordered(s), i, j)] for s, i, j in lists]
    for l, (s, i, j) in enumerate(lists):
        for p, key in enumerate(keyed[l]):
            rank = p + sum(bisect.bisect_left(keyed[m], key) for m in range(len(lists)) if m != l)
            if rank < kk:
                assert out[rank] is None
                out[rank] = (s[p], int(i[p]), int(j[p]))
    assert all(x is not None for x in out)
    return out


def multi_top_pairs(m, ids, G, n, block=16):
    N = len(m)
    total = N * (N - 1) // 2
    n = min(n, total)
    exact = np.dot(m, m.T)                                         # the oracle's matrix: re-scores are exact by construction
    m16 = (m * np.float32(4096)).astype(np.float16).astype(np.float32)
    coarse = (m16 @ m16.T) / np.float32(4096.0 * 4096.0)
    eps = eps_of(m)
    iu = np.triu_indices(N, k=1)
    assert np.abs(coarse[iu] - exact[iu]).max() <= eps                 # the margin the thresholds rely on
    row0, rows = shards(N, G)
    tasks = plan(rows)
    lists = [device_list(m, exact, coarse, row0, dev, tasks[dev], n, 2 * eps, block) for dev in range(G)]
    assert sum(len(s) for s, _, _ in lists) >= n
    return [(float(s), int(ids[a]), int(ids[b])) for s, a, b in rank_merge(lists, n)]


def reference(m, ids, n):
    """exact top n of the upper triangle of np.dot(M, M.T) under the engine's order"""
    N = len(m)
    i, j = np.triu_indices(N, k=1)
    s = np.dot(m, m.T)[i, j]
    o = engine_order(s, i, j)[:n]
    return [(float(s[x]), int(ids[i[x]]), int(ids[j[x]])) for x in o]


def _unit(rng, n, d):
    m = rng.standard_normal((n, d)).astype(np.float32)
    return (m / np.sqrt((m * m).sum(axis=1))[:, None]).astype(np.float32)


CASES = ["random", "all_top_in_one_shard", "all_top_in_one_cross_block", "duplicates_across_boundaries", "n_above_pairs"]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("G", [1, 2, 3, 5, 8])
def test_the_merged_answer_is_exact(case, G):
    rng = np.random.default_rng(zlib.crc32(f"{case}/{G}".encode()))
    N, d, n = 211, 16, 60
    m = _unit(rng, N, d)
    row0, rows = shards(N, G)
    if case == "all_top_in_one_shard":               # the last non-empty shard's rows are near-copies of one vector
        last = max(i for i in range(G) if rows[i] > 0)
        base = m[0]
        near = base[None, :] + 0.02 * rng.standard_normal((rows[last], d)).astype(np.float32)
        m[row0[last]:row0[last] + rows[last]] = near / np.linalg.norm(near, axis=1)[:, None]
    elif case == "all_top_in_one_cross_block":       # rows 2..9 (first shard) have near-copies at the end (last shard)
        base = _unit(rng, 1, d)[0]
        a = base[None, :] + 0.5 * _unit(rng, 8, d)
        a /= np.linalg.norm(a, axis=1)[:, None]
        b = a + 1e-3 * rng.standard_normal((8, d)).astype(np.float32)
        m[2:10] = a
        m[N - 9:N - 1] = b / np.linalg.norm(b, axis=1)[:, None]
        n = 8
    elif case == "duplicates_across_boundaries":     # exact ties: copies of one row on both sides of every boundary
        src = m[5].copy()
        for r0 in row0[1:]:
            for r in (r0 - 1, r0):
                if 0 <= r < N:
                    m[r] = src
        m[N - 1] = src
    elif case == "n_above_pairs":
        N = 23
        m = m[:N]
        n = N * (N - 1) // 2 + 40
    m = np.ascontiguousarray(m, dtype=np.float32)
    ids = np.cumsum(rng.integers(1, 4, size=len(m))).astype(np.int64)
    got = multi_top_pairs(m, ids, G, n)
    want = reference(m, ids, min(n, len(m) * (len(m) - 1) // 2))
    assert got == want
    if case == "all_top_in_one_cross_block":
        assert sorted((int(np.searchsorted(ids, a)), int(np.searchsorted(ids, b))) for _, a, b in want) == \
            [(2 + k, N - 9 + k) for k in range(8)]
    oracle.compare_pairs(got, oracle.top_pairwise(m, ids, n), np.dot(m, m.T), ids)


def test_a_device_that_sees_fewer_than_n_pairs_keeps_all_of_them():
    """5 rows on 8 devices: most devices have no pairs; the few that do keep everything (threshold stays at -inf)."""
    rng = np.random.default_rng(9)
    m = _unit(rng, 5, 8)
    ids = np.arange(10, 15, dtype=np.int64)
    for n in (1, 4, 10, 11, 50):
        assert multi_top_pairs(m, ids, 8, n, block=2) == reference(m, ids, min(n, 10))
