"""CPU: the bit-exact K1 reference (oracle/k1_exact.py) checked against rational arithmetic and brute force.

The GPU suites compare every exact path with this reference bit for bit, so it must itself be right: its FMA against
fractions.Fraction (random operands and constructed cases where a float64 product-sum rounded to fp32 rounds twice),
its summation order against test_filter8_bound.k1_scores on data where no double rounding can occur, and its
prefiltered top-k and top-pairs against emulating every row or pair."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import k1_exact as kx  # noqa: E402
from test_filter8_bound import k1_scores  # noqa: E402

F32 = np.float32


def _naive_fma(acc, a, b):
    return (acc.astype(np.float64) + a.astype(np.float64) * b.astype(np.float64)).astype(F32)


def _random_operands(rng, n):
    """fp32 operands over many binades, both signs, some zeros and subnormals."""
    def one():
        m = rng.uniform(1.0, 2.0, n)
        e = rng.integers(-40, 40, n).astype(float)
        e[rng.random(n) < 0.05] = -140.0                          # products and sums in the subnormal range
        x = (m * np.exp2(e) * rng.choice([-1.0, 1.0], n)).astype(F32)
        x[rng.random(n) < 0.02] = 0.0
        return x
    return one(), one(), one()


def test_fma_matches_rational_arithmetic_on_random_operands():
    rng = np.random.default_rng(1)
    acc, a, b = _random_operands(rng, 20_000)
    # a share of sums with cancellation: acc close to -a*b
    c = rng.random(len(acc)) < 0.2
    acc[c] = (-(a[c].astype(np.float64) * b[c].astype(np.float64))).astype(F32)
    got = kx.fma32(acc, a, b)
    want = np.array([kx.fma_fraction(x, y, z) for x, y, z in zip(acc, a, b)], F32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def _midpoint_cases(rng, n):
    """acc + a*b = acc + h (1 +- 2^-30) with h half an fp32 ulp of acc: the float64 sum lands exactly on the fp32
    midpoint and a single float64 -> fp32 rounding goes the wrong way for half of them (ties to even)."""
    acc = (rng.uniform(1.0, 2.0, n) * np.exp2(rng.integers(-60, 60, n).astype(float))).astype(F32)
    sign = rng.choice([-1.0, 1.0], n)
    acc = (acc * sign).astype(F32)
    e = np.floor(np.log2(np.abs(acc.astype(np.float64)))).astype(int)        # acc in [2^e, 2^(e+1))
    plus = rng.random(n) < 0.5
    fa = np.where(plus, 1025.0, 32769.0)                           # 1025 * 1047553 = 2^30 + 1
    fb = np.where(plus, 1047553.0, 32767.0)                        # 32769 * 32767 = 2^30 - 1
    split = rng.integers(-20, 20, n)
    a = (fa * np.exp2(split.astype(float))).astype(F32)
    b = (fb * np.exp2((e - 54 - split).astype(float)) * sign * rng.choice([-1.0, 1.0], n)).astype(F32)
    return acc, a, b


def test_fma_rounds_constructed_midpoints_like_rational_arithmetic():
    rng = np.random.default_rng(2)
    acc, a, b = _midpoint_cases(rng, 4000)
    got = kx.fma32(acc, a, b)
    want = np.array([kx.fma_fraction(x, y, z) for x, y, z in zip(acc, a, b)], F32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    wrong = (_naive_fma(acc, a, b).view(np.uint32) != want.view(np.uint32)).sum()
    assert wrong > 500, wrong                                      # the cases really are double roundings


def test_fma_special_values():
    big = F32(3.0e38)
    cases = [(F32(0.0), F32(-0.0), F32(1.0)), (F32(-0.0), F32(-0.0), F32(1.0)), (F32(-0.0), F32(0.0), F32(1.0)),
             (F32(1.0), F32(1.0), F32(-1.0)), (big, big, F32(1.0)), (big, F32(2.0), F32(1.7e38)),
             (F32(-big), F32(-2.0), F32(1.7e38)), (F32(1e-45), F32(1e-30), F32(1e-20)),
             (F32(3.4028235e38), F32(1.0), F32(1.0141204e31))]     # FLT_MAX + half an ulp: overflows to inf
    for acc, a, b in cases:
        got = kx.fma32(np.array([acc]), np.array([a]), np.array([b]))[0]
        want = kx.fma_fraction(acc, a, b)
        assert np.array_equal(np.array([got]).view(np.uint32), np.array([want]).view(np.uint32)), (acc, a, b, got, want)


@pytest.mark.parametrize("d", [1, 3, 4, 5, 127, 128, 129, 190, 1537, 3073, 12801])
def test_k1_exact_equals_the_float64_restatement_where_it_rounds_once(d):
    """Components with 12 significant bits: every product is exact in fp32 and every float64 product-sum is exact, so
    k1_scores' one rounding per FMA is a true FMA and the two restatements must agree bit for bit."""
    rng = np.random.default_rng(d)
    n = 64 if d > 3000 else 300
    s = int(np.ceil(np.log2(np.sqrt(d))))                          # rows of norm ~1, still 12-bit values
    M = (rng.integers(-2048, 2049, (n, d)) * 2.0 ** (-11 - s)).astype(F32)
    q = (rng.integers(-2048, 2049, d) * 2.0 ** -11).astype(F32)
    ld = (d + 3) & ~3
    Mp = np.zeros((n, ld), F32); Mp[:, :d] = M
    qp = np.zeros(ld, F32); qp[:d] = q
    assert np.array_equal(kx.k1_exact(M, q).view(np.uint32), k1_scores(Mp, qp).view(np.uint32))


def test_k1_exact_differs_from_one_accumulator_per_lane_above_128():
    """The order matters: one float4 accumulator per lane (the LDG kernel's order before it took K1's) gives other
    bits for most rows once a lane owns two chunks (d > 128), and the same bits up to d = 128."""
    def one_acc(M, q):
        n, d = M.shape
        ld = (d + 3) & ~3
        nch = -(-(ld // 4) // 32)
        Mp = np.zeros((n, nch * 128), F32); Mp[:, :d] = M
        qp = np.zeros(nch * 128, F32); qp[:d] = q
        acc = np.zeros((n, 32, 4), F32)
        for j in range(nch):
            acc = kx.fma32(acc, Mp.reshape(n, nch, 32, 4)[:, j], qp.reshape(nch, 32, 4)[j][None])
        v = (acc[..., 0] + acc[..., 1]) + (acc[..., 2] + acc[..., 3])
        for o in (16, 8, 4, 2, 1):
            v = v + v[:, np.arange(32) ^ o]
        return v[:, 0]
    rng = np.random.default_rng(7)
    for d, same in ((128, True), (1536, False)):
        M = rng.standard_normal((200, d)).astype(F32)
        q = rng.standard_normal(d).astype(F32)
        eq = kx.k1_exact(M, q).view(np.uint32) == one_acc(M, q).view(np.uint32)
        assert eq.all() if same else eq.mean() < 0.5


@pytest.mark.parametrize("case", ["normal", "ties", "tombstones", "k_above_live", "negative"])
def test_prefiltered_topk_equals_brute_force(case):
    rng = np.random.default_rng(len(case))
    n, d = 700, 37
    M = rng.standard_normal((n, d)).astype(F32)
    M /= np.sqrt((M.astype(np.float64) ** 2).sum(axis=1)).astype(F32)[:, None]
    q = rng.standard_normal(d).astype(F32)
    live = None
    if case == "ties":
        M[::7] = M[3]                                              # bit-equal scores: ordered by row
    if case in ("tombstones", "k_above_live"):
        live = rng.random(n) < (0.6 if case == "tombstones" else 0.05)
    if case == "negative":
        q = -np.abs(q); M = np.abs(M)                              # every score negative
    ids = np.cumsum(rng.integers(1, 5, n)).astype(np.int64)
    for k in (1, 10, 100, n, n + 5):
        b1, i1 = kx.k1_topk_exact(M, ids, q, k, live)
        b2, i2 = kx.k1_topk_brute(M, ids, q, k, live)
        assert np.array_equal(b1, b2) and np.array_equal(i1, i2), k
    if live is not None and k >= n:
        assert (b1[len(b1) - (~live).sum():] == kx.DEAD_BITS).all()


def test_pairs_reference_equals_brute_force():
    rng = np.random.default_rng(11)
    N, d = 90, 70
    M = rng.standard_normal((N, d)).astype(F32)
    M /= np.sqrt((M.astype(np.float64) ** 2).sum(axis=1)).astype(F32)[:, None]
    M[40] = M[3]; M[50] = M[3]                                     # identical rows: tied pair scores
    ids = np.arange(100, 100 + N, dtype=np.int64)
    ia, ib = np.triu_indices(N, k=1)
    sc = np.array([kx.pair_exact(M, i, j) for i, j in zip(ia, ib)], F32).view(np.uint32)
    order = np.lexsort((ib, ia, ~kx.ordered(sc)))
    for n in (1, 25, 600, len(ia), len(ia) + 3):
        got = kx.top_pairs_exact(M, ids, n)
        want = [(int(sc[o]), int(ids[ia[o]]), int(ids[ib[o]])) for o in order[:n]]
        assert got == want, n
    # row i plays the query; the product commutes, so the score is symmetric
    assert kx.pair_exact(M, 5, 9) == kx.pair_exact(M, 9, 5)
