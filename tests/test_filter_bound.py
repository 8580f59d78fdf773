"""CPU: the fp16 filter's error bound and candidate set (DESIGN.md section 4, K1f), restated in NumPy.

The coarse score is what gemv16_tma_kernel computes: rows rounded to fp16 after the 2^12 scale, the fp32 query, fp32
FMAs in the kernel's lane / accumulator layout, the warp's xor tree, x 2^-12.  The exact score is K1's fp32 arithmetic
(gemv_tma_kernel).  FMAs are emulated as one float64 product-sum rounded to fp32.  On adversarial data this checks
|coarse - exact| <= eps for every row and that the rows with coarse >= T (the threshold filter_threshold_kernel derives
from the group maxima) contain the exact top-k."""
import numpy as np
import pytest

SCALE = np.float32(4096.0)


def eps_coef(d):
    f = np.float32
    return f(f(9.765625e-4) + f(2.384185791015625e-7)) + f(d) * f(f(2.384185791015625e-7) + f(1.1920928955078125e-7))


def _fma(acc, a, b):
    return (acc.astype(np.float64) + a.astype(np.float64) * b.astype(np.float64)).astype(np.float32)


def _combine_and_tree(a0, a1):
    f = np.float32
    v = ((a0[..., 0] + a1[..., 0]).astype(f) + (a0[..., 1] + a1[..., 1]).astype(f)).astype(f) + \
        ((a0[..., 2] + a1[..., 2]).astype(f) + (a0[..., 3] + a1[..., 3]).astype(f)).astype(f)
    v = v.astype(f)                                                  # [n, 32]
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = (v + v[:, lanes ^ o]).astype(f)
    return v[:, 0]


def k1_scores(M, q):
    """gemv_tma_kernel: lane l owns float4 chunks l, l+32, ...; even chunks into a0, odd into a1."""
    n, ld = M.shape
    d4 = ld // 4
    nq = -(-d4 // 32)
    Mp = np.zeros((n, nq * 32 * 4), np.float32); Mp[:, :ld] = M
    qp = np.zeros(nq * 32 * 4, np.float32); qp[:ld] = q
    Mc = Mp.reshape(n, nq, 32, 4); qc = qp.reshape(nq, 32, 4)
    a = [np.zeros((n, 32, 4), np.float32), np.zeros((n, 32, 4), np.float32)]
    for j in range(nq):
        a[j & 1] = _fma(a[j & 1], Mc[:, j], qc[j][None])
    return _combine_and_tree(a[0], a[1])


def filter_scores(M, q):
    """gemv16_tma_kernel: lane l owns 8-half chunks l, l+32, ...; halfs 0-3 into a0 (query floats 8c..8c+3), 4-7 into a1."""
    n, ld = M.shape
    ld16 = (ld + 7) & ~7
    c16 = ld16 // 8
    nc = -(-c16 // 32)
    H = np.zeros((n, nc * 32 * 8), np.float32)
    H[:, :ld] = (M * SCALE).astype(np.float16).astype(np.float32)
    qp = np.zeros(nc * 32 * 8, np.float32); qp[:ld] = q
    Hc = H.reshape(n, nc, 32, 2, 4); qc = qp.reshape(nc, 32, 2, 4)
    a0 = np.zeros((n, 32, 4), np.float32); a1 = np.zeros((n, 32, 4), np.float32)
    for j in range(nc):
        a0 = _fma(a0, Hc[:, j, :, 0], qc[j, :, 0][None])
        a1 = _fma(a1, Hc[:, j, :, 1], qc[j, :, 1][None])
    return (_combine_and_tree(a0, a1) * np.float32(1.0 / 4096.0)).astype(np.float32)


def group_shift_for(n):
    s = 6
    while ((n + (1 << s) - 1) >> s) > 16384:
        s += 1
    return s


def threshold(coarse, kk, eps):
    """filter_threshold_kernel: (kk-th largest group maximum) - 2 eps, rounded down; None = every row."""
    n = len(coarse)
    m = 1 << group_shift_for(n)
    G = -(-n // m)
    pad = np.full(G * m, -np.inf, np.float32); pad[:n] = coarse
    gmax = pad.reshape(G, m).max(axis=1)
    if G <= kk or not np.isfinite(eps):
        return None
    tau = np.sort(gmax)[::-1][kk - 1]
    t = np.float32(np.float64(tau) - 2.0 * np.float64(eps))
    if np.float64(t) > np.float64(tau) - 2.0 * np.float64(eps):
        t = np.nextafter(t, np.float32(-np.inf))
    return t


def exact_topk_rows(exact, k):
    order = np.lexsort((np.arange(len(exact)), -exact.astype(np.float64)))
    return order[:k]


def check(M, q, k):
    n, d = M.shape
    ld = (d + 3) & ~3
    Mp = np.zeros((n, ld), np.float32); Mp[:, :d] = M
    qp = np.zeros(ld, np.float32); qp[:d] = q
    exact = k1_scores(Mp, qp)
    coarse = filter_scores(Mp, qp)
    R = np.float32((1.0 + np.abs(np.linalg.norm(M.astype(np.float64), axis=1) - 1.0).max()) * 1.000001)
    assert R <= 8.0 * 1.000001
    qn = np.float32(np.sqrt(np.sum(qp.astype(np.float32) ** 2, dtype=np.float32)))
    eps = np.float64(eps_coef(d)) * np.float64(qn) * np.float64(R) + 1e-8
    err = np.abs(coarse.astype(np.float64) - exact.astype(np.float64))
    assert err.max() <= eps, (err.max(), eps)
    T = threshold(coarse, k, eps)
    cand = np.ones(n, bool) if T is None else coarse >= T
    top = exact_topk_rows(exact, k)
    assert cand[top].all(), (int((~cand[top]).sum()), T)
    return int(cand.sum())


def _unit(x):
    return (x / np.linalg.norm(x.astype(np.float64), axis=1, keepdims=True)).astype(np.float32)


@pytest.mark.parametrize("d", [100, 768])
def test_uniform_rows_as_the_bench(d):
    rng = np.random.default_rng(1)
    M = _unit(rng.random((8192, d), dtype=np.float32))
    q = _unit(rng.random((1, d), dtype=np.float32))[0]
    c = check(M, q, 100)
    assert c < 8192 // 4                       # the filter really filters


def test_near_ties():
    rng = np.random.default_rng(2)
    d = 256
    base = _unit(rng.random((1, d), dtype=np.float32))
    M = _unit(base + rng.standard_normal((6000, d)).astype(np.float32) * np.float32(1e-6))
    q = _unit(base + rng.standard_normal((1, d)).astype(np.float32) * np.float32(1e-3))[0]
    for k in (1, 100, 1000):
        check(M, q, k)


def test_rows_sorted_by_similarity():
    rng = np.random.default_rng(3)
    d = 384
    M = _unit(rng.standard_normal((8192, d)).astype(np.float32))
    q = _unit(rng.standard_normal((1, d)).astype(np.float32))[0]
    M = M[np.argsort(M @ q)]
    for k in (1, 100, 1000):
        check(M, q, k)
    check(M[::-1].copy(), q, 100)


def test_subnormal_range_components():
    """Components below 2^-26: their scaled fp16 value is subnormal (or zero), an absolute rounding error."""
    rng = np.random.default_rng(4)
    d = 200
    M = rng.standard_normal((4096, d)).astype(np.float32)
    tiny = rng.random((4096, d)) < 0.7
    M[tiny] *= np.float32(2.0 ** -30)
    M = _unit(M)
    M[:, :150] *= np.float32(2.0 ** -28)       # most of every row in the fp16 subnormal range after the scale
    M = _unit(M)
    q = rng.standard_normal(d).astype(np.float32)
    q /= np.float32(np.linalg.norm(q))
    for k in (1, 100):
        check(M, q, k)
    check(M, q * np.float32(1e3), 100)         # a long query: eps grows with ||q||


def test_row_norm_at_the_limit():
    rng = np.random.default_rng(5)
    d = 512
    M = _unit(rng.standard_normal((4096, d)).astype(np.float32))
    M *= rng.uniform(0.1, 8.0, (4096, 1)).astype(np.float32)
    M[7] = 0.0
    M[7, 3] = 8.0                              # 8 * 2^12 = 32768: the largest power of two below fp16's max
    q = _unit(rng.standard_normal((1, d)).astype(np.float32))[0]
    for k in (1, 100, 1000):
        check(M, q, k)


def test_identical_rows_take_every_row():
    rng = np.random.default_rng(6)
    d = 64
    M = np.repeat(_unit(rng.random((1, d), dtype=np.float32)), 5000, axis=0)
    q = _unit(rng.random((1, d), dtype=np.float32))[0]
    assert check(M, q, 100) == 5000
