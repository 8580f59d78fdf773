"""CPU: the single-query filter's error bound and candidate set on more inputs, through the int8 check.

Each case runs test_filter8_bound.check (the NumPy restatement of the int8 shadow, the query split, gemv8_tma_kernel's
coarse score, filter_threshold_kernel's eps and threshold, and K1's exact score): |coarse - exact| <= eps for every row,
and the rows with coarse >= T contain the exact top-k.  The inputs: uniform rows as the bench draws them, near ties,
rows sorted by similarity, components below 2^-26 (where most of every row rounds to 0), row norms up to the filter's
limit of 8, and identical rows."""
import numpy as np
import pytest

from test_filter8_bound import check as _check8


def check(M, q, k):
    return _check8(M, q, k)[0]


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
    """Components below 2^-26, far below each row's largest: they round to 0 in the shadow."""
    rng = np.random.default_rng(4)
    d = 200
    M = rng.standard_normal((4096, d)).astype(np.float32)
    tiny = rng.random((4096, d)) < 0.7
    M[tiny] *= np.float32(2.0 ** -30)
    M = _unit(M)
    M[:, :150] *= np.float32(2.0 ** -28)       # most of every row
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
    M[7, 3] = 8.0                              # a row of norm 8 in one component
    q = _unit(rng.standard_normal((1, d)).astype(np.float32))[0]
    for k in (1, 100, 1000):
        check(M, q, k)


def test_identical_rows_take_every_row():
    rng = np.random.default_rng(6)
    d = 64
    M = np.repeat(_unit(rng.random((1, d), dtype=np.float32)), 5000, axis=0)
    q = _unit(rng.random((1, d), dtype=np.float32))[0]
    assert check(M, q, 100) == 5000
