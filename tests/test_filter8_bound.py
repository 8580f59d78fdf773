"""CPU: the int8 filter's error bound and candidate set (DESIGN.md section 4, K1f8), restated in NumPy.

The shadow is what rows_to_i8_kernel writes: per row s_r = fp32(max|r_j| / 127), Q_r = clip(rint(r / s_r), +-127), and
E = max_r ||r - s_r Q_r|| (float64, rounded up).  The query split is q8_split: s1 = fp32(max|q_j| / 127),
s2 = fp32(s1 / 254), q_hi = clip(rint(q / s1)), q_lo = clip(rint(fma(-s1, q_hi, q) / s2)).  The coarse score is
gemv8_tma_kernel's: two exact integer dot products, then s_r * fma(s2, D_lo, s1 * D_hi) in fp32.  The exact score is K1's
fp32 arithmetic (test_filter_bound.k1_scores).  On adversarial data this checks |coarse - exact| <= eps (the bound of
filter_threshold_kernel) for every row and that the rows with coarse >= T contain the exact top-k."""
import numpy as np
import pytest

from test_filter_bound import exact_topk_rows, k1_scores, threshold

f32 = np.float32


def _round_q(x):
    return np.clip(np.rint(x), -127, 127).astype(np.int64)


def shadow(M, ld8):
    n, ld = M.shape
    amax = np.abs(M).max(axis=1) if ld else np.zeros(n, f32)
    s = (amax / f32(127)).astype(f32)
    Q = np.zeros((n, ld8), np.int64)
    nz = s > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        Q[nz, :ld] = _round_q((M[nz] / s[nz, None]).astype(f32))
    err = M.astype(np.float64) - s[:, None].astype(np.float64) * Q[:, :ld]
    e = np.sqrt((err * err).sum(axis=1)) * (1.0 + 2.0 ** -20)
    return Q, s, e


def round_up_f32(x):
    y = f32(x)
    return np.nextafter(y, f32(np.inf)) if np.float64(y) < x else y


def q8_split(q):
    s1 = f32(f32(np.abs(q).max()) / f32(127))
    s2 = f32(s1 / f32(254))
    hi = _round_q((q / s1).astype(f32)) if s1 > 0 else np.zeros(len(q), np.int64)
    res = (q.astype(np.float64) - np.float64(s1) * hi).astype(f32)            # fmaf(-s1, hi, q)
    lo = _round_q((res / s2).astype(f32)) if s2 > 0 else np.zeros(len(q), np.int64)
    return s1, s2, hi, lo


def coarse_scores(Q, s, q8):
    s1, s2, hi, lo = q8
    ld8 = Q.shape[1]
    h = np.zeros(ld8, np.int64); h[:len(hi)] = hi
    l_ = np.zeros(ld8, np.int64); l_[:len(lo)] = lo
    dh, dl = Q @ h, Q @ l_
    assert np.abs(dh).max(initial=0) < 2 ** 31 and np.abs(dl).max(initial=0) < 2 ** 31
    t = (f32(s1) * dh.astype(f32)).astype(f32)
    c = (np.float64(s2) * dl.astype(f32).astype(np.float64) + t.astype(np.float64)).astype(f32)   # fmaf
    return (s * c).astype(f32)


def eps8(q, q8, E, R, ld):
    s1, s2, hi, lo = q8
    with np.errstate(over="ignore"):                                         # fp32 ||q|| may overflow, as on the device
        qn = np.float64(np.sqrt(np.sum(q.astype(f32) ** 2, dtype=f32)))
    th, tl = np.float64(s1) * hi, np.float64(s2) * lo
    dq = np.sqrt(((q.astype(np.float64) - th - tl) ** 2).sum())
    Rh = np.float64(R) + np.float64(E)
    return ((qn * np.float64(E) + dq * Rh + ld * 2.0 ** -23 * qn * np.float64(R)
             + 2.0 ** -21 * (np.sqrt((th * th).sum()) + np.sqrt((tl * tl).sum())) * Rh) * (1.0 + 2.0 ** -10) + 1e-8)


def check(M, q, k, E_floor=0.0):
    """E_floor: an E raised by rows no longer part of this view (appends to a later generation only raise it)."""
    n, d = M.shape
    ld = (d + 3) & ~3
    ld8 = (ld + 15) & ~15
    Mp = np.zeros((n, ld), f32); Mp[:, :d] = M
    qp = np.zeros(ld, f32); qp[:d] = q
    Q, s, e = shadow(Mp, ld8)
    E = round_up_f32(max(e.max(initial=0.0), E_floor))
    q8 = q8_split(qp)
    exact = k1_scores(Mp, qp)
    coarse = coarse_scores(Q, s, q8)
    R = f32((1.0 + np.abs(np.linalg.norm(M.astype(np.float64), axis=1) - 1.0).max()) * 1.000001)
    eps = eps8(qp, q8, E, R, ld)
    if np.isfinite(eps):
        err = np.abs(coarse.astype(np.float64) - exact.astype(np.float64))
        assert err.max() <= eps, (err.max(), eps)
    T = threshold(coarse, k, eps)
    cand = np.ones(n, bool) if T is None else coarse >= T
    top = exact_topk_rows(exact, k)
    assert cand[top].all(), (int((~cand[top]).sum()), T)
    return int(cand.sum()), eps


def _unit(x):
    return (x / np.linalg.norm(x.astype(np.float64), axis=1, keepdims=True)).astype(f32)


@pytest.mark.parametrize("d", [64, 100, 768, 1536, 3072])
def test_uniform_rows_as_the_bench(d):
    rng = np.random.default_rng(1)
    n = 8192 if d <= 1536 else 4096
    M = _unit(rng.random((n, d), dtype=f32))
    q = _unit(rng.random((1, d), dtype=f32))[0]
    c, _ = check(M, q, 20)
    assert c < n // 4                          # the filter really filters


@pytest.mark.parametrize("k", [1, 10, 100, 1000, 2048])
def test_signed_rows_over_k(k):
    rng = np.random.default_rng(2)
    M = _unit(rng.standard_normal((6000, 256)).astype(f32))
    q = _unit(rng.standard_normal((1, 256)).astype(f32))[0]
    check(M, q, k)


def test_rows_with_one_large_component_and_zero_rows():
    rng = np.random.default_rng(3)
    d = 512
    M = rng.standard_normal((6000, d)).astype(f32)
    M[::5, rng.integers(0, d, 1200)] *= f32(300.0)    # a coarse scale: the rest of the row rounds to few levels
    M = _unit(M)
    M[10:40] = 0.0
    q = _unit(rng.standard_normal((1, d)).astype(f32))[0]
    for k in (1, 100, 1000):
        check(M, q, k)


def test_zero_query_and_a_query_with_one_huge_component():
    rng = np.random.default_rng(4)
    d = 384
    M = _unit(rng.standard_normal((5000, d)).astype(f32))
    c, eps = check(M, np.zeros(d, f32), 100)
    assert c == 5000 and eps == 1e-8               # no division by s1 = 0; every row re-scored
    q = np.full(d, 1e-3, f32)
    q[7] = 1e3                                     # the other components vanish from q_hi and mostly from q_lo
    check(M, q, 100)
    check(M, q * f32(1e-30), 100)                  # tiny scales
    q[7] = 1e30                                    # ||q|| overflows in fp32: no threshold
    c, _ = check(M, q, 100)
    assert c == 5000


def test_identical_rows_take_every_row():
    rng = np.random.default_rng(5)
    M = np.repeat(_unit(rng.random((1, 64), dtype=f32)), 5000, axis=0)
    q = _unit(rng.random((1, 64), dtype=f32))[0]
    assert check(M, q, 100)[0] == 5000


def test_rows_appended_later_raise_e():
    """E only grows: the bound holds for the old rows under the E raised by coarser appended rows, and for all rows."""
    rng = np.random.default_rng(6)
    d = 768
    old = _unit(rng.random((4000, d), dtype=f32))
    new = rng.random((500, d), dtype=f32)
    new[:, 0] = 40.0                                # one large component: a larger quantisation step
    new = _unit(new)
    _, _, e_new = shadow(np.ascontiguousarray(new), d)
    _, _, e_old = shadow(np.ascontiguousarray(old), d)
    assert e_new.max() > 2 * e_old.max()
    q = _unit(rng.random((1, d), dtype=f32))[0]
    check(old, q, 100, E_floor=e_new.max())
    check(np.concatenate([old, new]), q, 100)
    q2 = new[3] + f32(1e-3)
    check(np.concatenate([old, new]), q2, 10)


def test_rows_sorted_by_similarity_and_near_ties():
    rng = np.random.default_rng(7)
    d = 256
    base = _unit(rng.random((1, d), dtype=f32))
    M = _unit(base + rng.standard_normal((6000, d)).astype(f32) * f32(1e-4))
    q = _unit(base + rng.standard_normal((1, d)).astype(f32) * f32(1e-3))[0]
    M = M[np.argsort(M @ q)]
    for k in (1, 100, 1000):
        check(M, q, k)
