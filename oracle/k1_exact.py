"""Bit-exact CPU restatement of K1, the fp32 similarity kernel (svs_b200/csrc/gemv.cu: gemv_tma_kernel).

Every exact path of the engine promises the bits of svsb_query: the multi-query passes, the filters' re-score, the
batched refine, the pair re-score and the LDG variant all use K1's summation order.  This module computes those bits on
the CPU, so the GPU paths can be compared with ground truth instead of only with each other:

- the row is zero-padded to ld = (d + 3) & ~3 and read as float4 chunks;
- lane l of the warp owns chunks l, l + 32, l + 64, ...; the lane's even chunks accumulate into a0, its odd ones into
  a1, one fp32 FMA (round to nearest even) per component;
- the combine ((a0.x + a1.x) + (a0.y + a1.y)) + ((a0.z + a1.z) + (a0.w + a1.w)), then the xor tree over the 32 lanes
  (offsets 16, 8, 4, 2, 1).

The FMA is exact: acc + a * b is formed in float64 (the product of two fp32 values is exact there), TwoSum recovers
the residual of that sum, and only when the float64 sum sits exactly on an fp32 rounding midpoint with a non-zero
residual is the rounding direction taken from the residual.  Values near fp32's overflow threshold go through
fractions.Fraction.  (A float64 product-sum simply rounded to fp32 rounds twice and is not an FMA.)
"""
from __future__ import annotations

from fractions import Fraction
from typing import List, Optional, Tuple

import numpy as np

F32, F64 = np.float32, np.float64
DEAD_BITS = np.uint32(0xFFFFFFFF)           # common.cuh: dead_score(), the score of a tombstoned row
_HUGE = 2.0 ** 127                          # at and above this the fp32 midpoint test runs into the overflow threshold


# ---------------------------------------------------------------------------------------------------------------------
# exact fp32 FMA
# ---------------------------------------------------------------------------------------------------------------------
def round_fraction_f32(x: Fraction, zero_sign: float = 1.0) -> np.float32:
    """Round the rational x to fp32, to nearest, ties to even (subnormals and overflow to inf included).  An exact
    zero gets the sign of zero_sign."""
    if x == 0:
        return F32(np.copysign(0.0, zero_sign))
    neg = x < 0
    a = -x if neg else x
    e = a.numerator.bit_length() - a.denominator.bit_length()        # 2^e <= a < 2^(e+2)
    if Fraction(2) ** e > a:
        e -= 1
    elif Fraction(2) ** (e + 1) <= a:
        e += 1
    quantum = Fraction(2) ** max(e - 23, -149)
    m = a / quantum
    fl = m.numerator // m.denominator
    rem = m - fl
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and fl & 1):
        fl += 1
    v = fl * quantum
    if v >= Fraction(2) ** 128:
        r = np.inf
    else:
        r = float(v)                                                  # exact: v is an fp32 value
    return F32(-r if neg else r)


def fma_fraction(acc, a, b) -> np.float32:
    """fmaf(a, b, acc) by rational arithmetic: the definition the fast emulation is tested against."""
    acc, a, b = F32(acc), F32(a), F32(b)
    p = Fraction(float(a)) * Fraction(float(b))
    x = Fraction(float(acc)) + p
    # IEEE 754 exact zero sum: +0 under round-to-nearest unless both addends are -0
    prod_neg_zero = p == 0 and (np.signbit(a) != np.signbit(b))
    zs = -1.0 if (x == 0 and np.signbit(acc) and prod_neg_zero) else 1.0
    return round_fraction_f32(x, zs)


def fma32(acc: np.ndarray, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Element-wise fmaf(a, b, acc) on fp32 arrays (broadcasting), correctly rounded to nearest even."""
    acc, a, b = np.broadcast_arrays(np.asarray(acc, F32), np.asarray(a, F32), np.asarray(b, F32))
    acc64 = acc.astype(F64)
    p = a.astype(F64) * b.astype(F64)                                # exact: 48 significant bits, exponents in range
    with np.errstate(invalid="ignore", over="ignore"):
        s = acc64 + p
        bb = s - acc64                                               # TwoSum: s + e == acc + p exactly
        e = (acc64 - (s - bb)) + (p - bb)
        r = s.astype(F32)
    r = np.array(r, copy=True)
    fin = np.isfinite(s)
    huge = fin & (np.abs(s) >= _HUGE)
    check = fin & ~huge & (e != 0) & (r.astype(F64) != s)
    if check.any():
        idx = np.nonzero(check)
        rr = r[idx]
        ss = s[idx]
        other = np.nextafter(rr, np.where(ss > rr.astype(F64), F32(np.inf), F32(-np.inf)).astype(F32))
        mid = (rr.astype(F64) + other.astype(F64)) * 0.5             # exact: 25 significant bits
        at_mid = ss == mid
        if at_mid.any():
            up = e[idx] > 0
            hi = np.maximum(rr, other); lo = np.minimum(rr, other)
            fixed = np.where(up, hi, lo)
            rr = np.where(at_mid, fixed, rr)
            r[idx] = rr
    if huge.any():
        for ix in zip(*np.nonzero(huge)):
            r[ix] = fma_fraction(acc[ix], a[ix], b[ix])
    return r


# ---------------------------------------------------------------------------------------------------------------------
# K1
# ---------------------------------------------------------------------------------------------------------------------
def _pad4(x: np.ndarray) -> np.ndarray:
    x = np.asarray(x, F32)
    d = x.shape[-1]
    ld = (d + 3) & ~3
    if ld == d:
        return x
    out = np.zeros(x.shape[:-1] + (ld,), F32)
    out[..., :d] = x
    return out


def _combine_and_tree(a0: np.ndarray, a1: np.ndarray) -> np.ndarray:
    v = ((a0[..., 0] + a1[..., 0]) + (a0[..., 1] + a1[..., 1])) + ((a0[..., 2] + a1[..., 2]) + (a0[..., 3] + a1[..., 3]))
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = v + v[..., lanes ^ o]
    return v[..., 0]


def k1_exact_rows(M: np.ndarray, Q: np.ndarray) -> np.ndarray:
    """Scores of rows M[i] against queries Q[i] (Q may be one row, broadcast): float32[n] with K1's bits."""
    M = _pad4(np.atleast_2d(M)); Q = _pad4(np.atleast_2d(Q))
    n, ld = M.shape
    assert Q.shape[1] == ld and Q.shape[0] in (1, n)
    d4 = ld // 4
    nch = -(-d4 // 32)                                               # chunk rounds per lane
    Mp = np.zeros((n, nch * 128), F32); Mp[:, :ld] = M
    Qp = np.zeros((Q.shape[0], nch * 128), F32); Qp[:, :ld] = Q
    Mc = Mp.reshape(n, nch, 32, 4); Qc = Qp.reshape(Q.shape[0], nch, 32, 4)
    acc = [np.zeros((n, 32, 4), F32), np.zeros((n, 32, 4), F32)]
    lane_has = (np.arange(32)[None, :] + 32 * np.arange(nch)[:, None]) < d4    # [nch, 32]: chunk exists for the lane
    for j in range(nch):
        new = fma32(acc[j & 1], Mc[:, j], Qc[:, j])
        acc[j & 1] = np.where(lane_has[j][None, :, None], new, acc[j & 1])
    return _combine_and_tree(acc[0], acc[1]).astype(F32)


def k1_exact(M: np.ndarray, q: np.ndarray) -> np.ndarray:
    """What gemv_tma_kernel writes for the rows of M (n, d) and the query q (d,): float32[n]."""
    return k1_exact_rows(M, np.asarray(q, F32)[None, :])


def bits(x) -> np.ndarray:
    return np.asarray(x, F32).view(np.uint32)


def ordered(b: np.ndarray) -> np.ndarray:
    """common.cuh: f32_to_ordered on score bits -- unsigned order == the engine's score order."""
    b = np.asarray(b, np.uint32)
    return np.where(b & np.uint32(0x80000000), ~b, b | np.uint32(0x80000000)).astype(np.uint32)


def _margin(absdot: np.ndarray, d: int) -> np.ndarray:
    """Proven bound on |K1's fp32 score - the float64 score|: d + 8 roundings of relative size 2^-24 of sum |m_i q_i|
    each, doubled, plus the float64 dot product's own error."""
    return (d + 8) * 2.0 ** -23 * absdot * (1 + 1e-9) + 1e-300


def k1_topk_exact(M: np.ndarray, ids: np.ndarray, q: np.ndarray, k: int,
                  live: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
    """Expected (score bits uint32[c], ids int64[c]), c = min(k, n), of svsb_query: order (score desc, row asc), the
    tombstoned rows (live[r] == 0) last with dead_score()'s bits.  Only rows that can reach the top k under a proven
    margin around their float64 score are emulated exactly."""
    M = np.asarray(M, F32); q = np.asarray(q, F32)
    n, d = M.shape
    k = min(int(k), n)
    if k <= 0:
        return np.zeros(0, np.uint32), np.zeros(0, np.int64)
    alive = np.ones(n, bool) if live is None else np.asarray(live).astype(bool)
    rows = np.nonzero(alive)[0]
    out_b: List[np.ndarray] = []
    out_r: List[np.ndarray] = []
    if len(rows):
        M64 = M[rows].astype(F64); q64 = q.astype(F64)
        s64 = M64 @ q64
        mg = _margin(np.abs(M64) @ np.abs(q64), d)
        kk = min(k, len(rows))
        lo = np.partition(s64 - mg, len(rows) - kk)[len(rows) - kk]   # kk-th largest lower bound
        cand = rows[s64 + mg >= lo]
        sc = bits(k1_exact(M[cand], q))
        order = np.lexsort((cand, ~ordered(sc)))
        out_b.append(sc[order][:kk]); out_r.append(cand[order][:kk])
    if k > len(rows):
        dead = np.nonzero(~alive)[0][:k - len(rows)]
        out_b.append(np.full(len(dead), DEAD_BITS, np.uint32)); out_r.append(dead)
    r = np.concatenate(out_r)
    return np.concatenate(out_b), np.asarray(ids, np.int64)[r]


def k1_topk_brute(M: np.ndarray, ids: np.ndarray, q: np.ndarray, k: int,
                  live: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
    """k1_topk_exact without the prefilter: every row emulated.  The check of the prefilter on small inputs."""
    M = np.asarray(M, F32)
    n = M.shape[0]
    sc = bits(k1_exact(M, q))
    if live is not None:
        sc = np.where(np.asarray(live).astype(bool), sc, DEAD_BITS)
    order = np.lexsort((np.arange(n), ~ordered(sc)))[:min(int(k), n)]
    return sc[order], np.asarray(ids, np.int64)[order]


# ---------------------------------------------------------------------------------------------------------------------
# pairs
# ---------------------------------------------------------------------------------------------------------------------
def pair_exact(M: np.ndarray, i: int, j: int) -> np.float32:
    """pairs_rescore_kernel's score of rows (i, j): row i plays the query, row j the matrix row."""
    M = np.asarray(M, F32)
    return k1_exact(M[j][None, :], M[i])[0]


def top_pairs_exact(M: np.ndarray, ids: np.ndarray, n: int) -> List[Tuple[int, int, int]]:
    """Expected svsb_top_pairs: [(score bits, id of row a, id of row b)] of the n best pairs a < b, ordered by score
    desc, then row a asc, then row b asc.  Same prefilter as k1_topk_exact."""
    M = np.asarray(M, F32)
    N, d = M.shape
    n = min(int(n), N * (N - 1) // 2)
    if n <= 0:
        return []
    M64 = M.astype(F64)
    s64 = M64 @ M64.T
    A = np.abs(M64)
    mg = _margin(A @ A.T, d)
    ia, ib = np.triu_indices(N, k=1)
    s = s64[ia, ib]; m = mg[ia, ib]
    lo = np.partition(s - m, len(s) - n)[len(s) - n]
    keep = s + m >= lo
    ia, ib = ia[keep], ib[keep]
    sc = bits(k1_exact_rows(M[ib], M[ia]))
    order = np.lexsort((ib, ia, ~ordered(sc)))[:n]
    ids = np.asarray(ids, np.int64)
    return [(int(sc[o]), int(ids[ia[o]]), int(ids[ib[o]])) for o in order]
