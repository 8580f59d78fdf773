"""GPU: the tensor-core coarse pass's error bound, measured and attacked.

The batched path is exact only if |coarse - exact| <= eps = coarse_eps_coef(d) * ||q|| * R + 1e-8 for every (row,
query) (kernels.cuh; DESIGN.md section 6 item 4).  Its accumulation term d * 2^-22 rests on how tcgen05.mma kind::f16
accumulates in fp32, which NVIDIA does not document.  These tests read the coarse scores back
(Engine.batch_candidates) on matrices built so that every row is a candidate of every query: the rows of a matrix are
permutations of one multiset of components and the queries are constant vectors, so all exact scores agree up to fp32
rounding and every row lies inside the 2 eps band.  Per data family and d they check |coarse - K1| <= eps for every
pair, that eps is the formula's, and how large the accumulator's own error is: the coarse score against the float64
sum of the fp16-rounded operands, as a share of the d * 2^-22 term.  Then the batch must still return K1's bits in
both threshold modes.  The families:
  a  components just below fp16 rounding midpoints (after the 2^12 scale): every operand rounds down, aligned with q
  b  cancellation: pairs of terms near +-1/sqrt(d) that sum to nearly 0
  c  16-element blocks of one large term followed by 15 just under half its fp32 ulp
  d  rows of norm just below 8 and queries of norm just below 8
  e  most components in fp16's subnormal range after the scale
Set SVSB_COARSE_REPORT=<file> to append the measured ratios to a file."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import k1_exact as kx  # noqa: E402

pytestmark = pytest.mark.gpu

F32 = np.float32
N_ROWS = 4096


def eps_coef(d):
    f = F32
    return f(f(9.765625e-4) + f(2.384185791015625e-7)) + f(d) * f(f(2.384185791015625e-7) + f(1.1920928955078125e-7))


def _fp16_operand(x):
    return (np.asarray(x, F32) * F32(4096.0)).astype(np.float16).astype(np.float64)


def _multiset(fam, d, rng):
    """One row's components; every row of the matrix is a permutation of them (blocks of 16 kept whole for c)."""
    if fam in ("a", "d"):
        h = rng.uniform(0.5, 1.0, d) * np.sqrt(1.0 / d) * 4096.0       # scaled magnitudes
        h16 = h.astype(np.float16).astype(np.float64)
        ulp = np.spacing(np.abs(h16).astype(np.float16)).astype(np.float64)
        v = (h16 + 0.5 * ulp * (1 - 2.0 ** -9)) / 4096.0                # just below the midpoint: rounds down
        v = v.astype(F32)
    elif fam == "b":
        half = d // 2
        x = (rng.uniform(0.9, 1.1, half) / np.sqrt(d)).astype(F32)
        y = (x * (F32(1) + F32(2.0 ** -20) * rng.choice([-1, 1], half).astype(F32))).astype(F32)
        v = np.concatenate([x, -y, np.full(d - 2 * half, F32(0.5 / np.sqrt(d)), F32)])
    elif fam == "c":
        nb = -(-d // 16)
        L = (rng.uniform(0.9, 1.1, nb) * np.sqrt(1.0 / nb)).astype(F32)
        v = np.empty(nb * 16, F32)
        for j in range(nb):
            v[16 * j] = L[j]
            v[16 * j + 1:16 * j + 16] = F32(float(L[j]) * 2.0 ** -24 * 0.96)
        v = v[:d]
    elif fam == "e":
        v = (rng.uniform(0.5, 1.0, d) * 2.0 ** -28).astype(F32)          # scaled: 2^-16 .. 2^-17, fp16 subnormal
        big = max(1, d // 16)
        v[:big] = F32(np.sqrt(1.0 / big))
    else:
        raise ValueError(fam)
    norm = np.sqrt((v.astype(np.float64) ** 2).sum())
    if fam == "d":
        return (v * F32(8.0 * (1 - 2e-6) / norm)).astype(F32)
    return (v * F32(2.0 ** np.floor(np.log2(1.0 / norm)))).astype(F32)  # a power of two keeps the fp16 structure


def family(fam, d, b, seed):
    rng = np.random.default_rng(seed)
    v = _multiset(fam, d, rng)
    if fam == "c":
        nb = -(-d // 16)
        blocks = np.concatenate([v, np.zeros(nb * 16 - d, F32)]).reshape(nb, 16)
        M = np.stack([blocks[rng.permutation(nb)].reshape(-1)[:d] for _ in range(N_ROWS)])
    else:
        M = np.stack([v[rng.permutation(d)] for _ in range(N_ROWS)])
    qn = 8.0 * (1 - 4e-6) if fam == "d" else 1.0
    c = np.array([qn / np.sqrt(d) * (1 + 0.013 * j) / (1 + 0.013 * (b - 1)) for j in range(b)])
    Q = np.repeat(c[:, None], d, axis=1).astype(F32)
    return M.astype(F32), Q


def _topk(exact_bits, ids, k):
    order = np.lexsort((np.arange(len(exact_bits)), ~kx.ordered(exact_bits)))[:k]
    return exact_bits[order], ids[order]


def _report(line):
    path = os.environ.get("SVSB_COARSE_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(line + "\n")


@pytest.mark.parametrize("d", [16, 24, 768, 3072, 13000])
@pytest.mark.parametrize("fam", ["a", "b", "c", "d", "e"])
def test_coarse_error_within_eps_for_every_pair(fam, d, monkeypatch):
    import svs_b200
    monkeypatch.setenv("SVSB_MQ_MAX", "1")
    monkeypatch.setenv("SVSB_BATCH_CAND_CAP", str(N_ROWS))
    b = 4 if d >= 3072 else 8
    M, Q = family(fam, d, b, seed=d * 7 + ord(fam))
    ids = np.arange(1, N_ROWS + 1, dtype=np.int64) * 2
    R = float(F32(1.0) + F32(abs(np.sqrt((M.astype(np.float64) ** 2).sum(axis=1)) - 1.0).max()))
    worst_acc, worst_eps = 0.0, 0.0
    exact = [kx.k1_exact(M, q) for q in Q]
    with svs_b200.Engine() as e:
        e.load(M, ids)
        for guaranteed in ("0", "1"):
            monkeypatch.setenv("SVSB_BATCH_GUARANTEED", guaranteed)
            s, i, c = e.query_batch(Q, 10)
            flags = e.batch_stats(b)[2]
            assert (flags == 0).all(), flags
            for j in range(b):                                     # end to end: K1's bits whatever the coarse errors
                wb, wi = _topk(exact[j].view(np.uint32), ids, 10)
                assert np.array_equal(s[j, :c[j]].view(np.uint32), wb) and np.array_equal(i[j, :c[j]], wi), (guaranteed, j)
        M16 = _fp16_operand(M)
        for j in range(b):
            cs, rows, cnt, eps = e.batch_candidates(j)
            assert cnt == N_ROWS and len(rows) == N_ROWS, cnt      # every row is a candidate
            order = np.argsort(rows)
            cs, rows = cs[order].astype(np.float64), rows[order]
            assert np.array_equal(rows, np.arange(N_ROWS))
            qn = float(np.sqrt((Q[j].astype(np.float64) ** 2).sum()))
            formula = float(eps_coef(d)) * qn * 1.000001 * R * 1.000001 + 1e-8
            assert abs(eps - formula) <= 1e-5 * formula, (eps, formula)
            err = np.abs(cs - exact[j].astype(np.float64))
            assert err.max() <= eps, (fam, d, j, err.max(), eps)
            ref16 = (M16 @ _fp16_operand(Q[j])) * 2.0 ** -24       # the fp16 operands' exact products, summed in float64
            acc = np.abs(cs - ref16).max()
            worst_acc = max(worst_acc, acc / (d * 2.0 ** -22 * qn * R))
            worst_eps = max(worst_eps, err.max() / eps)
    _report(f"family {fam}  d {d:5d}  max |coarse - fp16-operand sum| / (d 2^-22 |q| R) = {worst_acc:.4f}  "
            f"max |coarse - K1| / eps = {worst_eps:.4f}")
    assert worst_acc <= 1.0, worst_acc


def test_query_norm_gate(monkeypatch):
    """queries_to_f16_kernel flags a query whose norm, inflated by 1.000001 for its own rounding, exceeds 8: a query of
    norm exactly 8 is answered by the exact single-query kernels, one a little shorter by the coarse path."""
    import svs_b200
    monkeypatch.setenv("SVSB_MQ_MAX", "1")
    rng = np.random.default_rng(3)
    d = 64
    M = rng.standard_normal((N_ROWS, d)).astype(F32)
    M /= np.sqrt((M.astype(np.float64) ** 2).sum(axis=1)).astype(F32)[:, None]
    ids = np.arange(N_ROWS, dtype=np.int64)
    Q = M[100:108].copy()                                          # a batch of 8: smaller ones take the exact kernels
    Q[:3] = 0.0
    Q[0, 5] = 8.0                                                  # norm exactly 8
    Q[1, 5] = np.nextafter(F32(8.0), F32(np.inf))
    Q[2, 5] = F32(8.0 * (1 - 4e-6))
    with svs_b200.Engine() as e:
        e.load(M, ids)
        s, i, c = e.query_batch(Q, 20)
        flags = e.batch_stats(len(Q))[2]
        assert flags[0] != 0 and flags[1] != 0 and (flags[2:] == 0).all(), flags
        for j in range(len(Q)):
            wb, wi = kx.k1_topk_exact(M, ids, Q[j], 20)
            assert np.array_equal(s[j, :c[j]].view(np.uint32), wb) and np.array_equal(i[j, :c[j]], wi), j


def test_row_norm_gate(monkeypatch):
    """batch_plan takes the coarse path while R = 1 + max | ||row|| - 1 | <= 8; one row just longer turns it off for
    the generation.  Either way the batch returns K1's bits."""
    import svs_b200
    monkeypatch.setenv("SVSB_MQ_MAX", "1")
    rng = np.random.default_rng(4)
    d = 32
    M = rng.standard_normal((N_ROWS, d)).astype(F32)
    M /= np.sqrt((M.astype(np.float64) ** 2).sum(axis=1)).astype(F32)[:, None]
    M[17] = 0.0
    M[17, 3] = 8.0                                                 # norm exactly 8: R = 8
    ids = np.arange(N_ROWS, dtype=np.int64) + 100
    Q = M[[1, 2, 3, 4, 5, 6, 7, 17]].copy()
    Q[7] /= F32(8.0)
    for above in (False, True):
        if above:
            M[17, 3] = np.nextafter(F32(8.0), F32(np.inf))
        with svs_b200.Engine() as e:
            e.load(M, ids)
            s, i, c = e.query_batch(Q, 15)
            if not above:
                assert (e.batch_stats(len(Q))[2] == 0).all()
            for j in range(len(Q)):
                wb, wi = kx.k1_topk_exact(M, ids, Q[j], 15)
                assert np.array_equal(s[j, :c[j]].view(np.uint32), wb) and np.array_equal(i[j, :c[j]], wi), (above, j)


def _boundary_case(d, k):
    """Row A carries the exact top score, but every product of A rounds down twice (its component and the query's, each
    just below an fp16 midpoint) while the k rows B, on the other half of the components, round up twice: coarse(A) is
    about 2^-10 * A.q below exact and coarse(B) as far above, and exact(A) - exact(B) is a small fraction of that.
    Then A survives the refine's cut-off coarse >= tau - 2 eps only because eps really covers both fp16 roundings of
    every product: with the 2^-10 term of eps halved this batch loses A."""
    h = d // 2
    r0 = 2.0 ** -np.floor(np.log2(np.sqrt(h)))                     # powers of two keep the fp16 midpoints
    s0 = 2.0 ** -np.floor(np.log2(np.sqrt(d)))
    lo, hi = 1 + 2.0 ** -11 - 2.0 ** -20, 1 + 2.0 ** -11 + 2.0 ** -20   # just below / above the first fp16 midpoint
    q = np.empty(d); q[:h] = lo * s0; q[h:] = hi * s0
    A = np.zeros(d); A[:h] = lo * r0
    B = np.zeros(d); B[h:] = hi * r0
    q = q.astype(F32); A = A.astype(F32); B = B.astype(F32)
    # trim B's last component to an fp16-exact value (no rounding error) that puts exact(B) just below exact(A)
    sa = float(A.astype(np.float64) @ q.astype(np.float64))
    v = np.float16(B[-1] * 4096.0)
    while (B[:-1].astype(np.float64) @ q[:-1].astype(np.float64)) + float(v) / 4096.0 * float(q[-1]) >= sa:
        v = np.nextafter(v, np.float16(0))
    B[-1] = F32(float(v) / 4096.0)
    rng = np.random.default_rng(d)
    fill = rng.standard_normal((N_ROWS - 1 - k, d)).astype(F32)
    fill /= np.sqrt((fill.astype(np.float64) ** 2).sum(axis=1)).astype(F32)[:, None]
    fill *= np.where(fill @ q > 0, F32(-1), F32(1))[:, None]       # filler rows score below 0
    M = np.concatenate([fill[:1000], np.repeat(B[None, :], k, axis=0), A[None, :], fill[1000:]]).astype(F32)
    return M, q


@pytest.mark.parametrize("guaranteed", ["0", "1"])
@pytest.mark.parametrize("d", [32, 128])
def test_boundary_between_opposite_coarse_errors(d, guaranteed, monkeypatch):
    import svs_b200
    monkeypatch.setenv("SVSB_MQ_MAX", "1")
    monkeypatch.setenv("SVSB_BATCH_GUARANTEED", guaranteed)
    k = 5
    M, q = _boundary_case(d, k)
    ids = np.arange(N_ROWS, dtype=np.int64) * 3 + 1
    exact = kx.k1_exact(M, q).view(np.uint32)
    a_row = 1000 + k
    wb, wi = _topk(exact, ids, k)
    assert ids[a_row] == wi[0]                                     # A is the exact top row
    Q = np.repeat(q[None, :], 6, axis=0)
    with svs_b200.Engine() as e:
        e.load(M, ids)
        s, i, c = e.query_batch(Q, k)
        assert (e.batch_stats(len(Q))[2] == 0).all()
        cs, rows, cnt, eps = e.batch_candidates(0)
        ca = float(cs[rows == a_row][0]) if (rows == a_row).any() else None
        cb = float(cs[rows == 1000][0]) if (rows == 1000).any() else None
    assert ca is not None and cb is not None
    # the construction really is adversarial: the coarse order of A and B is reversed by more than eps
    assert cb - ca > eps, (cb, ca, eps)
    for j in range(len(Q)):
        assert np.array_equal(s[j, :c[j]].view(np.uint32), wb) and np.array_equal(i[j, :c[j]], wi), j
