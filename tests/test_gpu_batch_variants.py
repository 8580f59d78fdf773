"""GPU: the batched path's kernel variants that are chosen once per process, against the bit-exact K1 reference.

SVSB_COARSE_CTAS, SVSB_REFINE, SVSB_REFINE_MINB, SVSB_RESCORE_SPLIT and SVSB_SAMPLE_GENERIC are read into static
variables on first use, so they cannot be switched inside one test process.  Each variant runs in a child process
(this file run as a script) that answers a fixed set of hard cases of tests/test_gpu_batch.py through the
tensor-core path and one top_pairs case, and writes the answers to an .npz; the parent compares every answer with
oracle/k1_exact.py bit for bit."""
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import k1_exact as kx  # noqa: E402


def _unit(x):
    return (x / np.sqrt((x.astype(np.float64) ** 2).sum(axis=1)).astype(np.float32)[:, None]).astype(np.float32)


def cases():
    """name -> (rows, ids, queries, k); regenerated identically in the child and the parent."""
    out = {}
    rng = np.random.default_rng(1)
    n, d = 20_000, 768                                             # packed uniform scores (0.75 +- 0.007)
    out["packed_uniform"] = (_unit(rng.random((n, d), dtype=np.float32)), np.arange(3, 3 * n + 3, 3, dtype=np.int64),
                             _unit(rng.random((40, d), dtype=np.float32)), 100)
    rng = np.random.default_rng(2)
    n, d = 60_000, 128                                             # 2 500 survivors per query: the refine spills
    m = _unit(rng.standard_normal((n, d)).astype(np.float32))
    centre = _unit(rng.standard_normal((1, d)).astype(np.float32))[0]
    m[rng.choice(n, 2500, replace=False)] = _unit(centre[None, :] + 2e-4 * rng.standard_normal((2500, d)).astype(np.float32))
    out["survivors"] = (m, np.arange(10, n + 10, dtype=np.int64),
                        _unit(centre[None, :] + 0.05 * rng.standard_normal((8, d)).astype(np.float32)), 100)
    rng = np.random.default_rng(3)
    n, d = 300_000, 64                                             # best rows first: statistical thresholds fail verification
    base = _unit(rng.standard_normal((1, d)).astype(np.float32))[0]
    m = _unit(rng.standard_normal((n, d)).astype(np.float32))
    m = m[np.argsort(-(m @ base), kind="stable")]
    out["sorted_rows"] = (m, np.arange(1, n + 1, dtype=np.int64),
                          _unit(base[None, :] + 0.05 * rng.standard_normal((16, d)).astype(np.float32)), 20)
    rng = np.random.default_rng(4)
    n, d = 40_000, 128                                             # identical rows: every coarse score ties
    out["identical_rows"] = (np.repeat(_unit(rng.standard_normal((1, d)).astype(np.float32)), n, axis=0),
                             np.arange(n, dtype=np.int64), _unit(rng.standard_normal((4, d)).astype(np.float32)), 50)
    rng = np.random.default_rng(5)
    n, d = 5_000, 96                                               # one partial query tile
    out["partial_tile"] = (_unit(rng.standard_normal((n, d)).astype(np.float32)), np.cumsum(rng.integers(1, 4, n)),
                           _unit(rng.standard_normal((8, d)).astype(np.float32)), 10)
    rng = np.random.default_rng(6)
    n, d = 40_000, 256
    out["k1"] = (_unit(rng.standard_normal((n, d)).astype(np.float32)), np.arange(n, dtype=np.int64),
                 _unit(rng.standard_normal((20, d)).astype(np.float32)), 1)
    rng = np.random.default_rng(7)
    n, d = 12_345, 3072
    out["k1000"] = (_unit(rng.random((n, d), dtype=np.float32)), np.arange(5, n + 5, dtype=np.int64),
                    _unit(rng.random((6, d), dtype=np.float32)), 1000)
    return out


def pairs_case():
    rng = np.random.default_rng(8)
    n, d = 3000, 128
    m = _unit(rng.standard_normal((n, d)).astype(np.float32))
    m[2000] = m[17]
    return m, np.arange(1, n + 1, dtype=np.int64), 300


def _child(path):
    import svs_b200
    res = {}
    with svs_b200.Engine() as e:
        for name, (m, ids, q, k) in cases().items():
            e.load(m, ids)
            s, i, c = e.query_batch(q, k)
            res[name + "_s"], res[name + "_i"], res[name + "_c"] = s, i, c
            res[name + "_flags"] = e.batch_stats(len(q))[2]
        m, ids, n = pairs_case()
        e.load(m, ids)
        p = e.top_pairs(n)
        res["pairs"] = np.array([(int(np.array([s], np.float32).view(np.uint32)[0]), a, b) for s, a, b in p], np.int64)
    np.savez(path, **res)


VARIANTS = {
    "default": {},
    "cta_pair": {"SVSB_COARSE_CTAS": "2"},
    "refine_split": {"SVSB_REFINE": "split"},
    "refine_fused": {"SVSB_REFINE": "fused"},
    "refine_minb3": {"SVSB_REFINE_MINB": "3"},
    "refine_minb5": {"SVSB_REFINE_MINB": "5"},
    "rescore_split1": {"SVSB_RESCORE_SPLIT": "1"},
    "rescore_split16": {"SVSB_RESCORE_SPLIT": "16"},
    "sample_generic": {"SVSB_SAMPLE_GENERIC": "1"},
}

_EXPECTED = {}


def _expected():
    if not _EXPECTED:
        for name, (m, ids, q, k) in cases().items():
            _EXPECTED[name] = [kx.k1_topk_exact(m, ids, qq, k) for qq in q]
        m, ids, n = pairs_case()
        _EXPECTED["pairs"] = np.array(kx.top_pairs_exact(m, ids, n), np.int64)
    return _EXPECTED


if __name__ == "__main__":
    _child(sys.argv[1])
else:
    import pytest

    @pytest.mark.gpu
    @pytest.mark.parametrize("variant", list(VARIANTS))
    def test_variant_answers_hard_cases_with_k1_bits(variant, tmp_path):
        out = tmp_path / "answers.npz"
        env = dict(os.environ)
        for key in ("SVSB_COARSE_CTAS", "SVSB_REFINE", "SVSB_REFINE_FUSED", "SVSB_REFINE_MINB", "SVSB_RESCORE_SPLIT",
                    "SVSB_SAMPLE_GENERIC", "SVSB_MQ_MAX", "SVSB_BATCH_GUARANTEED"):
            env.pop(key, None)
        env.update(VARIANTS[variant])
        env["SVSB_MQ_MAX"] = "1"                                   # every batch through the tensor-core path
        env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
        r = subprocess.run([sys.executable, os.path.abspath(__file__), str(out)], env=env, cwd=ROOT,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
        got = np.load(out)
        want = _expected()
        for name, (m, ids, q, k) in cases().items():
            s, i, c = got[name + "_s"], got[name + "_i"], got[name + "_c"]
            if name != "identical_rows":
                assert (got[name + "_flags"] == 0).all(), (name, got[name + "_flags"])
            for j, (wb, wi) in enumerate(want[name]):
                assert c[j] == len(wb), (name, j)
                gb = s[j, :c[j]].view(np.uint32)
                bad = np.nonzero((gb != wb) | (i[j, :c[j]] != wi))[0]
                assert len(bad) == 0, f"{name} query {j}: {len(bad)} ranks differ, first {bad[0]}"
        assert np.array_equal(got["pairs"], want["pairs"])
