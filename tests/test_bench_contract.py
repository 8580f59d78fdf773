"""bench.py's JSON contract, as far as a CPU-only container can exercise it: the reference arm (`--impl reference`) runs
here and must print ONE JSON line with the keys the driver reads; under a fake torchrun environment only rank 0 works;
our own arm must fail loudly without a GPU (no CPU fallback).  On a GPU, --dump-outputs writes the same answers run after
run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=300):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, env=e)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run(["--impl", "reference", "--workload", "c1", "--steps", "2", "--warmup", "1"], env={"OMP_NUM_THREADS": "1"})
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "retrieve_queries_per_sec" and j["unit"] == "queries/s"
    assert j["higher_is_better"] is True and j["steps"] == 2 and j["warmup"] == 1 and j["value"] > 0
    assert j["config"]["rows"] == 10_548 and j["config"]["dims"] == 1536 and j["config"]["k"] == 10
    cb = j["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["value"] == j["value"] and "np.dot + get_top_k" in cb["sample"]
    # torchrun exports OMP_NUM_THREADS=1; the arm must undo that and report the threads BLAS really uses
    assert cb["cores"] >= 1 and (cb["cores"] > 1 or (os.cpu_count() or 1) == 1)
    assert j["e2e"] == {"value": j["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["gpu_launches"] == 0 and j["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_without_work():
    r = _run(["--impl", "reference", "--workload", "c1", "--gpus", "2", "--steps", "1", "--warmup", "0"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, timeout=60)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_our_arm_fails_loudly_without_a_gpu():
    try:
        import torch
        if torch.cuda.is_available():
            import pytest
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    r = _run(["--workload", "c1", "--steps", "1", "--no-cpu-baseline"], timeout=120)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout) or "svs_b200 has no CPU path" in (r.stderr + r.stdout)


def test_bench_refuses_zero_steps_and_dumping_the_reference_arm(tmp_path):
    r = _run(["--impl", "reference", "--workload", "c1", "--steps", "0"], timeout=60)
    assert r.returncode == 2 and "--steps" in r.stderr
    r = _run(["--impl", "reference", "--workload", "c1", "--steps", "1", "--dump-outputs", str(tmp_path / "o")], timeout=60)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "o").exists()


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step_and_repeat_bit_for_bit(tmp_path):
    """Two runs with the same arguments write the same answers: one row of k per query of the last timed step, the
    oracle's top-k over the same synthetic rows."""
    import numpy as np
    from _util import oracle
    import svs_b200
    args = ["--workload", "c1", "--only", "--steps", "3", "--warmup", "1", "--no-cpu-baseline"]
    got = []
    for tag in ("a", "b"):
        r = _run(args + ["--dump-outputs", str(tmp_path / tag)], timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
        assert sorted(os.listdir(tmp_path / tag)) == ["c1_ids.npy", "c1_scores.npy"]
        got.append((np.load(tmp_path / tag / "c1_scores.npy"), np.load(tmp_path / tag / "c1_ids.npy")))
    (s, i), (s2, i2) = got
    assert s.dtype == np.float32 and i.dtype == np.float64 and s.shape == i.shape == (64, 10)
    assert np.array_equal(s.view(np.uint32), s2.view(np.uint32)) and np.array_equal(i, i2)
    # the same rows the benchmark loads (svsb_load_synthetic, ids 1..n), read back and judged by the oracle
    n, d, k = 10_548, 1536, 10
    with svs_b200.Engine([0]) as e:
        e.load_synthetic(n, d, seed=0, id0=1, id_step=1)
        m, ids = e.read_rows(0, n)
    rng = np.random.default_rng(1)                          # bench.py's unit_queries(128, d, 1)
    qs = rng.random((128, d), dtype=np.float32)
    qs /= np.sqrt((qs * qs).sum(axis=1))[:, None]
    for j in (0, 31, 63):
        want = oracle.superheavy(m, ids, qs[j], k)
        oracle.compare_retrieval([(float(a), int(b)) for a, b in zip(s[j], i[j])], want, oracle.scores_of(m, qs[j]), ids)
