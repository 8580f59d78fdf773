#!/usr/bin/env python
"""bench.py -- retrieve queries/sec on B200 for the SVS hot path (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2] [--configs c1,c5,c3,c4 | --only]
                    [--impl reference] [--dump-outputs DIR]

A "step" is one batch of QUERIES_PER_STEP single-query retrieves (distinct query vectors) against the
resident matrix: similarity (fp32 GEMV over all rows) + exact top-k, i.e. the body of the reference's
`superheavy()` (src/svs/kb.py:1622-1627).  Headline workload: BASELINE.json configs[1] = 1M x 1536 fp32,
top-100 ("c2").  With N>1 (torchrun, one rank per GPU) the SAME matrix is row-sharded over the ranks
(strong scaling): every rank computes its local top-k and the k-candidate records are exchanged by the
kernels themselves over NVLink peer memory (svs_b200/sharded.py).

ONE JSON line (rank 0).  The top-level keys are the headline workload's; the other BASELINE.json configs
run as short legs of the same invocation and are attached under "configs": {"c1": {...}, "c5": {...},
"c3": {...}, "c4": {...}}, each with value, e2e, roofline and parity.  Extra keys of every leg:
`roofline` (dominant kernel, algorithmic bytes or flops per launch over its in-loop CUDA-event duration,
against MEASURED_PEAKS.json), `e2e` (the same metric through the C ABI with HOST buffers: the query goes in
from host memory and the k results come back to host memory inside every call), `parity` (a sample of the
timed queries judged by the oracle's streamed superheavy() over ALL rows read back from the device; a
mismatch fails the run), `cpu_baseline` (headline only: the reference's NumPy path timed on this host).

--dump-outputs DIR (one process only) writes, after the timed steps of every leg, what that leg's timed path computed in
its last step: DIR/<config>_scores.npy (float32, one row of k scores per query of the step) and DIR/<config>_ids.npy
(float64 embeddings.id, exact below 2**53).  A row the path left short (a batched query it routes to the exact path)
is padded with NaN / -1.  Inputs are seeded, so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The reference arm must run on all the host threads OpenBLAS can use, but torchrun exports OMP_NUM_THREADS=1 to
# every rank: undo that BEFORE NumPy loads its BLAS (rank 0 alone runs the arm).
if "--impl" in sys.argv and sys.argv[sys.argv.index("--impl") + 1:][:1] == ["reference"]:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

sys.dont_write_bytecode = True          # a benchmark run writes nothing into the tree it runs from, which may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

QUERIES_PER_STEP = 64
BATCH = 1024          # queries per step of the batched workload (c3)
WORKLOADS = {
    # name: (rows, dims, k, description)
    "c1": (10_548, 1536, 10, "10,548 x 1536 fp32 top-10 (dad-jokes shape, synthetic unit rows)"),
    "c2": (1_000_000, 1536, 100, "1M x 1536 fp32 top-100 (README 'One Million Documents' shape)"),
    "c3": (1_000_000, 768, 100, "1M x 768 fp32, batches of 1024 queries, top-100 (batched tensor-core path)"),
    "c4": (10_000_000, 1536, 100, "10M x 1536 fp32 top-100, row-sharded"),
    "c5": (1_000_000, 3072, 1000, "1M x 3072 fp32 top-1000"),
}
PARITY_QUERIES = 4    # timed queries per leg judged by the oracle


def config_of(name: str) -> dict:
    """The `config` object: identical in our arm and in the reference arm."""
    n, d, k, desc = WORKLOADS[name]
    mb = n * d * 4 / 1e6
    l2 = ("inputs larger than L2 (matrix %.2f GB, distinct queries)" % (mb / 1e3) if mb > 200 else
          "matrix %.1f MB is L2-resident by design of the config (distinct queries)" % mb)
    return {"workload": desc, "rows": n, "dims": d, "k": k, "l2": l2}


def measured_peaks() -> dict:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def measured_peak_tflops():
    """(sustained, burst, source): a batch step is ~1.5 ms, i.e. a kernel timed alone -> the BURST figure is the
    applicable denominator; the sustained one is reported next to it."""
    j = measured_peaks()
    if "bf16_tflops" in j:
        return float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), float(j["bf16_tflops"]), \
            "measured (MEASURED_PEAKS.json bf16_tflops = burst; cuBLAS 16-bit dense)"
    return 1400.0, 1650.0, "fallback (B200_PROFILING.md)"


def measured_peak_gbs():
    j = measured_peaks()
    if "hbm_gbs" in j:
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def replayed_traffic(name: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed ncu capture
    (profiles/); NOT measured in this run -- ncu cannot run inside a timed bench."""
    for fn in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", fn)
        if os.path.exists(p):
            try:
                v = json.load(open(p)).get(name)
                if v is not None:
                    return v, f"replayed from profiles/{fn} (one `ncu --set full` capture of this kernel on this workload), not measured in this run"
            except Exception:
                pass
    return None, "no ncu capture of this workload under profiles/"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def unit_queries(count: int, d: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    q = rng.random((count, d), dtype=np.float32)
    q /= np.sqrt((q * q).sum(axis=1))[:, None]
    return q


# ---------------------------------------------------------------------------------------------------
# reference / CPU arm: the reference's own NumPy path on the host cores
# ---------------------------------------------------------------------------------------------------
def _reference_get_top_k():
    """svs.util.get_top_k from the byte-compiled reference (oracle/_ref) if present, else the oracle port."""
    ref = os.path.join(ROOT, "oracle", "_ref", "svs_ref.bin")    # zip of the byte-compiled reference
    if os.path.isfile(ref):
        try:
            sys.path.insert(0, ref)
            from svs.util import get_top_k          # the reference's own code
            return get_top_k, "reference"
        except Exception:
            sys.path.remove(ref)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from svs_oracle import get_top_k                # CPU restatement (checker), timed only as the baseline
    return get_top_k, "port"


def blas_threads() -> int:
    """Threads the BLAS behind np.dot actually uses (what `cores` must report)."""
    try:
        from threadpoolctl import threadpool_info
        n = [int(p.get("num_threads", 0)) for p in threadpool_info() if p.get("user_api") == "blas"]
        if n and max(n) > 0:
            return max(n)
    except Exception:
        pass
    return os.cpu_count() or 1


def cpu_matrix(n: int, d: int, seed: int = 0) -> np.ndarray:
    """The notebook's recipe (uniform [0,1) rows / L2 norm) in chunks, float32."""
    rng = np.random.default_rng(seed)
    m = np.empty((n, d), dtype=np.float32)
    step = 65536
    for a in range(0, n, step):
        b = min(n, a + step)
        blk = rng.random((b - a, d), dtype=np.float32)
        blk /= np.sqrt(np.einsum("ij,ij->i", blk, blk))[:, None]
        m[a:b] = blk
    return m


def cpu_arm(n: int, d: int, k: int):
    """Returns (matrix rows used, function running one query, kind)."""
    get_top_k, kind = _reference_get_top_k()
    try:
        avail = int(next(l for l in open("/proc/meminfo") if l.startswith("MemAvailable")).split()[1]) * 1024
    except Exception:
        avail = 8 << 30
    rows = n
    while rows * d * 4 > avail * 0.4 and rows > 50_000:
        rows //= 2
    m = cpu_matrix(rows, d, 0)
    ids = np.arange(1, rows + 1, dtype=np.int64)

    def one_query(qv):
        x = np.dot(m, qv)                                      # src/svs/kb.py:1623
        return [(s, int(ids[i])) for s, i in get_top_k(x, k)]  # src/svs/kb.py:1625-1626
    return rows, one_query, kind


def cpu_baseline_of(name: str, queries: np.ndarray, per_query_note: str = "") -> dict:
    n, d, k, _ = WORKLOADS[name]
    rows, one_query, kind = cpu_arm(n, d, k)
    for i in range(2):
        one_query(queries[i])
    t0 = time.perf_counter(); cnt = 0
    while cnt < 10 or (time.perf_counter() - t0 < 5.0 and cnt < 40):
        one_query(queries[cnt % len(queries)]); cnt += 1
    dt = time.perf_counter() - t0
    scale = rows / n
    return {"value": cnt / dt * scale, "unit": "queries/s", "cores": blas_threads(), "kind": kind,
            "sample": f"{cnt} queries of np.dot + get_top_k on {rows} x {d} host rows" + per_query_note
                      + ("" if rows == n else f", scaled x{scale:.3f}")}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                                  # other ranks exit 0 without work
    n, d, k, _ = WORKLOADS[args.workload]
    rows, one_query, kind = cpu_arm(n, d, k)
    qs = unit_queries(8, d, 1)
    per_step = 2                                                # bounded sample: 2 queries per step
    for w in range(args.warmup):
        one_query(qs[w % len(qs)])
    t0 = time.perf_counter()
    for s in range(args.steps):
        for j in range(per_step):
            one_query(qs[(s * per_step + j) % len(qs)])
    dt = time.perf_counter() - t0
    scale = rows / n                                            # < 1 only if the host lacks RAM for n rows
    qps = args.steps * per_step / dt * scale
    sample = (f"{args.steps} steps x {per_step} queries of np.dot + get_top_k on {rows} x {d} host rows"
              + ("" if rows == n else f", scaled x{scale:.3f} to {n} rows (host RAM bound)"))
    line = {
        "impl": "reference", "metric": "retrieve_queries_per_sec", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": blas_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# parity: the oracle's superheavy() streamed over ALL rows of the device matrix (checker only; after the timed region)
# ---------------------------------------------------------------------------------------------------
def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import svs_oracle                                           # test infrastructure: the checker, never the thing measured
    return svs_oracle


def oracle_local_scores(read_rows, n_local: int, queries: np.ndarray, slab: int = 16384):
    """np.dot(slab, q) (src/svs/kb.py:1623) per query over every row of this engine, read back from the device slab by
    slab (a slab stays in the host's cache across the queries).  Returns (scores (nq, n_local) f32, ids (n_local,))."""
    oracle = _oracle()
    x = np.empty((len(queries), n_local), dtype=np.float32)
    ids = np.empty(n_local, dtype=np.int64)
    for a in range(0, n_local, slab):
        cnt = min(slab, n_local - a)
        rows, rid = read_rows(a, cnt)
        ids[a:a + cnt] = rid
        for j, q in enumerate(queries):
            x[j, a:a + cnt] = oracle.scores_of(rows, q)
    return x, ids


def judge(got_lists, want_lists, score_maps) -> dict:
    """The tolerance-aware comparator of SURVEY.md section 8c (oracle.compare_retrieval) per query; raises on a mismatch.
    score_maps[j]: {embeddings.id: oracle score} covering every id of got_lists[j] and want_lists[j]."""
    oracle = _oracle()
    exact, max_rel = 0, 0.0
    for got, want, smap in zip(got_lists, want_lists, score_maps):
        ids_sub = np.fromiter(smap.keys(), dtype=np.int64, count=len(smap))
        x_sub = np.fromiter(smap.values(), dtype=np.float32, count=len(smap))
        rep = oracle.compare_retrieval(got, want, x_sub, ids_sub)
        exact += 1 if [g[1] for g in got] == [w[1] for w in want] else 0
        max_rel = max(max_rel, rep["max_rel_score_err"])
    if max_rel > 1e-5:
        raise AssertionError(f"parity: relative score error {max_rel:.3e} > 1e-5")
    return {"checked": len(got_lists), "exact": exact, "tolerance_ok": len(got_lists), "max_rel_err": max_rel,
            "tolerance": "<= 1e-5 relative score error; rank swaps only among scores closer than that (BASELINE.json north_star)",
            "oracle": "np.dot + get_top_k (oracle/svs_oracle.py = src/svs/kb.py:1622-1627, util.py:190-203) over ALL rows, read back from the device"}


def parity_single(eng, n: int, k: int, queries: np.ndarray, got_lists) -> dict:
    oracle = _oracle()
    x, ids = oracle_local_scores(eng.read_rows, n, queries)
    want, maps = [], []
    row_of = None
    for j in range(len(queries)):
        w = [(s, int(ids[i])) for s, i in oracle.get_top_k(x[j], k)]            # src/svs/kb.py:1625-1626
        want.append(w)
        if row_of is None:
            step = int(ids[1] - ids[0]) if n > 1 else 1                          # synthetic ids: id0 + row * step
            row_of = lambda e, i0=int(ids[0]), st=step: (int(e) - i0) // st
        smap = {}
        for _s, e in list(got_lists[j]) + w:
            r = row_of(e)
            assert 0 <= r < n and int(ids[r]) == int(e), f"parity: id {e} is not in the matrix"
            smap[int(e)] = float(x[j, r])
        maps.append(smap)
    return judge(got_lists, want, maps)


def parity_sharded(dist, rank, world, sr, k: int, queries: np.ndarray, got_lists) -> dict:
    """Every rank scores ITS shard with the oracle; rank 0 merges the per-shard oracle lists under the reference's order
    (score desc, index desc: util.py:203) and judges the engine's answer (identical on every rank)."""
    oracle = _oracle()
    n_local = sr.local_rows
    x, ids = oracle_local_scores(sr.backend.engine.read_rows, n_local, queries) if n_local else \
        (np.empty((len(queries), 0), np.float32), np.empty(0, np.int64))
    part = []
    for j in range(len(queries)):
        loc = [(s, sr.row0 + i, int(ids[i])) for s, i in oracle.get_top_k(x[j], k)] if n_local else []
        look = {}
        if n_local:
            want_ids = np.array([e for _s, e in got_lists[j]], dtype=np.int64)
            pos = np.searchsorted(ids, want_ids)                                  # ids ascend with the row
            for e, p in zip(want_ids, pos):
                if p < n_local and ids[p] == e:
                    look[int(e)] = float(x[j, p])
        part.append((loc, look))
    gathered = [None] * world
    dist.all_gather_object(gathered, part)
    if rank != 0:
        return {}
    want, maps = [], []
    for j in range(len(queries)):
        allc = sorted([c for g in gathered for c in g[j][0]], key=lambda c: (c[0], c[1]), reverse=True)[:k]
        want.append([(s, e) for s, _r, e in allc])
        smap = {e: s for s, _r, e in allc}
        for g in gathered:
            smap.update(g[j][1])
        maps.append(smap)
    return judge(got_lists, want, maps)


# ---------------------------------------------------------------------------------------------------
# our arm, one GPU
# ---------------------------------------------------------------------------------------------------
def e2e_pipelined(eng, queries: np.ndarray, k: int, steps: int, in_flight: int = 3):
    """The e2e metric with `in_flight` queries pending (Engine.submit / Pending.result): host query in, host result out for
    every query.  The warm-up keeps `in_flight` queries pending too, so that every query context (stream, workspace,
    pinned staging: created on first use) exists before the clock starts -- warming up one query at a time left the
    second and third context's allocations inside the timed pass (4 % at C2, 20 % at C5).  Two passes of
    steps x QUERIES_PER_STEP queries, the better one reported, both listed.
    Returns (queries/s, the first len(queries) results, [queries/s of every pass])."""
    import gc
    first = []
    warm = [eng.submit(queries[i], k) for i in range(in_flight)]
    for i in range(in_flight, 4 * in_flight):
        warm.pop(0).result()
        warm.append(eng.submit(queries[i % len(queries)], k))
    for p in warm:
        p.result()
    nq = steps * QUERIES_PER_STEP
    rates = []
    for _pass in range(2):
        pend = []
        gc.collect(); gc.disable()
        try:
            t0 = time.perf_counter()
            for j in range(nq):
                pend.append(eng.submit(queries[j % len(queries)], k))
                if len(pend) == in_flight:
                    r = pend.pop(0).result()
                    if len(first) < len(queries):
                        first.append(r)
            for p in pend:
                r = p.result()
                if len(first) < len(queries):
                    first.append(r)
            rates.append(nq / (time.perf_counter() - t0))
        finally:
            gc.enable()
    return max(rates), first, rates


def step_arrays(lists, k: int):
    """[(score, emb_id), ...] per query -> (scores (nq, k) float32, ids (nq, k) float64), short rows padded NaN / -1."""
    s = np.full((len(lists), k), np.nan, dtype=np.float32)
    i = np.full((len(lists), k), -1.0, dtype=np.float64)
    for j, res in enumerate(lists):
        s[j, :len(res)] = [a for a, _ in res]
        i[j, :len(res)] = [b for _, b in res]
    return s, i


def last_step_single(eng, queries: np.ndarray, k: int):
    """What the device-resident loop (svsb_bench_run) computes in every step: the answers to queries 0 .. QUERIES_PER_STEP-1.
    The loop keeps only its last query's answer, so each query goes through the same loop once on its own; the uploaded
    queries are restored afterwards."""
    res = []
    for j in range(QUERIES_PER_STEP):
        eng.bench_set_queries(queries[j % len(queries)][None])
        eng.bench_run(k, 1)
        res.append(eng.bench_last_result(k))
    eng.bench_set_queries(queries)
    return res


def incremental_probe(eng, n: int, d: int, k: int) -> dict:
    """SURVEY.md section 8f rank 4: a one-document add (and a delete) on the resident matrix, then the next retrieve --
    what the reference answers with a full rebuild (src/svs/kb.py:1523, 573-618).  The new row must come back first."""
    rng = np.random.default_rng(99)
    out = {}
    next_id = n + 1                                               # synthetic ids are 1..n
    for tag in ("first_add_then_retrieve_ms", "next_add_then_retrieve_ms"):
        row = rng.random((1, d), dtype=np.float32)
        row /= np.sqrt((row * row).sum())
        t0 = time.perf_counter()
        eng.apply_mutations([], [next_id], row)
        s, i = eng.query(row[0], k)
        out[tag] = (time.perf_counter() - t0) * 1e3
        if int(i[0]) != next_id or abs(float(s[0]) - 1.0) > 1e-5:
            raise AssertionError("incremental add: the new row is not the best match of itself")
        next_id += 1
    t0 = time.perf_counter()
    eng.apply_mutations([next_id - 1, 17], [], None)
    s, i = eng.query(row[0], k)
    out["delete_then_retrieve_ms"] = (time.perf_counter() - t0) * 1e3
    if next_id - 1 in i.tolist() or 17 in i.tolist():
        raise AssertionError("incremental delete: a tombstoned row was returned")
    phys, live = eng.generation_rows()
    out.update({"rows_physical": phys, "rows_live": live,
                "note": "a loaded shard carries 0.4 % head-room, so adds append in place; a shard that fills up is re-allocated with 12.5 % head-room (one device-to-device copy)"})
    return out


def leg_single(name: str, steps: int, warmup: int, headline: bool, cpu: bool, outputs: dict | None = None) -> dict:
    """Single-query workloads (c1, c2, c4, c5) on one GPU.  `outputs`, when given, receives the last step's answers."""
    import svs_b200
    from svs_b200.engine import Engine
    n, d, k, _ = WORKLOADS[name]
    queries = unit_queries(128, d, 1)                            # distinct queries: never L2-useful
    peak, peak_src = measured_peak_gbs()
    eng = Engine([0])
    t_load = time.perf_counter()
    eng.load_synthetic(n, d, seed=0, id0=1, id_step=1)
    load_s = time.perf_counter() - t_load
    eng.bench_set_queries(queries)
    for _ in range(warmup):
        eng.bench_run(k, QUERIES_PER_STEP)
    sampler = ClockSampler(0)
    sampler.start()
    total_ms = gemv_ms = 0.0
    launches = 0
    for _ in range(steps):                                       # each step: events on the launching stream, sync on both sides
        r = eng.bench_run(k, QUERIES_PER_STEP, with_gemv=True)
        total_ms += r["total_ms"]; gemv_ms += r["gemv_ms"]; launches += r["launches"]
    clocks = sampler.stop()
    last_timed = eng.bench_last_result(k)                        # answer of the LAST query of the timed loop
    nq = steps * QUERIES_PER_STEP
    value = nq / (total_ms / 1e3)
    # latency: one query in flight, host-visible (host buffers in and out)
    lat = []
    for i in range(40):
        t0 = time.perf_counter(); eng.query(queries[i % len(queries)], k); lat.append(time.perf_counter() - t0)
    # e2e: the public C-ABI call with host buffers, H2D + D2H inside every call
    for i in range(8):
        eng.query(queries[i], k)
    t0 = time.perf_counter()
    for s in range(steps):
        for j in range(QUERIES_PER_STEP):
            eng.query(queries[(s * QUERIES_PER_STEP + j) % len(queries)], k)
    e2e_sync_qps = nq / (time.perf_counter() - t0)
    e2e_qps, piped, e2e_passes = e2e_pipelined(eng, queries, k, steps)
    # parity of the timed paths: PARITY_QUERIES of the e2e calls' answers judged by the oracle over all rows, and the
    # device-resident loop's last answer must equal the e2e call's for the same query, bit for bit
    pq = [0, 1, QUERIES_PER_STEP // 2, (QUERIES_PER_STEP - 1) % len(queries)][:PARITY_QUERIES]
    got = [eng.retrieve(queries[j], k) for j in pq]
    for j in pq:                                                 # the pipelined e2e loop returned the same bits
        s_, i_ = piped[j]
        if [(float(a), int(b)) for a, b in zip(s_, i_)] != got[pq.index(j)]:
            raise AssertionError(f"{name}: svsb_query_submit/wait and svsb_query disagree")
    parity = parity_single(eng, n, k, queries[pq], got)
    parity["device_resident_loop_bits_equal_e2e"] = bool(last_timed == eng.retrieve(queries[(QUERIES_PER_STEP - 1) % len(queries)], k))
    if not parity["device_resident_loop_bits_equal_e2e"]:
        raise AssertionError(f"{name}: the device-resident loop and svsb_query disagree")
    if outputs is not None:                                      # before the incremental probe changes the matrix
        step = last_step_single(eng, queries, k)
        if step[-1] != last_timed:
            raise AssertionError(f"{name}: a query run alone and the timed loop's last query disagree")
        outputs[name] = step_arrays(step, k)
    algo_bytes = n * d * 4
    achieved = algo_bytes * nq / (gemv_ms / 1e3) / 1e9
    traffic, traffic_src = replayed_traffic(name)
    line = {
        "metric": "retrieve_queries_per_sec", "value": value, "unit": "queries/s", "n_gpus": 1,
        "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(name),
        "run": {"queries_per_step": QUERIES_PER_STEP, "parallelism": "1 GPU"},
        "ms_per_query": total_ms / nq, "latency_ms": {"median": float(np.median(lat)) * 1e3, "min": float(min(lat)) * 1e3},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": "gemv_tma_kernel", "peak_source": peak_src,
                     "timed_launches": "1 in 8 bracketed with CUDA events inside the timed loop",
                     "algorithmic_bytes_per_launch": algo_bytes, "frac_of_nominal_8TBs": achieved / 8000.0,
                     "whole_query_frac": (algo_bytes * nq / (total_ms / 1e3) / 1e9) / peak},
        "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": QUERIES_PER_STEP * d * 4,
                "d2h_bytes_per_step": QUERIES_PER_STEP * (k * 12 + 4),
                "how": "svsb_query_submit / svsb_query_wait from one host thread, 3 queries in flight; every query goes in from host "
                       "memory and its k results come back to host memory inside the timed region",
                "one_query_in_flight": e2e_sync_qps, "passes": e2e_passes, "reported": "the better of two passes of steps x 64 queries"},
        "parity": parity,
        "gpu_launches": int(launches), "clocks": clocks, "load_synthetic_s": load_s,
    }
    if headline:
        line["incremental_update"] = incremental_probe(eng, n, d, k)
    if cpu:
        line["cpu_baseline"] = cpu_baseline_of(name, queries)
    eng.close()
    return line


def leg_batch(name: str, steps: int, warmup: int, headline: bool, cpu: bool, outputs: dict | None = None) -> dict:
    """c3 on one GPU: one step = one batch of BATCH queries through svsb_query_batch's pipeline.  `outputs`, when given,
    receives the last step's answers."""
    from svs_b200 import pinned_empty
    from svs_b200.engine import Engine
    n, d, k, _ = WORKLOADS[name]
    queries = unit_queries(BATCH, d, 2)
    peak_sus, peak_burst, peak_src = measured_peak_tflops()
    eng = Engine([0])
    t_load = time.perf_counter()
    eng.load_synthetic(n, d, seed=0, id0=1, id_step=1)
    load_s = time.perf_counter() - t_load
    eng.bench_set_queries(queries)
    for _ in range(warmup):                                      # a batch is ~1.5 ms: 10 per warm-up step lets the clocks ramp
        eng.bench_run_batch(k, 10)
    sampler = ClockSampler(0)
    sampler.start()
    total_ms = coarse_ms = 0.0
    launches = 0
    for _ in range(steps):                                       # the timed steps: the product's pipeline, nothing else in the stream
        r = eng.bench_run_batch(k, 1)
        total_ms += r["total_ms"]; launches += r["launches"]
    clocks = sampler.stop()
    if outputs is not None:                                      # the last timed batch, still in the pipeline's output buffers
        outputs[name] = step_arrays([eng.bench_batch_result(qi, k)[0] for qi in range(BATCH)], k)
    for _ in range(steps):                                       # the filter pass's own duration (roofline numerator), bracketed in a
        coarse_ms += eng.bench_run_batch(k, 1, with_coarse=True)["coarse_ms"]   # separate pass: the bracket's host sync idles the GPU ~20 us
    cand, resc, flags = eng.batch_stats(BATCH)
    # the timed path must compute the answer: a few queries of the device-resident batch against the single-query kernels
    agree = True
    for qi in (0, BATCH // 2, BATCH - 1):
        got, flag = eng.bench_batch_result(qi, k)
        agree = agree and flag == 0 and got == eng.retrieve(queries[qi], k)
    # e2e: the public C-ABI call with host buffers (H2D of the batch from pinned host memory, D2H of the results
    # into pinned host memory, inside every call)
    hq = pinned_empty((BATCH, d), np.float32)
    hq[:] = queries
    out = (pinned_empty((BATCH, k), np.float32), pinned_empty((BATCH, k), np.int64), np.zeros(BATCH, dtype=np.int32))
    eng.query_batch(hq, k, out=out)
    t0 = time.perf_counter()
    for s in range(steps):
        eng.query_batch(hq, k, out=out)
    e2e_qps = steps * BATCH / (time.perf_counter() - t0)
    ref_s, ref_i, _ = eng.query_batch(queries, k)                # pageable buffers take the staged path: same answer
    agree = agree and np.array_equal(out[0].view(np.uint32), ref_s.view(np.uint32)) and np.array_equal(out[1], ref_i)
    if not agree:
        raise AssertionError(f"{name}: the batched path and the single-query kernels disagree")
    pq = [0, 1, BATCH // 2, BATCH - 1][:PARITY_QUERIES]
    got = [[(float(s), int(i)) for s, i in zip(out[0][j, :out[2][j]], out[1][j, :out[2][j]])] for j in pq]
    parity = parity_single(eng, n, k, queries[pq], got)
    parity["batched_path_bits_equal_single_query"] = bool(agree)
    nq = steps * BATCH
    flop = 2.0 * n * d * BATCH
    achieved = flop * steps / (coarse_ms / 1e3) / 1e12
    traffic, traffic_src = replayed_traffic(name)
    line = {
        "metric": "retrieve_queries_per_sec", "value": nq / (total_ms / 1e3), "unit": "queries/s", "n_gpus": 1,
        "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 results (f16 tensor-core coarse pass + exact f32 re-score)", "data": "synthetic",
        "config": config_of(name),
        "run": {"queries_per_step": BATCH, "parallelism": "1 GPU", "f16_shadow_gb": n * d * 2 / 1e9},
        "ms_per_query": total_ms / nq,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_burst, "unit": "TFLOP/s", "frac": achieved / peak_burst,
                     "frac_of_sustained_peak": achieved / peak_sus, "peak_sustained": peak_sus,
                     "whole_batch_frac": flop * steps / (total_ms / 1e3) / 1e12 / peak_burst,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": "coarse_gemm_kernel<0> (filter pass)",
                     "peak_source": peak_src, "algorithmic_flop_per_launch": flop, "coarse_ms_per_batch": coarse_ms / steps,
                     "hbm_floor_ms": n * d * 2 / 1e9 / measured_peak_gbs()[0] * 1e3},
        "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": BATCH * d * 4, "d2h_bytes_per_step": BATCH * (k * 12 + 8)},
        "parity": parity,
        "gpu_launches": int(launches), "clocks": clocks, "load_synthetic_s": load_s,
        "batch_stats": {"candidates_mean": float(cand.mean()), "candidates_max": int(cand.max()), "rescored_mean": float(resc.mean()),
                        "rescored_max": int(resc.max()), "fallback_queries": int((flags != 0).sum()),
                        "agrees_with_single_query_bits": bool(agree)},
    }
    if cpu:
        line["cpu_baseline"] = cpu_baseline_of(name, queries, " (the reference has no batched API: a batch is a loop)")
    eng.close()
    return line


# ---------------------------------------------------------------------------------------------------
# our arm, N > 1: one rank per GPU (torchrun), row shards
# ---------------------------------------------------------------------------------------------------
class Spmd:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.exchange = args.exchange
        torch.cuda.set_device(self.local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.cpu_group = dist.new_group(backend="gloo")          # host-side barriers that put no kernel on any GPU

    def cpu_barrier(self):
        self.dist.barrier(group=self.cpu_group)

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]


def leg_sharded(sp: Spmd, name: str, steps: int, warmup: int) -> dict:
    import svs_b200
    from svs_b200.sharded import ShardedRetriever, MICRO_BATCH
    torch, dist, rank, world = sp.torch, sp.dist, sp.rank, sp.world
    n, d, k, _ = WORKLOADS[name]
    queries = unit_queries(128, d, 1)
    peak, peak_src = measured_peak_gbs()
    l0 = svs_b200.launch_count()
    sr = ShardedRetriever(rank, world, sp.local_rank, exchange=sp.exchange)
    sr.load_synthetic(n, d, seed=0, id0=1, id_step=1)
    sr.set_queries(queries)
    for _ in range(warmup):
        sr.run_queries(k, QUERIES_PER_STEP)
    sampler = ClockSampler(sp.local_rank)
    if rank == 0:
        sampler.start()
    dist.barrier(); torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    gemv_ms = 0.0
    for _ in range(steps):
        gemv_ms += sr.run_queries(k, QUERIES_PER_STEP, time_gemv=True)
    ev1.record()
    torch.cuda.synchronize(); dist.barrier()
    total_ms, gemv_ms = sp.max_over_ranks(ev0.elapsed_time(ev1), gemv_ms)
    clocks = sampler.stop() if rank == 0 else None
    nq = steps * QUERIES_PER_STEP
    # the device-resident loop's last micro-batch is still in its output buffers: query (QUERIES_PER_STEP - 1) sits in row
    # (QUERIES_PER_STEP - 1) % MICRO_BATCH
    o_s, o_i, o_c = sr._buffers(k)[2]
    jl = (QUERIES_PER_STEP - 1) % MICRO_BATCH
    cl = int(o_c[jl].item())
    last_timed = [(float(a), int(b)) for a, b in zip(o_s[jl, :cl].cpu().numpy(), o_i[jl, :cl].cpu().numpy())]
    # e2e: host query in, host result out, every call
    for i in range(4):
        sr.retrieve_arrays(queries[i], k)
    dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(steps):
        for j in range(QUERIES_PER_STEP):                       # host query in, host (scores, ids) arrays out, as Engine.query at N=1
            sr.retrieve_arrays(queries[(s * QUERIES_PER_STEP + j) % len(queries)], k)
    torch.cuda.synchronize(); dist.barrier()
    (e2e_sync_s,) = sp.max_over_ranks(time.perf_counter() - t0)
    # the same with 3 queries in flight (svsb_query_peer_submit / _wait): every query still goes in from host memory and
    # comes back to host memory inside the timed region
    piped = []
    warm = [sr.submit(queries[i], k) for i in range(3)]           # warm up with all three tickets in flight
    for i in range(3, 9):
        sr.wait(warm.pop(0)); warm.append(sr.submit(queries[i], k))
    for p in warm:
        sr.wait(p)
    dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    pend = []
    for j in range(nq):
        pend.append(sr.submit(queries[j % len(queries)], k))
        if len(pend) == 3:
            r = sr.wait(pend.pop(0))
            if len(piped) < QUERIES_PER_STEP:
                piped.append(r)
    for p in pend:
        r = sr.wait(p)
        if len(piped) < QUERIES_PER_STEP:
            piped.append(r)
    torch.cuda.synchronize(); dist.barrier()
    (e2e_s,) = sp.max_over_ranks(time.perf_counter() - t0)
    # parity: the e2e path's answers for PARITY_QUERIES of the timed queries, judged by the oracle on every shard
    pq = [0, 1, QUERIES_PER_STEP // 2, (QUERIES_PER_STEP - 1) % len(queries)][:PARITY_QUERIES]
    got = [sr.retrieve(queries[j], k) for j in pq]
    same = bool(last_timed == got[-1])
    for j in pq:
        s_, i_ = piped[j]
        same = same and [(float(a), int(b)) for a, b in zip(s_, i_)] == got[pq.index(j)]
    parity = parity_sharded(dist, rank, world, sr, k, queries[pq], got)
    launches = torch.tensor([svs_b200.launch_count() - l0], device="cuda", dtype=torch.int64)
    shard_bytes = sr.local_rows * d * 4
    exchange = sr.exchange
    sr.close()
    if rank != 0:
        return {}
    if not same:
        raise AssertionError(f"{name}: the device-resident loop, svsb_query_peer and svsb_query_peer_submit/wait disagree")
    parity["device_resident_loop_bits_equal_e2e"] = same
    achieved = shard_bytes * nq / (gemv_ms / 1e3) / 1e9
    return {
        "metric": "retrieve_queries_per_sec", "value": nq / (total_ms / 1e3), "unit": "queries/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(name),
        "run": {"queries_per_step": QUERIES_PER_STEP, "per_gpu_shard_gb": shard_bytes / 1e9,
                "parallelism": (f"row-sharded over {world} GPUs, k-candidate records pushed into every rank's window over "
                                "NVLink peer memory by the selection kernel, merge kernel waits on flags (no collective call)"
                                if exchange == "peer" else
                                f"row-sharded over {world} GPUs, NCCL all-gather of k candidates + merge kernel")},
        "ms_per_query": total_ms / nq,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "traffic_source": "ncu captures are single-GPU (profiles/)",
                     "kernel": "gemv_tma_kernel (per GPU, rank-max of the sampled launches)", "peak_source": peak_src,
                     "timed_launches": "1 in 8 bracketed with CUDA events inside the timed loop",
                     "algorithmic_bytes_per_launch": shard_bytes,
                     "whole_query_frac": (shard_bytes * nq / (total_ms / 1e3) / 1e9) / peak},
        "e2e": {"value": nq / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": QUERIES_PER_STEP * d * 4,
                "d2h_bytes_per_step": QUERIES_PER_STEP * (k * 12 + 4),
                "how": "svsb_query_peer_submit / _wait on every rank, 3 queries in flight; host query in, host result out",
                "one_query_in_flight": nq / e2e_sync_s},
        "parity": parity,
        "gpu_launches": int(launches[0]), "clocks": clocks,
    }


def leg_batch_sharded(sp: Spmd, name: str, steps: int, warmup: int) -> dict:
    """c3 on N GPUs: rows sharded, every rank runs the batched pipeline on its shard, ONE all-gather of 1024 records
    per rank and ONE merge launch per batch."""
    import svs_b200
    from svs_b200.sharded import ShardedRetriever
    torch, dist, rank, world = sp.torch, sp.dist, sp.rank, sp.world
    n, d, k, _ = WORKLOADS[name]
    steps = steps * 8                      # a sharded batch is a fraction of a millisecond: time 8x as many of them
    queries = unit_queries(BATCH, d, 2)
    l0 = svs_b200.launch_count()
    sr = ShardedRetriever(rank, world, sp.local_rank, exchange=sp.exchange)
    sr.load_synthetic(n, d, seed=0, id0=1, id_step=1)
    sr.set_queries(queries)
    for _ in range(warmup * 10):
        sr.run_batch(k, defer=True)
    sr.flush_batches()
    sampler = ClockSampler(sp.local_rank)
    if rank == 0:
        sampler.start()
    dist.barrier(); torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        sr.run_batch(k, defer=True)       # a stream of batches: each batch's merge goes behind the next batch's first phase
    sr.flush_batches()                    # ... and the last one's inside the timed region
    ev1.record()
    torch.cuda.synchronize(); dist.barrier()
    (total_ms,) = sp.max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop() if rank == 0 else None
    fallbacks = sr.last_fallbacks + sr.last_batch_unanswered()    # queries of the last timed batch the coarse pass did not answer
    global_plan = sr._global_plan(k)
    batch_peer = bool(global_plan) and sr._batch_peer_ready
    # e2e: host queries in (a page-locked tensor, DMA'd as is -- as the one-GPU leg passes page-locked arrays to
    # svsb_query_batch), host results out (page-locked buffers), every batch; pageable NumPy arrays give the same answer
    hq = torch.from_numpy(queries).pin_memory()
    for _ in range(2):
        sr.retrieve_many_pinned(hq, k)
    dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = sr.retrieve_many_pinned(hq, k)                      # host (b, d) in, host (b, k) arrays out
    torch.cuda.synchronize(); dist.barrier()
    (e2e_s,) = sp.max_over_ranks(time.perf_counter() - t0)
    out = tuple(a.copy() for a in out)
    ref = sr.retrieve_many_arrays(queries, k)
    if not (np.array_equal(out[0].view(np.uint32), ref[0].view(np.uint32)) and np.array_equal(out[1], ref[1]) and np.array_equal(out[2], ref[2])):
        raise AssertionError(f"{name}: page-locked and pageable batch calls disagree")
    pq = [0, 1, BATCH // 2, BATCH - 1][:PARITY_QUERIES]
    got = [[(float(s), int(i)) for s, i in zip(out[0][j, :out[2][j]], out[1][j, :out[2][j]])] for j in pq]
    parity = parity_sharded(dist, rank, world, sr, k, queries[pq], got)
    launches = svs_b200.launch_count() - l0
    local_rows = sr.local_rows
    sr.close()
    if rank != 0:
        return {}
    nq = steps * BATCH
    peak_sus, peak_burst, peak_src = measured_peak_tflops()
    flop_per_gpu = 2.0 * local_rows * d * BATCH
    achieved = flop_per_gpu * steps / (total_ms / 1e3) / 1e12
    return {
        "metric": "retrieve_queries_per_sec", "value": nq / (total_ms / 1e3), "unit": "queries/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 results (f16 tensor-core coarse pass + exact f32 re-score)", "data": "synthetic",
        "config": config_of(name),
        "run": {"queries_per_step": BATCH, "per_gpu_f16_shadow_gb": local_rows * d * 2 / 1e9,
                "parallelism": (
                    (f"row-sharded over {world} GPUs, no collective: ONE filter threshold per query for all ranks (order statistic {global_plan[0]} of "
                     f"the union of the ranks' samples), every rank's sample maxima and its <= {global_plan[2]} exact candidates per query stored "
                     "into every rank's batch window over NVLink peer memory by the kernels that produce them, consumers behind flag waits, "
                     "one verifying merge launch; no host synchronisation" if batch_peer else
                     f"row-sharded over {world} GPUs; per batch: one all-gather of {BATCH} x 32 sample maxima (ONE filter threshold per query for "
                     f"all ranks, order statistic {global_plan[0]} of the union sample), one all-gather of {BATCH} records of <= {global_plan[2]} "
                     "candidates per rank, one verifying merge launch; no host synchronisation in between") if global_plan else
                    f"row-sharded over {world} GPUs, per-rank thresholds, one NCCL all-gather of {BATCH} k-candidate records per rank per batch + merge kernel")},
        "ms_per_query": total_ms / nq,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_burst, "unit": "TFLOP/s", "frac": achieved / peak_burst,
                     "traffic": None, "kernel": "whole batch step per GPU (coarse passes + refine + exchange + merge), rank-max time",
                     "peak_source": peak_src, "algorithmic_flop_per_launch": flop_per_gpu},
        "e2e": {"value": nq / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": BATCH * d * 4,
                "d2h_bytes_per_step": BATCH * (k * 12 + 4)},
        "parity": parity,
        "gpu_launches": int(launches), "clocks": clocks, "batch_stats": {"fallback_queries_rank0": int(fallbacks)},
    }


def leg_inprocess(sp: Spmd, name: str, steps: int, warmup: int) -> dict:
    """The SAME workload on the SAME GPUs through ONE process: `svs_b200.Engine(devices=[0..N-1])`, the engine that
    `svs_b200.install(svs, devices=[...])` puts behind KB.retrieve (src/svs/kb.py:1608-1640).  Rank 0 drives all N GPUs
    (one worker thread per device, records pushed into device 0's window over NVLink); the other ranks have freed
    their shards and wait on a host-side barrier."""
    import svs_b200
    from svs_b200.engine import Engine
    sp.torch.cuda.empty_cache()
    sp.cpu_barrier()
    out = {}
    if sp.rank == 0:
        n, d, k, _ = WORKLOADS[name]
        world = sp.world
        queries = unit_queries(128, d, 1)
        peak, peak_src = measured_peak_gbs()
        eng = Engine(list(range(world)))
        eng.load_synthetic(n, d, seed=0, id0=1, id_step=1)
        eng.bench_set_queries(queries)
        for _ in range(warmup):
            eng.bench_run(k, QUERIES_PER_STEP)
        total_ms = gemv_ms = 0.0
        launches = 0
        for _ in range(steps):
            r = eng.bench_run(k, QUERIES_PER_STEP, with_gemv=True)
            total_ms += r["total_ms"]; gemv_ms += r["gemv_ms"]; launches += r["launches"]
        last_timed = eng.bench_last_result(k)
        nq = steps * QUERIES_PER_STEP
        for i in range(8):
            eng.query(queries[i], k)
        t0 = time.perf_counter()
        for j in range(nq):
            eng.query(queries[j % len(queries)], k)
        e2e_sync_qps = nq / (time.perf_counter() - t0)
        e2e_qps, piped, e2e_passes = e2e_pipelined(eng, queries, k, steps)
        pq = [0, 1, QUERIES_PER_STEP // 2, (QUERIES_PER_STEP - 1) % len(queries)][:PARITY_QUERIES]
        got = [eng.retrieve(queries[j], k) for j in pq]
        same = last_timed == got[-1]
        for j in pq:
            s_, i_ = piped[j]
            same = same and [(float(a), int(b)) for a, b in zip(s_, i_)] == got[pq.index(j)]
        if not same:
            raise AssertionError(f"{name} in-process: device-resident loop, svsb_query and svsb_query_submit/wait disagree")
        parity = parity_single(eng, n, k, queries[pq], got)
        parity["device_resident_loop_bits_equal_e2e"] = True
        shard_bytes = -(-n // world) * d * 4
        achieved = shard_bytes * nq / (gemv_ms / 1e3) / 1e9
        out = {
            "value": nq / (total_ms / 1e3), "unit": "queries/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "ms_per_query": total_ms / nq, "dtype": "f32", "config": config_of(name), "scaling": "strong",
            "run": {"queries_per_step": QUERIES_PER_STEP,
                    "parallelism": f"ONE process, {world} GPUs: a shard engine + a host worker thread per device, k-candidate records pushed "
                                   "into device 0's window over NVLink peer memory by the selection kernels, one waiting merge kernel; "
                                   "3 queries in flight"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "kernel": "gemv_tma_kernel (device 0's shard, sampled launches)", "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": shard_bytes,
                         "whole_query_frac": (shard_bytes * nq / (total_ms / 1e3) / 1e9) / peak},
            "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": QUERIES_PER_STEP * d * 4,
                    "d2h_bytes_per_step": QUERIES_PER_STEP * (k * 12 + 4),
                    "how": "svsb_query_submit / svsb_query_wait from one host thread, 3 queries in flight", "one_query_in_flight": e2e_sync_qps},
            "parity": parity, "gpu_launches": int(launches),
        }
        eng.close()
    sp.cpu_barrier()
    return out


def summary_of(leg: dict) -> dict:
    """What a sub-config contributes to the headline line."""
    keep = ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "ms_per_query", "latency_ms", "dtype", "config", "run",
            "roofline", "e2e", "parity", "gpu_launches", "clocks", "batch_stats", "scaling")
    return {k: leg[k] for k in keep if k in leg}


DUMP_MAX_BYTES = 64 << 20


def write_outputs(out_dir: str, outputs: dict) -> None:
    """--dump-outputs: {config: (scores, ids)} -> out_dir/<config>_scores.npy, out_dir/<config>_ids.npy."""
    total = sum(a.nbytes for pair in outputs.values() for a in pair)
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes, more than {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, (scores, ids) in outputs.items():
        np.save(os.path.join(out_dir, f"{name}_scores.npy"), scores)
        np.save(os.path.join(out_dir, f"{name}_ids.npy"), ids)


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS), help="the headline workload (top-level keys)")
    ap.add_argument("--configs", default=None, help="comma list of the other configs to attach under 'configs' (default: all the others)")
    ap.add_argument("--only", action="store_true", help="headline workload only")
    ap.add_argument("--config-steps", type=int, default=5, help="timed steps of each attached config leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-inprocess", action="store_true", help="N>1: skip the one-process-all-GPUs leg of the headline workload")
    ap.add_argument("--exchange", default="peer", choices=["peer", "collective"],
                    help="N>1, single queries: fused push over NVLink peer memory (default) or NCCL all-gather + merge")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write every leg's answers of its last timed step to DIR/<config>_{scores,ids}.npy (one process only)")
    args = ap.parse_args()
    if args.steps < 1 or args.config_steps < 1:
        ap.error("--steps and --config-steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes what the engine computed: it needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if world > 1 and args.dump_outputs is not None:
        raise SystemExit("--dump-outputs runs in one process (--gpus 1) only")
    import svs_b200                                             # fails loudly if the CUDA library is missing  # noqa: F401

    if args.only:
        extra = []
    elif args.configs is not None:
        extra = [c for c in args.configs.split(",") if c and c != args.workload]
    else:
        extra = [c for c in ("c1", "c5", "c3", "c4") if c != args.workload]
    for c in extra:
        if c not in WORKLOADS:
            raise SystemExit(f"unknown config {c}")

    if world == 1:
        outputs = {} if args.dump_outputs is not None else None

        def run(name, steps, headline):
            fn = leg_batch if name == "c3" else leg_single
            return fn(name, steps, args.warmup, headline, headline and not args.no_cpu_baseline, outputs)
        line = run(args.workload, args.steps, True)
        if extra:
            line["configs"] = {}
            for c in extra:
                try:
                    line["configs"][c] = summary_of(run(c, args.config_steps, False))
                except AssertionError:
                    raise                                           # a parity failure fails the run
                except Exception as ex:                             # e.g. not enough free HBM for c4 next to another tenant
                    line["configs"][c] = {"error": f"{type(ex).__name__}: {ex}"}
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
        return

    sp = Spmd(args)

    def run_n(name, steps):
        fn = leg_batch_sharded if name == "c3" else leg_sharded
        return fn(sp, name, steps, args.warmup)
    line = run_n(args.workload, args.steps)
    if not args.no_inprocess and args.workload != "c3":
        inproc = leg_inprocess(sp, args.workload, args.steps, args.warmup)
        if sp.rank == 0:
            line["inprocess"] = inproc
    if extra:
        cfgs = {}
        for c in extra:
            leg = run_n(c, args.config_steps)
            if sp.rank == 0:
                cfgs[c] = summary_of(leg)
        if sp.rank == 0:
            line["configs"] = cfgs
    if sp.rank == 0:
        print(json.dumps(line), flush=True)
    sp.dist.destroy_process_group()


if __name__ == "__main__":
    main()
