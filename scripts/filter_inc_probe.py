"""Incremental update with the single-query filter on and off: load 1M x 1536, then three times add one row and
query it twice, timing svsb_apply_mutations and each query on the host (profiles/r05_filter_ab.txt)."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from svs_b200.engine import Engine
n, d, k = 1_000_000, 1536, 100
for f in ("1", "0", "1"):
    os.environ["SVSB_FILTER"] = f
    e = Engine([0]); e.load_synthetic(n, d, seed=0, id0=1, id_step=1)
    rng = np.random.default_rng(99)
    q = rng.random(d, dtype=np.float32); q /= np.sqrt((q*q).sum())
    for _ in range(5): e.query(q, k)
    nid = n + 1
    for rep in range(3):
        row = rng.random((1, d), dtype=np.float32); row /= np.sqrt((row*row).sum())
        t0 = time.perf_counter(); e.apply_mutations([], [nid], row); t1 = time.perf_counter()
        s, i = e.query(row[0], k); t2 = time.perf_counter()
        s, i = e.query(row[0], k); t3 = time.perf_counter()
        print(f"FILTER={f} add#{rep}: apply {1e3*(t1-t0):.2f} ms, first query {1e3*(t2-t1):.2f} ms, second query {1e3*(t3-t2):.2f} ms, top={i[0]==nid}", flush=True)
        nid += 1
    e.close()
