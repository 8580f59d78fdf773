"""The single-query filter (DESIGN.md section 4, K1f8) against K1: real bytes and rates, candidates per query.

    python scripts/filter_roofline.py [--iters 256] [--sweep] [--c4]

For each shape the device-resident loop (svsb_bench_run, pipelined, the bench's loop) runs with SVSB_FILTER=0 (K1) and
=1 (automatic: the int8 filter wherever its shadow exists), in turn, twice each.  Reported per query: the step time, the
bracketed similarity-kernel time, the REAL bytes the kernel streams (K1: n*ld*4; int8 filter: n*ld8 + 4n for the row
scales) over that time, the rows re-scored exactly and the bytes they re-read (rows * ld * 4), and whether every route
returned the same last answer (bit for bit).  bench.py's `roofline` key keeps dividing n*d*4 by the bracketed kernel,
which for the filter is an effective figure, ~4x the real one.
--sweep: matrices from 10 548 rows (the bench's C1) up, to place the size cut-off (SVSB_FILTER_MIN_MB).
--c4: also the bench's C4 (10M x 1536, top-100; ~107 GB of device memory with both shadows)."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from svs_b200.engine import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=256)
ap.add_argument("--sweep", action="store_true")
ap.add_argument("--c4", action="store_true")
args = ap.parse_args()

shapes = [(1_000_000, 1536, 100, "c2"), (1_000_000, 3072, 1000, "c5")]
if args.c4:
    shapes.append((10_000_000, 1536, 100, "c4"))
if args.sweep:
    shapes = [(10_548, 1536, 10, "c1"), (40_000, 1536, 100, ""), (80_000, 1536, 100, ""),
              (160_000, 1536, 100, ""), (320_000, 1536, 100, "")]
os.environ["SVSB_FILTER_MIN_MB"] = "0"          # every shape gets its shadows; SVSB_FILTER picks the route per call
os.environ.pop("SVSB_FILTER", None)

for n, d, k, name in shapes:
    rng = np.random.default_rng(1)
    Q = rng.random((64, d), dtype=np.float32)
    Q /= np.sqrt((Q.astype(np.float64) ** 2).sum(axis=1)).astype(np.float32)[:, None]
    e = Engine([0])
    e.load_synthetic(n, d, seed=0, id0=1, id_step=1)
    e.bench_set_queries(Q)
    ld = (d + 3) & ~3
    real_bytes = {0: n * ld * 4, 8: n * ((d + 15) & ~15) + 4 * n}
    last = {}
    for f in ("0", "1", "0", "1"):
        os.environ["SVSB_FILTER"] = f
        e.bench_run(k, 16, with_gemv=True)                   # warm-up
        r = e.bench_run(k, args.iters, with_gemv=True)
        _, rescored = e.bench_filter_stats()
        route = e.bench_filter_route()
        step_us = r["total_ms"] / args.iters * 1e3
        kern_us = r["gemv_ms"] / args.iters * 1e3
        real = real_bytes[route]
        res = e.bench_last_result(k)
        last.setdefault(route, res)
        assert last[route] == res
        print(f"{name or '-':>3} n={n} d={d} k={k} SVSB_FILTER={f:>2} route={route:>2}: step {step_us:8.1f} us, kernel {kern_us:8.1f} us, "
              f"real {real / kern_us / 1e3:7.1f} GB/s ({real / 1e9:.3f} GB), effective n*d*4 {n * d * 4 / kern_us / 1e3:7.1f} GB/s, "
              f"re-scored {rescored} rows ({rescored * ld * 4 / 1e6:.2f} MB)", flush=True)
    bits = {rt: [(np.float32(s).view(np.uint32), i) for s, i in v] for rt, v in last.items()}
    same = all(b == bits[0] for b in bits.values())
    print(f"{name or '-':>3} n={n}: last answers of every route bit-identical: {same}", flush=True)
    assert same
    e.close()
os.environ.pop("SVSB_FILTER", None)
