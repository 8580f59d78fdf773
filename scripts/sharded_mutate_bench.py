"""Run under torchrun: incremental updates on the one-process-per-GPU deployment (ShardedRetriever.apply_mutations,
compact) against loading the same rows again.  Prints the card and its power limit, then one JSON line per shape with,
in ms (host clock around calls that end in a device synchronise; slowest rank):

  add1_ms / add1_retrieve_ms        a one-document add, then the next retrieve (k = 100)
  del1000_ms / del1000_retrieve_ms  a 1000-id delete spread over the ranks, then the next retrieve
  compact_ms                        compact() of the tombstoned shards
  load_synthetic_ms                 load_synthetic of the same shape (the rows a reload would stream)
  load_global_ms                    load_global of the shape from host memory (only where the global matrix fits, --global-max)
  qps_before / qps_after_append     single retrieves per second (k = 100, host query in) before and after a 1 % append,
                                    which all goes to the last rank

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29641 \
        scripts/sharded_mutate_bench.py [--rows 1000000] [--c4] [--dims 1536] [--reps 5]

--c4 adds 10M x 1536.  One process per GPU; N = 1 runs on one GPU.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from svs_b200.sharded import ShardedRetriever                    # noqa: E402


def card(local: int) -> str:
    try:
        return subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        return f"{torch.cuda.get_device_name(local)} (nvidia-smi failed: {ex})"


def slowest(ms: float) -> float:
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return round(float(t.item()), 3)


def clock(fn) -> float:
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return slowest((time.perf_counter() - t0) * 1e3)


def rows_of(rng, n: int, d: int) -> np.ndarray:
    m = rng.standard_normal((n, d)).astype(np.float32)
    return m / np.linalg.norm(m, axis=1, keepdims=True).astype(np.float32)


def qps(sr, qs) -> float:
    sr.retrieve_arrays(qs[0], 100)                               # warm-up
    dist.barrier()
    t0 = time.perf_counter()
    for q in qs:
        sr.retrieve_arrays(q, 100)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return round(len(qs) / float(t.item()), 1)


def median(fn, reps: int) -> float:
    return float(np.median([fn() for _ in range(reps)]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dims", type=int, default=1536)
    ap.add_argument("--c4", action="store_true")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--queries", type=int, default=500)
    ap.add_argument("--global-max", type=int, default=2_000_000, help="largest n timed through load_global")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cards = [None] * world
    dist.all_gather_object(cards, card(local))
    if rank == 0:
        for r, c in enumerate(cards):
            print(f"rank {r}: {c}", flush=True)
    rng = np.random.default_rng(1)
    for n, d in [(args.rows, args.dims)] + ([(10_000_000, 1536)] if args.c4 else []):
        qs = rows_of(np.random.default_rng(7), args.queries, d)
        out = {"rows": n, "dims": d, "world": world}
        sr = ShardedRetriever(rank, world, local)
        out["load_synthetic_ms"] = median(lambda: clock(lambda: sr.load_synthetic(n, d, seed=0, id0=1, id_step=1)), args.reps)
        out["qps_before"] = qps(sr, qs)
        next_id = n + 1                                          # synthetic ids are 1 .. n
        adds, retr = [], []
        for _ in range(args.reps):
            row = rows_of(rng, 1, d)
            adds.append(clock(lambda: sr.apply_mutations([], [next_id], row)))
            retr.append(clock(lambda: sr.retrieve_arrays(qs[0], 100)))
            next_id += 1
        out["add1_ms"], out["add1_retrieve_ms"] = float(np.median(adds)), float(np.median(retr))
        dels, retr = [], []
        for r in range(args.reps):
            ids = np.random.default_rng(100 + r).choice(np.arange(1 + r, n + 1, args.reps), size=1000, replace=False)   # disjoint per rep
            dels.append(clock(lambda: sr.apply_mutations(ids, [], None)))
            retr.append(clock(lambda: sr.retrieve_arrays(qs[0], 100)))
        out["del1000_ms"], out["del1000_retrieve_ms"] = float(np.median(dels)), float(np.median(retr))
        out["compact_ms"] = clock(sr.compact)
        n_app = n // 100
        step = 100_000
        for a in range(0, n_app, step):                          # 1 % more rows, all on the last rank
            c = min(step, n_app - a)
            sr.apply_mutations([], np.arange(next_id, next_id + c, dtype=np.int64), rows_of(rng, c, d))
            next_id += c
        out["last_shard_rows"] = sr._shard_live[-1]
        out["largest_other_shard_rows"] = max(sr._shard_live[:-1], default=0)
        out["qps_after_append"] = qps(sr, qs)
        sr.close()
        del sr
        torch.cuda.empty_cache()
        if n <= args.global_max:
            m = rows_of(np.random.default_rng(3), n, d)
            ids = np.arange(1, n + 1, dtype=np.int64)
            sr = ShardedRetriever(rank, world, local)
            out["load_global_ms"] = median(lambda: clock(lambda: sr.load_global(m, ids)), args.reps)
            sr.close()
            del sr, m
            torch.cuda.empty_cache()
        else:
            out["load_global_ms"] = "not measured (the global matrix does not fit host memory)"
        if rank == 0:
            print(json.dumps(out), flush=True)
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
