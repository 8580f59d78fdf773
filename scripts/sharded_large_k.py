"""Run under torchrun: ShardedRetriever.retrieve above 2048 results per query (full sort per shard, one all-gather of
the sorted records, rank merge on every rank) against the in-process engine on the same devices.  Prints the card and
its power limit, then one JSON line per (shape, k): ms per retrieve (median over --reps, host query in, host arrays
out, slowest rank) for both, and whether the answers are identical on every rank and equal, bit for bit, to the
in-process engine's.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29631 \
        scripts/sharded_large_k.py [--rows 1000000] [--dims 1536] [--c4] [--reps 5]

--c4 adds synthetic C4 rows (10M x 1536).  Sharded and in-process engines are loaded one after the other, so that a
shape fits once on the devices.
"""
import argparse
import hashlib
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
import svs_b200                                                   # noqa: E402
from svs_b200.sharded import ShardedRetriever                    # noqa: E402


def card(local: int) -> str:
    try:
        return subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        return f"{torch.cuda.get_device_name(local)} (nvidia-smi failed: {ex})"


def queries(nq: int, d: int) -> np.ndarray:
    q = np.random.default_rng(7).random((nq, d), dtype=np.float32)
    return q / np.linalg.norm(q, axis=1, keepdims=True).astype(np.float32)


def timed(fn, reps: int) -> float:
    fn()                                                         # warm-up: buffers, sort scratch, modules
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def digest(s: np.ndarray, i: np.ndarray) -> str:
    return hashlib.sha256(s.view(np.uint32).tobytes() + i.tobytes()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dims", type=int, default=1536)
    ap.add_argument("--c4", action="store_true")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cards = [None] * world
    dist.all_gather_object(cards, card(local))
    if rank == 0:
        for r, c in enumerate(cards):
            print(f"rank {r}: {c}", flush=True)
    shapes = [(args.rows, args.dims)] + ([(10_000_000, 1536)] if args.c4 else [])
    for n, d in shapes:
        q = queries(1, d)[0]
        ks = [k for k in (2049, 10_000, 100_000, n) if k <= n]
        sr = ShardedRetriever(rank, world, local)
        sr.load_synthetic(n, d, seed=0, id0=1, id_step=1)
        sharded = {}
        for k in ks:
            dist.barrier()
            ms = timed(lambda: sr.retrieve_arrays(q, k), args.reps)
            s, i = sr.retrieve_arrays(q, k)
            digests = [None] * world
            dist.all_gather_object(digests, digest(s, i))
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sharded[k] = (float(t.item()), len(set(digests)) == 1, s, i)
        sr.close()
        del sr
        torch.cuda.empty_cache()
        dist.barrier()
        if rank == 0:                                            # the in-process engine over the same devices
            with svs_b200.Engine(list(range(world))) as eng:
                eng.load_synthetic(n, d, seed=0, id0=1, id_step=1)
                for k in ks:
                    ms = timed(lambda: eng.query(q, k), args.reps)
                    s, i = eng.query(q, k)
                    sms, same_ranks, ss, si = sharded[k]
                    equal = len(s) == len(ss) == min(k, n) and np.array_equal(s.view(np.uint32), ss.view(np.uint32)) and np.array_equal(i, si)
                    print(json.dumps({"rows": n, "dims": d, "k": k, "world": world, "sharded_ms": round(sms, 3),
                                      "in_process_ms": round(ms, 3), "identical_on_every_rank": same_ranks,
                                      "equal_to_in_process": bool(equal)}), flush=True)
        dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
