"""Pairwise top pairs: svsb_top_pairs vs the reference's np.dot(M, M.T) + get_top_pairs on the host.

    python scripts/pairs_bench.py [rows] [dims] [n_pairs] [--devices 0,1,...]... [--calls K] [--normal] [--no-cpu]
    python -m torch.distributed.run --nproc-per-node G scripts/pairs_bench.py [rows] [dims] [n_pairs] --sharded [--calls K] [--normal]
Default = the dad-jokes notebook's shape (examples/dad_jokes/Build Dad Jokes KB.ipynb:338-340: 4,875 x 1536, 10,000 pairs,
0.47 s + 0.03 s on the author's i3-8100).

--devices (repeatable): device lists to run, in one process, on the same matrix; a repeated id means virtual shards of
one GPU (SVSB_ALLOW_DUP_DEVICES=1).  Default: one list, device 0.  Every list is timed after a warm-up call that builds
the fp16 shadows (median and best of K calls, host clock around a call that returns its answer to the host); the first
list's answer is the reference the others must equal bit for bit.  The NumPy reference (and the oracle parity check)
runs where np.dot(M, M.T) fits in host RAM (<= 50,000 rows) unless --no-cpu.
Rows are uniform in [0, 1) (all pair scores in a narrow band around 0.75) unless --normal (Gaussian components: scores
spread around 0).  On the uniform rows of 200,000 x 768 and up, more pairs lie within the coarse pass's 2 eps margin of
the n-th best score than a candidate list holds: the engine refuses (SVSB_E_NOMEM) and the drop-in hands the call to
the reference's host path.

--sharded: the one-process-per-GPU deployment, one rank per GPU (NCCL cannot run two ranks on one GPU).  Every rank
generates the same seeded matrix and keeps its slice; ShardedRetriever.top_pairs is timed after a warm-up call that
exports and connects the shards and builds the fp16 shadows: host clock from a barrier to the answer on the host
followed by a device synchronize, max over ranks, median / best / worst of K calls.  Rank 0 then runs a single-device
engine over the whole matrix and checks that the answer is bit-identical.
"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import svs_b200  # noqa: E402
import svs_oracle as oracle  # noqa: E402  (checker / CPU baseline only)


def _opt_values(flag):
    out = []
    for i, a in enumerate(sys.argv):
        if a == flag and i + 1 < len(sys.argv):
            out.append(sys.argv[i + 1])
        elif a.startswith(flag + "="):
            out.append(a.split("=", 1)[1])
    return out


argv = sys.argv[1:]
args = [a for i, a in enumerate(argv) if not a.startswith("--") and not (i > 0 and argv[i - 1] in ("--devices", "--calls"))]
N = int(args[0]) if len(args) > 0 else 4875
d = int(args[1]) if len(args) > 1 else 1536
n = int(args[2]) if len(args) > 2 else 10000
calls = int((_opt_values("--calls") or ["5"])[0])
dev_lists = [[int(x) for x in v.split(",")] for v in _opt_values("--devices")] or [[0]]


def run_sharded(m, ids):
    import torch
    import torch.distributed as dist
    from svs_b200.sharded import ShardedRetriever
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    sr = ShardedRetriever(rank, world, local)
    sr.load_global(m, ids)
    got = sr.top_pairs(n)                               # export + connect, fp16 shadows
    ts = []
    for _ in range(calls):
        dist.barrier()
        t0 = time.perf_counter(); got = sr.top_pairs(n); torch.cuda.synchronize(); dt = time.perf_counter() - t0
        every = [None] * world
        dist.all_gather_object(every, dt)
        ts.append(max(every))
    if rank == 0:
        with svs_b200.Engine([local]) as e:
            e.load(m, ids)
            want = e.top_pairs(n)
        same = (len(got) == len(want) and
                np.array_equal(np.array([s for s, _, _ in got], np.float32).view(np.uint32),
                               np.array([s for s, _, _ in want], np.float32).view(np.uint32)) and
                [(a, b) for _, a, b in got] == [(a, b) for _, a, b in want])
        dist_name = "normal" if "--normal" in sys.argv else "uniform"
        med = float(np.median(ts))
        print(f"sharded top_pairs: {N} x {d} {dist_name}, n={n}, {world} ranks (one per GPU): median {med * 1e3:.2f} ms, "
              f"best {min(ts) * 1e3:.2f} ms, worst {max(ts) * 1e3:.2f} ms over {calls} calls (max over ranks; "
              f"{float(N) * float(N - 1) * d / med / 1e12:.1f} useful TFLOP/s at the median), "
              f"answer vs one device: {'bit-identical' if same else 'DIFFERENT'}", flush=True)
    dist.barrier()
    sr.close()
    dist.destroy_process_group()


try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=60).stdout.strip().replace("\n", "; ")
except Exception as ex:  # noqa: BLE001
    card = f"nvidia-smi unavailable ({ex})"
if os.environ.get("RANK", "0") == "0":
    print(f"GPUs: {card}")

rng = np.random.default_rng(0)
m = rng.standard_normal((N, d), dtype=np.float32) if "--normal" in sys.argv else rng.random((N, d), dtype=np.float32)
m /= np.sqrt((m * m).sum(axis=1))[:, None]
ids = np.arange(1, N + 1, dtype=np.int64)
if "--sharded" in sys.argv:
    run_sharded(m, ids)
    sys.exit(0)
useful = float(N) * float(N - 1) * d                    # N(N-1)d: the FLOP of the upper triangle's dot products, counted twice
first = None
base_t = None
for devs in dev_lists:
    if len(set(devs)) != len(devs):
        os.environ["SVSB_ALLOW_DUP_DEVICES"] = "1"
    e = svs_b200.Engine(devs)
    e.load(m, ids)
    got = e.top_pairs(n)                                # first call builds the fp16 shadows
    l0 = svs_b200.launch_count()
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter(); got = e.top_pairs(n); ts.append(time.perf_counter() - t0)
    launches = (svs_b200.launch_count() - l0) / calls
    e.close()
    med = float(np.median(ts))
    if first is None:
        first, base_t = got, med
        same = "reference"
    else:
        same = "bit-identical" if (len(got) == len(first) and
                                   np.array_equal(np.array([s for s, _, _ in got], np.float32).view(np.uint32),
                                                  np.array([s for s, _, _ in first], np.float32).view(np.uint32)) and
                                   [(a, b) for _, a, b in got] == [(a, b) for _, a, b in first]) else "DIFFERENT"
    dist = "normal" if "--normal" in sys.argv else "uniform"
    print(f"svs_b200 top_pairs: {N} x {d} {dist}, n={n}, devices {devs}: median {med * 1e3:.2f} ms, best {min(ts) * 1e3:.2f} ms "
          f"over {calls} calls ({useful / med / 1e12:.1f} useful TFLOP/s at the median, x{base_t / med:.2f} vs {dev_lists[0]}), "
          f"{launches:.0f} launches per call, answer vs {dev_lists[0]}: {same}", flush=True)


def _host_gb_available():
    try:
        with open("/proc/meminfo") as f:
            return next(int(line.split()[1]) for line in f if line.startswith("MemAvailable:")) / 2 ** 20
    except Exception:  # noqa: BLE001
        return 0.0


# the reference's path holds the N x N fp32 matrix and its upper triangle's int64 indices (~ 28 N^2 bytes with copies)
if "--no-cpu" not in sys.argv and N <= 50_000 and 28.0 * N * N / 2 ** 30 > _host_gb_available():
    print(f"reference NumPy path skipped: needs ~{28.0 * N * N / 2 ** 30:.0f} GB of host RAM, {_host_gb_available():.0f} GB available")
elif "--no-cpu" not in sys.argv and N <= 50_000:
    t0 = time.perf_counter()
    want = oracle.top_pairwise(m, ids, n)
    dt = time.perf_counter() - t0
    print(f"reference NumPy path on {os.cpu_count()} host cores: {dt * 1e3:.1f} ms  -> {dt / base_t:.0f}x vs {dev_lists[0]}")
    print("parity:", oracle.compare_pairs(first, want, np.dot(m, m.T), ids))
