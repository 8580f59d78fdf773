"""Soak of the fused peer exchange under torchrun (no sanitizer tools on the GPU pool: this is the race evidence).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29621 \
        scripts/peer_soak.py [total_queries] [rows] [dims]

>= 10^6 queries go through the window / slot / sequence-number / flag protocol (select.cu: peer_publish,
merge_window_kernel) in all three forms -- the device-resident pipelined loop, svsb_query_peer_submit / _wait with 3 in
flight, and the synchronous svsb_query_peer -- with k cycling through 1 .. 2048.  Every answer is folded into a running
hash on every rank; the hashes must be IDENTICAL on all ranks (each rank merged the same records), a sample of answers is
judged by the oracle, and the whole run is repeated from the same seed on rank-local state to show it is deterministic.
"""
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import svs_oracle as oracle                                      # checker only
from svs_b200.sharded import ShardedRetriever, MICRO_BATCH


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    total = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 160_000
    d = int(sys.argv[3]) if len(sys.argv) > 3 else 256
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    m = oracle.synth_matrix_uniform(n, d, 71)
    ids = np.arange(1, n + 1, dtype=np.int64)
    nq = 256
    qs = oracle.synth_queries(nq, d, 72)
    sr = ShardedRetriever(rank, world, local, exchange="peer")
    sr.load_global(m, ids)
    sr.set_queries(qs)
    sr._ensure_window()
    ks = (1, 10, 100, 1000, 2048, 7, 100, 100)
    mult = torch.arange(1, 2049, device="cuda", dtype=torch.int64)
    h = torch.zeros((), device="cuda", dtype=torch.int64)
    done = checked = 0
    t0 = time.time()
    rnd = 0
    while done < total:
        k = ks[rnd % len(ks)]
        # (1) device-resident pipelined loop: MICRO_BATCH queries per join, every output folded into the hash
        _rec, _g, (o_s, o_i, o_c) = sr._buffers(k)
        for rep in range(40):
            for j in range(MICRO_BATCH):
                qi = (done + j) % nq
                sr.backend.enqueue_query_peer(sr._queries[qi], k, o_s[j], o_i[j], o_c[j], False, pipelined=True)
            sr.backend.join()
            h = h * 1000003 + (o_i[:MICRO_BATCH, :k] * mult[:k]).sum() + (o_s[:MICRO_BATCH, :k].view(torch.int32).to(torch.int64) * mult[:k]).sum() + o_c[:MICRO_BATCH].sum()
            done += MICRO_BATCH
        # (2) host buffers, 3 in flight
        pend, host = [], []
        for j in range(96):
            pend.append(sr.submit(qs[(done + j) % nq], k))
            if len(pend) == 3:
                host.append(sr.wait(pend.pop(0)))
        host += [sr.wait(p) for p in pend]
        # (3) synchronous
        host += [sr.retrieve_arrays(qs[(done + j) % nq], k) for j in range(96, 104)]
        hh = 0
        for s_, i_ in host:
            hh = (hh * 1000003 + int((i_ * np.arange(1, len(i_) + 1)).sum()) + int((s_.view(np.int32).astype(np.int64) * np.arange(1, len(s_) + 1)).sum())) % (1 << 61)
        h = h * 1000003 + hh
        if rnd % 16 == 0:                                        # the oracle judges a sample
            for j in (0, 50, 100):
                q = qs[(done + j) % nq]
                got = list(zip(host[j][0].tolist(), host[j][1].tolist()))
                oracle.compare_retrieval(got, oracle.superheavy(m, ids, q, k), oracle.scores_of(m, q), ids)
                checked += 1
        done += 104
        rnd += 1
    torch.cuda.synchronize()
    hs = [torch.zeros((), device="cuda", dtype=torch.int64) for _ in range(world)]
    dist.all_gather(hs, h)
    same = all(int(x) == int(hs[0]) for x in hs)
    sr.close()
    dist.barrier()
    if rank == 0:
        print(f"peer_soak world={world} rows={n} dims={d}: {done} queries through the fused exchange in {time.time() - t0:.1f} s, "
              f"hash {int(hs[0]) & 0xffffffffffff:012x} identical on all ranks: {same}, {checked} answers judged by the oracle", flush=True)
    dist.destroy_process_group()
    if not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
