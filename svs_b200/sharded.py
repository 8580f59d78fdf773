"""Row-sharded retrieve, one process per GPU (SURVEY.md section 8e; BASELINE.json north star item 4).

Rank r owns the contiguous rows [r*ceil(N/G), min(N, (r+1)*ceil(N/G))) of the scan order together with
their embeddings.ids.  A query is answered by
  1. every rank: similarity + exact local top-k on its shard (libsvsb200.so, on the caller's stream),
     written as ONE packed int64 record [keys(k) | ids(k) | count];
  2. the ONE exchange step: `all_gather_into_tensor` of those records (NCCL over NVLink/NVSwitch;
     k=100 -> 1.6 KB per rank per query), micro-batched over 16 queries per collective;
  3. every rank: one merge kernel per micro-batch (one CTA per query) -> global top-k under the same
     total order (score desc, global row asc), so all ranks hold the identical answer.
No reduction over scores is needed: rows are independent (splitting D instead would need an all-reduce
of N floats).

k > 2048 (up to the full ranking n = N) takes its own path under either exchange: every rank fully sorts its shard's
keys into one record of cap = min(k, ceil(N / world)) entries -- no shard holds more rows, so every record is complete
--, the ranks agree on the outcome of that local phase, all-gather the records and rank-merge the sorted lists on every
rank (include/svsb200.h svsb_enqueue_merge_sorted_records).

Single queries do not call a collective at all by default (`exchange="peer"`): steps 2 and 3 are fused into the
kernels over NVLink / NVSwitch peer memory -- the selection kernel's epilogue stores its record into every rank's
gather window and publishes it with a release store, and each rank's merge kernel waits for the `world` flags of
its own window (include/svsb200.h "peer exchange").  The windows are exchanged once, as CUDA IPC handles, through
torch.distributed.  `exchange="collective"` keeps the NCCL all-gather (the baseline the fused path is measured
against; also what batches use: one all-gather per batch is already amortised).

Pairwise top pairs (`top_pairs`, document_top_pairwise_scores) run over the same shards: once per load every rank
exports its shard (CUDA IPC handles of its fp32 rows, fp16 shadow and ids) and opens its peers'; per call every rank
runs its share of a static plan over the shard pairs -- the triangle of its own shard and rectangles against blocks of
its peers' rows -- with its own threshold, re-scores its survivors exactly and keeps its top n; one all-gather of the
lists (at most 20 bytes x n per rank) and a rank merge on every rank give every rank the single-device answer, bit for
bit (include/svsb200.h svsb_pairs_*).

The collective / packing / batching logic is backend-agnostic so that it can be exercised on CPU with
`gloo` (tests/test_sharded_gloo.py and tests/test_sharded_pairs_gloo.py inject NumPy backends); the product backend is
`CudaShardBackend`.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple

import numpy as np

from ._lib import K_FAST_MAX, SVSB_E_CUDA, SVSB_E_NOMEM, EngineError

MICRO_BATCH = 16
TIME_EVERY = 8        # bracket one similarity launch in 8 with timing events (two records cost ~5 us of stream time)


def partition(n: int, world: int, rank: int) -> Tuple[int, int]:
    """(first global row, row count) of `rank`'s shard: contiguous ranges of the scan order."""
    per = (n + world - 1) // world
    row0 = min(n, rank * per)
    return row0, min(n, (rank + 1) * per) - row0


class CudaShardBackend:
    """The shard's compute, on `cuda:device_index`, through the C ABI.  Torch owns streams and buffers."""

    def __init__(self, device_index: int):
        import torch
        from . import _lib
        from .engine import Engine
        self.torch = torch
        self._lib = _lib.load()
        self._check = _lib.check
        self._last_error = _lib.last_error
        self._desc_bytes = _lib.PAIRS_DESC_BYTES
        self.device = torch.device("cuda", device_index)
        self.engine = Engine([device_index])
        self.d = 0
        self.ld = 0

    # -- data ------------------------------------------------------------------------------------
    def set_shard(self, global_row0: int) -> None:
        self._check(self._lib.svsb_set_shard(self.engine._h, global_row0))

    def load_rows(self, rows: np.ndarray, emb_ids: np.ndarray) -> None:
        self.engine.load(rows, emb_ids)
        self.d = rows.shape[1]
        self.ld = (self.d + 3) & ~3

    def load_synthetic(self, n_local: int, d: int, seed: int, id0: int, id_step: int) -> None:
        self.engine.load_synthetic(n_local, d, seed, id0, id_step)
        self.d = d
        self.ld = (d + 3) & ~3

    def device_queries(self, Q: np.ndarray):
        """(nq, d) host float32 -> (nq, ld) device tensor, zero padded, staged through a cached pinned buffer."""
        t = self.torch
        Q = np.ascontiguousarray(Q, dtype=np.float32)
        key = (Q.shape[0], self.ld)
        stage = getattr(self, "_stage", None)
        if stage is None or stage[0] != key:                       # pinning is slow (ms): once per shape, not per call
            stage = (key, t.zeros(key, dtype=t.float32).pin_memory(), t.cuda.Event())
            self._stage = stage
        else:
            stage[2].synchronize()                                 # the previous upload out of this buffer has finished
        host = stage[1]
        host[:, :Q.shape[1]] = t.from_numpy(Q)
        dev = host.to(self.device, non_blocking=True)
        stage[2].record(t.cuda.current_stream(self.device))
        return dev

    def new_records(self, count: int, k: int):
        return self.torch.zeros((count, 2 * k + 1), dtype=self.torch.int64, device=self.device)

    def new_outputs(self, count: int, k: int):
        t = self.torch
        return (t.zeros((count, k), dtype=t.float32, device=self.device),
                t.zeros((count, k), dtype=t.int64, device=self.device),
                t.zeros((count,), dtype=t.int32, device=self.device))

    # -- compute ---------------------------------------------------------------------------------
    def enqueue_local(self, query_row, k: int, record_row, time_kernel: bool = False, seq: int = 0) -> None:
        """Similarity on the current stream, selection pipelined on the engine's side stream (slots alternate with
        `seq`, so the selection of one query overlaps the similarity pass of the next).  Call join() before the
        records are consumed.  k > 2048: the shard's keys are fully sorted, unpipelined, on the current stream."""
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_enqueue_local_topk(self.engine._h, C.c_void_p(st), seq & 1, C.c_void_p(query_row.data_ptr()),
                                                      k, C.c_void_p(record_row.data_ptr()), (1 if time_kernel else 0) | 2))

    def batch_local(self, queries, k: int, records) -> int:
        """Local top-k records of all rows of the device tensor `queries` (b, ld) in one call: tensor-core coarse pass
        + exact refine where the shard allows it.  Returns how many queries took the single-query kernels."""
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        nfb = C.c_int32()
        self._check(self._lib.svsb_batch_local_records(self.engine._h, C.c_void_p(st), C.c_void_p(queries.data_ptr()),
                                                       queries.shape[0], k, C.c_void_p(records.data_ptr()), C.byref(nfb)))
        return nfb.value

    # -- batches with one GLOBAL filter threshold per query (include/svsb200.h svsb_batch_global_*) --------
    def batch_global_probe(self, k: int) -> Tuple[bool, int, int, float]:
        """(eligible, sample rows, local rows, max row norm) of this shard for the global-threshold batch path."""
        el, sr, lr, nr = C.c_int32(), C.c_int64(), C.c_int64(), C.c_float()
        self._check(self._lib.svsb_batch_global_probe(self.engine._h, k, C.byref(el), C.byref(sr), C.byref(lr), C.byref(nr)))
        return bool(el.value), sr.value, lr.value, float(nr.value)

    def new_tops(self, count: int):
        return self.torch.zeros((count, 32), dtype=self.torch.float32, device=self.device)

    def batch_sample_tops(self, queries, k: int, max_row_norm: float, tops) -> None:
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_batch_sample_tops(self.engine._h, C.c_void_p(st), C.c_void_p(queries.data_ptr()), queries.shape[0], k,
                                                     C.c_float(max_row_norm), C.c_void_p(tops.data_ptr())))

    def batch_global_records(self, queries, k: int, tops_all, world: int, sample_rank: int, rec_cap: int, records) -> None:
        """records: (b, 2 * rec_cap + 1) int64 -- at most rec_cap entries per query are shipped."""
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_batch_global_records(self.engine._h, C.c_void_p(st), C.c_void_p(queries.data_ptr()), queries.shape[0], k,
                                                        C.c_void_p(tops_all.data_ptr()), world, sample_rank, rec_cap,
                                                        C.c_void_p(records.data_ptr())))

    def enqueue_merge_verified(self, gathered, n_lists: int, batch: int, rec_cap: int, k: int, verify_k: int, out_scores, out_ids,
                               out_counts) -> None:
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_enqueue_merge_batch_records(self.engine._h, C.c_void_p(st), C.c_void_p(gathered.data_ptr()),
                                                               n_lists, batch, rec_cap, k, verify_k, C.c_void_p(out_scores.data_ptr()),
                                                               C.c_void_p(out_ids.data_ptr()), C.c_void_p(out_counts.data_ptr())))

    # -- the batch protocol with both exchanges fused into the kernels over peer memory (svsb_bxchg_*, svsb_batch_peer) ----
    BATCH_WINDOW_CAP = 128          # entries per record the batch window is sized for

    def batch_exchange_handle(self, world: int, rank: int, rec_cap: int = BATCH_WINDOW_CAP) -> bytes:
        buf = C.create_string_buffer(64)
        self._check(self._lib.svsb_bxchg_create(self.engine._h, world, rank, rec_cap, buf))
        return buf.raw

    def batch_exchange_connect(self, handles: List[bytes]) -> None:
        self._check(self._lib.svsb_bxchg_connect(self.engine._h, C.c_char_p(b"".join(handles))))

    def batch_exchange_connect_local(self, backends: List["CudaShardBackend"]) -> None:
        self._check(self._lib.svsb_bxchg_connect_local(self.engine._h, self._engines(backends)))

    def batch_exchange_disconnect(self) -> None:
        self._check(self._lib.svsb_bxchg_disconnect(self.engine._h))

    def batch_peer_prepare(self, b: int, k: int) -> None:
        self._check(self._lib.svsb_batch_peer_prepare(self.engine._h, b, k))

    def batch_peer(self, queries, k: int, max_row_norm: float, sample_rank: int, rec_cap: int, out_scores, out_ids, out_counts,
                   defer_merge: bool = False) -> None:
        """One whole batch (<= 2048 device queries) on the current stream, no collective: see include/svsb200.h.
        defer_merge: the verifying merge is enqueued by the next batch_peer call (behind its first phase) or batch_peer_flush."""
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_batch_peer(self.engine._h, C.c_void_p(st), C.c_void_p(queries.data_ptr()), queries.shape[0], k,
                                              C.c_float(max_row_norm), sample_rank, rec_cap, C.c_void_p(out_scores.data_ptr()),
                                              C.c_void_p(out_ids.data_ptr()), C.c_void_p(out_counts.data_ptr()), 1 if defer_merge else 0))

    def batch_peer_flush(self) -> None:
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_batch_peer_flush(self.engine._h, C.c_void_p(st)))

    # -- peer exchange (fused selection + exchange over NVLink peer memory) -------------------------
    def exchange_handle(self, world: int, rank: int, k_max: int = 2048) -> bytes:
        """Allocate this rank's gather window; returns its CUDA IPC handle (64 bytes) for the other ranks."""
        buf = C.create_string_buffer(64)
        self._check(self._lib.svsb_xchg_create(self.engine._h, world, rank, k_max, buf))
        return buf.raw

    def exchange_connect(self, handles: List[bytes]) -> None:
        blob = b"".join(handles)
        self._check(self._lib.svsb_xchg_connect(self.engine._h, C.c_char_p(blob)))

    def exchange_connect_local(self, backends: List["CudaShardBackend"]) -> None:
        """All ranks live in this process (tests; one process driving several GPUs): plain pointers, no IPC."""
        self._check(self._lib.svsb_xchg_connect_local(self.engine._h, self._engines(backends)))

    def exchange_disconnect(self) -> None:
        self._check(self._lib.svsb_xchg_disconnect(self.engine._h))

    def enqueue_query_peer(self, query_row, k: int, out_scores, out_ids, out_count, time_kernel: bool = False,
                           pipelined: bool = True) -> None:
        """Similarity + selection with the fused push + waiting merge for one device-resident query; the GLOBAL top-k
        lands in the output rows (identical on every rank).  pipelined: call join() before consuming them."""
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_enqueue_query_peer(self.engine._h, C.c_void_p(st), C.c_void_p(query_row.data_ptr()), k,
                                                      C.c_void_p(out_scores.data_ptr()), C.c_void_p(out_ids.data_ptr()),
                                                      C.c_void_p(out_count.data_ptr()),
                                                      (1 if time_kernel else 0) | (2 if pipelined else 0)))

    def query_peer(self, q: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray]:
        """Host query in, host (scores, ids) out, one synchronous C call (svsb_query_peer)."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        s = np.empty(k, dtype=np.float32)
        i = np.empty(k, dtype=np.int64)
        cnt = C.c_int32()
        self._check(self._lib.svsb_query_peer(self.engine._h, q.ctypes.data, q.shape[0], k, s.ctypes.data, i.ctypes.data,
                                              C.byref(cnt)))
        return s[:cnt.value], i[:cnt.value]

    def query_peer_submit(self, q: np.ndarray, k: int) -> int:
        """Start a host-buffer query (svsb_query_peer_submit); up to 3 may be pending.  Returns the ticket."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        t = C.c_int32()
        self._check(self._lib.svsb_query_peer_submit(self.engine._h, q.ctypes.data, q.shape[0], k, C.byref(t)))
        return t.value

    def query_peer_wait(self, ticket: int, k: int) -> Tuple[np.ndarray, np.ndarray]:
        s = np.empty(k, dtype=np.float32)
        i = np.empty(k, dtype=np.int64)
        cnt = C.c_int32()
        self._check(self._lib.svsb_query_peer_wait(self.engine._h, ticket, s.ctypes.data, i.ctypes.data, C.byref(cnt)))
        return s[:cnt.value], i[:cnt.value]

    def join(self) -> None:
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_enqueue_join(self.engine._h, C.c_void_p(st)))

    def enqueue_merge(self, gathered, n_lists: int, batch: int, k: int, out_scores, out_ids, out_counts) -> None:
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_enqueue_merge_records(self.engine._h, C.c_void_p(st), C.c_void_p(gathered.data_ptr()),
                                                         n_lists, batch, k, C.c_void_p(out_scores.data_ptr()),
                                                         C.c_void_p(out_ids.data_ptr()), C.c_void_p(out_counts.data_ptr())))

    def enqueue_merge_sorted(self, gathered, n_lists: int, cap: int, k: int, out_scores, out_ids, out_count) -> None:
        """Any k: rank-merge n_lists sorted records of cap entries (gathered: [n_lists][2 * cap + 1]) into out_scores[k],
        out_ids[k], out_count[1] (-1: a record was truncated)."""
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_enqueue_merge_sorted_records(self.engine._h, C.c_void_p(st), C.c_void_p(gathered.data_ptr()),
                                                                n_lists, cap, k, C.c_void_p(out_scores.data_ptr()),
                                                                C.c_void_p(out_ids.data_ptr()), C.c_void_p(out_count.data_ptr())))

    # -- pairwise top pairs over the ranks' shards (include/svsb200.h svsb_pairs_*) ---------------------------------
    def pairs_export(self) -> Tuple[bytes, int, str, float]:
        """Pin the resident generation and describe it for the peers: (descriptor, status, message, max_dev).  A refusal
        comes back as its SVSB_E_* status instead of raising, so that every rank can learn it."""
        buf = C.create_string_buffer(self._desc_bytes)
        max_dev, rows = C.c_float(), C.c_int64()
        rc = self._lib.svsb_pairs_export(self.engine._h, C.byref(max_dev), C.byref(rows), buf)
        return buf.raw, rc, self._last_error() if rc else "", float(max_dev.value)

    def pairs_connect(self, world: int, rank: int, descs: List[bytes]) -> None:
        self._check(self._lib.svsb_pairs_connect(self.engine._h, world, rank, C.c_char_p(b"".join(descs))))

    def pairs_connect_local(self, world: int, rank: int, backends: List["CudaShardBackend"]) -> None:
        """All ranks live in this process (tests; one process driving several GPUs): plain pointers, no IPC."""
        self._check(self._lib.svsb_pairs_connect_local(self.engine._h, world, rank, self._engines(backends)))

    def pairs_disconnect(self) -> None:
        self._check(self._lib.svsb_pairs_disconnect(self.engine._h))

    def new_pair_lists(self, count: int, lists: int = 1):
        """(scores float32, first rows int64, second rows int64), each (lists, count), on the device."""
        t = self.torch
        return (t.zeros((lists, count), dtype=t.float32, device=self.device), t.zeros((lists, count), dtype=t.int64, device=self.device),
                t.zeros((lists, count), dtype=t.int64, device=self.device))

    def pairs_local(self, n: int, max_row_norm: float, out) -> Tuple[int, str, int]:
        """This rank's top list into row 0 of `out` (new_pair_lists(n)): (status, message, entries)."""
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        cnt = C.c_int64()
        rc = self._lib.svsb_pairs_local(self.engine._h, C.c_void_p(st), n, C.c_float(max_row_norm), C.c_void_p(out[0].data_ptr()),
                                        C.c_void_p(out[1].data_ptr()), C.c_void_p(out[2].data_ptr()), C.byref(cnt))
        return rc, self._last_error() if rc else "", cnt.value

    def pairs_merge(self, lists, counts: List[int], n: int, out) -> int:
        """Merge the all-gathered lists (new_pair_lists(stride, world), counts[l] valid in list l) into row 0 of `out`
        (new_pair_lists(n)), rows mapped to embeddings.id.  Returns the merged count (synchronises)."""
        t = self.torch
        world, stride = lists[0].shape
        d_counts = t.tensor(counts, dtype=t.int32).to(self.device)
        d_out = t.zeros(1, dtype=t.int32, device=self.device)
        st = t.cuda.current_stream(self.device).cuda_stream
        self._check(self._lib.svsb_pairs_merge(self.engine._h, C.c_void_p(st), C.c_void_p(lists[0].data_ptr()), C.c_void_p(lists[1].data_ptr()),
                                               C.c_void_p(lists[2].data_ptr()), C.c_void_p(d_counts.data_ptr()), world, stride, n,
                                               C.c_void_p(out[0].data_ptr()), C.c_void_p(out[1].data_ptr()), C.c_void_p(out[2].data_ptr()),
                                               C.c_void_p(d_out.data_ptr())))
        return int(d_out.item())

    def collect_kernel_ms(self) -> float:
        ms = C.c_float()
        self._check(self._lib.svsb_kernel_time_collect(self.engine._h, C.byref(ms)))
        return ms.value

    @staticmethod
    def _engines(backends: List["CudaShardBackend"]):
        """The backends' engine handles as the C array the *_connect_local entry points take."""
        return (C.c_void_p * len(backends))(*[b.engine._h for b in backends])

    def synchronize(self) -> None:
        self.torch.cuda.current_stream(self.device).synchronize()

    def close(self) -> None:
        self.engine.close()


class ShardedRetriever:
    """All ranks construct one and call the same methods in the same order (SPMD)."""

    def __init__(self, rank: int, world: int, device_index: int = 0, backend=None, group=None, exchange: str = "peer"):
        import torch.distributed as dist
        self.dist = dist
        self.rank, self.world, self.group = rank, world, group
        self.backend = backend if backend is not None else CudaShardBackend(device_index)
        if exchange not in ("peer", "collective"):
            raise ValueError("exchange must be 'peer' or 'collective'")
        # the fused peer exchange needs a backend that owns device windows; injected CPU backends use the collective
        self.exchange = exchange if hasattr(self.backend, "exchange_handle") and world <= 16 else "collective"
        self._peer_ready = False
        self._batch_peer_ready = False
        self.n = 0
        self.d = 0
        self.row0 = 0
        self.local_rows = 0
        self._queries = None
        self._bufs = {}
        self._big = None                 # (cap, record, gathered records, outputs) of the large-k path: one set at a time
        self._plans = {}
        self._epoch = 0
        self.last_fallbacks = 0
        self._last_counts = None
        self._pairs_epoch = None         # load epoch of the connected pair export (None: not connected)
        self._pairs_norm = 1.0

    # -- load ------------------------------------------------------------------------------------
    def load_synthetic(self, n: int, d: int, seed: int = 0, id0: int = 0, id_step: int = 1) -> None:
        self.n, self.d = n, d
        self._epoch += 1
        self._big = None
        self.row0, self.local_rows = partition(n, self.world, self.rank)
        self.backend.set_shard(self.row0)
        self.backend.load_synthetic(self.local_rows, d, seed, id0, id_step)

    def load_global(self, rows: np.ndarray, emb_ids: np.ndarray) -> None:
        """Every rank passes the same global (n, d) matrix / ids and keeps only its slice (tests, small KBs)."""
        self.n, self.d = rows.shape
        self._epoch += 1
        self._big = None
        self.row0, self.local_rows = partition(self.n, self.world, self.rank)
        self.backend.set_shard(self.row0)
        sl = slice(self.row0, self.row0 + self.local_rows)
        self.backend.load_rows(np.ascontiguousarray(rows[sl]), np.ascontiguousarray(emb_ids[sl]))

    def _all_gather_object(self, obj) -> list:
        if self.world == 1:
            return [obj]
        out: list = [None] * self.world
        self.dist.all_gather_object(out, obj, group=self.group)
        return out

    def _ensure_window(self, batch: bool = False) -> None:
        """One-time window exchange: every rank allocates its gather window (`batch`: its batch window), all-gathers the
        IPC handles and opens its peers' windows."""
        if self._batch_peer_ready if batch else self._peer_ready:
            return
        be = self.backend
        create, connect = (be.batch_exchange_handle, be.batch_exchange_connect) if batch else (be.exchange_handle, be.exchange_connect)
        connect(self._all_gather_object(create(self.world, self.rank)))
        if self.world > 1:
            self.dist.barrier(group=self.group)                    # every window is open before the first push
        if batch:
            self._batch_peer_ready = True
        else:
            self._peer_ready = True

    # -- queries ---------------------------------------------------------------------------------
    def set_queries(self, Q: np.ndarray) -> None:
        self._queries = self.backend.device_queries(Q)

    def _buffers(self, k: int):
        if k not in self._bufs:
            rec = self.backend.new_records(MICRO_BATCH, k)
            gath = self.backend.new_records(self.world * MICRO_BATCH, k)
            outs = self.backend.new_outputs(MICRO_BATCH, k)
            self._bufs[k] = (rec, gath, outs)
        return self._bufs[k]

    def _micro_batch(self, qrows, k: int, time_gemv: bool):
        """Local top-k for len(qrows) device queries, one all-gather, one merge.  Returns output views."""
        rec, gath, (o_s, o_i, o_c) = self._buffers(k)
        nb = len(qrows)
        if self.exchange == "peer":
            self._ensure_window()
            for j, q in enumerate(qrows):                          # no collective, no separate merge launch per batch
                self.backend.enqueue_query_peer(q, k, o_s[j], o_i[j], o_c[j], time_gemv and j % TIME_EVERY == 0, pipelined=True)
            self.backend.join()
            return o_s[:nb], o_i[:nb], o_c[:nb]
        for j, q in enumerate(qrows):
            self.backend.enqueue_local(q, k, rec[j], time_gemv and j % TIME_EVERY == 0, seq=j)
        self.backend.join()                                        # records complete before the exchange
        recw = 2 * k + 1
        g = gath.view(-1)[: self.world * nb * recw]
        self.dist.all_gather_into_tensor(g, rec[:nb].reshape(-1), group=self.group)
        self.backend.enqueue_merge(g, self.world, nb, k, o_s, o_i, o_c)
        return o_s[:nb], o_i[:nb], o_c[:nb]

    def run_queries(self, k: int, count: int, time_gemv: bool = False) -> float:
        """`count` retrieves over the uploaded queries, device-resident end to end (bench path)."""
        assert self._queries is not None, "set_queries first"
        nq = self._queries.shape[0]
        done = timed = 0
        if self.exchange == "peer":
            # no collective and nothing consumed on the host: enqueue every query back to back (outputs cycle through the
            # micro-batch buffers in stream order) and join once -- ranks couple only through the window flags
            self._ensure_window()
            _rec, _gath, (o_s, o_i, o_c) = self._buffers(k)
            for done in range(count):
                j = done % MICRO_BATCH
                t = time_gemv and done % TIME_EVERY == 0
                timed += 1 if t else 0
                self.backend.enqueue_query_peer(self._queries[done % nq], k, o_s[j], o_i[j], o_c[j], t, pipelined=True)
            self.backend.join()
            return self.backend.collect_kernel_ms() * count / timed if time_gemv else 0.0
        while done < count:
            nb = min(MICRO_BATCH, count - done)
            self._micro_batch([self._queries[(done + j) % nq] for j in range(nb)], k, time_gemv)
            done += nb
            timed += (nb + TIME_EVERY - 1) // TIME_EVERY
        # similarity-kernel time of the run, estimated as (mean bracketed launch) x launches
        return self.backend.collect_kernel_ms() * count / timed if time_gemv else 0.0

    # -- batches ---------------------------------------------------------------------------------
    def _global_plan(self, k: int):
        """(sample_rank, max_row_norm, entries shipped per rank) if EVERY rank can run the batched pipeline with one global filter threshold per
        query (include/svsb200.h svsb_batch_global_*), else None.  Agreed once per (k, load) through one object
        all-gather of the ranks' probes, so that all ranks take the same branch."""
        key = (k, self._epoch)
        if key not in self._plans:
            plan = None
            if self.world > 1 and hasattr(self.backend, "batch_global_probe"):
                probes: List[Optional[tuple]] = [None] * self.world
                self.dist.all_gather_object(probes, self.backend.batch_global_probe(k), group=self.group)
                if all(p[0] for p in probes):
                    f = max(min(1.0, p[1] / max(1, p[2])) for p in probes)      # largest sample fraction of any rank
                    lam = min(k, self.n) * f
                    rank = int(np.ceil(lam + 6.0 * np.sqrt(lam) + 4.0))         # P(the sample holds `rank` of the top k) ~ 1e-9
                    if rank <= 32:
                        # entries shipped per rank and query: a shard holds Binomial(k, 1/world) of the global top k; a
                        # rank with more says so and the merge checks whether that mattered (-1 -> exact path)
                        share = min(k, self.n) / self.world
                        cap = min(k, int(np.ceil(share + 6.0 * np.sqrt(share) + 4.0)))
                        if self.world * cap > 2048 or self.world > 16:
                            cap = k
                        plan = (rank, max(p[3] for p in probes), cap)
            self._plans[key] = plan
        return self._plans[key]

    def _batch(self, dq, k: int, defer: bool = False):
        """b device queries -> (scores (b, k), ids (b, k), counts (b,)) device tensors, identical on every rank:
        per-rank batched candidate records, ONE all-gather of b records per rank, ONE merge launch (a CTA per query).
        With a global plan the ranks first agree on one filter threshold per query (a b x 32-float all-gather), each
        keeps and re-scores only what can reach the GLOBAL top k, and a query the coarse pass could not vouch for has
        count -1 on every rank (the caller redoes it with the exact path); nothing synchronises with the host."""
        b = dq.shape[0]
        plan = self._global_plan(k)
        cap = k if plan is None else plan[2]
        key = ("batch", k, b, cap)                                  # cap changes with the plan (a reload can switch it on or off)
        if key not in self._bufs:
            self._bufs[key] = (self.backend.new_records(b, cap), self.backend.new_records(self.world * b, cap),
                               self.backend.new_outputs(b, k))
        rec, gath, (o_s, o_i, o_c) = self._bufs[key]
        if plan is None:
            self.last_fallbacks = self.backend.batch_local(dq, k, rec)
            self.dist.all_gather_into_tensor(gath.view(-1), rec.view(-1), group=self.group)
            self.backend.enqueue_merge(gath, self.world, b, k, o_s, o_i, o_c)
            self._last_counts = None
            return o_s, o_i, o_c
        sample_rank, max_row_norm, cap = plan
        self.last_fallbacks = 0
        if self.exchange == "peer" and hasattr(self.backend, "batch_peer") and cap <= self.backend.BATCH_WINDOW_CAP:
            # both exchanges fused into the kernels over NVLink peer memory: no collective call at all
            self._ensure_window(batch=True)
            for c0 in range(0, b, 2048):                           # chunks pipeline: merge of chunk c behind the first phase of c+1
                bc = min(2048, b - c0)
                self.backend.batch_peer(dq[c0:c0 + bc], k, max_row_norm, sample_rank, cap, o_s[c0:c0 + bc], o_i[c0:c0 + bc], o_c[c0:c0 + bc],
                                        defer_merge=True)
            if not defer:
                self.backend.batch_peer_flush()
            self._last_counts = o_c
            return o_s, o_i, o_c
        tkey = ("tops", b)
        if tkey not in self._bufs:
            self._bufs[tkey] = (self.backend.new_tops(min(b, 2048)), self.backend.new_tops(self.world * min(b, 2048)))
        tops, tops_all = self._bufs[tkey]
        for c0 in range(0, b, 2048):
            bc = min(2048, b - c0)
            self.backend.batch_sample_tops(dq[c0:c0 + bc], k, max_row_norm, tops)
            self.dist.all_gather_into_tensor(tops_all[:self.world * bc].view(-1), tops[:bc].view(-1), group=self.group)
            self.backend.batch_global_records(dq[c0:c0 + bc], k, tops_all, self.world, sample_rank, cap, rec[c0:c0 + bc])
        self.dist.all_gather_into_tensor(gath.view(-1), rec.view(-1), group=self.group)
        self.backend.enqueue_merge_verified(gath, self.world, b, cap, k, min(k, self.n), o_s, o_i, o_c)
        self._last_counts = o_c
        return o_s, o_i, o_c

    def last_batch_unanswered(self) -> int:
        """Queries of the last global-threshold batch that came out with count -1 (synchronises); 0 otherwise."""
        self.flush_batches()
        return 0 if self._last_counts is None else int((self._last_counts < 0).sum().item())

    def run_batch(self, k: int, defer: bool = False) -> None:
        """One batch of ALL uploaded queries, device-resident end to end (bench path).  defer: in a stream of batches the
        batch's verifying merge goes behind the next batch's first phase (flush_batches() ends the stream)."""
        assert self._queries is not None, "set_queries first"
        self._batch(self._queries, k, defer=defer)

    def flush_batches(self) -> None:
        if self._batch_peer_ready:
            self.backend.batch_peer_flush()

    def retrieve_many_arrays(self, query_vecs: np.ndarray, n: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """superheavy() for every row of query_vecs on every rank, as arrays: host queries in; host
        (scores (b, k) float32, embeddings.id (b, k) int64, counts (b,) int32) out, row j valid up to counts[j]."""
        Q = np.ascontiguousarray(query_vecs, dtype=np.float32)
        if Q.ndim != 2 or Q.shape[1] != self.d or self.n == 0:
            raise ValueError(f"shapes ({self.n},{self.d if self.n else 0}) and {Q.shape} not aligned")
        if n <= 0 or Q.shape[0] == 0:
            return (np.zeros((Q.shape[0], 0), np.float32), np.zeros((Q.shape[0], 0), np.int64), np.zeros(Q.shape[0], np.int32))
        k = min(int(n), self.n)                                     # get_top_k clips n to the row count (util.py:198-199)
        if k > K_FAST_MAX:
            return self._retrieve_many_big(Q, k)
        o_s, o_i, o_c = self._batch(self.backend.device_queries(Q), k)
        cnt = o_c.cpu().numpy()                                     # synchronises the stream
        s, i = o_s.cpu().numpy(), o_i.cpu().numpy()
        if (cnt == -2).any():
            raise RuntimeError("sharded batch: a peer's part of the batch did not arrive (SVSB_XCHG_TIMEOUT_MS)")
        redo = np.nonzero(cnt < 0)[0]                               # the coarse pass could not vouch for these (same on every rank)
        self.last_fallbacks += len(redo)
        for j in redo:
            sj, ij = self.retrieve_arrays(Q[j], k)
            cnt[j] = len(sj); s[j, :len(sj)] = sj; i[j, :len(ij)] = ij
        return s, i, cnt

    def retrieve_many_pinned(self, queries, n: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """retrieve_many_arrays without pageable staging: `queries` is a PINNED torch tensor (b, d) float32 (torch
        `pin_memory()`), DMA'd to the device as is; the results come back into page-locked buffers owned by this object and
        are returned as NumPy views of them -- valid until the next call.  Same answers as retrieve_many_arrays.  Above
        2048 results per query the answers come back in new arrays instead, one query at a time."""
        t = self.backend.torch
        if not (isinstance(queries, t.Tensor) and queries.is_pinned() and queries.dtype == t.float32 and queries.dim() == 2
                and queries.is_contiguous()):
            raise ValueError("retrieve_many_pinned: a contiguous pinned float32 torch tensor (b, d) is required")
        if queries.shape[1] != self.d or self.n == 0:
            raise ValueError(f"shapes ({self.n},{self.d if self.n else 0}) and {tuple(queries.shape)} not aligned")
        b = queries.shape[0]
        if n <= 0 or b == 0:
            return (np.zeros((b, 0), np.float32), np.zeros((b, 0), np.int64), np.zeros(b, np.int32))
        k = min(int(n), self.n)
        if k > K_FAST_MAX:
            return self._retrieve_many_big(queries.numpy(), k)
        ld = (self.d + 3) & ~3
        dq = queries.to(self.backend.device, non_blocking=True)
        if ld != self.d:
            dq = t.nn.functional.pad(dq, (0, ld - self.d))
        o_s, o_i, o_c = self._batch(dq, k)
        key = ("pinned_out", b, k)
        if key not in self._bufs:
            self._bufs[key] = (t.empty((b, k), dtype=t.float32).pin_memory(), t.empty((b, k), dtype=t.int64).pin_memory(),
                               t.empty((b,), dtype=t.int32).pin_memory())
        h_s, h_i, h_c = self._bufs[key]
        h_s.copy_(o_s, non_blocking=True); h_i.copy_(o_i, non_blocking=True); h_c.copy_(o_c, non_blocking=True)
        t.cuda.current_stream(self.backend.device).synchronize()
        s, i, cnt = h_s.numpy(), h_i.numpy(), h_c.numpy()
        if (cnt == -2).any():
            raise RuntimeError("sharded batch: a peer's part of the batch did not arrive (SVSB_XCHG_TIMEOUT_MS)")
        redo = np.nonzero(cnt < 0)[0]
        self.last_fallbacks += len(redo)
        for j in redo:
            sj, ij = self.retrieve_arrays(queries[j].numpy(), k)
            cnt[j] = len(sj); s[j, :len(sj)] = sj; i[j, :len(ij)] = ij
        return s, i, cnt

    def retrieve_many(self, query_vecs: np.ndarray, n: int) -> List[List[Tuple[float, int]]]:
        """superheavy() for every row of query_vecs on every rank: host queries in, host lists out."""
        s, i, cnt = self.retrieve_many_arrays(query_vecs, n)
        return [[(float(a), int(x)) for a, x in zip(s[j, :cnt[j]], i[j, :cnt[j]])] for j in range(s.shape[0])]

    def retrieve_arrays(self, query_vec: np.ndarray, n: int) -> Tuple[np.ndarray, np.ndarray]:
        """superheavy() on every rank as host arrays: (scores float32[c], embeddings.id int64[c]), c = min(n, N)
        (the sharded counterpart of Engine.query: host query in, host buffers out, one synchronous call)."""
        q = np.ascontiguousarray(query_vec, dtype=np.float32)
        if q.ndim != 1 or q.shape[0] != self.d or self.n == 0:
            raise ValueError(f"shapes ({self.n},{self.d if self.n else 0}) and ({q.shape[0]},) not aligned")
        if n <= 0:
            return np.zeros(0, np.float32), np.zeros(0, np.int64)
        k = min(int(n), self.n)                                     # get_top_k clips n to the row count (util.py:198-199)
        if k > K_FAST_MAX:
            return self._retrieve_big(q, k)
        if self.exchange == "peer":
            self._ensure_window()
            return self.backend.query_peer(q, k)                   # one synchronous C call, result written to host
        dq = self.backend.device_queries(q[None, :])
        o_s, o_i, o_c = self._micro_batch([dq[0]], k, False)
        cnt = int(o_c[0].item())                                   # synchronises the stream
        return o_s[0, :cnt].cpu().numpy(), o_i[0, :cnt].cpu().numpy()

    def submit(self, query_vec: np.ndarray, n: int):
        """Start a retrieve (host query in) and return a handle for `wait`; up to 3 may be pending, every rank submits the
        same sequence.  The next query's matrix pass overlaps this one's selection, exchange, merge and host round trip."""
        q = np.ascontiguousarray(query_vec, dtype=np.float32)
        if q.ndim != 1 or q.shape[0] != self.d or self.n == 0:
            raise ValueError(f"shapes ({self.n},{self.d if self.n else 0}) and ({q.shape[0]},) not aligned")
        k = min(int(n), self.n)
        if k <= 0 or k > K_FAST_MAX or self.exchange != "peer":
            return ("done", self.retrieve_arrays(q, n))           # nothing to overlap: answered synchronously
        self._ensure_window()
        return ("ticket", self.backend.query_peer_submit(q, k), k)

    def wait(self, handle) -> Tuple[np.ndarray, np.ndarray]:
        """(scores, embeddings.id) of a submitted retrieve; oldest first."""
        if handle[0] == "done":
            return handle[1]
        return self.backend.query_peer_wait(handle[1], handle[2])

    def retrieve(self, query_vec: np.ndarray, n: int) -> List[Tuple[float, int]]:
        """The reference's superheavy() result, on every rank: host query in, host list out."""
        s, i = self.retrieve_arrays(query_vec, n)
        return [(float(a), int(b)) for a, b in zip(s, i)]

    # -- k > 2048: full sort per shard, one all-gather of the sorted records, rank merge on every rank ----------------
    def _big_buffers(self, cap: int):
        """The large-k path's one buffer set, replaced when cap changes: this rank's record, the gathered records and
        outputs of world * cap >= k entries.  A full ranking of 10M rows on 8 ranks gathers ~160 MB per rank: it is
        not kept once for every k ever asked."""
        if self._big is None or self._big[0] != cap:
            self._big = None                                       # the old set goes before the new one is allocated
            be = self.backend
            self._big = (cap, be.new_records(1, cap), be.new_records(self.world, cap), be.new_outputs(1, self.world * cap))
        return self._big[1:]

    def _retrieve_big(self, q: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray]:
        """superheavy() for 2048 < k <= N, on every rank, through the collective under either exchange (the peer
        windows are sized for k <= 2048)."""
        cap = min(k, -(-self.n // self.world))                     # rows of the largest shard (partition) bound every record
        try:
            rec, gath, (o_s, o_i, o_c) = self._big_buffers(cap)
            self.backend.enqueue_local(self.backend.device_queries(q[None, :])[0], cap, rec[0])
            self.backend.join()
            outcome = (0, "")
        except EngineError as ex:
            outcome = (ex.code, ex.message)
        except (MemoryError, RuntimeError) as ex:                  # a buffer the framework could not allocate
            outcome = (SVSB_E_NOMEM, f"sharded retrieve, n = {k}: {ex}")
        # every rank learns every rank's outcome before the collective: one refusal raises the same error everywhere
        # instead of leaving the others blocked in the all-gather
        self._agree(self._all_gather_object(outcome))
        self.dist.all_gather_into_tensor(gath.view(-1), rec.view(-1), group=self.group)
        self.backend.enqueue_merge_sorted(gath, self.world, cap, k, o_s[0], o_i[0], o_c[0])
        cnt = int(o_c[0].item())                                   # synchronises the stream
        if cnt != k:
            raise EngineError(SVSB_E_CUDA, f"sharded retrieve: the large-k merge returned {cnt} of {k} entries")
        return o_s[0, :cnt].cpu().numpy(), o_i[0, :cnt].cpu().numpy()

    def _retrieve_many_big(self, Q: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """retrieve_many_arrays for k > 2048: one large-k retrieve per query into (b, k) outputs."""
        s, i = np.zeros((Q.shape[0], k), np.float32), np.zeros((Q.shape[0], k), np.int64)
        for j in range(Q.shape[0]):
            s[j], i[j] = self._retrieve_big(np.ascontiguousarray(Q[j]), k)
        self.last_fallbacks, self._last_counts = 0, None
        return s, i, np.full(Q.shape[0], k, np.int32)

    # -- pairwise top pairs ---------------------------------------------------------------------------
    @staticmethod
    def _agree(outcomes) -> None:
        """Every rank raises the first refusal any rank reported: ranks never disagree about answering."""
        for status, message in outcomes:
            if status != 0:
                raise EngineError(status, message)

    def _pairs_disconnect(self) -> None:
        """Every rank's last pair call has returned before any rank unmaps its peers and releases its export."""
        if self.world > 1:
            self.dist.barrier(group=self.group)
        self.backend.pairs_disconnect()
        self._pairs_epoch = None

    def _ensure_pairs(self) -> None:
        """Export, all-gather, connect: once per load (a reload re-exports)."""
        if self._pairs_epoch == self._epoch:
            return
        if self._pairs_epoch is not None:
            self._pairs_disconnect()
        desc, status, message, max_dev = self.backend.pairs_export()
        got = self._all_gather_object((desc, status, message, max_dev))
        self._agree([(g[1], g[2]) for g in got])
        self.backend.pairs_connect(self.world, self.rank, [g[0] for g in got])
        if self.world > 1:
            self.dist.barrier(group=self.group)                    # every rank has opened its peers' shards
        self._pairs_norm = max(1.0 + g[3] for g in got)            # one coarse error bound for every rank
        self._pairs_epoch = self._epoch

    def top_pairs(self, n: int) -> List[Tuple[float, int, int]]:
        """document_top_pairwise_scores' superheavy() over the global matrix, on every rank: [(score, emb_id_1,
        emb_id_2)] of the n best pairs of distinct rows, equal to Engine.top_pairs on one device bit for bit."""
        n = min(int(n), self.n * (self.n - 1) // 2)
        if n <= 0 or self.d == 0:
            return []
        self._ensure_pairs()
        be = self.backend
        own = be.new_pair_lists(n)
        outcomes = self._all_gather_object(be.pairs_local(n, self._pairs_norm, own))
        self._agree([(s, m) for s, m, _ in outcomes])
        counts = [c for _, _, c in outcomes]
        stride = max(1, max(counts))
        lists = be.new_pair_lists(stride, self.world)
        for whole, mine in zip(lists, own):
            self.dist.all_gather_into_tensor(whole.view(-1), mine[0, :stride].contiguous(), group=self.group)
        out = be.new_pair_lists(n)
        c = be.pairs_merge(lists, counts, n, out)
        if c != n:
            raise EngineError(SVSB_E_CUDA, f"sharded top_pairs: the merge returned {c} of {n} pairs")
        s, a, b = (x[0, :c].cpu().numpy() for x in out)
        return [(float(x), int(y), int(z)) for x, y, z in zip(s, a, b)]

    def close(self) -> None:
        """Collective when an exchange is up: unmap the peers' memory everywhere before any rank frees its own."""
        if self._pairs_epoch is not None:
            self._pairs_disconnect()
            if self.world > 1:
                self.dist.barrier(group=self.group)
        if self._peer_ready or self._batch_peer_ready:
            if self._peer_ready and hasattr(self.backend, "exchange_disconnect"):
                self.backend.exchange_disconnect()
            if self._batch_peer_ready:
                self.backend.batch_exchange_disconnect()
            if self.world > 1:
                self.dist.barrier(group=self.group)
            self._peer_ready = self._batch_peer_ready = False
        self._big = None
        self.backend.close()
