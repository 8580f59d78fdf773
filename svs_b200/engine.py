"""`Engine`: a thin, torch-free Python face of the C ABI (include/svsb200.h).

Everything numeric happens in libsvsb200.so on the GPU; this module only marshals NumPy buffers.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import check


def _f32c(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def clamp_k(k, n_rows: int) -> int:
    """get_top_k clips top_k to len(scores) and answers [] for k <= 0 (src/svs/util.py:198-201).  Done HERE, before any
    buffer is sized by k and before k passes through a 32-bit C argument: retrieve(q, n=10**12) must return all N rows,
    not allocate terabytes or wrap around."""
    return min(max(int(k), 0), max(int(n_rows), 0), 0x7fffffff)


class Engine:
    """One engine == one cached device matrix (the replacement of `_EmbeddingsMatrix`' two arrays,
    reference src/svs/kb.py:856-893) plus the kernels that query it.

    devices: list of CUDA device indices; more than one row-shards the matrix across them.
    """

    def __init__(self, devices: Optional[Sequence[int]] = None):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        if devices is None:
            check(self._lib.svsb_create(None, 0, C.byref(self._h)))
            self.devices = [0]
        else:
            devs = (C.c_int32 * len(devices))(*devices)
            check(self._lib.svsb_create(devs, len(devices), C.byref(self._h)))
            self.devices = list(devices)

    # ---- lifetime ---------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.svsb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- load path --------------------------------------------------------------------------
    def load_begin(self, n: int, d: int, normalize: bool = False) -> None:
        check(self._lib.svsb_load_begin(self._h, n, d, _lib.NORM_NORMALIZE if normalize else _lib.NORM_CHECK))

    def load_rows(self, rows: np.ndarray, emb_ids: np.ndarray) -> None:
        rows = _f32c(rows)
        emb_ids = np.ascontiguousarray(emb_ids, dtype=np.int64)
        if rows.ndim != 2 or emb_ids.ndim != 1 or rows.shape[0] != emb_ids.shape[0]:
            raise ValueError("rows must be (count, d) and emb_ids (count,)")
        check(self._lib.svsb_load_rows(self._h, rows.ctypes.data, emb_ids.ctypes.data, rows.shape[0]))

    def acquire_slab(self, d: int) -> Tuple[np.ndarray, np.ndarray]:
        """Borrow a pinned staging slab: returns (rows_u8 view of capacity*d*4 bytes, ids view)."""
        p_rows, p_ids, cap = C.c_void_p(), C.c_void_p(), C.c_int64()
        check(self._lib.svsb_load_acquire_slab(self._h, C.byref(p_rows), C.byref(p_ids), C.byref(cap)))
        n = cap.value
        if n == 0:
            return np.empty(0, dtype=np.uint8), np.empty(0, dtype=np.int64)
        rows = np.ctypeslib.as_array((C.c_uint8 * (n * d * 4)).from_address(p_rows.value))
        ids = np.ctypeslib.as_array((C.c_int64 * n).from_address(p_ids.value))
        return rows, ids

    def commit_slab(self, count: int) -> None:
        check(self._lib.svsb_load_commit_slab(self._h, count))

    def load_end(self) -> int:
        gen = C.c_uint64()
        check(self._lib.svsb_load_end(self._h, C.byref(gen)))
        return gen.value

    def load_abort(self) -> None:
        check(self._lib.svsb_load_abort(self._h))

    def load(self, rows: np.ndarray, emb_ids: Optional[np.ndarray] = None, normalize: bool = False) -> int:
        """Load a whole host matrix (n, d) float32 and its ids (default 0..n-1)."""
        rows = _f32c(rows)
        if rows.ndim != 2:
            raise ValueError("rows must be 2-D")
        n, d = rows.shape
        if emb_ids is None:
            emb_ids = np.arange(n, dtype=np.int64)
        self.load_begin(n, d, normalize)
        if n:
            self.load_rows(rows, emb_ids)
        return self.load_end()

    def load_chunks(self, n: int, d: int, chunks: Iterable[Tuple[np.ndarray, np.ndarray]], normalize: bool = False) -> int:
        self.load_begin(n, d, normalize)
        for rows, ids in chunks:
            self.load_rows(rows, ids)
        return self.load_end()

    def load_sqlite(self, path: str, normalize: bool = False, threads: int = 0) -> Tuple[int, int]:
        """build_embeddings_matrix (src/svs/kb.py:573-618) natively: scan the `embeddings` table of the SQLite file at
        `path` on private read-only connections (include/svsb200.h: svsb_load_sqlite).  Returns (n, d).  Raises
        EngineError(SVSB_E_STATE) when the native scan does not apply; the caller then uses the generic load path."""
        gen, n, d = C.c_uint64(), C.c_int64(), C.c_int32()
        check(self._lib.svsb_load_sqlite(self._h, os.fsencode(str(path)), _lib.NORM_NORMALIZE if normalize else _lib.NORM_CHECK,
                                         int(threads), C.byref(gen), C.byref(n), C.byref(d)))
        return n.value, d.value

    def load_synthetic(self, n: int, d: int, seed: int = 0, id0: int = 0, id_step: int = 1) -> int:
        gen = C.c_uint64()
        check(self._lib.svsb_load_synthetic(self._h, n, d, seed, id0, id_step, C.byref(gen)))
        return gen.value

    def invalidate(self) -> None:
        check(self._lib.svsb_invalidate(self._h))

    def is_loaded(self) -> bool:
        return bool(self._lib.svsb_is_loaded(self._h))

    @property
    def shape(self) -> Tuple[int, int]:
        n, d = C.c_int64(), C.c_int32()
        check(self._lib.svsb_shape(self._h, C.byref(n), C.byref(d)))
        # the reference's empty matrix has shape (0, 0) (src/svs/kb.py:595-601)
        return (n.value, d.value)

    def norm_stats(self) -> Tuple[float, int]:
        dev, bad = C.c_float(), C.c_int64()
        check(self._lib.svsb_norm_stats(self._h, C.byref(dev), C.byref(bad)))
        return dev.value, bad.value

    def read_rows(self, row0: int, count: int) -> Tuple[np.ndarray, np.ndarray]:
        n, d = self.shape
        rows = np.empty((count, d), dtype=np.float32)
        ids = np.empty(count, dtype=np.int64)
        check(self._lib.svsb_read_rows(self._h, row0, count, rows.ctypes.data, ids.ctypes.data))
        return rows, ids

    # ---- hot path ---------------------------------------------------------------------------
    def query(self, q: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray]:
        """Top-k of M @ q.  Returns (scores float32[c], emb_ids int64[c]), c = min(k, N); k <= 0 -> empty."""
        q = _f32c(q)
        if q.ndim != 1:
            raise ValueError("query vector must be 1-D")
        cap = clamp_k(k, self._rows_or_zero())
        k = cap if int(k) > 0 else int(max(k, -1))
        scores = np.empty(cap, dtype=np.float32)
        ids = np.empty(cap, dtype=np.int64)
        cnt = C.c_int32()
        check(self._lib.svsb_query(self._h, q.ctypes.data, q.shape[0], k, scores.ctypes.data, ids.ctypes.data, C.byref(cnt)))
        return scores[:cnt.value], ids[:cnt.value]

    def _rows_or_zero(self) -> int:
        """Rows of the resident matrix, 0 when nothing is resident (the C call then reports SVSB_E_NOT_LOADED)."""
        n = C.c_int64()
        return n.value if self._lib.svsb_shape(self._h, C.byref(n), None) == _lib.SVSB_OK else 0

    def submit(self, q: np.ndarray, k: int) -> "Pending":
        """Start a query and return at once; `.result()` of the returned handle blocks for its (scores, ids).  Keeping
        two or three in flight hides the per-call launch / selection / host round-trip latency behind the next query's
        similarity pass (include/svsb200.h: svsb_query_submit)."""
        q = _f32c(q)
        if q.ndim != 1:
            raise ValueError("query vector must be 1-D")
        cap = clamp_k(k, self._rows_or_zero())
        k = cap if int(k) > 0 else int(max(k, -1))
        h = C.c_void_p()
        check(self._lib.svsb_query_submit(self._h, q.ctypes.data, q.shape[0], k, C.byref(h)))
        return Pending(self, h, cap)

    def apply_mutations(self, del_ids, add_ids, add_rows: Optional[np.ndarray]) -> int:
        """Incremental update (include/svsb200.h: svsb_apply_mutations): tombstone the rows with embeddings.id in
        `del_ids`, append `add_rows` (n_add, d) with ids `add_ids` (ascending, above every live id).  Publishes a new
        generation that shares the matrix buffers with the old one; raises EngineError (SVSB_E_STATE) when the batch
        cannot be applied incrementally -- the caller then rebuilds."""
        dels = np.ascontiguousarray(np.asarray(del_ids, dtype=np.int64).reshape(-1))
        aids = np.ascontiguousarray(np.asarray(add_ids, dtype=np.int64).reshape(-1))
        n_add = int(aids.shape[0])
        if n_add:
            rows = _f32c(add_rows)
            if rows.ndim != 2 or rows.shape[0] != n_add:
                raise ValueError("add_rows must be (len(add_ids), d)")
            d = int(rows.shape[1])
        else:
            rows, d = np.zeros((0, 0), np.float32), 0
        gen = C.c_uint64()
        check(self._lib.svsb_apply_mutations(self._h, dels.ctypes.data if len(dels) else None, len(dels),
                                             rows.ctypes.data if n_add else None, aids.ctypes.data if n_add else None, n_add, d,
                                             C.byref(gen)))
        return gen.value

    def compact(self, global_row0: int = 0) -> int:
        """Gather the live rows of a tombstoned generation into a new buffer on the device and publish them as a
        tombstone-free generation whose first row is global row `global_row0` (include/svsb200.h: svsb_compact).  The
        result equals a fresh load of the live rows.  Single-device engines only; returns the new generation."""
        gen = C.c_uint64()
        check(self._lib.svsb_compact(self._h, int(global_row0), C.byref(gen)))
        return gen.value

    def generation_rows(self) -> Tuple[int, int]:
        """(physical rows incl. tombstoned ones, live rows) of the resident generation."""
        p, l = C.c_int64(), C.c_int64()
        check(self._lib.svsb_generation_rows(self._h, C.byref(p), C.byref(l)))
        return p.value, l.value

    def snapshot(self) -> "Snapshot":
        """Pin the resident generation (the reference's `embeddings_matrix, emb_id_lookup` references)."""
        return Snapshot(self)

    def query_batch(self, Q: np.ndarray, k: int, out=None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """b queries at once: (scores (b, k), emb_ids (b, k), counts (b,)).  Bit-identical to b calls of query();
        large batches run as one tensor-core contraction + exact refine (include/svsb200.h: svsb_query_batch).
        out: optional (scores, ids, counts) arrays to fill (C-contiguous, shapes as returned); with page-locked
        arrays (pinned_empty) for Q and out the library copies straight from / into them."""
        Q = _f32c(Q)
        if Q.ndim != 2:
            raise ValueError("Q must be (b, d)")
        b, d = Q.shape
        cap = clamp_k(k, self._rows_or_zero())
        k = cap if int(k) > 0 else int(max(k, -1))
        if out is None:
            scores = np.zeros((b, cap), dtype=np.float32)
            ids = np.full((b, cap), -1, dtype=np.int64)
            counts = np.zeros(b, dtype=np.int32)
        else:
            scores, ids, counts = out
            ok = (scores.shape == (b, cap) and ids.shape == (b, cap) and counts.shape == (b,) and scores.dtype == np.float32
                  and ids.dtype == np.int64 and counts.dtype == np.int32
                  and scores.flags.c_contiguous and ids.flags.c_contiguous and counts.flags.c_contiguous)
            if not ok:
                raise ValueError("out must be C-contiguous (float32 (b, k), int64 (b, k), int32 (b,)) arrays")
        check(self._lib.svsb_query_batch(self._h, Q.ctypes.data, b, d, k, scores.ctypes.data, ids.ctypes.data, counts.ctypes.data))
        return scores, ids, counts

    def retrieve(self, query_vec: np.ndarray, n: int) -> List[Tuple[float, int]]:
        """The reference's `superheavy()` result shape: [(score: float, emb_id: int), ...]
        (src/svs/kb.py:1622-1627)."""
        scores, ids = self.query(query_vec, n)
        return [(float(s), int(i)) for s, i in zip(scores, ids)]

    def top_pairs(self, n: int) -> List[Tuple[float, int, int]]:
        """The `superheavy()` of document_top_pairwise_scores (src/svs/kb.py:1650-1656): [(score, emb_id_1, emb_id_2)]
        of the n highest-scoring pairs of distinct rows (upper triangle), never materialising the N x N scores."""
        cap = max(int(n), 0)
        rows = self.shape[0]
        cap = min(cap, rows * (rows - 1) // 2)
        s = np.empty(cap, dtype=np.float32)
        a = np.empty(cap, dtype=np.int64)
        b = np.empty(cap, dtype=np.int64)
        cnt = C.c_int64()
        check(self._lib.svsb_top_pairs(self._h, cap, s.ctypes.data, a.ctypes.data, b.ctypes.data, C.byref(cnt)))
        c = cnt.value
        return [(float(x), int(y), int(z)) for x, y, z in zip(s[:c], a[:c], b[:c])]

    def topk_scores(self, scores: np.ndarray, k: int) -> List[Tuple[float, int]]:
        """get_top_k (src/svs/util.py:190-203) run by the device selection kernels on a host score
        vector; ties are ordered by ascending index (the engine's order), not descending."""
        scores = np.asarray(scores)
        assert scores.ndim == 1
        s32 = _f32c(scores)
        cap = max(min(int(k), len(s32)), 0)
        out_s = np.empty(cap, dtype=np.float32)
        out_i = np.empty(cap, dtype=np.int64)
        cnt = C.c_int32()
        check(self._lib.svsb_topk_scores(self._h, s32.ctypes.data, len(s32), int(k), out_s.ctypes.data, out_i.ctypes.data, C.byref(cnt)))
        return [(float(s), int(i)) for s, i in zip(out_s[:cnt.value], out_i[:cnt.value])]

    # ---- measurement ------------------------------------------------------------------------
    def bench_set_queries(self, Q: np.ndarray) -> None:
        Q = _f32c(Q)
        check(self._lib.svsb_bench_set_queries(self._h, Q.ctypes.data, Q.shape[0], Q.shape[1]))

    def bench_run(self, k: int, iters: int, with_gemv: bool = False) -> dict:
        total, gemv, launches = C.c_float(), C.c_float(), C.c_int64()
        check(self._lib.svsb_bench_run(self._h, k, iters, C.byref(total), C.byref(gemv) if with_gemv else None, C.byref(launches)))
        return {"total_ms": total.value, "gemv_ms": gemv.value if with_gemv else None, "launches": launches.value}

    def bench_run_batch(self, k: int, iters: int, with_coarse: bool = False) -> dict:
        """`iters` batches of ALL uploaded queries through the batched (tensor-core) path, device-resident."""
        total, coarse, launches = C.c_float(), C.c_float(), C.c_int64()
        check(self._lib.svsb_bench_run_batch(self._h, k, iters, C.byref(total), C.byref(coarse) if with_coarse else None,
                                             C.byref(launches)))
        return {"total_ms": total.value, "coarse_ms": coarse.value if with_coarse else None, "launches": launches.value}

    def bench_batch_result(self, qi: int, k: int) -> Tuple[List[Tuple[float, int]], int]:
        s = np.empty(k, dtype=np.float32)
        i = np.empty(k, dtype=np.int64)
        cnt, flag = C.c_int32(), C.c_int32()
        check(self._lib.svsb_bench_batch_result(self._h, qi, k, s.ctypes.data, i.ctypes.data, C.byref(cnt), C.byref(flag)))
        return [(float(a), int(b)) for a, b in zip(s[:cnt.value], i[:cnt.value])], flag.value

    def batch_stats(self, b: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """(coarse candidates, rows re-scored exactly, flag) per query of the last batch chunk."""
        cand = np.zeros(b, dtype=np.int32)
        resc = np.zeros(b, dtype=np.int32)
        flags = np.zeros(b, dtype=np.int32)
        check(self._lib.svsb_batch_stats(self._h, b, cand.ctypes.data, resc.ctypes.data, flags.ctypes.data))
        return cand, resc, flags

    def batch_candidates(self, q: int) -> Tuple[np.ndarray, np.ndarray, int, float]:
        """Query q's coarse candidates of the last batch chunk: (coarse scores float32[c], rows int64[c], count, eps).
        count above c means the list overflowed its capacity (SVSB_BATCH_CAND_CAP); rows are the shard's rows."""
        cnt, eps = C.c_int32(), C.c_float()
        check(self._lib.svsb_batch_candidates(self._h, int(q), 0, None, C.byref(cnt), C.byref(eps)))
        keys = np.zeros(max(cnt.value, 0), dtype=np.uint64)
        check(self._lib.svsb_batch_candidates(self._h, int(q), len(keys), keys.ctypes.data if len(keys) else None,
                                              C.byref(cnt), None))
        keys = keys[keys != 0]        # an overflowed list holds only its capacity; a real key is never 0 (its row < 2^32 - 1)
        hi = (keys >> np.uint64(32)).astype(np.uint32)               # key_score: the ordered transform, undone
        b = np.where(hi & np.uint32(0x80000000), hi & np.uint32(0x7FFFFFFF), ~hi).astype(np.uint32)
        rows = (~(keys & np.uint64(0xFFFFFFFF)).astype(np.uint32)).astype(np.int64)    # key_row
        return b.view(np.float32), rows, cnt.value, eps.value

    def bench_filter_stats(self) -> Tuple[bool, int]:
        """(took the int8 filter, rows the last query re-scored exactly) of the last bench_run."""
        f, r = C.c_int32(), C.c_int64()
        check(self._lib.svsb_bench_filter_stats(self._h, C.byref(f), C.byref(r)))
        return bool(f.value), int(r.value)

    def bench_filter_route(self) -> int:
        """Route of the last bench_run: 0 = fp32 similarity kernel, 8 = int8 filter."""
        r = C.c_int32()
        check(self._lib.svsb_bench_filter_route(self._h, C.byref(r)))
        return int(r.value)

    def batch_threshold_mode(self) -> int:
        """0 = verified statistical filter thresholds (default), 1 = proven-bound thresholds (see svsb200.h)."""
        rc = self._lib.svsb_batch_threshold_mode(self._h)
        if rc < 0:
            check(rc)
        return rc

    def bench_last_result(self, k: int) -> List[Tuple[float, int]]:
        s = np.empty(k, dtype=np.float32)
        i = np.empty(k, dtype=np.int64)
        cnt = C.c_int32()
        check(self._lib.svsb_bench_last_result(self._h, k, s.ctypes.data, i.ctypes.data, C.byref(cnt)))
        return [(float(a), int(b)) for a, b in zip(s[:cnt.value], i[:cnt.value])]


class Pending:
    """A query in flight (Engine.submit).  `.result()` must be called exactly once."""

    def __init__(self, engine: Engine, handle: C.c_void_p, cap: int):
        self._engine, self._h, self._cap = engine, handle, cap

    def result(self) -> Tuple[np.ndarray, np.ndarray]:
        if self._h is None:
            raise RuntimeError("result() was already taken")
        scores = np.empty(self._cap, dtype=np.float32)
        ids = np.empty(self._cap, dtype=np.int64)
        cnt = C.c_int32()
        h, self._h = self._h, None
        check(self._engine._lib.svsb_query_wait(self._engine._h, h, scores.ctypes.data, ids.ctypes.data, C.byref(cnt)))
        return scores[:cnt.value], ids[:cnt.value]

    def __del__(self):  # pragma: no cover - a handle nobody waited for still has to be released
        try:
            if self._h is not None and self._engine._h.value:
                self.result()
        except Exception:
            pass


class _PinnedBlock:
    """Owner of one svsb_host_alloc allocation; arrays made over it keep it alive through their .base chain."""

    def __init__(self, nbytes: int):
        self._lib = _lib.load()
        self._p = C.c_void_p()
        check(self._lib.svsb_host_alloc(nbytes, C.byref(self._p)))
        self.buf = (C.c_uint8 * max(nbytes, 1)).from_address(self._p.value)

    def __del__(self):
        try:
            if self._p.value:
                self._lib.svsb_host_free(self._p)
                self._p = C.c_void_p()
        except Exception:
            pass


def pinned_empty(shape, dtype) -> np.ndarray:
    """A page-locked (cudaHostAlloc) NumPy array: query batches / result buffers the engine can DMA without staging."""
    dtype = np.dtype(dtype)
    shape = (shape,) if isinstance(shape, int) else tuple(shape)
    n = int(np.prod(shape)) if shape else 1
    block = _PinnedBlock(n * dtype.itemsize)
    block.buf._owner = block          # the array's buffer exporter keeps the block alive (a cycle the GC frees later)
    return np.frombuffer(block.buf, dtype=dtype, count=n).reshape(shape)


class Snapshot:
    """A pinned generation: queries through it see the matrix that was resident when it was taken,
    even if the engine has been invalidated or re-loaded since (reference src/svs/kb.py:1178-1190)."""

    def __init__(self, engine: Engine):
        self._engine = engine
        self._lib = engine._lib
        self._s = C.c_void_p()
        check(self._lib.svsb_snapshot_acquire(engine._h, C.byref(self._s)))
        n, d, gen = C.c_int64(), C.c_int32(), C.c_uint64()
        check(self._lib.svsb_snapshot_shape(self._s, C.byref(n), C.byref(d), C.byref(gen)))
        self.shape = (n.value, d.value if n.value else 0)
        self.generation = gen.value
        p, l = C.c_int64(), C.c_int64()
        check(self._lib.svsb_snapshot_rows(self._s, C.byref(p), C.byref(l)))
        self.physical_rows, self.live_rows = p.value, l.value      # differ once rows were tombstoned (apply_mutations)

    def query(self, q: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray]:
        q = _f32c(q)
        if q.ndim != 1:
            raise ValueError("query vector must be 1-D")
        if not self._engine._h.value:
            raise _lib.EngineError(_lib.SVSB_E_STATE, "engine is closed")
        cap = clamp_k(k, self.shape[0])
        k = cap if int(k) > 0 else int(max(k, -1))
        scores = np.empty(cap, dtype=np.float32)
        ids = np.empty(cap, dtype=np.int64)
        cnt = C.c_int32()
        check(self._lib.svsb_snapshot_query(self._engine._h, self._s, q.ctypes.data, q.shape[0], k,
                                            scores.ctypes.data, ids.ctypes.data, C.byref(cnt)))
        return scores[:cnt.value], ids[:cnt.value]

    def retrieve(self, query_vec: np.ndarray, n: int) -> List[Tuple[float, int]]:
        scores, ids = self.query(query_vec, n)
        return [(float(s), int(i)) for s, i in zip(scores, ids)]

    def query_batch(self, Q: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """b queries against the pinned generation: (scores (b, k), emb_ids (b, k), counts (b,))."""
        Q = _f32c(Q)
        if Q.ndim != 2:
            raise ValueError("Q must be (b, d)")
        if not self._engine._h.value:
            raise _lib.EngineError(_lib.SVSB_E_STATE, "engine is closed")
        b, d = Q.shape
        cap = clamp_k(k, self.shape[0])
        k = cap if int(k) > 0 else int(max(k, -1))
        scores = np.zeros((b, cap), dtype=np.float32)
        ids = np.full((b, cap), -1, dtype=np.int64)
        counts = np.zeros(b, dtype=np.int32)
        check(self._lib.svsb_snapshot_query_batch(self._engine._h, self._s, Q.ctypes.data, b, d, k,
                                                  scores.ctypes.data, ids.ctypes.data, counts.ctypes.data))
        return scores, ids, counts

    def top_pairs(self, n: int) -> List[Tuple[float, int, int]]:
        """[(score, emb_id_1, emb_id_2)] of the n best pairs of distinct rows of the pinned generation."""
        if not self._engine._h.value:
            raise _lib.EngineError(_lib.SVSB_E_STATE, "engine is closed")
        rows = self.shape[0]
        cap = min(max(int(n), 0), rows * (rows - 1) // 2)
        s = np.empty(cap, dtype=np.float32)
        a = np.empty(cap, dtype=np.int64)
        b = np.empty(cap, dtype=np.int64)
        cnt = C.c_int64()
        check(self._lib.svsb_snapshot_top_pairs(self._engine._h, self._s, cap, s.ctypes.data, a.ctypes.data, b.ctypes.data,
                                                C.byref(cnt)))
        c = cnt.value
        return [(float(x), int(y), int(z)) for x, y, z in zip(s[:c], a[:c], b[:c])]

    def retrieve_many(self, query_vecs: np.ndarray, n: int) -> List[List[Tuple[float, int]]]:
        """superheavy() for every row of query_vecs, as ONE engine call."""
        scores, ids, counts = self.query_batch(query_vecs, n)
        return [[(float(s), int(i)) for s, i in zip(scores[j, :counts[j]], ids[j, :counts[j]])] for j in range(len(counts))]

    def release(self) -> None:
        if self._s is not None and self._s.value:
            self._lib.svsb_snapshot_release(self._s)
            self._s = C.c_void_p()

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.release()
        except Exception:
            pass


def sqlite_read(path: str, threads: int = 0) -> Tuple[np.ndarray, np.ndarray]:
    """The native table scan into host arrays (svsb_sqlite_read): (matrix float32 (n, d), embeddings.id int64 (n,)) in
    rowid order -- no device involved; what svsb_load_sqlite feeds the device with."""
    lib = _lib.load()
    n, d = C.c_int64(), C.c_int32()
    check(lib.svsb_sqlite_read(os.fsencode(str(path)), int(threads), None, None, 0, -1, C.byref(n), C.byref(d)))
    rows = np.empty((n.value, d.value), dtype=np.float32)
    ids = np.empty(n.value, dtype=np.int64)
    if n.value:
        check(lib.svsb_sqlite_read(os.fsencode(str(path)), int(threads), rows.ctypes.data, ids.ctypes.data, n.value, d.value,
                                   C.byref(n), C.byref(d)))
    return rows, ids


def launch_count() -> int:
    return int(_lib.load().svsb_launch_count())
