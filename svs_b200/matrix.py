"""Device-resident mirror of the reference's vector cache and matrix build.

`DeviceEmbeddingsMatrix` has the interface of `svs.kb._EmbeddingsMatrix` (reference
src/svs/kb.py:856-893): `get_sync(db)`, `async get(db)`, `invalidate()`.  Instead of two NumPy arrays
it hands back a `DeviceMatrix` handle whose `.retrieve(query_vec, n)` is the reference's `superheavy()`
closure (src/svs/kb.py:1622-1627) executed on the GPU.

`load_from_connection` is `_Querier.build_embeddings_matrix` (src/svs/kb.py:573-618): same three
statements against the same schema (src/svs/kb.py:80-83), same scan order, same asserts -- but the
blobs go straight into the engine's pinned staging slabs and on to the device, never through
`struct.unpack` lists.
"""
from __future__ import annotations

import asyncio
import logging
import os
import sqlite3
import threading
from typing import Any, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .engine import Engine, Snapshot
from .mutations import compaction_due

_LOG = logging.getLogger(__name__)


class DeviceMatrix:
    """Handle on one loaded generation: what `embeddings_matrix, emb_id_lookup` are to the reference."""

    def __init__(self, engine: Engine):
        self._engine = engine
        self._snap: Snapshot = engine.snapshot()    # pins this generation until the handle dies
        self.shape = self._snap.shape               # (N, D); (0, 0) for an empty table, like the reference
        self.generation = self._snap.generation
        # rows deleted since the last full build stay in the buffer as tombstones (incremental updates)
        self.has_tombstones = self._snap.physical_rows != self._snap.live_rows

    def __len__(self) -> int:
        return self.shape[0]

    def retrieve(self, query_vec: np.ndarray, n: int) -> List[Tuple[float, int]]:
        """superheavy(): [(score, emb_id)] of the n best rows.  Raises ValueError for a D mismatch or
        an empty matrix exactly where the reference's np.dot does."""
        return self._snap.retrieve(query_vec, n)

    def top_pairs(self, n: int) -> List[Tuple[float, int, int]]:
        """The `superheavy()` of document_top_pairwise_scores (src/svs/kb.py:1650-1656): np.dot(M, M.T) + get_top_pairs
        + emb_id_lookup, on the GPU, without materialising the N x N score matrix."""
        return self._snap.top_pairs(n)

    def retrieve_many(self, query_vecs: np.ndarray, n: int) -> List[List[Tuple[float, int]]]:
        """superheavy() for a batch of query vectors in one engine call (bit-identical to looping `retrieve`);
        large batches run as one tensor-core contraction (include/svsb200.h: svsb_query_batch)."""
        return self._snap.retrieve_many(query_vecs, n)


def _native_scan_applies(path: Any) -> bool:
    if path is None or os.environ.get("SVSB_NATIVE_LOAD", "1") == "0":
        return False
    p = str(path)
    return p != ":memory:" and not p.startswith("file:") and os.path.isfile(p)


def load_from_connection(engine: Engine, conn: sqlite3.Connection, normalize: bool = False, path: Any = None) -> DeviceMatrix:
    """build_embeddings_matrix (src/svs/kb.py:573-618) into the device cache.

    path: the database file behind `conn`, if known.  The scan then runs natively (svsb_load_sqlite: parallel read-only
    connections of libsqlite3 feeding pinned slabs, no per-row Python) -- same rows, same order; when that does not
    apply (in-memory database, no libsqlite3, anything it refuses) the generic scan through `conn` below does it."""
    if _native_scan_applies(path) and hasattr(engine, "load_sqlite"):
        try:
            engine.load_sqlite(path, normalize)
            return DeviceMatrix(engine)
        except _lib.EngineError as ex:
            if ex.code != _lib.SVSB_E_STATE:
                raise
            _LOG.info("native SQLite scan not applicable (%s); scanning through the connection", ex)
    n = conn.execute("SELECT COUNT(*) FROM embeddings;").fetchone()[0]
    assert isinstance(n, int)
    first = conn.execute("SELECT embedding FROM embeddings LIMIT 1;").fetchone()
    if first is not None:
        assert len(first[0]) % 4 == 0                       # embedding_from_bytes, embeddings/util.py:20-21
        d = len(first[0]) // 4
    else:
        d = 0
    engine.load_begin(n, d, normalize)
    try:
        loaded = 0
        if n and d:
            row_bytes = d * 4
            cur = conn.execute("SELECT id, embedding FROM embeddings;")
            # One memcpy per row, straight from the blob SQLite hands out into the pinned slab (measured: ~2x the
            # throughput of fetchmany + b"".join, which copies every byte three times).
            slab, slab_ids = engine.acquire_slab(d)
            cap, mv, idl, i = len(slab_ids), memoryview(slab), [], 0
            for emb_id, blob in cur:
                if cap == 0:
                    # rows beyond COUNT(*): the reference's `assert i == n-1` (kb.py:616)
                    raise AssertionError("more embedding rows than COUNT(*) reported")
                # every row must have the first row's length (kb.py:613)
                assert len(blob) == row_bytes, "embedding rows of unequal length"
                mv[i * row_bytes:(i + 1) * row_bytes] = blob
                idl.append(emb_id)
                i += 1
                if i == cap:
                    slab_ids[:i] = idl
                    del mv
                    engine.commit_slab(i)
                    loaded += i
                    slab, slab_ids = engine.acquire_slab(d)
                    cap, mv, idl, i = len(slab_ids), memoryview(slab), [], 0
            if i:
                slab_ids[:i] = idl
            del mv
            engine.commit_slab(i)
            loaded += i
        elif n:
            # zero-length blobs: nothing to copy, but ids still define N
            ids = np.fromiter((r[0] for r in conn.execute("SELECT id FROM embeddings;")), dtype=np.int64)
            engine.load_rows(np.zeros((len(ids), 0), dtype=np.float32), ids)
            loaded = len(ids)
        assert loaded == n, f"{loaded} embedding rows scanned, COUNT(*) said {n}"   # kb.py:616
        engine.load_end()
    except BaseException:
        # abandon the half-built generation; the previous one (if any) stays untouched
        try:
            engine.load_abort()
        except Exception:
            pass
        raise
    return DeviceMatrix(engine)


class DeviceEmbeddingsMatrix:
    """Drop-in for `_EmbeddingsMatrix` (src/svs/kb.py:856-893).

    `invalidate()` marks the device matrix stale instead of dropping it.  The next `get_sync` / `get` brings it up to
    date: incrementally (append + tombstone, `Engine.apply_mutations`) when the database object carries a mutation log
    that vouches for everything that happened since (`svs_b200.mutations`, attached by `install()`), else by the full
    rebuild inside a DB transaction exactly as the reference does (kb.py:870-877)."""

    def __init__(self, devices: Optional[Sequence[int]] = None, normalize: bool = False, incremental: bool = True) -> None:
        self._devices = list(devices) if devices is not None else None
        self._normalize = normalize
        self._incremental = incremental
        self._engine: Optional[Engine] = None        # created lazily on first load (SURVEY 3.5)
        self._matrix: Optional[DeviceMatrix] = None
        self._stale = False
        self._mu = threading.Lock()
        self.stats = {"full_builds": 0, "incremental_updates": 0, "incremental_fallbacks": 0}

    def _get_engine(self) -> Engine:
        if self._engine is None:
            self._engine = Engine(self._devices)
        return self._engine

    def prewarm(self) -> threading.Thread:
        """Create the engine (CUDA context, streams) on a daemon thread; a load that arrives first simply waits for it."""
        def work() -> None:
            try:
                with self._mu:
                    self._get_engine()
            except Exception as ex:                      # reported again, loudly, by the first load
                _LOG.warning("engine pre-warm failed: %s", ex)
        t = threading.Thread(target=work, name="svs_b200-prewarm", daemon=True)
        t.start()
        return t

    def invalidate(self) -> None:
        """kb.py:861-864.  In-flight queries keep the generation they started on.  The resident matrix is kept (stale)
        so that the next retrieve can update it in place of a rebuild; `drop()` frees it."""
        _LOG.info("invalidating cached device vectors; they'll be brought up to date next time you `retrieve()`")
        with self._mu:
            if self._matrix is not None:
                self._stale = True
            if not self._incremental:
                self._drop_locked()

    def _drop_locked(self) -> None:
        had = self._matrix is not None
        self._matrix = None
        self._stale = False
        if had and self._engine is not None:
            self._engine.invalidate()

    def drop(self) -> None:
        """Free the device matrix now (the pre-incremental behaviour of invalidate)."""
        with self._mu:
            self._drop_locked()

    def _try_incremental(self, db: Any) -> Optional[DeviceMatrix]:
        """Apply the committed mutations to the stale matrix.  None = not possible, do the full rebuild."""
        log = getattr(db, "_svsb_log", None)
        m = self._matrix
        if log is None or m is None or self._engine is None or not self._incremental:
            return None
        batch = log.take()
        if batch is None:
            return None
        dels, add_ids, blobs = batch
        if not dels and not add_ids:
            return m                                     # e.g. documents without embeddings were added / deleted
        d = m.shape[1]
        if m.shape[0] == 0 or any(len(b) != d * 4 for b in blobs):
            return None
        # past this fraction of dead rows a rebuild (which also compacts) is the better deal
        physical, live = self._engine.generation_rows()
        if compaction_due(physical + len(add_ids), physical - live + len(dels)):
            return None
        rows = np.frombuffer(b"".join(blobs), dtype="<f4").reshape(len(blobs), d) if blobs else None
        try:
            self._engine.apply_mutations(dels, add_ids, rows)
        except _lib.EngineError as ex:
            if ex.code != _lib.SVSB_E_STATE:
                raise
            _LOG.info("incremental update not applicable (%s); rebuilding", ex)
            self.stats["incremental_fallbacks"] += 1
            return None
        self.stats["incremental_updates"] += 1
        return DeviceMatrix(self._engine)

    def _build(self, q: Any, db: Any = None) -> DeviceMatrix:
        conn = q.conn if hasattr(q, "conn") else q
        log = getattr(db, "_svsb_log", None)
        if log is not None:
            log.take()                                   # the scan below sees everything committed so far
        with self._mu:
            self._drop_locked()                          # never two full generations resident at once
            engine = self._get_engine()
        self.stats["full_builds"] += 1
        return load_from_connection(engine, conn, self._normalize, path=getattr(db, "path", None))

    def _current(self, db: Any) -> Optional[DeviceMatrix]:
        m = self._matrix
        if m is not None and not self._stale:
            _LOG.info("using cached device vectors")
            return m
        if m is not None:
            m2 = self._try_incremental(db)
            if m2 is not None:
                _LOG.info("updated cached device vectors incrementally")
                self._matrix, self._stale = m2, False
                return m2
        return None

    def get_sync(self, db: Any, compact: bool = False) -> DeviceMatrix:
        """kb.py:866-877: cached handle, or bring it up to date (incrementally, else rebuild inside a DB transaction).
        compact: the caller needs a matrix without tombstones (the pairwise path)."""
        m = self._current(db)
        if m is not None and not (compact and m.has_tombstones):
            return m
        _LOG.info("re-building cached device vectors...")
        with db as q:
            m = self._build(q, db)
        _LOG.info("re-building cached device vectors... DONE!")
        self._matrix, self._stale = m, False
        return m

    async def get(self, db: Any, compact: bool = False) -> DeviceMatrix:
        """kb.py:879-893: same, with the heavy part in the default executor."""
        loop = asyncio.get_running_loop()
        m = self._matrix
        if m is not None and self._stale:
            m = await loop.run_in_executor(None, self._current, db)
        else:
            m = self._current(db)
        if m is not None and not (compact and m.has_tombstones):
            return m
        _LOG.info("re-building cached device vectors...")

        def heavy() -> DeviceMatrix:
            with db as q:
                return self._build(q, db)
        m = await loop.run_in_executor(None, heavy)
        _LOG.info("re-building cached device vectors... DONE!")
        self._matrix, self._stale = m, False
        return m

    def close(self) -> None:
        with self._mu:
            self._matrix = None
            self._stale = False
            if self._engine is not None:
                self._engine.close()
                self._engine = None
