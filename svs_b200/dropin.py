"""Make an imported `svs` package (Rhobota/svs 0.7.x) answer `retrieve` on the GPU.

    import svs, svs_b200
    svs_b200.install(svs)            # or install(svs, devices=[0, 1, 2, 3])
    kb = svs.KB('my.sqlite')         # unchanged public API, unchanged SQLite schema
    kb.retrieve('query', n=100)      # similarity + top-n now run in libsvsb200.so

What is replaced -- and nothing else (SURVEY.md section 8b):
  * `svs.kb._EmbeddingsMatrix` (reference src/svs/kb.py:856-893) gains a `.device` member, a
    `DeviceEmbeddingsMatrix`; `invalidate()` drops both caches, so every invalidation site of the
    reference (kb.py:984,1062,1086,1455,1523,1541) keeps working untouched.  The host NumPy cache
    stays in place (it is only filled if something still asks for it, e.g. the pairwise path of an
    install with pairwise=False, or a pairwise call the engine declines).
  * `KB.retrieve` (kb.py:1608-1640), `AsyncKB.retrieve` (kb.py:1171-1206): same orchestration --
    cache fetch, query embedding through the magnitude guard, SQL fetch of the n documents -- with the
    `superheavy()` closure (np.dot + get_top_k + emb_id_lookup) replaced by one engine call.
  * `AsyncKB.load` (kb.py:964-967) pre-warms the device cache instead of the host one.
  * `document_top_pairwise_scores` (kb.py:1642-1671, 1208-1243): same orchestration with `superheavy()` =
    np.dot(M, M.T) + get_top_pairs replaced by `svsb_top_pairs` (one device or several; SURVEY.md section 8f rank 2).
  * additive: `KB.retrieve_many` / `AsyncKB.retrieve_many` (one embedding call, one engine batch).

INTEGRATION.md shows the same change as a source patch to kb.py for a maintainer who prefers that.
"""
from __future__ import annotations

import asyncio
from typing import Any, List, Optional, Sequence

import numpy as np

from . import _lib
from .matrix import DeviceEmbeddingsMatrix
from .mutations import LoggingConnection, MutationLog

_ORIGINALS: dict = {}
# svsb_top_pairs refusals that the reference's np.dot(M, M.T) + get_top_pairs still answers (include/svsb200.h)
_PAIRS_DELEGATE = (_lib.SVSB_E_NOMEM, _lib.SVSB_E_INVALID)


class _Coalescer:
    """Dynamic batching of concurrent `AsyncKB.retrieve` calls (SURVEY.md section 8f rank 3).

    The reference runs every retrieve's `superheavy()` in the default executor without holding the KB lock
    (src/svs/kb.py:1190), so many can be in flight; on one GPU they would simply queue behind each other, one
    full pass over the matrix each.  Here the calls that arrive while a batch is on the GPU are collected and go out
    together as ONE `retrieve_many` (the tensor-core path from 4 queries up) -- results are bit-identical to the
    single-query kernels', so only the scheduling changes.  No added latency when idle: a lone call is issued at
    once.  Queries with different n share a batch (run at the largest n; a top-n list is a prefix of a top-k list).
    """

    def __init__(self) -> None:
        self._pending: List[Any] = []          # (matrix, vec, n, future)
        self._busy = False

    async def submit(self, matrix: Any, vec: np.ndarray, n: int) -> List[Any]:
        loop = asyncio.get_running_loop()
        fut = loop.create_future()
        self._pending.append((matrix, vec, n, fut))
        if not self._busy:
            self._busy = True
            loop.create_task(self._drain())
        return await fut

    async def _drain(self) -> None:
        loop = asyncio.get_running_loop()
        try:
            await asyncio.sleep(0)             # let every retrieve that is runnable in this tick join the batch
            while self._pending:
                matrix = self._pending[0][0]
                dim = self._pending[0][1].shape
                batch = [it for it in self._pending if it[0] is matrix and it[1].shape == dim]
                self._pending = [it for it in self._pending if not (it[0] is matrix and it[1].shape == dim)]
                # every caller's n is clipped to the row count first (get_top_k, src/svs/util.py:198-199): one caller's
                # oversized n must not size the whole batch's buffers
                rows = int(matrix.shape[0])
                k = max(min(max(int(it[2]), 0), rows) for it in batch)
                try:
                    if len(batch) == 1:
                        res = [await loop.run_in_executor(None, matrix.retrieve, batch[0][1], batch[0][2])]
                    else:
                        vecs = np.stack([it[1] for it in batch])
                        full = await loop.run_in_executor(None, matrix.retrieve_many, vecs, k)
                        res = [r[:max(it[2], 0)] for r, it in zip(full, batch)]
                    for it, r in zip(batch, res):
                        if not it[3].done():
                            it[3].set_result(r)
                except BaseException as ex:    # e.g. ValueError for a d mismatch: every caller of the batch sees it
                    for it in batch:
                        if not it[3].done():
                            it[3].set_exception(ex)
        finally:
            self._busy = False
            if self._pending:                  # arrivals that raced with the end of the loop
                self._busy = True
                loop.create_task(self._drain())


def install(svs_module: Any = None, devices: Optional[Sequence[int]] = None, normalize: bool = False,
            pairwise: Optional[bool] = None, coalesce: bool = True, prewarm: bool = True, incremental: bool = True) -> None:
    """Patch `svs` in place.  Idempotent.  `devices`: CUDA devices to row-shard the matrix over.
    `pairwise` (default on): also route document_top_pairwise_scores to the engine, on one device or several (each
    device runs a share of the pair search); False keeps the reference's host NumPy path for it.
    `coalesce`: batch concurrent AsyncKB.retrieve calls into one engine call (see _Coalescer).
    `prewarm` (default on): create the engine (= the CUDA context, ~2 s once per process on a B200 box,
    profiles/r01_first_query_probe.txt) on a background thread as soon as a KB object exists, instead of inside the
    first retrieve.
    `incremental` (default on): bulk adds / deletes UPDATE the device matrix (append + tombstone) instead of forcing the
    full rebuild the reference does (kb.py:1062, 1086, 1523, 1541): the querier's connection is wrapped so that every
    `INSERT INTO embeddings` / `DELETE FROM embeddings` of a committed transaction is logged (svs_b200.mutations)."""
    if pairwise is None:
        pairwise = True
    if svs_module is None:
        import svs as svs_module                         # type: ignore  (the host application)
    kb = svs_module.kb if hasattr(svs_module, "kb") else __import__(svs_module.__name__ + ".kb", fromlist=["kb"])
    if _ORIGINALS.get("module") is kb:
        return
    host_cls = kb._EmbeddingsMatrix
    log = kb._LOG

    class _EmbeddingsMatrix(host_cls):                   # type: ignore
        """Host cache (pairwise path, untouched) + device cache (retrieve path)."""

        def __init__(self) -> None:
            super().__init__()
            self.device = DeviceEmbeddingsMatrix(devices, normalize, incremental)
            self.coalescer = _Coalescer() if coalesce else None
            if prewarm:
                self.device.prewarm()

        def invalidate(self) -> None:
            super().invalidate()
            self.device.invalidate()

    def _fetch_docs(q: Any, emb_ids: List[Any], n: int) -> List[Any]:
        res = []
        for score, emb_id in emb_ids:
            doc_id = q.fetch_doc_with_emb_id(emb_id)
            res.append({'score': score, 'doc': q.fetch_doc(doc_id, include_embedding=False)})
        log.info(f"retrieved top {n} documents")
        return res

    def retrieve(self: Any, query: str, n: int) -> List[Any]:
        log.info(f"retrieving {n} documents with query string: {query}")
        assert self.db is not None
        matrix = self.embeddings_matrix.device.get_sync(self.db)
        func = self._get_embedding_func()
        awaitable = func([query])
        assert asyncio.iscoroutine(awaitable)
        query_vec = np.array(asyncio.run_coroutine_threadsafe(awaitable, self.loop).result()[0], dtype=np.float32)
        log.info("got embedding for query!")
        emb_ids = matrix.retrieve(query_vec, n)          # superheavy(), on the GPU
        log.info(f"computed {matrix.shape[0]} cosine similarities")
        with self.db as q:
            return _fetch_docs(q, emb_ids, n)

    async def aretrieve(self: Any, query: str, n: int) -> List[Any]:
        log.info(f"retrieving {n} documents with query string: {query}")
        loop = asyncio.get_running_loop()
        async with self._get_lock():
            db = await self._ensure_db()
            matrix = await self.embeddings_matrix.device.get(db)
        func = await self._get_embedding_func()
        query_vec = np.array((await func([query]))[0], dtype=np.float32)
        log.info("got embedding for query!")
        # the lock is NOT held here (as in the reference): `matrix` pins its generation, so a
        # concurrent bulk_add/bulk_del may invalidate the cache while this runs
        co = getattr(self.embeddings_matrix, "coalescer", None)
        if co is not None and query_vec.ndim == 1 and query_vec.shape[0] == matrix.shape[1] and matrix.shape[0] > 0:
            emb_ids = await co.submit(matrix, query_vec, n)      # joins whatever else is waiting for the GPU
        else:                                                    # shape errors surface exactly as in the single path
            emb_ids = await loop.run_in_executor(None, matrix.retrieve, query_vec, n)
        log.info(f"computed {matrix.shape[0]} cosine similarities")
        async with self._get_lock():
            db = await self._ensure_db()
            async with db as q:
                return await loop.run_in_executor(None, _fetch_docs, q, emb_ids, n)

    def retrieve_many(self: Any, queries: List[str], n: int) -> List[List[Any]]:
        """ADDITIVE API (the reference has none; its equivalent is a Python loop over retrieve, kb.py:1608-1640):
        embed all queries with ONE call of the embedding function (it takes a list, types.py EmbeddingFunc), run ONE
        engine batch, then fetch the documents.  Result j equals `retrieve(queries[j], n)`."""
        log.info(f"retrieving {n} documents for each of {len(queries)} query strings")
        assert self.db is not None
        matrix = self.embeddings_matrix.device.get_sync(self.db)
        if not queries:
            return []
        func = self._get_embedding_func()
        awaitable = func(list(queries))
        assert asyncio.iscoroutine(awaitable)
        vecs = np.array(asyncio.run_coroutine_threadsafe(awaitable, self.loop).result(), dtype=np.float32)
        log.info("got embeddings for the queries!")
        all_ids = matrix.retrieve_many(vecs, n)
        log.info(f"computed {matrix.shape[0]} x {len(queries)} cosine similarities")
        with self.db as q:
            return [_fetch_docs(q, emb_ids, n) for emb_ids in all_ids]

    async def aretrieve_many(self: Any, queries: List[str], n: int) -> List[List[Any]]:
        log.info(f"retrieving {n} documents for each of {len(queries)} query strings")
        loop = asyncio.get_running_loop()
        async with self._get_lock():
            db = await self._ensure_db()
            matrix = await self.embeddings_matrix.device.get(db)
        if not queries:
            return []
        func = await self._get_embedding_func()
        vecs = np.array(await func(list(queries)), dtype=np.float32)
        log.info("got embeddings for the queries!")
        all_ids = await loop.run_in_executor(None, matrix.retrieve_many, vecs, n)
        log.info(f"computed {matrix.shape[0]} x {len(queries)} cosine similarities")
        async with self._get_lock():
            db = await self._ensure_db()
            async with db as q:
                return await loop.run_in_executor(None, lambda: [_fetch_docs(q, emb_ids, n) for emb_ids in all_ids])

    def _pair_docs(q: Any, pairwise_scores: List[Any], n: int) -> List[Any]:
        # the reference's document fetch for pairs, verbatim in behaviour (kb.py:1658-1671)
        emb_id_to_doc_id = {}
        for emb_id in set(emb_id for _, e1, e2 in pairwise_scores for emb_id in (e1, e2)):
            emb_id_to_doc_id[emb_id] = q.fetch_doc_with_emb_id(emb_id)
        doc_lookup = {}
        for doc_id in emb_id_to_doc_id.values():
            doc_lookup[doc_id] = q.fetch_doc(doc_id, include_embedding=False)
        res = [(score, doc_lookup[emb_id_to_doc_id[e1]], doc_lookup[emb_id_to_doc_id[e2]]) for score, e1, e2 in pairwise_scores]
        log.info(f"retrieved top {n} document pairs")
        return res

    def top_pairwise(self: Any, n: int) -> List[Any]:
        """document_top_pairwise_scores (kb.py:1642-1671) with `superheavy()` = np.dot(M, M.T) + get_top_pairs replaced by
        one engine call that never materialises the N x N scores."""
        assert self.db is not None
        matrix = self.embeddings_matrix.device.get_sync(self.db, compact=True)   # the pair kernels want no tombstones
        n_docs = matrix.shape[0]
        log.info(f"computing pairwise similarity over {n_docs} documents")
        try:
            pairwise_scores = matrix.top_pairs(n)
        except _lib.EngineError as ex:
            if ex.code not in _PAIRS_DELEGATE:
                raise
            # The engine's pair list has fixed capacity (millions of near-tied pairs -- e.g. thousands of duplicate
            # documents, the typical use of this API -- or n > 2^22 overflow it) and its fp16 coarse pass needs rows near
            # unit norm.  The reference answers all of these: hand the call to its own host path (the host cache is kept).
            log.info(f"engine declined the pairwise query ({ex}); using the reference's host path")
            return _ORIGINALS["KB.pairs"](self, n)
        log.info(f"computed {n_docs * n_docs} pairwise cosine similarities")
        with self.db as q:
            return _pair_docs(q, pairwise_scores, n)

    async def atop_pairwise(self: Any, n: int) -> List[Any]:
        loop = asyncio.get_running_loop()
        async with self._get_lock():
            db = await self._ensure_db()
            matrix = await self.embeddings_matrix.device.get(db, compact=True)
        n_docs = matrix.shape[0]
        log.info(f"computing pairwise similarity over {n_docs} documents")
        try:
            pairwise_scores = await loop.run_in_executor(None, matrix.top_pairs, n)
        except _lib.EngineError as ex:
            if ex.code not in _PAIRS_DELEGATE:
                raise
            log.info(f"engine declined the pairwise query ({ex}); using the reference's host path")
            return await _ORIGINALS["AsyncKB.pairs"](self, n)
        log.info(f"computed {n_docs * n_docs} pairwise cosine similarities")
        async with self._get_lock():
            db = await self._ensure_db()
            async with db as q:
                return await loop.run_in_executor(None, _pair_docs, q, pairwise_scores, n)

    async def aload(self: Any) -> None:
        async with self._get_lock():
            db = await self._ensure_db()
            await self.embeddings_matrix.device.get(db)

    # ---- mutation log: the querier's connection tells the log about embeddings inserts / deletes; _DB.__exit__ commits
    #      or drops the transaction's records (kb.py:793-821).  __aenter__ / __aexit__ call these through `self`.
    db_cls = getattr(kb, "_DB", None)
    orig_enter = db_cls.__enter__ if db_cls is not None else None
    orig_exit = db_cls.__exit__ if db_cls is not None else None

    def db_enter(self: Any) -> Any:
        q = orig_enter(self)
        mlog = self.__dict__.get("_svsb_log")
        if mlog is None:
            mlog = self.__dict__["_svsb_log"] = MutationLog()
        mlog.begin()
        q.conn = LoggingConnection(q.conn, mlog)
        return q

    def db_exit(self: Any, exc_type: Any, exc_val: Any, exc_tb: Any) -> Any:
        mlog = self.__dict__.get("_svsb_log")
        try:
            ret = orig_exit(self, exc_type, exc_val, exc_tb)
        except BaseException:
            if mlog is not None:
                mlog.rollback()                          # the commit itself failed
            raise
        if mlog is not None:
            if exc_type is None:
                mlog.commit()
            else:
                mlog.rollback()
        return ret

    def kb_close(self: Any, *a: Any, **kw: Any) -> Any:
        try:
            return _ORIGINALS["KB.close"](self, *a, **kw)
        finally:
            self.embeddings_matrix.device.close()        # invalidate() keeps the (stale) matrix resident; close frees it

    async def akb_close(self: Any, *a: Any, **kw: Any) -> Any:
        try:
            return await _ORIGINALS["AsyncKB.close"](self, *a, **kw)
        finally:
            self.embeddings_matrix.device.close()

    _ORIGINALS.update({
        "_DB": db_cls, "_DB.__enter__": orig_enter, "_DB.__exit__": orig_exit,
        "KB.close": getattr(kb.KB, "close", None), "AsyncKB.close": getattr(kb.AsyncKB, "close", None),
        "module": kb, "_EmbeddingsMatrix": host_cls, "KB.retrieve": kb.KB.retrieve,
        "AsyncKB.retrieve": kb.AsyncKB.retrieve, "AsyncKB.load": kb.AsyncKB.load,
        "KB.pairs": kb.KB.document_top_pairwise_scores, "AsyncKB.pairs": kb.AsyncKB.document_top_pairwise_scores,
    })
    kb._EmbeddingsMatrix = _EmbeddingsMatrix
    kb.KB.retrieve = retrieve
    kb.AsyncKB.retrieve = aretrieve
    kb.AsyncKB.load = aload
    if pairwise:
        kb.KB.document_top_pairwise_scores = top_pairwise
        kb.AsyncKB.document_top_pairwise_scores = atop_pairwise
    kb.KB.retrieve_many = retrieve_many                  # additive: batched retrieve
    kb.AsyncKB.retrieve_many = aretrieve_many
    if incremental and db_cls is not None:
        db_cls.__enter__ = db_enter
        db_cls.__exit__ = db_exit
    if _ORIGINALS["KB.close"] is not None:
        kb.KB.close = kb_close
    if _ORIGINALS["AsyncKB.close"] is not None:
        kb.AsyncKB.close = akb_close


def uninstall() -> None:
    """Undo install()."""
    kb = _ORIGINALS.get("module")
    if kb is None:
        return
    kb._EmbeddingsMatrix = _ORIGINALS["_EmbeddingsMatrix"]
    kb.KB.retrieve = _ORIGINALS["KB.retrieve"]
    kb.AsyncKB.retrieve = _ORIGINALS["AsyncKB.retrieve"]
    kb.AsyncKB.load = _ORIGINALS["AsyncKB.load"]
    kb.KB.document_top_pairwise_scores = _ORIGINALS["KB.pairs"]
    kb.AsyncKB.document_top_pairwise_scores = _ORIGINALS["AsyncKB.pairs"]
    for cls in (kb.KB, kb.AsyncKB):
        if "retrieve_many" in cls.__dict__:
            delattr(cls, "retrieve_many")
    if _ORIGINALS.get("_DB") is not None:
        _ORIGINALS["_DB"].__enter__ = _ORIGINALS["_DB.__enter__"]
        _ORIGINALS["_DB"].__exit__ = _ORIGINALS["_DB.__exit__"]
    if _ORIGINALS.get("KB.close") is not None:
        kb.KB.close = _ORIGINALS["KB.close"]
    if _ORIGINALS.get("AsyncKB.close") is not None:
        kb.AsyncKB.close = _ORIGINALS["AsyncKB.close"]
    _ORIGINALS.clear()
