"""Mutation log of the `embeddings` table: what lets the device cache be UPDATED instead of rebuilt.

The reference invalidates its vector cache after every bulk add / delete (src/svs/kb.py:1062, 1086, 1523, 1541) and the
next `retrieve` rebuilds the whole matrix from SQLite (kb.py:573-618) -- seconds for a million rows even with this
package's loader, for a one-document add.  `_EmbeddingsMatrix.invalidate()` carries no arguments, so the drop-in
captures the mutations where they happen: every statement of the reference that changes the table

    INSERT INTO embeddings (embedding) VALUES (?);      kb.py:310 (add_doc), kb.py:557 (set_doc_embedding)
    DELETE FROM embeddings WHERE id = ?;                kb.py:403 (del_doc),  kb.py:548 (set_doc_embedding)

goes through `_Querier.conn.execute`; `install()` hands the querier a thin connection proxy (`LoggingConnection`) that
records (id, blob) / id per transaction, and `_DB.__exit__` (kb.py:804-821) turns the transaction's records into
committed ones on commit and drops them on rollback.  On the next `retrieve` the committed records are applied with
`svsb_apply_mutations` (append + tombstone).  Anything the log cannot vouch for -- another kind of statement touching
the table, an inconsistency, too many bytes to keep -- POISONS it and the cache falls back to the full rebuild, which
is correct by construction.  rowids may be recycled (INTEGER PRIMARY KEY without AUTOINCREMENT, kb.py:80-83: delete the
newest row, insert, and the same id comes back with a different blob -- the reference's own tests do it,
tests/test_kb.py:1592-1595); the log is keyed by what happened, not by id diffs, so that is an ordinary
"tombstone + append".
"""
from __future__ import annotations

import threading
from typing import Any, Dict, List, Optional, Tuple

_INSERT = "INSERT INTO EMBEDDINGS (EMBEDDING) VALUES (?);"
_DELETE = "DELETE FROM EMBEDDINGS WHERE ID = ?;"
_WRITE_VERBS = ("INSERT", "DELETE", "UPDATE", "REPLACE", "DROP", "ALTER", "CREATE", "VACUUM")



def compaction_due(physical: int, dead: int) -> bool:
    """Past this fraction of dead (tombstoned) rows among `physical` rows, compacting is the better deal than further
    incremental updates: every query still streams the dead rows."""
    return dead > 64 and dead * 4 > physical


class MutationLog:
    """Per-database log.  Thread-safe: AsyncKB runs the querier in executor threads."""

    def __init__(self, max_bytes: int = 256 << 20) -> None:
        self.max_bytes = max_bytes
        self._mu = threading.Lock()
        self._txn: Optional[List[Tuple[str, int, Optional[bytes]]]] = None
        self._adds: Dict[int, bytes] = {}         # committed inserts not yet applied, insertion order
        self._dels: List[int] = []                # committed deletes of rows that pre-date the log
        self._bytes = 0
        self._poison: Optional[str] = None

    # ---- transaction scope (called by the _DB hooks) --------------------------------------------------
    def begin(self) -> None:
        with self._mu:
            self._txn = []

    def record_insert(self, emb_id: int, blob: bytes) -> None:
        with self._mu:
            if self._txn is not None:
                self._txn.append(("ins", int(emb_id), bytes(blob)))
            else:
                self._poison = "insert outside a transaction"

    def record_delete(self, emb_id: int) -> None:
        with self._mu:
            if self._txn is not None:
                self._txn.append(("del", int(emb_id), None))
            else:
                self._poison = "delete outside a transaction"

    def poison(self, why: str) -> None:
        """Something changed the table in a way the log does not model: only a full rebuild is safe."""
        with self._mu:
            self._poison = why
            self._adds.clear(); self._dels.clear(); self._bytes = 0

    def rollback(self) -> None:
        with self._mu:
            self._txn = None

    def commit(self) -> None:
        with self._mu:
            txn, self._txn = self._txn, None
            if not txn or self._poison:
                return
            for op, emb_id, blob in txn:
                if op == "ins":
                    if emb_id in self._adds:
                        self._poison = f"id {emb_id} inserted twice"
                        break
                    self._adds[emb_id] = blob             # type: ignore[assignment]
                    self._bytes += len(blob or b"")
                elif emb_id in self._adds:                 # inserted and deleted before anyone looked
                    self._bytes -= len(self._adds.pop(emb_id))
                elif emb_id in self._dels:
                    self._poison = f"id {emb_id} deleted twice"
                    break
                else:
                    self._dels.append(emb_id)
            if self._bytes > self.max_bytes:
                self._poison = f"more than {self.max_bytes} bytes of pending rows"
            if self._poison:
                self._adds.clear(); self._dels.clear(); self._bytes = 0

    # ---- consumer (DeviceEmbeddingsMatrix) ------------------------------------------------------------
    def take(self) -> Optional[Tuple[List[int], List[int], List[bytes]]]:
        """(deleted ids, inserted ids, their blobs) committed since the last take -- or None if only a rebuild is safe.
        Either way the log starts afresh (the caller is about to bring the cache up to date one way or the other)."""
        with self._mu:
            poisoned = self._poison is not None
            dels, adds = self._dels, self._adds
            self._adds, self._dels, self._bytes, self._poison = {}, [], 0, None
            if poisoned:
                return None
            return list(dels), list(adds.keys()), list(adds.values())

    def pending(self) -> Tuple[int, int, Optional[str]]:
        with self._mu:
            return len(self._dels), len(self._adds), self._poison


class LoggingConnection:
    """What `_Querier.conn` is after install(): forwards everything to the sqlite3 connection and tells the log about
    the two statements that change `embeddings`."""

    def __init__(self, conn: Any, log: MutationLog) -> None:
        self._conn = conn
        self._log = log

    def execute(self, sql: str, parameters: Any = ()) -> Any:
        res = self._conn.execute(sql, parameters)
        if "embeddings" in sql or "EMBEDDINGS" in sql:
            norm = " ".join(sql.split()).upper()
            if norm == _INSERT:
                if res.lastrowid is None:
                    self._log.poison("insert without a rowid")
                else:
                    self._log.record_insert(res.lastrowid, parameters[0])
            elif norm == _DELETE:
                if res.rowcount == 1:
                    self._log.record_delete(parameters[0])
                elif res.rowcount != 0:
                    self._log.poison("delete touched several rows")
            elif norm.startswith(_WRITE_VERBS) and not norm.startswith("UPDATE DOCS"):
                self._log.poison("unmodelled statement on the embeddings table: " + norm[:60])
        return res

    def __getattr__(self, name: str) -> Any:
        return getattr(self._conn, name)
