"""install() with several devices routes document_top_pairwise_scores to the engine (svsb_top_pairs answers it on
multi-device engines); pairwise=False keeps the reference's host path.  No GPU: the recording fake of
test_host_logic.py stands in for the Engine."""
import asyncio
import os
import shutil
import sqlite3
import types

import pytest

from _util import GOLDEN
from test_host_logic import FakeEngine, _fake_svs_module

import svs_b200
from svs_b200 import matrix as matrix_mod


class _DB:
    """`with db as q:` yields a querier with .conn and the two document fetches _pair_docs uses (kb.py:1658-1671)."""

    def __init__(self, conn):
        self.conn = conn

    def __enter__(self):
        return types.SimpleNamespace(conn=self.conn, fetch_doc_with_emb_id=lambda emb_id: 1000 + emb_id,
                                     fetch_doc=lambda doc_id, include_embedding=False: {"id": doc_id})

    def __exit__(self, *a):
        return False


@pytest.fixture
def engines_made(monkeypatch):
    made = []

    def factory(devices=None):
        e = FakeEngine(devices)
        e.devices = devices
        made.append(e)
        return e
    monkeypatch.setattr(matrix_mod, "Engine", factory)
    return made


def test_multi_device_install_routes_pairwise_to_the_engine(engines_made, tmp_path):
    dst = tmp_path / "kb.sqlite"
    shutil.copy(os.path.join(GOLDEN, "kb_small.sqlite"), dst)
    mod = _fake_svs_module()
    host_sync, host_async = mod.kb.KB.document_top_pairwise_scores, mod.kb.AsyncKB.document_top_pairwise_scores
    svs_b200.install(mod, devices=[0, 1], prewarm=False)
    try:
        assert mod.kb.KB.document_top_pairwise_scores is not host_sync
        assert mod.kb.AsyncKB.document_top_pairwise_scores is not host_async
        kb = mod.kb.KB()
        kb.db = _DB(sqlite3.connect(str(dst), check_same_thread=False))
        res = kb.document_top_pairwise_scores(1)
        eng = engines_made[0]
        assert eng.devices == [0, 1]
        assert res == [(0.5, {"id": 1000 + int(eng.ids[0])}, {"id": 1000 + int(eng.ids[1])})]   # the fake engine's pair
    finally:
        svs_b200.uninstall()


def test_pairwise_false_keeps_the_host_path_on_several_devices(engines_made):
    mod = _fake_svs_module()
    svs_b200.install(mod, devices=[0, 1], pairwise=False, prewarm=False)
    try:
        assert mod.kb.KB().document_top_pairwise_scores(1) == "host pairs"
        assert asyncio.run(mod.kb.AsyncKB().document_top_pairwise_scores(1)) == "host pairs"
    finally:
        svs_b200.uninstall()
    assert engines_made == []
