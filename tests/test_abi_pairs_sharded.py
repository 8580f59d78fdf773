"""The sharded pair search's entry points (include/svsb200.h svsb_pairs_*) are declared, exported and bound."""
import ctypes
import os
import re

from _util import ROOT

PAIRS = ("svsb_pairs_export", "svsb_pairs_connect", "svsb_pairs_connect_local", "svsb_pairs_local", "svsb_pairs_merge",
         "svsb_pairs_disconnect")


def test_header_declares_library_exports_and_binding_binds_the_pair_entry_points():
    from svs_b200 import _lib, build
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "svsb200.h")).read(), flags=re.S)
    lib = ctypes.CDLL(build.build())
    for name in PAIRS:
        assert re.search(rf"\bint {name}\s*\(", text), name
        assert hasattr(lib, name), name
        assert name in _lib.SIGNATURES, name
    assert re.search(r"#define SVSB_PAIRS_DESC_BYTES (\d+)", text).group(1) == str(_lib.PAIRS_DESC_BYTES)
