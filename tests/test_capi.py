"""C-ABI surface checks that need no GPU: the library loads, exports every symbol that
include/b2slam.h declares, the ctypes table matches the header, and compute entry points
fail loudly (never fall back) when no CUDA device is present."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np

from conftest import ROOT
from b2slam import _lib

HEADER = os.path.join(ROOT, "include", "b2slam.h")


def _declared():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b2s_[a-z0-9_]+)\s*\(", text)))


def test_library_is_built_in_tree():
    assert os.path.isfile(_lib.LIB_PATH), "run __graft_entry__.build()"
    assert os.path.dirname(_lib.LIB_PATH).startswith(ROOT)


def test_every_declared_symbol_is_exported():
    L = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), "missing export %s" % n


def test_ctypes_table_matches_header():
    assert sorted(_lib.SIGNATURES) == _declared()


def test_header_cites_reference_lines():
    text = open(HEADER).read()
    for cite in ("[ICP]:38-88", "[ICP]:90-114", "[ICP]:149-179", "[MAP]:22-51", "[BRES]:2-58",
                 "[SLAM]:270-271"):
        assert cite in text


def test_status_strings_and_version():
    L = _lib.lib()
    assert L.b2s_version() >= 100
    assert L.b2s_status_string(0) == b"ok"
    assert b"non-finite" in L.b2s_status_string(_lib.ERR_NONFINITE)


def test_argument_validation_needs_no_device():
    L = _lib.lib()
    assert L.b2s_grid_raycast(None, None, 4, 4, 1.0, 0.0, 0.0, None, None, None, None, 1, 1,
                              None, None) == _lib.ERR_INVALID_ARG
    assert b"null pointer" in L.b2s_last_error()
    assert L.b2s_icp_batch_f32(None, None, 1, 0, 8, 30, 1e-3, None, None, None) == _lib.ERR_INVALID_ARG
    assert L.b2s_tune(b"grid_variant", 7) == _lib.ERR_INVALID_ARG
    assert L.b2s_tune(b"nope", 1) == _lib.ERR_INVALID_ARG
    # the ICP search switches: every documented value is accepted, the next one is not; the defaults are restored
    for key, good, bad, default in ((b"icp_prune", (0, 1, 2, 3, 4), 5, 4), (b"icp_block", (0, 8, 16, 32), 12, 0),
                                    (b"icp_layout", (0, 1, 2), 3, 2), (b"icp_src_per_thread", (0, 2, 3, 4), 1, 0)):
        for v in good:
            assert L.b2s_tune(key, v) == 0, (key, v)
        assert L.b2s_tune(key, bad) == _lib.ERR_INVALID_ARG, key
        assert L.b2s_tune(key, default) == 0


_NO_DEVICE_CHECK = """
import ctypes, sys
import pytest
sys.path.insert(0, sys.argv[1])
import b2slam
from b2slam import _lib
assert _lib.device_count() == 0
with pytest.raises(_lib.B2SlamError):
    b2slam.ICP()
with pytest.raises(_lib.B2SlamError):
    b2slam.Mapping(200, 200, 0.1)
with pytest.raises(_lib.B2SlamError):
    from b2slam import bresenham as drawing
    drawing.bresenham([0, 0], [3, 1])
h = ctypes.c_void_p()
assert _lib.lib().b2s_mapping_create(ctypes.byref(h), 8, 8, 0.1, 20.0, 0.01, 10.0, -1) == _lib.ERR_CUDA
"""


def test_no_cpu_fallback_without_device():
    """In a child process from which the GPUs are hidden, so that the no-device path is checked on any machine."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK, ROOT], env=env, check=True, timeout=300)


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "a-2d-lidar-based-slam-system-for-wheeled-mobile-robots_b200")
    bad = re.compile(r"^\s*(from|import)\s+oracle\b|liboracle|oracle\.(corc|pyref)", re.M)
    seen = 0
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                seen += 1
                assert not bad.search(open(os.path.join(dirpath, f)).read()), f
    assert seen >= 8
