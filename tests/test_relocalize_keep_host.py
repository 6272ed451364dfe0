"""Host-side checks of the coarse-to-fine relocalization (no GPU): argument validation of its C entry points without a
device."""
import os
import subprocess
import sys

from conftest import ROOT

_NO_DEVICE_CHECK = """
import ctypes, sys
sys.path.insert(0, sys.argv[1])
from b2slam import _lib
L = _lib.lib()
assert _lib.device_count() == 0
bad = _lib.ERR_INVALID_ARG
d = ctypes.c_double(0.0)
p = ctypes.byref(d)
nan = float("nan")
# b2s_icp_relocalize_keep: keep < 1, coarse_iters outside [1, max_iter], K * min(keep, H) > 2^31 - 1, then the checks
# of b2s_icp_relocalize under its own name
def args(K=1, H=4, n=8, inc=0.1, max_iter=30, keep=2, coarse=5):
    return (None, p, p, p, 0.0, K, H, n, -3.1, inc, 100.0, max_iter, 1e-3, keep, coarse, p, p, None, None, None, None)
assert L.b2s_icp_relocalize_keep(*args(keep=0)) == bad
assert b"keep must be >= 1" in L.b2s_last_error()
assert L.b2s_icp_relocalize_keep(*args(keep=-3)) == bad
assert L.b2s_icp_relocalize_keep(*args(coarse=0)) == bad
assert b"coarse_iters" in L.b2s_last_error()
assert L.b2s_icp_relocalize_keep(*args(coarse=31)) == bad
assert b"coarse_iters" in L.b2s_last_error()
assert L.b2s_icp_relocalize_keep(*args(K=70000, H=40000, keep=40000)) == bad
assert b"2^31 - 1" in L.b2s_last_error()
assert L.b2s_icp_relocalize_keep(*args(H=0)) == bad
assert L.b2s_last_error() == b"b2s_icp_relocalize_keep: bad sizes"
assert L.b2s_icp_relocalize_keep(*args(n=2305)) == bad
assert b"2304" in L.b2s_last_error()
assert L.b2s_icp_relocalize_keep(*args(inc=nan)) == bad
assert b"angle_increment" in L.b2s_last_error()
assert L.b2s_icp_relocalize_keep(*args()) == bad
assert L.b2s_last_error() == b"b2s_icp_relocalize_keep: null handle"
# the exhaustive call keeps its own texts
assert L.b2s_icp_relocalize(None, p, p, p, 0.0, 1, 4, 8, -3.1, 0.1, 100.0, 30, 1e-3, p, p, None, None, None) == bad
assert L.b2s_last_error() == b"b2s_icp_relocalize: null handle"
# b2s_relocalize_keep: H <= 0, keep < 1, K * H > 2^31 - 1, null pointers
assert L.b2s_relocalize_keep(p, p, 1, 0, 1, p, p, None) == bad
assert L.b2s_relocalize_keep(p, p, 1, 4, 0, p, p, None) == bad
assert L.b2s_relocalize_keep(p, p, 70000, 40000, 1, p, p, None) == bad
assert L.b2s_relocalize_keep(None, p, 1, 4, 1, p, p, None) == bad
assert L.b2s_relocalize_keep(p, p, 1, 4, 1, None, p, None) == bad
assert L.b2s_relocalize_keep(p, p, 1, 4, 1, p, None, None) == bad
assert b"null pointer" in L.b2s_last_error()
# b2s_relocalize_select_kept: keep <= 0, null pointers
assert L.b2s_relocalize_select_kept(p, p, p, p, 1, 0, p, p, None) == bad
assert L.b2s_relocalize_select_kept(p, p, p, None, 1, 4, p, p, None) == bad
assert L.b2s_relocalize_select_kept(None, p, p, p, 1, 4, p, p, None) == bad
assert b"null pointer" in L.b2s_last_error()
# no scans: nothing to do, nothing dereferenced
assert L.b2s_relocalize_keep(None, None, 0, 4, 1, None, None, None) == 0
assert L.b2s_relocalize_select_kept(None, None, None, None, 0, 4, None, None, None) == 0
print("ok")
"""


def test_new_entry_points_validate_without_a_device():
    """In a child process from which the GPUs are hidden, so that the no-device path is checked on any machine."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK, ROOT], env=env, check=True, timeout=300,
                         capture_output=True, text=True)
    assert out.stdout.strip() == "ok"

