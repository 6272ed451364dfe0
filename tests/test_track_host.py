"""Host-side checks of pose tracking (no GPU): argument and shape validation of ICP.track and of its C entry points
without a device, and the agreement of their ctypes signatures with the header."""
import os
import re
import subprocess
import sys

from conftest import ROOT
from b2slam import _lib

_NO_DEVICE_CHECK = """
import ctypes, math, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import b2slam
from b2slam import _lib
L = _lib.lib()
assert _lib.device_count() == 0
bad = _lib.ERR_INVALID_ARG
d = ctypes.c_double(0.0)
p = ctypes.byref(d)
nan = float("nan")
# b2s_icp_track: K < 1, H <= 0, K * H > 2^31 - 1, N > 2304, a NaN angle increment, then a null handle
def args(K=2, H=4, n=8, inc=0.1):
    return (None, p, p, p, 0.0, K, H, n, -3.1, inc, 100.0, 30, 1e-3, p, p, None, None, None, None)
for kw in (dict(K=0), dict(K=-1), dict(H=0), dict(K=70000, H=40000)):
    assert L.b2s_icp_track(*args(**kw)) == bad, kw
    assert L.b2s_last_error() == b"b2s_icp_track: bad sizes", kw
assert L.b2s_icp_track(*args(n=2305)) == bad
assert b"2304" in L.b2s_last_error()
assert L.b2s_icp_track(*args(inc=nan)) == bad
assert L.b2s_last_error() == b"b2s_icp_track: angle_increment"
assert L.b2s_icp_track(*args()) == bad
assert L.b2s_last_error() == b"b2s_icp_track: null handle"
# b2s_track_step: H <= 0, a negative stage, null pointers, odometry without next_prior and the reverse
def step(H=4, stage=0, T=p, odo=None, nxt=None, joint=p):
    return L.b2s_track_step(T, p, odo, H, stage, p, p, nxt, joint, p, None)
assert step(H=0) == bad and b"bad sizes" in L.b2s_last_error()
assert step(stage=-1) == bad and b"bad sizes" in L.b2s_last_error()
assert step(T=None) == bad and b"null pointer" in L.b2s_last_error()
assert step(joint=None) == bad and b"null pointer" in L.b2s_last_error()
assert step(odo=p) == bad and b"go together" in L.b2s_last_error()
assert step(nxt=p) == bad and b"go together" in L.b2s_last_error()
# b2s_track_select: H <= 0, null pointers
assert L.b2s_track_select(p, p, 0, p, None) == bad and b"bad sizes" in L.b2s_last_error()
assert L.b2s_track_select(None, p, 4, p, None) == bad and b"null pointer" in L.b2s_last_error()
assert L.b2s_track_select(p, p, 4, None, None) == bad and b"null pointer" in L.b2s_last_error()

# ICP.track's own shape checks run before the library is called; an object without a device handle reaches the
# library's null-handle error once the shapes are right
icp = b2slam.ICP.__new__(b2slam.ICP)
icp._L, icp._h, icp.max_iter, icp.tolerance = L, None, 30, 1e-3
ranges = np.ones((3, 360), dtype=np.float32)
starts = np.zeros((5, 3))
def raises(text, *a, **kw):
    try:
        icp.track(*a, **kw)
    except ValueError as e:
        assert text in str(e), (text, str(e))
        return
    raise AssertionError("no ValueError for %r" % (text,))
pi = math.pi
raises("expected ranges (K,N)", ranges[:0], starts, -pi, pi)
raises("expected ranges (K,N)", ranges[0], starts, -pi, pi)
raises("expected ranges (K,N)", ranges[:, :0], starts, -pi, pi)
raises("expected starts (H,3)", ranges, starts[:0], -pi, pi)
raises("expected starts (H,3)", ranges, starts[:, :2], -pi, pi)
raises("expected starts (H,3)", ranges, starts[None], -pi, pi)
raises("one-beam scan", ranges[:, :1], starts, -pi, pi)
raises("exceeds 2^31 - 1", np.ones((70000, 2), dtype=np.float32), np.zeros((40000, 3)), -pi, pi)
raises("2304", np.ones((2, 2305), dtype=np.float32), starts, -pi, pi)
raises("null handle", ranges, starts, -pi, pi)
raises("null handle", ranges, starts[0], -pi, pi)
print("ok")
"""


def test_track_validates_without_a_device():
    """In a child process from which the GPUs are hidden, so that the no-device path is checked on any machine."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK, ROOT], env=env, check=True, timeout=300,
                         capture_output=True, text=True)
    assert out.stdout.strip() == "ok"


def test_track_signatures_match_the_header():
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b2slam.h")).read(), flags=re.S)
    for name in ("b2s_icp_track", "b2s_track_step", "b2s_track_select"):
        m = re.search(r"\bint\s+%s\s*\(([^)]*)\)" % name, text)
        assert m, name
        assert len(m.group(1).split(",")) == len(_lib.SIGNATURES[name][1]), name
        assert _lib.SIGNATURES[name][0] is _lib.SIGNATURES["b2s_icp_relocalize"][0], name
