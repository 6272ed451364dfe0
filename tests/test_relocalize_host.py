"""Host-side checks of the relocalization (no GPU): argument validation of its C entry points without a device, and
the seeded room workload with its candidate grid."""
import math
import os
import subprocess
import sys

import numpy as np

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
# b2s_icp_relocalize: H <= 0, N > 2304, a NaN angle increment, then a null handle
args = lambda K, H, n, inc: (None, p, p, p, 0.0, K, H, n, -3.1, inc, 100.0, 30, 1e-3, p, p, None, None, None)
assert L.b2s_icp_relocalize(*args(1, 0, 8, 0.1)) == bad
assert L.b2s_icp_relocalize(*args(1, -2, 8, 0.1)) == bad
assert L.b2s_icp_relocalize(*args(1, 4, 2305, 0.1)) == bad
assert b"2304" in L.b2s_last_error()
assert L.b2s_icp_relocalize(*args(1, 4, 8, nan)) == bad
assert b"angle_increment" in L.b2s_last_error()
assert L.b2s_icp_relocalize(*args(1, 4, 8, 0.1)) == bad
assert b"null handle" in L.b2s_last_error()
# b2s_relocalize_select: H <= 0, null pointers
assert L.b2s_relocalize_select(p, p, p, 1, 0, p, p, None) == bad
assert L.b2s_relocalize_select(None, p, p, 1, 4, p, p, None) == bad
assert L.b2s_relocalize_select(p, p, None, 1, 4, p, p, None) == bad
assert L.b2s_relocalize_select(p, p, p, 1, 4, None, p, None) == bad
assert b"null pointer" in L.b2s_last_error()
# b2s_icp_batch_f64_err: null pointers, more than 2304 source points
assert L.b2s_icp_batch_f64_err(None, None, 1, 8, 8, 30, 1e-3, None, None, p, None) == bad
assert L.b2s_icp_batch_f64_err(p, p, 1, 2305, 8, 30, 1e-3, p, None, p, None) == bad
assert b"2304" in L.b2s_last_error()
print("ok")
"""


def test_new_entry_points_validate_without_a_device():
    """In a child process from which the GPUs are hidden, so that the no-device path is checked on any machine."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK, ROOT], env=env, check=True, timeout=300,
                         capture_output=True, text=True)
    assert out.stdout.strip() == "ok"


def _inside(poly, x, y):
    """Winding number of the polygon around (x, y) is non-zero (independent of synth's even-odd test)."""
    ang = np.arctan2(poly[:, 1] - y, poly[:, 0] - x)
    d = np.diff(np.append(ang, ang[0]))
    d = (d + np.pi) % (2 * np.pi) - np.pi
    return abs(d.sum()) > np.pi


def test_room_relocalization_workload():
    from b2slam import synth
    a = synth.room_relocalization(9001, 8, 360)
    b = synth.room_relocalization(9001, 8, 360)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert a["ranges"].dtype == np.float32 and a["ranges"].shape == (8, 360)
    cand, poly = a["candidates"], a["poly"]
    assert cand.shape == (27324, 3) and cand.dtype == np.float64
    # the true poses and ranges are those of room_sequence, and the map that of room_map_observation
    xy, poses = synth.room_sequence(9001, 8, 360)
    assert np.array_equal(poses, a["poses"])
    phi = synth.beam_angles(360)
    np.testing.assert_allclose(xy[:, 0], a["ranges"] * np.cos(phi), rtol=1e-6, atol=1e-6)
    assert np.array_equal(a["obstacles_course"], synth.room_map_observation(9001, 8, 360)["obstacles_course"])
    # every candidate inside the room, at least 0.3 m from every wall; 36 yaws per cell, 10 degrees apart
    xy = np.unique(cand[:, :2], axis=0)
    assert len(xy) * 36 == len(cand)
    for x, y in xy:
        assert _inside(poly, x, y)
        for p, q in zip(poly, np.roll(poly, -1, axis=0)):
            e = q - p
            t = min(1.0, max(0.0, ((x - p[0]) * e[0] + (y - p[1]) * e[1]) / (e @ e)))
            assert math.hypot(x - p[0] - t * e[0], y - p[1] - t * e[1]) >= 0.3
    np.testing.assert_allclose(np.diff(np.unique(cand[:, 2])), math.radians(10), rtol=0, atol=1e-12)
    # the grid is 0.5 m on the origin
    assert np.allclose(xy / 0.5, np.round(xy / 0.5), rtol=0, atol=1e-12)
    # a finer grid has more candidates
    assert len(synth.room_relocalization(9001, 2, 360, xy_step=0.25)["candidates"]) > 3 * len(cand)
