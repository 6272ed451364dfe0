"""Host-side checks of the map observation (no GPU): argument validation of the new C entry points without a device,
the seeded room workload and the composed reference of the map observation, which the GPU tests also use."""
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
# b2s_virtual_scan_batch: null obstacles / poses / outputs, bad sizes, a missing or misaligned beam table
assert L.b2s_virtual_scan_batch(None, None, 5, p, 1, -3.1, 0.1, 8, 100.0, None, p, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, None, 1, -3.1, 0.1, 8, 100.0, None, p, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, p, 1, -3.1, 0.1, 8, 100.0, None, None, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, p, 1, -3.1, 0.1, 8, 100.0, None, None, p, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, p, 1, -3.1, 0.1, 0, 100.0, None, p, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, -1, p, 1, -3.1, 0.1, 8, 100.0, None, p, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, p, -1, -3.1, 0.1, 8, 100.0, None, p, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, p, 1, -3.1, 0.1, 6145, 100.0, None, p, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, p, 1, -3.1, 0.0, 8, 100.0, None, p, None, None) == bad
assert L.b2s_virtual_scan_batch(p, p, 1, p, 1, -3.1, float("nan"), 8, 100.0, None, p, None, None) == bad
# b2s_icp_set_map / b2s_icp_map_observation: null handle, null obstacles, bad sizes
assert L.b2s_icp_set_map(None, p, p, 1) == bad
assert L.b2s_icp_map_observation(None, None, None, None, 0.0, 1, 8, -3.1, 0.1, 100.0, 30, 1e-3, None, None,
                                 None) == bad
assert b"null handle" in L.b2s_last_error()
print("ok")
"""


def test_new_entry_points_validate_without_a_device():
    """In a child process from which the GPUs are hidden, so that the no-device path is checked on any machine."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK, ROOT], env=env, check=True, timeout=300,
                         capture_output=True, text=True)
    assert out.stdout.strip() == "ok"


def test_room_map_observation_workload():
    from b2slam import synth
    a = synth.room_map_observation(9001, 400, 360)
    b = synth.room_map_observation(9001, 400, 360)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert a["ranges"].dtype == np.float32 and a["ranges"].shape == (400, 360)
    assert a["poses"].shape == a["prior"].shape == (400, 3)
    d = np.abs(a["prior"] - a["poses"])
    assert 0 < d[:, :2].max() < 0.2 and 0 < d[:, 2].max() < 0.1
    # the trajectory and ranges are those of room_sequence
    xy, poses = synth.room_sequence(9001, 400, 360)
    assert np.array_equal(poses, a["poses"])
    phi = synth.beam_angles(360)
    np.testing.assert_allclose(xy[:, 0], a["ranges"] * np.cos(phi), rtol=1e-6, atol=1e-6)
    course, fine = a["obstacles_course"], a["obstacles_fine"]
    assert 500 < course.shape[1] < 2000 and fine.shape[1] >= 200000
    # cell centres on the course map's grid: 129 x 129 at 0.155 m centred on the origin
    idx = (course + 129 * 0.155 / 2.0) / 0.155 - 0.5
    assert np.allclose(idx, np.round(idx), atol=1e-9) and idx.min() >= 0 and idx.max() <= 128


def pyref_map_observation(obstacle_xy, ranges, pose, angle_min, angle_max, angle_increment, clamp_inf_to=None,
                          far_range=100.0, max_iter=30, tolerance=1e-3):
    """calc_map_observation, W9 localization.py:152-157, for one scan, composed from the literal oracle pieces:
    target = laserToNumpy(laserEstimation at `pose`), source = laserToNumpy(ranges), then ICP.process(target, source)
    (oracle.pyref.icp_process with the vectorised nearest search, same values).  Returns (T, iterations, virtual)."""
    from oracle import pyref
    virtual = pyref.virtual_scan(obstacle_xy, pose, angle_min, angle_increment, len(ranges), far_range)
    tar = pyref.laser_to_points(virtual, angle_min, angle_max)
    src = pyref.laser_to_points(ranges, angle_min, angle_max, clamp_inf_to)
    T, iters = pyref.icp_process(tar, src, max_iter, tolerance, nearest=pyref.nearest_targets_vec)
    return T, iters, virtual


def test_composed_reference_map_observation():
    """The composed reference (virtual_scan + laser_to_points + the literal ICP) agrees with the C oracle's ICP on the
    same point pairs."""
    from b2slam import synth
    from oracle import corc, pyref
    w = synth.room_map_observation(9001, 40, 120)
    obs = w["obstacles_course"]
    for k in (3, 29):
        T, it, virt = pyref_map_observation(obs, w["ranges"][k], w["prior"][k], -math.pi, math.pi, 2 * math.pi / 119)
        assert np.array_equal(virt, pyref.virtual_scan(obs, w["prior"][k], -math.pi, 2 * math.pi / 119, 120))
        tar = pyref.laser_to_points(virt, -math.pi, math.pi)[:2]
        src = pyref.laser_to_points(w["ranges"][k], -math.pi, math.pi)[:2]
        wT, wit = corc.icp_batch(tar[None], src[None], 30, 1e-3)
        assert it == wit[0]
        np.testing.assert_allclose(T, wT[0], rtol=0, atol=1e-9)
