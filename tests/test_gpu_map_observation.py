"""GPU parity: the map observation of W9 localization (calc_map_observation, [LOC9]:152-157).

b2s_virtual_scan_batch must give the bytes of one b2s_virtual_scan call per pose (and the reference's own
laserEstimation bins); ICP.map_observation must give the transforms of ICP.process_batch on the float64 point pairs
that laser_to_points makes of the virtual and the measured scans, bit for bit."""
import math

import numpy as np
import pytest

from conftest import load_golden
from test_map_observation_host import pyref_map_observation

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

NAN_TEXT = "cannot convert float NaN to integer"


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, scan, synth
    from oracle import corc, pyref
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.lib, e.dev, e.scan, e.synth, e.corc, e.pyref = b2slam, _lib, devapi, scan, synth, corc, pyref
    e.icp = b2slam.ICP()
    e.room = synth.room_map_observation(9001, 3000, 360)
    return e


def _batch(env, obstacle_xy, poses, angle_min, angle_max, inc, beams, far=100.0, with_ranges=True, with_tar=True):
    """devapi.virtual_scan_batch -> (ranges or None, tar_xy or None) on the host."""
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")
    K = len(poses)
    ranges = torch.empty((K, beams), dtype=torch.float64, device="cuda") if with_ranges else None
    tar = torch.empty((K, 2, beams), dtype=torch.float64, device="cuda") if with_tar else None
    cs = cuda(env.scan.beam_table(angle_min, angle_max, beams)) if with_tar else None
    env.dev.virtual_scan_batch(cuda(obstacle_xy[0]), cuda(obstacle_xy[1]), cuda(np.reshape(poses, (K, 3))), angle_min,
                               inc, beams, far, beam_cs=cs, ranges=ranges, tar_xy=tar)
    torch.cuda.synchronize()
    return (None if ranges is None else ranges.cpu().numpy()), (None if tar is None else tar.cpu().numpy())


def _check_batch(env, obstacle_xy, poses, angle_min, angle_max, beams, far=100.0):
    """Ranges and targets of the batched call, with and without the other output, against single-pose calls."""
    inc = (angle_max - angle_min) / (beams - 1) if beams > 1 else 2 * math.pi
    want = np.stack([env.scan.virtual_scan(obstacle_xy, p, angle_min, inc, beams, far) for p in poses])
    want_tar = np.stack([env.scan.laser_to_points(w, angle_min, angle_max)[:2] for w in want])
    r, t = _batch(env, obstacle_xy, poses, angle_min, angle_max, inc, beams, far)
    assert r.tobytes() == want.tobytes()
    assert t.tobytes() == want_tar.tobytes()
    r, _ = _batch(env, obstacle_xy, poses, angle_min, angle_max, inc, beams, far, with_tar=False)
    assert r.tobytes() == want.tobytes()
    _, t = _batch(env, obstacle_xy, poses, angle_min, angle_max, inc, beams, far, with_ranges=False)
    assert t.tobytes() == want_tar.tobytes()
    return want


@pytest.mark.parametrize("beams", [1, 90, 120, 360, 361, 1080, 2304])
def test_batch_equals_single_pose_calls_on_the_course_map(env, beams):
    poses = np.concatenate([env.room["prior"][:6], env.room["poses"][2000:2003]])
    want = _check_batch(env, env.room["obstacles_course"], poses, -math.pi, math.pi, beams)
    assert beams == 1 or (want < 100.0).mean(axis=1).min() > 0.1   # every pose really sees the map


def test_batch_edge_cases(env):
    course = env.room["obstacles_course"]
    poses = env.room["prior"][:4]
    # no obstacles: every bin stays far_range
    want = _check_batch(env, np.zeros((2, 0)), poses, -math.pi, math.pi, 360)
    assert (want == 100.0).all()
    # obstacles beyond far_range never win; 30 m as far_range cuts the room's far walls
    far = np.stack([150.0 * np.cos(np.linspace(0, 6, 500)), 150.0 * np.sin(np.linspace(0, 6, 500))])
    assert (_check_batch(env, far, poses, -math.pi, math.pi, 360) == 100.0).all()
    _check_batch(env, course, poses, -math.pi, math.pi, 360, far=3.0)
    # an obstacle exactly at the pose (distance 0, atan2(0, 0))
    at = course[:, 100]
    want = _check_batch(env, course, [(at[0], at[1], 0.3), (at[0], at[1], -2.0)], -math.pi, math.pi, 360)
    assert (want == 0.0).any()
    # a partial sweep, and one pose
    _check_batch(env, course, poses, -2.0, 2.5, 270)
    _check_batch(env, course, poses[:1], -math.pi, math.pi, 360)
    # +-inf poses and obstacles: no bin is won through them, exactly as in the single-pose kernel
    inf_map = np.concatenate([course, [[np.inf, -np.inf, 1.0], [0.5, 2.0, np.inf]]], axis=1)
    _check_batch(env, inf_map, [(np.inf, 0.0, 0.1), (0.0, -np.inf, 0.1), (0.2, 0.1, np.inf), (0.2, 0.1, 0.3)],
                 -math.pi, math.pi, 360)


def test_batch_multi_slice_path_on_a_large_map(env):
    """Few poses over > 2e5 cells: the obstacles are cut into slices merged with a global atomicMin."""
    fine = env.room["obstacles_fine"]
    assert fine.shape[1] >= 200000
    _check_batch(env, fine, env.room["prior"][:3], -math.pi, math.pi, 360)
    _check_batch(env, fine, env.room["prior"][5:6], -2.0, 2.5, 1080)


def test_batch_matches_reference_laserEstimation_golden(env):
    """Every next_rows.npz vscan case through the batched call: the reference's bins, ranges to 1e-13 relative."""
    z = load_golden("next_rows.npz")
    for i in range(int(z["vscan_count"])):
        g = lambda k: z["vscan%d_%s" % (i, k)]
        beams = int(g("beams"))
        obs = np.stack([g("obs_x"), g("obs_y")])
        got, _ = _batch(env, obs, [g("pose")], float(g("angle_min")), 0.0, float(g("angle_increment")), beams,
                        with_tar=False)
        want = g("ranges")
        assert np.array_equal(got[0] == 100.0, want == 100.0), i
        np.testing.assert_allclose(got[0], want, rtol=1e-13, atol=0)


def _pairs(env, virtual, ranges, clamp=None):
    tar = np.stack([env.scan.laser_to_points(v, -math.pi, math.pi)[:2] for v in virtual])
    src = np.stack([env.scan.laser_to_points(r, -math.pi, math.pi, clamp)[:2] for r in ranges])
    return tar, src


def test_map_observation_equals_process_batch_on_the_point_pairs(env):
    """3000 scans x 360 beams (more than one automatic chunk), without and with the 30 m clamp, with inf ranges."""
    room = env.room
    env.icp.set_static_map(room["obstacles_course"])
    ranges = room["ranges"].copy()
    ranges[::7, 40:60] = np.inf
    for clamp in (None, 30.0):
        T, it, virt = env.icp.map_observation(ranges, room["prior"], -math.pi, math.pi, clamp_inf_to=clamp,
                                              return_virtual=True)
        want_v = np.stack([env.scan.virtual_scan(room["obstacles_course"], p, -math.pi, 2 * math.pi / 359, 360)
                           for p in room["prior"][::97]])
        assert virt[::97].tobytes() == want_v.tobytes()
        tar, src = _pairs(env, virt, ranges, clamp)
        wT, wit = env.icp.process_batch(tar, src)
        assert T.tobytes() == wT.tobytes() and it.tobytes() == wit.tobytes(), clamp
    T, it = env.icp.map_observation(room["ranges"], room["prior"], -math.pi, math.pi)
    assert (it > 1).mean() > 0.5 and np.median(np.abs(T[:, :2, 2])) < 0.5   # small corrections of the prior


def test_map_observation_against_the_oracle(env):
    room = env.room
    rng = np.random.Generator(np.random.PCG64(64))
    pick = np.sort(rng.choice(3000, 64, replace=False))
    obs = room["obstacles_course"]
    env.icp.set_static_map(obs)
    T, it, virt = env.icp.map_observation(room["ranges"][pick], room["prior"][pick], -math.pi, math.pi,
                                          return_virtual=True)
    want_v = np.stack([env.pyref.virtual_scan(obs, p, -math.pi, 2 * math.pi / 359, 360) for p in room["prior"][pick]])
    assert np.array_equal(virt == 100.0, want_v == 100.0)
    np.testing.assert_allclose(virt, want_v, rtol=1e-13, atol=0)
    tar, src = _pairs(env, want_v, room["ranges"][pick])
    wT, wit = env.corc.icp_batch(tar, src, 30, 1e-3)
    assert np.array_equal(it, wit)
    np.testing.assert_allclose(T, wT, rtol=0, atol=1e-9)
    # the composed reference, literal ICP included, on two of them
    for k in (0, 33):
        rT, rit, rv = pyref_map_observation(obs, room["ranges"][pick[k]], room["prior"][pick[k]], -math.pi, math.pi,
                                            2 * math.pi / 359)
        assert rit == it[k]
        np.testing.assert_allclose(T[k], rT, rtol=0, atol=1e-9)


def test_pipeline_depth_gives_identical_bytes(env):
    room = env.room
    env.icp.set_static_map(room["obstacles_course"])
    L = env.lib.lib()
    outs = []
    try:
        for chunks in (0, 1, 3, 16):
            assert L.b2s_tune(b"h2d_chunks", chunks) == 0
            outs.append(env.icp.map_observation(room["ranges"], room["prior"], -math.pi, math.pi, clamp_inf_to=30.0,
                                                return_virtual=True))
    finally:
        L.b2s_tune(b"h2d_chunks", 0)
    for o in outs[1:]:
        for a, b in zip(o, outs[0]):
            assert a.tobytes() == b.tobytes()


def test_map_lifecycle(env):
    room = env.room
    icp = env.b2slam.ICP()
    icp.set_static_map(room["obstacles_course"])
    T1, it1, v1 = icp.map_observation(room["ranges"][:200], room["prior"][:200], -math.pi, math.pi,
                                      return_virtual=True)
    T0, it0 = icp.map_observation(room["ranges"][:200], room["prior"][:200], -math.pi, math.pi)
    assert T0.tobytes() == T1.tobytes() and it0.tobytes() == it1.tobytes()
    # one scan
    T, it = icp.map_observation(room["ranges"][7:8], room["prior"][7:8], -math.pi, math.pi)
    assert T.shape == (1, 3, 3) and T.tobytes() == T1[7:8].tobytes() and it[0] == it1[7]
    # a LaserScan's own angle_increment may differ from (max - min) / (N - 1)
    _, _, vi = icp.map_observation(room["ranges"][:5], room["prior"][:5], -math.pi, math.pi,
                                   angle_increment=2 * math.pi / 360, return_virtual=True)
    want = np.stack([env.scan.virtual_scan(room["obstacles_course"], p, -math.pi, 2 * math.pi / 360, 360)
                     for p in room["prior"][:5]])
    assert vi.tobytes() == want.tobytes()
    # replacing the map changes the result
    icp.set_static_map(room["obstacles_course"][:, ::2])
    T2, _, v2 = icp.map_observation(room["ranges"][:200], room["prior"][:200], -math.pi, math.pi, return_virtual=True)
    assert not np.array_equal(v2, v1) and not np.array_equal(T2, T1)
    want = np.stack([env.scan.virtual_scan(room["obstacles_course"][:, ::2], p, -math.pi, 2 * math.pi / 359, 360)
                     for p in room["prior"][:3]])
    assert v2[:3].tobytes() == want.tobytes()
    # clearing it
    icp.set_static_map(np.zeros((2, 0)))
    with pytest.raises(ValueError, match="no static map"):
        icp.map_observation(room["ranges"][:2], room["prior"][:2], -math.pi, math.pi)


def test_errors_leave_the_object_usable(env):
    room = env.room
    icp = env.b2slam.ICP()
    with pytest.raises(ValueError, match="no static map"):
        icp.map_observation(room["ranges"][:2], room["prior"][:2], -math.pi, math.pi)
    icp.set_static_map(room["obstacles_course"])
    ranges, prior = room["ranges"][:300], room["prior"][:300]
    want = icp.map_observation(ranges, prior, -math.pi, math.pi, return_virtual=True)
    for k, col in ((0, 0), (299, 2), (150, 1)):
        bad = prior.copy()
        bad[k, col] = np.nan
        with pytest.raises(ValueError, match=NAN_TEXT):
            icp.map_observation(ranges, bad, -math.pi, math.pi)
        got = icp.map_observation(ranges, prior, -math.pi, math.pi, return_virtual=True)
        assert all(a.tobytes() == b.tobytes() for a, b in zip(got, want))
    bad_map = room["obstacles_course"].copy()
    bad_map[1, 17] = np.nan
    with pytest.raises(ValueError, match=NAN_TEXT):
        icp.set_static_map(bad_map)
    with pytest.raises(ValueError, match="no static map"):   # the rejected map is not half-set
        icp.map_observation(ranges, prior, -math.pi, math.pi)
    icp.set_static_map(room["obstacles_course"])
    got = icp.map_observation(ranges, prior, -math.pi, math.pi, return_virtual=True)
    assert all(a.tobytes() == b.tobytes() for a, b in zip(got, want))
    # +-inf poses and obstacles do not raise, and give the single-pose bytes
    inf_map = np.concatenate([room["obstacles_course"], [[np.inf, -np.inf], [1.0, np.inf]]], axis=1)
    icp.set_static_map(inf_map)
    poses = prior[:4].copy()
    poses[0, 0], poses[1, 1], poses[2, 2] = np.inf, -np.inf, np.inf
    _, _, virt = icp.map_observation(ranges[:4], poses, -math.pi, math.pi, return_virtual=True)
    single = np.stack([env.scan.virtual_scan(inf_map, p, -math.pi, 2 * math.pi / 359, 360) for p in poses])
    assert virt.tobytes() == single.tobytes()
    with pytest.raises(ValueError, match="2304"):
        icp.map_observation(np.ones((2, 2305), np.float32), prior[:2], -math.pi, math.pi)


def test_devapi_equals_the_host_calls(env):
    room = env.room
    obs, poses = room["obstacles_course"], room["prior"][:500]
    env.icp.set_static_map(obs)
    _, _, virt = env.icp.map_observation(room["ranges"][:500], poses, -math.pi, math.pi, return_virtual=True)
    r, t = _batch(env, obs, poses, -math.pi, math.pi, 2 * math.pi / 359, 360)
    assert r.tobytes() == virt.tobytes()
    want_tar, _ = _pairs(env, virt, room["ranges"][:500])
    assert t.tobytes() == want_tar.tobytes()
