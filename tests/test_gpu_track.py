"""GPU checks of ICP.track: pose hypotheses carried through consecutive scans in the static map.

Every stage must be the map observation relocalize computes at the stage's prior, the priors must chain the poses by
process_scans' odometry, the joint score must be the ascending sum and the selection the lowest-index finite rule;
on the room workload one track must follow the robot and the full grid must find it from a few scans."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

NAN_TEXT = "cannot convert float NaN to integer"
INC = 2 * math.pi / 359
EVERY = 6  # the W9 node matches one scan in six


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, scan, synth
    from oracle import pyref
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.dev, e.scan, e.pyref = b2slam, devapi, scan, pyref
    e.w = synth.room_relocalization(9001, 300 * EVERY, 360)
    e.ranges = e.w["ranges"][::EVERY]
    e.truth = e.w["poses"][::EVERY]
    e.icp = b2slam.ICP()
    e.icp.set_static_map(e.w["obstacles_course"])
    return e


def _step(p, t):
    """The pose-chain step p (+) t of [ICP]:185-190."""
    x, y, yaw = p
    c, s = math.cos(yaw), math.sin(yaw)
    return np.array([x + c * t[0, 2] - s * t[1, 2], y + s * t[0, 2] + c * t[1, 2], yaw + math.atan2(t[1, 0], t[0, 0])])


def _starts(env):
    """The true start, a wrong one from the grid, a duplicate of the true start, and a start 8 cm / 0.03 rad off."""
    t0 = env.truth[0]
    return np.stack([t0, env.w["candidates"][4321], t0, t0 + np.array([0.06, -0.05, 0.03])])


def test_one_scan_is_relocalize(env):
    rng = np.random.Generator(np.random.PCG64(17))
    cand = env.w["candidates"][np.sort(rng.choice(len(env.w["candidates"]), 2000, replace=False))].copy()
    cand[7] = env.truth[0] + np.array([0.03, -0.02, 0.01])
    best, pose, score, it, joint = env.icp.track(env.ranges[:1], cand, -math.pi, math.pi)
    rbest, rpose, rscore, rit, rT = env.icp.relocalize(env.ranges[:1], cand, -math.pi, math.pi, return_T=True)
    assert pose.shape == (2000, 1, 3) and score.shape == it.shape == (2000, 1) and joint.shape == (2000,)
    assert np.int32(best).tobytes() == rbest[0].tobytes() and best >= 0
    assert score[:, 0].tobytes() == rscore[0].tobytes()
    assert it[:, 0].tobytes() == rit[0].tobytes()
    assert joint.tobytes() == (0.0 + rscore[0]).tobytes()
    np.testing.assert_allclose(pose[best, 0], rpose[0], rtol=0, atol=1e-12)
    want = np.stack([_step(cand[h], rT[0, h]) for h in range(len(cand))])
    np.testing.assert_allclose(pose[:, 0], want, rtol=0, atol=1e-12)


def test_stages_decompose(env):
    icp, ranges, starts = env.icp, env.ranges[:6], _starts(env)
    best, pose, score, it, joint, prior = icp.track(ranges, starts, -math.pi, math.pi, return_priors=True)
    assert prior.shape == pose.shape == (4, 6, 3)
    assert prior[:, 0].tobytes() == starts.tobytes()
    odo, _ = icp.process_scans(ranges, -math.pi, math.pi)
    for h in range(len(starts)):
        for k in range(6):
            if k > 0:
                np.testing.assert_allclose(prior[h, k], _step(pose[h, k - 1], odo[k - 1]), rtol=0, atol=1e-12)
            _, _, rscore, rit = icp.relocalize(ranges[k:k + 1], prior[h, k][None], -math.pi, math.pi)
            assert score[h, k].tobytes() == rscore[0, 0].tobytes(), (h, k)
            assert it[h, k].tobytes() == rit[0, 0].tobytes(), (h, k)
            T, _ = icp.map_observation(ranges[k:k + 1], prior[h, k][None], -math.pi, math.pi)
            np.testing.assert_allclose(pose[h, k], _step(prior[h, k], T[0]), rtol=0, atol=1e-12)


def _select_ref(score, pose, joint):
    ok = np.isfinite(score).all(axis=1) & np.isfinite(pose).all(axis=(1, 2))
    if not ok.any():
        return -1
    return int(np.flatnonzero(ok & (joint == joint[ok].min()))[0])


def test_joint_score_and_selection(env):
    inf = np.inf
    starts = np.concatenate([_starts(env), [[inf, 0.0, 0.0], [0.0, -inf, 0.3], [1.0, 1.0, inf], [-inf, inf, -inf]]])
    best, pose, score, it, joint = env.icp.track(env.ranges[:4], starts, -math.pi, math.pi)
    for h in range(len(starts)):
        j = 0.0
        for k in range(4):
            j += score[h, k]
        assert np.float64(j).tobytes() == joint[h].tobytes(), h
    assert joint[0].tobytes() == joint[2].tobytes() and score[0].tobytes() == score[2].tobytes()
    # a track near the truth wins, and the true start ahead of its duplicate at 2
    assert best == _select_ref(score, pose, joint) and best in (0, 3)
    # +-inf starts run to the end with a non-finite pose, never win, and alone give -1
    assert not np.isfinite(pose[4:]).all(axis=(1, 2)).any()
    best, pose, score, it, joint = env.icp.track(env.ranges[:4], starts[4:], -math.pi, math.pi)
    assert best == -1
    assert np.isfinite(score).all()  # what excludes them is the pose: their virtual scans are the far_range circle
    assert np.isnan(pose[2:, :, :2]).all()  # an infinite yaw: cos and sin are NaN


def _reference(env, prior, ranges, max_iter=30, tolerance=1e-3):
    """The literal reference loop (oracle.pyref.icp_process, [ICP]:38-88) on the composed map observation at `prior`:
    (T, iterations, mean_error of the last iteration)."""
    p = env.pyref
    virtual = p.virtual_scan(env.w["obstacles_course"], prior, -math.pi, INC, len(ranges))
    tar_pc = p.laser_to_points(virtual, -math.pi, math.pi)
    src_pc = p.laser_to_points(ranges, -math.pi, math.pi)
    first = np.array(src_pc[:2, :], dtype=np.float64)
    tar = np.ones((3, tar_pc.shape[1]))
    tar[:2, :] = tar_pc[:2, :]
    cur = np.ones((3, first.shape[1]))
    cur[:2, :] = first
    prev_err, err, done = 0, 0.0, 0
    for _ in range(max_iter):
        dist, idx = p.nearest_targets_vec(cur[:2, :].transpose(), tar[:2, :].transpose())
        step = p.rigid_fit_svd(cur[:2, :].transpose(), tar[:2, idx].transpose())
        cur = np.dot(step, cur)
        done += 1
        err = np.sum(dist) / dist.size
        if abs(prev_err - err) < tolerance:
            break
        prev_err = err
    return p.rigid_fit_svd(first.transpose(), cur[:2, :].transpose()), done, err


def test_stages_are_the_reference_loop(env):
    ranges, starts = env.ranges[:4], _starts(env)[[0, 1, 3]]
    best, pose, score, it, joint, prior = env.icp.track(ranges, starts, -math.pi, math.pi, return_priors=True)
    for h in range(len(starts)):
        for k in range(4):
            rT, rit, rerr = _reference(env, prior[h, k], ranges[k])
            assert rit == it[h, k], (h, k)
            assert abs(score[h, k] - rerr) <= 1e-12, (h, k, score[h, k], rerr)
            np.testing.assert_allclose(pose[h, k], _step(prior[h, k], rT), rtol=0, atol=1e-9)


def _errors(pose, truth):
    d_xy = np.hypot(pose[..., 0] - truth[..., 0], pose[..., 1] - truth[..., 1])
    d_yaw = np.abs((pose[..., 2] - truth[..., 2] + math.pi) % (2 * math.pi) - math.pi)
    return d_xy, d_yaw


def test_one_track_follows_the_robot(env):
    best, pose, score, it, joint = env.icp.track(env.ranges, env.truth[0], -math.pi, math.pi)
    assert best == 0 and pose.shape == (300, 3)
    d_xy, d_yaw = _errors(pose, env.truth)
    # measured on a B200 over the 300 stages: 0.101 m / 0.081 rad at most, 0.050 m / 0.044 rad on average (the course
    # map's cells are 0.155 m, and the observation is taken as the pose without an EKF)
    assert d_xy.max() < 0.15 and d_xy.mean() < 0.08, (d_xy.max(), d_xy.mean())
    assert d_yaw.max() < 0.12 and d_yaw.mean() < 0.07, (d_yaw.max(), d_yaw.mean())


def test_the_grid_finds_the_robot_from_four_scans(env):
    best, pose, score, it, joint = env.icp.track(env.ranges[:4], env.w["candidates"], -math.pi, math.pi)
    assert best >= 0 and pose.shape == (len(env.w["candidates"]), 4, 3)
    d_xy, d_yaw = _errors(pose[best, 3], env.truth[3])
    # measured on a B200: 0.038 m and 0.008 rad from the truth of the last scan
    assert d_xy < 0.10, d_xy
    assert d_yaw < 0.05, d_yaw


def test_layer1_pieces_compose_the_call(env):
    icp, dev, scan = env.icp, env.dev, env.scan
    ranges, starts = env.ranges[:5], _starts(env)
    K, H = len(ranges), len(starts)
    want = icp.track(ranges, starts, -math.pi, math.pi, return_priors=True)
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    obs = env.w["obstacles_course"]
    ox, oy, cs = cuda(obs[0]), cuda(obs[1]), cuda(scan.beam_table(-math.pi, math.pi, 360))
    odo = cuda(icp.process_scans(ranges, -math.pi, math.pi)[0])
    prior = torch.empty((K, H, 3), dtype=torch.float64, device="cuda")
    prior[0] = cuda(starts)
    pose = torch.empty_like(prior)
    score = torch.empty((K, H), dtype=torch.float64, device="cuda")
    iters = torch.empty((K, H), dtype=torch.int32, device="cuda")
    joint = torch.empty(H, dtype=torch.float64, device="cuda")
    finite = torch.empty(H, dtype=torch.int32, device="cuda")
    tar = torch.empty((H, 2, 360), dtype=torch.float64, device="cuda")
    for k in range(K):
        dev.virtual_scan_batch(ox, oy, prior[k], -math.pi, INC, 360, beam_cs=cs, tar_xy=tar)
        src = cuda(np.repeat(scan.laser_to_points(ranges[k], -math.pi, math.pi)[:2][None], H, axis=0))
        T, _, _ = dev.icp_batch_err(tar, src, iters_out=iters[k], err_out=score[k])
        last = k == K - 1
        dev.track_step(T, score[k], prior[k], pose[k], joint, finite, k, odometry=None if last else odo[k],
                       next_prior=None if last else prior[k + 1])
    best = dev.track_select(joint, finite)
    torch.cuda.synchronize()
    got = (int(best.cpu()[0]), pose.cpu().numpy().transpose(1, 0, 2), score.cpu().numpy().T, iters.cpu().numpy().T,
           joint.cpu().numpy(), prior.cpu().numpy().transpose(1, 0, 2))
    assert got[0] == want[0]
    for a, b in zip(got[1:], want[1:]):
        assert np.ascontiguousarray(a).tobytes() == b.tobytes()


def test_repeatable_and_errors_leave_the_object_usable(env):
    icp = env.icp
    ranges, starts = env.ranges[:3], _starts(env)
    first = icp.track(ranges, starts, -math.pi, math.pi, return_priors=True)
    one = icp.track(ranges, starts[0], -math.pi, math.pi)
    assert one[0] == 0 and one[1].shape == (3, 3) and one[2].shape == (3,) and one[4].shape == ()
    bad = starts.copy()
    bad[2, 1] = np.nan
    with pytest.raises(ValueError, match=NAN_TEXT):
        icp.track(ranges, bad, -math.pi, math.pi)
    with pytest.raises(ValueError, match="2304"):
        icp.track(np.ones((2, 2305), dtype=np.float32), starts, -math.pi, math.pi)
    with pytest.raises(ValueError):
        icp.track(ranges, starts[:0], -math.pi, math.pi)
    with pytest.raises(ValueError):
        icp.track(ranges[:0], starts, -math.pi, math.pi)
    with pytest.raises(ValueError):
        icp.track(ranges, starts[:, :2], -math.pi, math.pi)
    fresh = env.b2slam.ICP()
    with pytest.raises(ValueError, match="no static map"):
        fresh.track(ranges, starts, -math.pi, math.pi)
    again = icp.track(ranges, starts, -math.pi, math.pi, return_priors=True)
    assert first[0] == again[0]
    for a, b in zip(first[1:], again[1:]):
        assert a.tobytes() == b.tobytes()
