"""GPU checks of ICP.relocalize: the map observation at many candidate poses, scored and chosen on the device.

Every hypothesis must equal ICP.map_observation at its candidate bit for bit; the score must be the reference's own
mean_error of the last iteration; the selection must follow the lowest-index, finite-only rule whatever the number of
hypotheses; and on the room workload the chosen pose must be the robot's."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

NAN_TEXT = "cannot convert float NaN to integer"
INC = 2 * math.pi / 359


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, synth
    from oracle import pyref
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.lib, e.dev, e.synth, e.pyref = b2slam, _lib, devapi, synth, pyref
    e.w = synth.room_relocalization(9001, 8, 360)
    e.icp = b2slam.ICP()
    e.icp.set_static_map(e.w["obstacles_course"])
    return e


def _sample(env, count, seed, near_truth_of=None):
    """`count` candidates drawn from the grid; with near_truth_of=k, one of them (index 7) lies within 5 cm of the
    true pose of scan k."""
    grid = env.w["candidates"]
    rng = np.random.Generator(np.random.PCG64(seed))
    cand = grid[np.sort(rng.choice(grid.shape[0], count, replace=False))].copy()
    if near_truth_of is not None:
        cand[7] = env.w["poses"][near_truth_of] + np.array([0.03, -0.02, 0.01])
    return cand


def _select_ref(score, T, cand):
    """The selection rule in NumPy: lowest-index argmin over the hypotheses whose score and T are finite."""
    best = np.full(score.shape[0], -1, dtype=np.int32)
    pose = np.full((score.shape[0], 3), np.nan)
    for k in range(score.shape[0]):
        ok = np.isfinite(score[k]) & np.isfinite(T[k].reshape(len(cand), 9)).all(axis=1)
        if ok.any():
            s = np.where(ok, score[k], np.inf)
            b = int(np.flatnonzero(ok & (s == s[ok].min()))[0])
            best[k] = b
            x, y, yaw = cand[b]
            t = T[k, b]
            pose[k] = (x + math.cos(yaw) * t[0, 2] - math.sin(yaw) * t[1, 2],
                       y + math.sin(yaw) * t[0, 2] + math.cos(yaw) * t[1, 2], yaw + math.atan2(t[1, 0], t[0, 0]))
    return best, pose


@pytest.mark.parametrize("with_inf", [False, True])
@pytest.mark.parametrize("clamp", [None, 30.0])
def test_hypotheses_equal_map_observation(env, with_inf, clamp):
    ranges = env.w["ranges"][[0, 5]].copy()
    if with_inf:
        ranges[:, ::17] = np.inf
    cand = _sample(env, 2000, 11, near_truth_of=0)
    H = len(cand)
    best, pose, score, it, T = env.icp.relocalize(ranges, cand, -math.pi, math.pi, clamp_inf_to=clamp, return_T=True)
    wT, wit = env.icp.map_observation(np.repeat(ranges, H, axis=0), np.tile(cand, (2, 1)), -math.pi, math.pi,
                                      clamp_inf_to=clamp)
    assert T.shape == (2, H, 3, 3) and score.shape == it.shape == (2, H)
    assert T.tobytes() == wT.tobytes()
    assert it.tobytes() == wit.reshape(2, H).tobytes()
    # the selection and the pose follow the documented rule on what the call returned
    want_best, want_pose = _select_ref(score, T, cand)
    assert np.array_equal(best, want_best)
    np.testing.assert_allclose(pose, want_pose, rtol=0, atol=1e-12)


def _reference_score(env, cand, ranges, max_iter=30, tolerance=1e-3):
    """The literal reference loop (oracle.pyref.icp_process, [ICP]:38-88) on the composed map observation, returning
    the mean_error of its last iteration as well: (T, iterations, mean_error)."""
    p = env.pyref
    virtual = p.virtual_scan(env.w["obstacles_course"], cand, -math.pi, INC, len(ranges))
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


def test_score_is_the_reference_mean_error(env):
    cand = _sample(env, 64, 64, near_truth_of=2)
    ranges = env.w["ranges"][2]
    best, pose, score, it, T = env.icp.relocalize(ranges, cand, -math.pi, math.pi, return_T=True)
    assert score.shape == it.shape == (64,) and T.shape == (64, 3, 3) and pose.shape == (3,)
    for h in range(64):
        rT, rit, rerr = _reference_score(env, cand[h], ranges)
        assert rit == it[h], h
        assert abs(score[h] - rerr) <= 1e-12, (h, score[h], rerr)
        np.testing.assert_allclose(T[h], rT, rtol=0, atol=1e-9)


def test_duplicated_candidates_score_alike_and_the_lower_index_wins(env):
    cand = _sample(env, 700, 5, near_truth_of=3)
    both = np.concatenate([cand, cand])
    best, pose, score, it = env.icp.relocalize(env.w["ranges"][[3, 4]], both, -math.pi, math.pi)
    H = len(cand)
    assert score[:, :H].tobytes() == score[:, H:].tobytes()
    assert it[:, :H].tobytes() == it[:, H:].tobytes()
    assert (best >= 0).all() and (best < H).all()  # every winner has a twin at best + H with the same score


def _crafted(H, K=4, seed=3):
    rng = np.random.Generator(np.random.PCG64(seed + H))
    score = rng.uniform(0.05, 2.0, size=(K, H))
    th = rng.uniform(-0.2, 0.2, size=(K, H))
    T = np.zeros((K, H, 3, 3))
    T[..., 0, 0] = T[..., 1, 1] = np.cos(th)
    T[..., 1, 0] = np.sin(th)
    T[..., 0, 1] = -np.sin(th)
    T[..., 0, 2] = rng.uniform(-0.3, 0.3, size=(K, H))
    T[..., 1, 2] = rng.uniform(-0.3, 0.3, size=(K, H))
    T[..., 2, 2] = 1.0
    cand = np.stack([rng.uniform(-5, 5, H), rng.uniform(-5, 5, H), rng.uniform(-math.pi, math.pi, H)], axis=1)
    want = {}
    # scan 0: ties at the lowest score
    lo = [H - 1, H // 2, H // 3] if H > 1 else [0]
    score[0, lo] = 0.01
    want[0] = min(lo)
    # scan 1: NaN and +-inf scores below, around and above every finite one
    bad = [0, H // 2, H - 1] if H > 2 else [0]
    score[1, bad[0]] = -np.inf
    if H > 2:
        score[1, bad[1]], score[1, bad[2]] = np.nan, np.inf
    if H > 3:
        score[1, H // 4] = 0.001
        want[1] = H // 4
    # scan 2: the smallest score goes with a transform that is not finite
    score[2, H - 1] = 0.0001
    T[2, H - 1, 1, 2] = np.nan
    if H > 1:
        score[2, 0] = 0.0002
        want[2] = 0
    else:
        want[2] = -1
    # scan 3: nothing finite
    score[3, ::2] = np.nan
    T[3, 1::2, 0, 0] = np.inf
    want[3] = -1
    return score, T, cand, want


@pytest.mark.parametrize("H", [1, 1025, 57600])
def test_layer1_selection(env, H):
    score, T, cand, want = _crafted(H)
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    best, pose = env.dev.relocalize_select(cuda(score), cuda(T), cuda(cand))
    torch.cuda.synchronize()
    best, pose = best.cpu().numpy(), pose.cpu().numpy()
    wbest, wpose = _select_ref(score, T, cand)
    assert np.array_equal(best, wbest)
    for k, b in want.items():
        assert best[k] == b, (k, best[k], b)
    assert np.isnan(pose[best < 0]).all()
    np.testing.assert_allclose(pose[best >= 0], wpose[best >= 0], rtol=0, atol=1e-12)


def test_layer1_solve_reports_the_score(env):
    """b2s_icp_batch_f64_err: same T and iterations as b2s_icp_batch_f64, and the score of ICP.relocalize."""
    from b2slam import scan
    cand = _sample(env, 300, 9, near_truth_of=1)
    ranges = env.w["ranges"][1]
    _, _, score, it, T = env.icp.relocalize(ranges, cand, -math.pi, math.pi, return_T=True)
    virt = np.stack([scan.virtual_scan(env.w["obstacles_course"], c, -math.pi, INC, 360) for c in cand])
    tar = np.stack([scan.laser_to_points(v, -math.pi, math.pi)[:2] for v in virt])
    src = np.repeat(scan.laser_to_points(ranges, -math.pi, math.pi)[:2][None], len(cand), axis=0)
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    dT, dit, derr = env.dev.icp_batch_err(cuda(tar), cuda(src))
    pT, pit = env.dev.icp_batch(cuda(tar), cuda(src))
    torch.cuda.synchronize()
    assert dT.cpu().numpy().tobytes() == pT.cpu().numpy().tobytes() == T.tobytes()
    assert dit.cpu().numpy().tobytes() == pit.cpu().numpy().tobytes() == it.tobytes()
    assert derr.cpu().numpy().tobytes() == score.tobytes()


def test_it_finds_the_robot(env):
    w = env.w
    best, pose, score, it = env.icp.relocalize(w["ranges"], w["candidates"], -math.pi, math.pi)
    assert score.shape == (8, len(w["candidates"])) and (best >= 0).all()
    d_xy = np.hypot(pose[:, 0] - w["poses"][:, 0], pose[:, 1] - w["poses"][:, 1])
    d_yaw = np.abs((pose[:, 2] - w["poses"][:, 2] + math.pi) % (2 * math.pi) - math.pi)
    assert d_xy.max() < 0.10, d_xy
    assert d_yaw.max() < 0.05, d_yaw


def test_repeatable_and_errors_leave_the_object_usable(env):
    w = env.w
    icp = env.icp
    cand = _sample(env, 500, 21, near_truth_of=6)
    ranges = w["ranges"][6:8]
    first = icp.relocalize(ranges, cand, -math.pi, math.pi, return_T=True)
    mo = icp.map_observation(ranges, cand[:2], -math.pi, math.pi)
    bad = cand.copy()
    bad[123, 2] = np.nan
    with pytest.raises(ValueError, match=NAN_TEXT):
        icp.relocalize(ranges, bad, -math.pi, math.pi)
    with pytest.raises(ValueError, match="2304"):
        icp.relocalize(np.ones((1, 2305), dtype=np.float32), cand, -math.pi, math.pi)
    with pytest.raises(ValueError):
        icp.relocalize(ranges, cand[:0], -math.pi, math.pi)
    with pytest.raises(ValueError):
        icp.relocalize(ranges, cand[:, :2], -math.pi, math.pi)
    with pytest.raises(ValueError):
        icp.relocalize(ranges[None], cand, -math.pi, math.pi)
    fresh = env.b2slam.ICP()
    with pytest.raises(ValueError, match="no static map"):
        fresh.relocalize(ranges, cand, -math.pi, math.pi)
    again = icp.relocalize(ranges, cand, -math.pi, math.pi, return_T=True)
    for a, b in zip(first, again):
        assert a.tobytes() == b.tobytes()
    for a, b in zip(mo, icp.map_observation(ranges, cand[:2], -math.pi, math.pi)):
        assert a.tobytes() == b.tobytes()
