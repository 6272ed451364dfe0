"""GPU checks of the coarse-to-fine relocalization, ICP.relocalize(keep=...).

The coarse stage must be relocalize(max_iter=coarse_iters); the survivors must be the first min(keep, H) of the keep
order, computed here in NumPy from that call; every survivor's refined values must be the exhaustive call's entries bit
for bit; and the winner must be the exhaustive winner whenever it survives.  The layer-1 keep kernel and the kept form
of the selection are checked on crafted scores."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

NAN_TEXT = "cannot convert float NaN to integer"
A0, A1 = -math.pi, math.pi


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, icp, synth
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.dev, e.icpmod = b2slam, devapi, icp
    e.w = synth.room_relocalization(9001, 8, 360)
    e.fine = synth.room_relocalization(9001, 1, 360, xy_step=0.25)["candidates"]
    e.icp = b2slam.ICP()
    e.icp.set_static_map(e.w["obstacles_course"])
    return e


def _sample(grid, count, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return np.ascontiguousarray(grid[np.sort(rng.choice(grid.shape[0], count, replace=False))])


def _keep_ref(score, T, keep):
    """The keep order in NumPy: finite (score and all of T) hypotheses by (score, h), -0 == +0, then the rest by h; the
    first min(keep, H) of each scan, in ascending h."""
    K, H = score.shape
    fin = np.isfinite(score) & np.isfinite(T.reshape(K, H, 9)).all(axis=2)
    M = min(keep, H)
    out = np.empty((K, M), dtype=np.int32)
    for k in range(K):
        f = np.flatnonzero(fin[k])
        order = np.concatenate([f[np.argsort(score[k, f], kind="stable")], np.flatnonzero(~fin[k])])
        out[k] = np.sort(order[:M])
    return out


def _check_staged(env, ranges, cand, keep, coarse, clamp=None):
    """One staged call against the exhaustive and the coarse calls on the same input."""
    icp = env.icp
    best, pose, score, it, kept, T = icp.relocalize(ranges, cand, A0, A1, clamp_inf_to=clamp, keep=keep,
                                                    coarse_iters=coarse, return_T=True)
    xb, xp, xs, xit, xT = icp.relocalize(ranges, cand, A0, A1, clamp_inf_to=clamp, return_T=True)
    _, _, cs, _, cT = icp.relocalize(ranges, cand, A0, A1, clamp_inf_to=clamp, max_iter=coarse, return_T=True)
    K, H = xs.shape
    M = min(keep, H)
    assert kept.dtype == np.int32 and kept.shape == score.shape == it.shape == (K, M) and T.shape == (K, M, 3, 3)
    assert np.array_equal(kept, _keep_ref(cs, cT, keep))
    rows = np.arange(K)[:, None]
    assert score.tobytes() == xs[rows, kept].tobytes()
    assert it.tobytes() == xit[rows, kept].tobytes()
    assert T.tobytes() == xT[rows, kept].tobytes()
    for k in range(K):
        if xb[k] >= 0 and xb[k] in kept[k]:
            assert best[k] == xb[k] and pose[k].tobytes() == xp[k].tobytes(), k
        elif best[k] >= 0:
            assert xb[k] >= 0 and xs[k, best[k]] >= xs[k, xb[k]], k
        if best[k] >= 0:
            assert best[k] in kept[k]
    return best, pose, kept


@pytest.mark.parametrize("with_inf,clamp", [(False, None), (True, None), (True, 30.0)])
@pytest.mark.parametrize("extra", [0, 5])
def test_keep_at_least_H_is_the_exhaustive_call(env, with_inf, clamp, extra):
    ranges = env.w["ranges"][[0, 5]].copy()
    if with_inf:
        ranges[:, ::17] = np.inf
    cand = _sample(env.w["candidates"], 2000, 11)
    H = len(cand)
    best, pose, score, it, kept, T = env.icp.relocalize(ranges, cand, A0, A1, clamp_inf_to=clamp, keep=H + extra,
                                                        return_T=True)
    xb, xp, xs, xit, xT = env.icp.relocalize(ranges, cand, A0, A1, clamp_inf_to=clamp, return_T=True)
    assert np.array_equal(kept, np.tile(np.arange(H, dtype=np.int32), (2, 1)))
    assert best.tobytes() == xb.tobytes() and pose.tobytes() == xp.tobytes()
    assert score.tobytes() == xs.tobytes() and it.tobytes() == xit.tobytes() and T.tobytes() == xT.tobytes()


@pytest.mark.parametrize("H", [2000, 57600])
@pytest.mark.parametrize("keep", [1, 7, 256])
def test_survivors_and_refined_values(env, H, keep):
    cand = _sample(env.fine, H, H + keep)
    _check_staged(env, env.w["ranges"][[1, 4]], cand, keep, env.icpmod.RELOCALIZE_COARSE_ITERS)


@pytest.mark.parametrize("coarse", [1, 3, 30])
def test_other_coarse_iterations_and_clamped_inf_ranges(env, coarse):
    ranges = env.w["ranges"][[2, 6, 7]].copy()
    ranges[:, 5::23] = np.inf
    _check_staged(env, ranges, _sample(env.fine, 3000, coarse), 64, coarse, clamp=30.0)


def test_it_finds_the_robot(env):
    """The default coarse_iters with the keep INTEGRATION.md recommends, on the full grid."""
    w = env.w
    keep = env.icpmod.RELOCALIZE_KEEP_RECOMMENDED
    best, pose, score, it, kept = env.icp.relocalize(w["ranges"], w["candidates"], A0, A1, keep=keep)
    assert kept.shape == (8, keep) and (best >= 0).all()
    d_xy = np.hypot(pose[:, 0] - w["poses"][:, 0], pose[:, 1] - w["poses"][:, 1])
    d_yaw = np.abs((pose[:, 2] - w["poses"][:, 2] + math.pi) % (2 * math.pi) - math.pi)
    assert d_xy.max() < 0.10, d_xy
    assert d_yaw.max() < 0.05, d_yaw


def test_errors_repeatability_and_one_scan(env):
    w = env.w
    icp = env.icp
    cand = _sample(env.fine, 1500, 21)
    ranges = w["ranges"][6:8]
    first = icp.relocalize(ranges, cand, A0, A1, keep=40, return_T=True)
    for kw in ({"keep": 0}, {"keep": -1}, {"keep": 4, "coarse_iters": 0}, {"keep": 4, "coarse_iters": 31},
               {"keep": 4, "coarse_iters": 11, "max_iter": 10}, {"coarse_iters": 3}):
        with pytest.raises(ValueError):
            icp.relocalize(ranges, cand, A0, A1, **kw)
    with pytest.raises(ValueError, match="2\\^31 - 1"):  # K * M' > 2^31 - 1, before any device work
        icp.relocalize(np.ones((70000, 1), dtype=np.float32), np.zeros((40000, 3)), A0, A1, angle_increment=0.1,
                       keep=40000)
    bad = cand.copy()
    bad[123, 2] = np.nan
    with pytest.raises(ValueError, match=NAN_TEXT):
        icp.relocalize(ranges, bad, A0, A1, keep=8)
    with pytest.raises(ValueError, match="2304"):
        icp.relocalize(np.ones((1, 2305), dtype=np.float32), cand, A0, A1, keep=8)
    with pytest.raises(ValueError):
        icp.relocalize(ranges, cand[:0], A0, A1, keep=8)
    with pytest.raises(ValueError):
        icp.relocalize(ranges, cand[:, :2], A0, A1, keep=8)
    with pytest.raises(ValueError, match="no static map"):
        env.b2slam.ICP().relocalize(ranges, cand, A0, A1, keep=8)
    again = icp.relocalize(ranges, cand, A0, A1, keep=40, return_T=True)
    for a, b in zip(first, again):
        assert a.tobytes() == b.tobytes()
    one = icp.relocalize(ranges[1], cand, A0, A1, keep=40, return_T=True)
    assert one[0].shape == () and one[1].shape == (3,) and one[2].shape == one[3].shape == one[4].shape == (40,)
    assert one[5].shape == (40, 3, 3)
    for a, b in zip(one, first):
        assert a.tobytes() == b[1].tobytes()


def _crafted_coarse(K, H, seed):
    """Scores on a coarse grid of values (so that many tie), with -0 and +0, NaN and +-inf scores, and non-finite T."""
    rng = np.random.Generator(np.random.PCG64(seed))
    score = rng.integers(0, max(2, H // 8), size=(K, H)).astype(np.float64) * 0.125 - 0.5
    T = np.zeros((K, H, 3, 3))
    T[..., 0, 0] = T[..., 1, 1] = T[..., 2, 2] = 1.0
    n_bad = max(1, H // 50)
    for k in range(K):
        zs = rng.choice(H, min(H, 6), replace=False)
        score[k, zs[::2]] = -0.0
        score[k, zs[1::2]] = 0.0
        idx = rng.choice(H, min(H, 4 * n_bad), replace=False)
        score[k, idx[0::4]] = np.nan
        score[k, idx[1::4]] = np.inf
        score[k, idx[2::4]] = -np.inf
        T[k, idx[3::4], 1, 2] = np.nan
    return score, T


@pytest.mark.parametrize("K,H", [(64, 1), (1, 57600), (64, 2000), (1, 2 ** 20 + 3)])
def test_layer1_keep_kernel(env, K, H):
    score, T = _crafted_coarse(K, H, K * 7 + H)
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    ds, dT = cuda(score), cuda(T)
    for keep in sorted({1, 3, max(1, H // 3), H - 1 if H > 1 else 1, H, H + 9}):
        kept = env.dev.relocalize_keep(ds, dT, keep)
        torch.cuda.synchronize()
        assert np.array_equal(kept.cpu().numpy(), _keep_ref(score, T, keep)), keep


def test_layer1_keep_ties_straddle_the_boundary(env):
    """Equal scores around rank keep go to the lower h; -0 and +0 are one value; non-finite ones go last, by h."""
    H = 40
    score = np.full((3, H), 2.0)
    T = np.zeros((3, H, 3, 3))
    score[0, [30, 5, 17, 2]] = 1.0         # 4 below, then 36 tied at 2.0: keep 6 takes 2, 5, 17, 30 and h 0, 1
    score[1, ::2] = -0.0                   # 20 tied zeros of both signs
    score[1, 1::2] = 0.0
    score[1, [3, 4]] = np.nan
    score[2, :] = np.inf                   # nothing finite: the first keep by h
    score[2, 7] = 5.0
    T[2, 8, 0, 0] = np.nan
    score[2, 8] = 0.1
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    kept = env.dev.relocalize_keep(cuda(score), cuda(T), 6)
    torch.cuda.synchronize()
    kept = kept.cpu().numpy()
    assert kept[0].tolist() == [0, 1, 2, 5, 17, 30]
    assert kept[1].tolist() == [0, 1, 2, 5, 6, 7]
    assert kept[2].tolist() == [0, 1, 2, 3, 4, 7]
    assert np.array_equal(kept, _keep_ref(score, T, 6))


def test_layer1_selection_with_kept(env):
    rng = np.random.Generator(np.random.PCG64(5))
    C, K, M = 500, 4, 9
    cand = np.stack([rng.uniform(-5, 5, C), rng.uniform(-5, 5, C), rng.uniform(-math.pi, math.pi, C)], axis=1)
    kept = np.sort(np.stack([rng.choice(C, M, replace=False) for _ in range(K)]), axis=1).astype(np.int32)
    score = rng.uniform(0.1, 1.0, size=(K, M))
    th = rng.uniform(-0.2, 0.2, size=(K, M))
    T = np.zeros((K, M, 3, 3))
    T[..., 0, 0] = T[..., 1, 1] = np.cos(th)
    T[..., 1, 0], T[..., 0, 1] = np.sin(th), -np.sin(th)
    T[..., 0, 2], T[..., 1, 2], T[..., 2, 2] = 0.1, -0.2, 1.0
    score[0, [6, 2, 8]] = 0.01             # ties: the lowest j, which is the lowest original h
    score[1, 0] = np.nan                   # non-finite ones never win
    score[1, 1] = -np.inf
    T[1, 2, 0, 1] = np.inf
    score[1, 2] = 0.001
    score[2, :] = np.nan                   # nothing finite
    T[3, :, 1, 2] = np.nan
    cuda = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
    best, pose = env.dev.relocalize_select(cuda(score), cuda(T), cuda(cand), kept=cuda(kept))
    torch.cuda.synchronize()
    best, pose = best.cpu().numpy(), pose.cpu().numpy()
    j1 = 3 + int(np.argmin(score[1, 3:]))
    assert best.tolist() == [kept[0, 2], kept[1, j1], -1, -1]
    assert np.isnan(pose[2:]).all()
    for k, j in ((0, 2), (1, j1)):
        x, y, yaw = cand[kept[k, j]]
        t = T[k, j]
        want = (x + math.cos(yaw) * t[0, 2] - math.sin(yaw) * t[1, 2],
                y + math.sin(yaw) * t[0, 2] + math.cos(yaw) * t[1, 2], yaw + math.atan2(t[1, 0], t[0, 0]))
        np.testing.assert_allclose(pose[k], want, rtol=0, atol=1e-12)
