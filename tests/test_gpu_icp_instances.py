"""Every instance of the batched ICP kernel that computes a relocalization score (b2s_icp_batch_f64_err) or solves raw
ranges (b2s_icp_batch_ranges), checked on the device against the C oracle.

b2s_icp_dispatch names the instance (R, PRUNE, NN_BLK) each call takes; tests/test_icp_instances_host.py pins it to a
model and derives the sets of instances that can be reached.  Here every one of them runs: the score must lie within
the rounding bound of the oracle's mean error of the last iteration, T within 1e-9, the iterations equal, and all of it
bit-identical across the search modes and block sizes.  The module fails if an instance of either set was not run."""
import math

import numpy as np
import pytest

from test_icp_instances_host import library_dispatch, reachable_instances, restore_tuning, score_bound, set_tuning

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

A0, A1 = -math.pi, math.pi
T_ATOL = 1e-9
REACHED = {"scored": set(), "ranges": set()}
TUNINGS = [(prune, block) for prune in (0, 1, 2, 3, 4) for block in (0, 8, 16, 32)]


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
    e.b2slam, e.L, e.dev, e.scan, e.synth, e.corc, e.pyref = b2slam, _lib.lib(), devapi, scan, synth, corc, pyref
    e.icp = b2slam.ICP()
    e.room = synth.room_relocalization(9001, 1, 360)  # the map and the candidate grid do not depend on the beam count
    e.icp.set_static_map(e.room["obstacles_course"])
    return e


@pytest.fixture(autouse=True)
def default_tuning(env):
    """Every test starts and ends with the default search, whatever it set or however it ended."""
    restore_tuning(env.L)
    try:
        yield
    finally:
        restore_tuning(env.L)


def _cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a), device="cuda")


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def check_score(score, want, n, T, want_T, src, max_iter):
    """score within the summation bound of the oracle's.  After the first iteration the two solves move the source
    points by transforms that differ in the last bits, so the distances of the last iteration differ by up to that
    movement: the disagreement of the final transforms at the source points, counted twice."""
    for p in range(len(score)):
        if np.isnan(want[p]):
            assert np.isnan(score[p]), p
            continue
        drift = 0.0
        if max_iter > 1:
            d = np.einsum("ij,jn->in", (T[p] - want_T[p])[:2], np.vstack([src[p], np.ones(src.shape[2])]))
            d = np.hypot(d[0], d[1])
            d = d[np.isfinite(d)]
            drift = 2.0 * float(d.max()) if d.size else 0.0
        assert abs(score[p] - want[p]) <= score_bound(n, want[p]) + drift, (p, score[p], want[p], drift)


# ---------------------------------------------------------------------------------------------------- scored layer 1

def _clouds(env, seed, pairs, n_src, n_tar):
    """float64 (pairs, 2, M) targets and (pairs, 2, N) sources from synth.icp_pairs (one room profile sampled at both
    densities); pair 1 has NaN and inf targets, pair 3 a NaN source point (it matches nothing), pair 2 starts 1.8 m off
    its targets, so that the first iteration's pruning bounds are loose."""
    tar = env.synth.icp_pairs(seed, pairs, n_tar)[0].astype(np.float64)
    src = env.synth.icp_pairs(seed, pairs, n_src)[1].astype(np.float64)
    tar[1, 0, 3] = np.nan
    tar[1, :, n_tar // 2] = np.inf
    tar[1, 1, n_tar - 1] = -np.inf
    src[2] += np.array([[1.5], [-1.0]])
    src[3, 0, n_src // 3] = np.nan
    return np.ascontiguousarray(tar), np.ascontiguousarray(src)


# n_tar chosen so that each R reaches all 13 (PRUNE, NN_BLK): 300 targets take the queued search with 8 and 16 targets
# per block (PRUNE 4), 600 the second-level warp test with 8 (PRUNE 5) and PRUNE 4 with 16, 1700 PRUNE 5 with both
# and more than 48 KB of shared memory for the collective searches; the 1500 sources of the first shape give the
# queued instances more than 48 KB as well.
SCORED_SHAPES = [(1500, 300), (97, 600), (200, 1700)]


@pytest.mark.parametrize("n_src,n_tar", SCORED_SHAPES)
def test_scored_instances_vs_oracle(env, n_src, n_tar):
    tar, src = _clouds(env, 7000 + n_tar, 4, n_src, n_tar)
    dtar, dsrc = _cuda(tar), _cuda(src)
    for max_iter, tol in ((30, 1e-3), (1, 1e-3), (5, 0.0)):
        oT, oit, oerr = env.corc.icp_batch(tar, src, max_iter, tol, return_err=True)
        if tol == 0.0:
            assert (oit == max_iter).all()
        for R in (2, 3, 4):
            first = None
            for prune, block in TUNINGS:
                set_tuning(env.L, icp_prune=prune, icp_block=block, icp_src_per_thread=R)
                inst = library_dispatch(env.L, n_src, n_tar, 8, False)
                assert inst is not None and inst[0] == R
                T, it, err = (t.cpu().numpy() for t in env.dev.icp_batch_err(dtar, dsrc, max_iter, tol))
                pT, pit = (t.cpu().numpy() for t in env.dev.icp_batch(dtar, dsrc, max_iter, tol))
                tag = (max_iter, tol, inst, prune, block)
                assert _same(T, pT) and np.array_equal(it, pit), tag
                if first is None:
                    first = (T, it, err)
                    assert np.array_equal(it, oit), (tag, it, oit)
                    np.testing.assert_allclose(T, oT, rtol=0, atol=T_ATOL, err_msg=str(tag))
                    check_score(err, oerr, n_src, T, oT, src, max_iter)
                else:  # bit-identical to every other search mode and block size, the score included
                    assert _same(T, first[0]) and np.array_equal(it, first[1]) and _same(err, first[2]), tag
                REACHED["scored"].add(inst)


def test_scored_misaligned_view(env):
    """Targets at an odd float64 offset (no bulk copy into shared memory) give the aligned call's bits."""
    n_src, n_tar = 97, 600
    tar, src = _clouds(env, 7600, 4, n_src, n_tar)
    buf = torch.empty(tar.size + 1, dtype=torch.float64, device="cuda")
    view = buf[1:].view(tar.shape)
    view.copy_(_cuda(tar))
    assert view.data_ptr() % 16 == 8 and view.is_contiguous()
    oT, oit, oerr = env.corc.icp_batch(tar, src, 30, 1e-3, return_err=True)
    for R in (2, 3, 4):
        set_tuning(env.L, icp_src_per_thread=R)
        want = [t.cpu().numpy() for t in env.dev.icp_batch_err(_cuda(tar), _cuda(src))]
        got = [t.cpu().numpy() for t in env.dev.icp_batch_err(view, _cuda(src))]
        assert all(_same(a, b) for a, b in zip(got, want)), R
        assert np.array_equal(got[1], oit)
        np.testing.assert_allclose(got[0], oT, rtol=0, atol=T_ATOL)
        check_score(got[2], oerr, n_src, got[0], oT, src, 30)


# ---------------------------------------------------------------------------------------------------- relocalization

# the default instances (2, 4, 8), (4, 4, 8), (3, 4, 8), (3, 5, 8), (3, 5, 16) and the beam counts on both sides of
# the boundaries of the dispatch: R 2 -> 3 (129), PRUNE 4 -> 5 (513), 8 -> 16 targets per block (2033)
RELOC_BEAMS = [100, 128, 129, 200, 360, 512, 513, 1080, 2032, 2033, 2304]


def _hypotheses(env, truth, count, seed):
    """`count` candidates: three within a few cm of the true pose of the scan, the rest drawn from the grid."""
    rng = np.random.Generator(np.random.PCG64(seed))
    grid = env.room["candidates"]
    cand = grid[np.sort(rng.choice(grid.shape[0], count, replace=False))].copy()
    cand[:3] = truth + np.array([[0.03, -0.02, 0.01], [-0.05, 0.04, -0.02], [0.0, 0.1, 0.03]])
    return cand


def _reference_score(env, cand, ranges):
    """The whole map observation by the literal reference: pyref's virtual scan and laserToNumpy, then the reference
    loop.  Returns (T, iterations, mean_error of the last iteration)."""
    from test_icp_instances_host import reference_loop
    p, n = env.pyref, len(ranges)
    virtual = p.virtual_scan(env.room["obstacles_course"], cand, A0, (A1 - A0) / (n - 1), n)
    return reference_loop(p.laser_to_points(virtual, A0, A1)[:2], p.laser_to_points(ranges, A0, A1)[:2])


@pytest.mark.parametrize("n", RELOC_BEAMS)
def test_relocalize_vs_oracle(env, n):
    w = env.synth.room_relocalization(9001, 1, n)
    count = 24 if n <= 600 else 8 if n <= 1200 else 3  # the oracle's work grows as n^2
    cand = _hypotheses(env, w["poses"][0], count, n)
    inst = library_dispatch(env.L, n, n, 8, False)
    for clamp in (None, 30.0):
        ranges = w["ranges"].copy()
        ranges[0, 5::17] = np.inf
        best, pose, score, it, T = env.icp.relocalize(ranges, cand, A0, A1, clamp_inf_to=clamp, return_T=True)
        H = len(cand)
        _, _, virt = env.icp.map_observation(np.repeat(ranges, H, axis=0), cand, A0, A1, clamp_inf_to=clamp,
                                             return_virtual=True)
        tar = np.stack([env.scan.laser_to_points(v, A0, A1)[:2] for v in virt])
        src = np.repeat(env.scan.laser_to_points(ranges[0], A0, A1, clamp_inf_to=clamp)[:2][None], H, axis=0)
        oT, oit, oerr = env.corc.icp_batch(tar, src, 30, 1e-3, return_err=True)
        assert np.array_equal(it[0], oit), (n, clamp)
        np.testing.assert_allclose(T[0], oT, rtol=0, atol=T_ATOL, err_msg=str((n, clamp)))
        check_score(score[0], oerr, n, T[0], oT, src, 30)
        if clamp is not None:
            assert best[0] >= 0
    REACHED["scored"].add(inst)
    # two hypotheses, one near the truth and one far, end to end against the literal reference loop (its virtual scan
    # takes hypot from libm, the device's from CUDA: last-bit differences, hence the tolerance of test_gpu_relocalize)
    ranges = w["ranges"][0]
    pick = cand[[0, count - 1]]
    _, _, score, it, T = env.icp.relocalize(ranges, pick, A0, A1, return_T=True)
    for h in range(2):
        rT, rit, rerr = _reference_score(env, pick[h], ranges)
        assert rit == it[h], (n, h)
        assert abs(score[h] - rerr) <= 1e-12, (n, h, score[h], rerr)
        np.testing.assert_allclose(T[h], rT, rtol=0, atol=T_ATOL)


@pytest.mark.parametrize("n", [1080, 2304])
def test_relocalize_keep(env, n):
    from test_gpu_relocalize_keep import _check_staged
    w = env.synth.room_relocalization(9001, 1, n)
    rng = np.random.Generator(np.random.PCG64(n))
    grid = env.room["candidates"]
    cand = np.ascontiguousarray(grid[np.sort(rng.choice(grid.shape[0], 600, replace=False))])
    ranges = w["ranges"].copy()
    ranges[0, 3::29] = np.inf
    _check_staged(env, ranges, cand, 16, 3, clamp=30.0)
    REACHED["scored"].add(library_dispatch(env.L, n, n, 8, False))


# ---------------------------------------------------------------------------------------------------- raw ranges

# 300 beams reach the queued (4, 8), (4, 16) and every collective instance, 700 (5, 8), 1100 (5, 16)
@pytest.mark.parametrize("n", [300, 700, 1100])
def test_raw_range_instances(env, n):
    xy, _ = env.synth.room_sequence(9300 + n, 6, n)
    base = np.hypot(xy[:, 0, :], xy[:, 1, :]).astype(np.float32)
    for clamp in (30.0, None):
        r = base.copy()
        if clamp is not None:
            r[[1, 3, 4], [7, n // 2, n - 1]] = np.inf
        else:
            r[[2, 5], [11, n // 3]] = np.nan
        clouds = np.stack([env.scan.laser_to_points(r[k], A0, A1, clamp_inf_to=clamp)[:2] for k in range(6)])
        oT, oit = env.corc.icp_batch(clouds[:-1], clouds[1:], 30, 1e-3)
        for R in (2, 3, 4):  # (R sets the order of the CTA's sums: the bits are R's)
            first = None
            for prune, block in TUNINGS:
                set_tuning(env.L, icp_prune=prune, icp_block=block, icp_src_per_thread=R)
                inst = library_dispatch(env.L, n, n, 4, True)
                assert inst is not None and inst[0] == R
                T, it = env.icp.process_scans(r, A0, A1, clamp_inf_to=clamp)
                want_T, want_it = env.icp.process_sequence(clouds)
                tag = (n, clamp, inst, prune, block)
                assert np.array_equal(it, want_it) and _same(T, want_T), tag
                if first is None:
                    first = (T, it)
                    assert np.array_equal(it, oit), tag
                    np.testing.assert_allclose(T, oT, rtol=0, atol=T_ATOL, err_msg=str(tag))
                else:
                    assert _same(T, first[0]) and np.array_equal(it, first[1]), tag
                REACHED["ranges"].add(inst)


# ---------------------------------------------------------------------------------------------------- coverage

def test_every_reachable_instance_ran():
    """(Last in the module: the tests above record the instances they ran.)"""
    want = reachable_instances()
    for key in ("scored", "ranges"):
        missing = sorted(want[key] - REACHED[key])
        assert not missing, "%s instances never run: %s" % (key, missing)
    assert len(want["scored"]) == 39 and len(want["ranges"]) == 21
