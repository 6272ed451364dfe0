"""Which instance of the batched ICP kernel a call launches, and the oracle's score, checked without a GPU.

b2s_icp_dispatch is the library's one copy of the choice of (R source points per thread, search PRUNE, NN_BLK targets
per block) that b2s_icp_batch_f32 / _f64 / _f64_err / _ranges launch.  Every search mode gives the same bits by
design, so a wrong choice shows in no result: it is compared here with a model written from the dispatch's comments,
over every scan size up to 2304 and every value of the ICP tuning keys.  The model also gives the reachable instance
sets that tests/test_gpu_icp_instances.py must cover on the device.

orc_icp_batch_err, the oracle's score (the mean error of the last iteration, [ICP]:75), is checked against the
literal reference loop."""
import ctypes
import functools
import math

import numpy as np
import pytest

from b2slam import _lib

QSUP_MIN, QBLOCKS, MAX_POINTS = 64, 254, 2304
PRUNES, BLOCKS, SPTS = (0, 1, 2, 3, 4), (0, 8, 16, 32), (0, 2, 3, 4)
DEFAULT_TUNING = {"icp_prune": 4, "icp_block": 0, "icp_src_per_thread": 0, "icp_layout": 2}


def set_tuning(L, **keys):
    for k, v in keys.items():
        assert L.b2s_tune(k.encode(), int(v)) == 0, (k, v)


def restore_tuning(L):
    set_tuning(L, **DEFAULT_TUNING)


# ---------------------------------------------------------------------------------------------------- the model

def _cdiv(a, b):
    return -(-a // b)


def _threads(n, r):
    return max(64, _cdiv(_cdiv(n, r), 32) * 32)


def points_per_thread(n, spt):
    """R: forced by icp_src_per_thread, else 3 unless it takes over 10 % more register slots (threads x R, idle ones
    included) than the leanest choice, then 4, then 2; a CTA holds at most 768 threads (R <= 3) or 576 (R = 4)."""
    if spt:
        return spt
    slots = {c: _threads(n, c) * c for c in (2, 3, 4) if _threads(n, c) <= (768 if c <= 3 else 576)}
    least = min(slots.values())
    return next((c for c in (3, 4, 2) if c in slots and slots[c] * 10 <= least * 11), 3)


def smem_bytes(prune, blk, r, m, in_bytes, threads):
    """The CTA's dynamic shared memory: header, reduction scratch, staged input rows (reused for the block bounds),
    then the padded targets, moved sources and per-warp queues of the queued search, or the plain target array."""
    nblk = _cdiv(m, blk)
    stage = (max(in_bytes, (nblk + _cdiv(nblk, 32)) * 16) + 15) // 16 * 16
    b = 16 + max(2 * (threads // 32) * 10, 128) * 8 + stage
    if prune >= 4:
        b += nblk * (blk + 1) * 16 + r * threads * 16 + (threads // 32) * r * 3 * 32 * 12
    else:
        b += m * 16
    return b


def model_dispatch(n_src, n_tar, in_bytes, ranges, prune, block, spt):
    """(R, PRUNE, NN_BLK) of one call, or None where the library refuses it."""
    if n_src <= 0 or n_tar <= 0 or in_bytes not in (4, 8) or (ranges and (n_src != n_tar or in_bytes != 4)):
        return None
    if n_src > MAX_POINTS:
        return None
    r = points_per_thread(n_src, spt)
    q8, q16 = _cdiv(n_tar, 8), _cdiv(n_tar, 16)
    queued8 = (5 if q8 > QSUP_MIN else 4, 8)
    queued16 = (5 if q16 > QSUP_MIN else 4, 16)
    if ranges:
        # queued for icp_prune 4 (8-target blocks by default), the collective search (PRUNE 2) for every other value
        blk = block or (8 if prune == 4 or n_tar <= 600 else 16)
        if prune == 4 and blk == 8 and q8 <= QBLOCKS:
            p, b = queued8
        elif prune == 4 and q16 <= QBLOCKS:
            p, b = queued16
        else:
            p, b = 2, blk
    else:
        blk = block or (8 if prune == 4 else (8 if n_tar <= 600 else 16) if prune >= 2 else (16 if n_tar <= 600 else 32))
        fits = _cdiv(n_tar, blk) * 16 <= 2 * n_tar * in_bytes  # the block bounds reuse the staged input rows
        if prune == 0 or not fits:
            p, b = 0, 16
        elif prune == 4 and blk == 8 and q8 <= QBLOCKS:
            p, b = queued8
        elif prune == 4 and q16 <= QBLOCKS:
            p, b = queued16
        elif prune >= 2:
            p, b = (3 if prune == 3 else 2), blk
        else:
            p, b = 1, (32 if blk == 32 else 16)
    threads = _threads(n_src, r)
    if threads > 1024:
        return None
    if smem_bytes(p, b, r, n_tar, (1 if ranges else 2) * n_tar * in_bytes, threads) > 227 * 1024:
        return None
    return r, p, b


@functools.lru_cache(maxsize=None)
def reachable_instances():
    """{"scored": the float64 instances (b2s_icp_batch_f64_err), "ranges": the raw-range instances} that any scan
    size N = n_src = n_tar <= 2304 reaches under any tuning, by the model."""
    out = {"scored": set(), "ranges": set()}
    for prune in PRUNES:
        for block in BLOCKS:
            for spt in SPTS:
                for n in range(1, MAX_POINTS + 1):
                    for key, ib, rg in (("scored", 8, False), ("ranges", 4, True)):
                        got = model_dispatch(n, n, ib, rg, prune, block, spt)
                        if got is not None:
                            out[key].add(got)
    return {k: frozenset(v) for k, v in out.items()}


def default_boundaries():
    """Beam counts N at which the default float64 instance (N = n_src = n_tar) differs from that of N - 1."""
    prev, out = None, []
    for n in range(1, MAX_POINTS + 1):
        got = model_dispatch(n, n, 8, False, 4, 0, 0)
        if prev is not None and got != prev:
            out.append(n)
        prev = got
    return out


def library_dispatch(L, n_src, n_tar, in_bytes, ranges):
    r, p, b = ctypes.c_int(-1), ctypes.c_int(-1), ctypes.c_int(-1)
    rc = L.b2s_icp_dispatch(n_src, n_tar, in_bytes, int(ranges), ctypes.byref(r), ctypes.byref(p), ctypes.byref(b))
    if rc != _lib.OK:
        assert rc == _lib.ERR_INVALID_ARG, rc
        return None
    return r.value, p.value, b.value


# ---------------------------------------------------------------------------------------------------- dispatch

@pytest.fixture
def L():
    L = _lib.lib()
    restore_tuning(L)
    try:
        yield L
    finally:
        restore_tuning(L)


@pytest.mark.parametrize("prune", PRUNES)
def test_dispatch_table_equals_the_model(L, prune):
    """Every N = n_src = n_tar in 1..2304 (and 2305, refused), every icp_block and icp_src_per_thread, float32 and
    float64 clouds and raw ranges."""
    for block in BLOCKS:
        for spt in SPTS:
            set_tuning(L, icp_prune=prune, icp_block=block, icp_src_per_thread=spt)
            for ib, rg in ((4, False), (8, False), (4, True)):
                for n in range(1, MAX_POINTS + 2):
                    want = model_dispatch(n, n, ib, rg, prune, block, spt)
                    assert library_dispatch(L, n, n, ib, rg) == want, (n, ib, rg, prune, block, spt)


def test_dispatch_with_unequal_clouds_and_refusals(L):
    """n_src != n_tar (targets up to the shared-memory limit, where icp_prune 4 leaves the queued search), and the
    arguments the calls refuse."""
    rng = np.random.Generator(np.random.PCG64(2024))
    refused = 0
    for _ in range(4000):
        prune, block, spt = int(rng.choice(PRUNES)), int(rng.choice(BLOCKS)), int(rng.choice(SPTS))
        n_src, n_tar = int(rng.integers(1, 2400)), int(rng.integers(1, 9000))
        ib = int(rng.choice([4, 8]))
        set_tuning(L, icp_prune=prune, icp_block=block, icp_src_per_thread=spt)
        want = model_dispatch(n_src, n_tar, ib, False, prune, block, spt)
        refused += want is None
        assert library_dispatch(L, n_src, n_tar, ib, False) == want, (n_src, n_tar, ib, prune, block, spt)
    assert refused > 100
    restore_tuning(L)
    for args in ((0, 5, 8, 0), (5, 0, 8, 0), (5, 5, 2, 0), (5, 5, 16, 0), (5, 6, 4, 1), (5, 5, 8, 1), (2305, 5, 8, 0),
                 (2305, 2305, 4, 1), (-1, 5, 8, 0)):
        assert library_dispatch(L, *args) is None, args
    r = ctypes.c_int()
    assert L.b2s_icp_dispatch(5, 5, 8, 0, None, ctypes.byref(r), ctypes.byref(r)) == _lib.ERR_INVALID_ARG
    # the shared-memory limit: float64 targets beyond about 7000 points
    assert library_dispatch(L, 100, 7000, 8, False) is not None and library_dispatch(L, 100, 7500, 8, False) is None


def test_default_instances_and_their_boundaries(L):
    """The default instance of a relocalization or an odometry stream (N beams on both sides): R changes from 2 to 3
    at 129 beams, the second level of the warp test starts at 65 blocks of 8 (513 beams) and 16-target blocks at
    255 blocks of 8 (2033 beams); a single float32 point has no room for its block bound and takes the brute force."""
    inst = {n: library_dispatch(L, n, n, 8, False) for n in range(1, MAX_POINTS + 1)}
    assert {inst[n] for n in inst} == {(2, 4, 8), (3, 4, 8), (4, 4, 8), (3, 5, 8), (3, 5, 16)}
    b = default_boundaries()
    assert 129 in b and inst[128] == (2, 4, 8) and inst[129] == (3, 4, 8)
    assert 513 in b and inst[512][1] == 4 and inst[513] == (3, 5, 8)
    assert 2033 in b and inst[2032] == (3, 5, 8) and inst[2033] == (3, 5, 16)
    assert all(inst[n] == (3, 5, 8) for n in range(513, 2033)) and all(inst[n] == (3, 5, 16) for n in range(2033, 2305))
    assert inst[100] == (2, 4, 8) and inst[200] == (4, 4, 8) and inst[360] == (3, 4, 8) and inst[1080] == (3, 5, 8)
    assert library_dispatch(L, 1, 1, 4, False) == (2, 0, 16) and library_dispatch(L, 1, 1, 8, False) == (2, 4, 8)
    assert library_dispatch(L, 2, 2, 4, False) == (2, 4, 8)
    assert library_dispatch(L, 1, 1, 4, True) == (2, 4, 8)  # (the raw form stages no points: no such test)


def test_reachable_instance_sets():
    """39 scored instances (R 2..4 x the 13 (PRUNE, NN_BLK) of the point form) and 21 raw-range ones (R x (4, 8),
    (5, 8), (4, 16), (5, 16) and the collective (2, 8 / 16 / 32))."""
    got = reachable_instances()
    pb = {(5, 8), (4, 8), (5, 16), (4, 16), (3, 8), (3, 16), (3, 32), (2, 8), (2, 16), (2, 32), (1, 16), (1, 32), (0, 16)}
    assert got["scored"] == {(r, p, b) for r in (2, 3, 4) for p, b in pb}
    pb = {(4, 8), (5, 8), (4, 16), (5, 16), (2, 8), (2, 16), (2, 32)}
    assert got["ranges"] == {(r, p, b) for r in (2, 3, 4) for p, b in pb}


# ---------------------------------------------------------------------------------------------------- oracle score

def score_bound(n, ref):
    """Two sums of the same n non-negative float64 distances, one left to right, one by a tree, differ by at most
    2 (n - 1) 2^-53 times their sum; each is then divided by n (one rounding each)."""
    return 2.0 * (n - 1) * 2.0 ** -53 * abs(ref) + 2.0 * np.spacing(abs(ref))


def _nearest(src, tar):
    """pyref.nearest_targets_vec with the reference loop's rule for non-finite distances ([ICP]:99-106): a NaN never
    wins (np.argmin would take it), and a point that matches nothing keeps index 0 and distance 0."""
    from oracle import pyref
    if np.isfinite(src).all() and np.isfinite(tar).all():
        return pyref.nearest_targets_vec(src, tar)
    with np.errstate(invalid="ignore"):
        dx = src[:, None, 0] - tar[None, :, 0]
        dy = src[:, None, 1] - tar[None, :, 1]
        d = np.sqrt(dx * dx + dy * dy)
    d = np.where(np.isnan(d), np.inf, d)
    which = np.argmin(d, axis=1)
    dist = d[np.arange(src.shape[0]), which]
    which = np.where(np.isfinite(dist), which, 0)
    return np.where(np.isfinite(dist), dist, 0.0), which


def _fit(src, tar):
    """pyref.rigid_fit_svd; its closed form where the matched points are not finite (the SVD does not converge on
    them, the reference's fit gives NaN there like the closed form)."""
    from oracle import pyref
    if np.isfinite(src).all() and np.isfinite(tar).all():
        return pyref.rigid_fit_svd(src, tar)
    with np.errstate(invalid="ignore"):
        return pyref.rigid_fit_closed_form(src, tar)


def reference_loop(tar, src, max_iter=30, tolerance=1e-3):
    """The literal reference loop ([ICP]:38-88) on one pair, tar (2,M), src (2,N): (T, iterations, mean_error of the
    last iteration)."""
    first = np.array(src, dtype=np.float64)
    cur = np.ones((3, first.shape[1]))
    cur[:2] = first
    tar = np.asarray(tar, dtype=np.float64)
    prev_err, err, done = 0, 0.0, 0
    for _ in range(max_iter):
        dist, idx = _nearest(cur[:2].T, tar.T)
        with np.errstate(invalid="ignore"):
            cur = np.dot(_fit(cur[:2].T, tar[:, idx].T), cur)
        done += 1
        err = np.sum(dist) / dist.size
        if abs(prev_err - err) < tolerance:
            break
        prev_err = err
    with np.errstate(invalid="ignore"):
        return _fit(first.T, cur[:2].T), done, err


def _pairs(seed, count, n, m):
    rng = np.random.Generator(np.random.PCG64(seed))
    tar = rng.normal(0.0, 3.0, (count, 2, m))
    pick = rng.integers(0, m, (count, n))
    src = np.take_along_axis(tar, pick[:, None, :].repeat(2, axis=1), axis=2).copy()
    th = rng.uniform(-0.1, 0.1, count)[:, None]
    c, s = np.cos(th), np.sin(th)
    src = np.stack([c * src[:, 0] - s * src[:, 1] + 0.1, s * src[:, 0] + c * src[:, 1] - 0.05], axis=1)
    return tar, src + rng.normal(0.0, 0.02, src.shape)


@pytest.mark.parametrize("n,m", [(1, 1), (1, 7), (5, 3), (17, 40), (64, 64), (100, 37)])
@pytest.mark.parametrize("max_iter,tol", [(30, 1e-3), (1, 1e-3), (4, 0.0)])
def test_oracle_score_is_the_reference_mean_error(n, m, max_iter, tol):
    from oracle import corc
    tar, src = _pairs(n * 1000 + m, 4, n, m)
    if m > 2:
        tar[1, 0, 1] = np.nan
        tar[2, :, m - 1] = np.inf
        tar[3, 1, 0] = -np.inf
    if n > 2:
        src[3, :, n // 2] = np.inf  # a beam with an infinite range, no clamp: it matches nothing
    T, it, err = corc.icp_batch(tar, src, max_iter, tol, return_err=True)
    T0, it0 = corc.icp_batch(tar, src, max_iter, tol)
    assert T.tobytes() == T0.tobytes() and it.tobytes() == it0.tobytes()  # the old entry is unchanged
    for p in range(4):
        rT, rit, rerr = reference_loop(tar[p], src[p], max_iter, tol)
        assert it[p] == rit, (p, it[p], rit)
        if tol == 0.0:
            assert rit == max_iter
        np.testing.assert_allclose(T[p], rT, rtol=0, atol=1e-9)
        if max_iter == 1:  # the same distances summed in another order; pyref squares them without the fused
            # multiply-add of the oracle and the kernel, which moves each by at most one rounding of the square root
            assert abs(err[p] - rerr) <= score_bound(n, rerr) + 2.0 ** -52 * abs(rerr), (p, err[p], rerr)
        else:
            assert math.isclose(err[p], rerr, rel_tol=1e-9, abs_tol=1e-12), (p, err[p], rerr)


def test_oracle_score_edges():
    from oracle import corc
    tar, src = _pairs(5, 2, 9, 11)
    T, it, err = corc.icp_batch(tar, src, 0, 1e-3, return_err=True)
    assert (it == 0).all() and (err == 0).all() and np.array_equal(T, np.broadcast_to(np.identity(3), (2, 3, 3)))
    # a source cloud on top of its targets: mean error 0 in the first iteration, which stops it
    T, it, err = corc.icp_batch(tar, tar, 30, 1e-3, return_err=True)
    assert (it == 1).all() and (err == 0).all()
