"""Mapping's host-buffer pipeline (b2s_mapping_update* / submit* / wait) at every pipeline depth.

Every entry point, at the automatic chunk count and with b2s_tune("h2d_chunks", k) forcing k chunks, must apply a good
batch exactly as the oracle does, and take a rejected batch -- a NaN in the first or the last scan, an inf in oy, a beam
longer than B2S_MAX_PATH_CELLS -- back out of the counts to the byte, with the status code and error text of its kind.
A streamed step submitted behind a rejected one stays applied."""
import ctypes
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

G, RESO = 1024, 0.05
K, N = 3000, 360        # 1.08 M beams: more than one ~1 M-beam chunk at the automatic depth
SMALL = 16              # scans of the good step submitted behind a rejected streamed one
CHUNKS = (0, 1, 3, 16)  # 0: automatic

NAN_TEXT = "cannot convert float NaN to integer"
INF_TEXT = "cannot convert float infinity to integer"
LONG_TEXT = "1 beam(s) longer than %d cells: batch rejected" % (1 << 22)


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, scan, synth
    from oracle import corc
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.lib, e.scan, e.corc = b2slam, _lib, scan, corc
    S, Hx, Hy = devapi.grid_scale(G, G, RESO)
    e.beam_cs = scan.beam_table(-math.pi, math.pi, N)
    e.pts = synth.grid_scans(71, K, N, half_extent_m=20.0)
    e.ranges, e.poses = synth.grid_scan_ranges(72, K, N, half_extent_m=20.0)

    def oracle(form, s1):
        oh = np.zeros((G, G), dtype=np.int32)
        om = np.zeros((G, G), dtype=np.int32)
        if form == "pts":
            e.corc.grid_raycast(oh, om, S, Hx, Hy, *[a[:s1] for a in e.pts])
        else:
            e.corc.grid_raycast_ranges(oh, om, S, Hx, Hy, e.ranges[:s1], scan.pose_table(e.poses[:s1]), e.beam_cs, 30.0)
        return oh, om
    e.want = {form: oracle(form, K) for form in ("pts", "ranges")}
    e.small = {form: oracle(form, SMALL) for form in ("pts", "ranges")}
    return e


# ----------------------------------------------------------------------------- entry points
# Each takes (env, Mapping, batch) and returns the int8 map of the call, or raises what the Mapping methods raise.
# Endpoint batches are (ox, oy, cx, cy), raw batches (ranges, poses).

def _checked(env, m, rc):
    m._raise_nonfinite(rc)
    env.lib.check(rc)


def _update_batch_f32(env, m, b):
    return m.update_batch(*b)


def _update_batch_f64(env, m, b):
    return m.update_batch(*[a.astype(np.float64) for a in b])


def _update_incremental(env, m, b):
    """Mapping.update's call (b2s_mapping_update_incremental_f64) with the whole batch, so that it is chunked."""
    ox, oy, cx, cy = [np.ascontiguousarray(a, dtype=np.float64) for a in b]
    count = ctypes.c_int(-1)
    tiles = np.empty(1024, dtype=np.int32)
    p = env.lib.ptr
    _checked(env, m, m._L.b2s_mapping_update_incremental_f64(m._h, p(ox), p(oy), p(cx), p(cy), ox.shape[0], ox.shape[1],
                                                             p(m._pmap8), p(tiles), tiles.shape[0], ctypes.byref(count)))
    return m._pmap8


def _update_scans(env, m, b):
    return m.update_scans(b[0], b[1], -math.pi, math.pi)


def _update_ranges(env, m, b):
    """b2s_mapping_update_ranges: the pose table [x, y, cos, sin] made by the caller."""
    ranges, table = np.ascontiguousarray(b[0], dtype=np.float32), env.scan.pose_table(b[1])
    p = env.lib.ptr
    _checked(env, m, m._L.b2s_mapping_update_ranges(m._h, p(ranges), p(table), p(env.beam_cs), 30.0, ranges.shape[0],
                                                    ranges.shape[1], p(m._pmap8)))
    return m._pmap8


def _submit_batch(env, m, b):
    return m.submit_batch(*b)


def _submit_scans(env, m, b):
    return m.submit_scans(b[0], b[1], -math.pi, math.pi)


BLOCKING = {"update_batch_f32": (_update_batch_f32, "pts"), "update_batch_f64": (_update_batch_f64, "pts"),
            "update_incremental": (_update_incremental, "pts"), "update_scans": (_update_scans, "ranges"),
            "update_ranges": (_update_ranges, "ranges")}
STREAMED = {"submit_batch": (_submit_batch, "pts"), "submit_scans": (_submit_scans, "ranges")}


def _good(env, form, s1=K):
    return tuple(a[:s1] for a in (env.pts if form == "pts" else (env.ranges, env.poses)))


def _bad(env, form):
    """(name, batch, exception, status, error text) of every rejected batch of one input form."""
    nan = (ValueError, env.lib.ERR_NONFINITE, NAN_TEXT)
    inf = (OverflowError, env.lib.ERR_NONFINITE, INF_TEXT)
    too_long = (env.lib.B2SlamError, env.lib.ERR_TOO_LONG, LONG_TEXT)
    if form == "pts":   # (name, array of (ox, oy, cx, cy), scan, beam, value, verdict)
        good = env.pts
        cases = [("nan in the first scan", 1, 0, 5, np.nan, nan), ("nan in the last scan", 1, K - 1, 7, np.nan, nan),
                 ("inf in oy", 1, K // 2, 3, np.inf, inf), ("beam too long", 0, K // 2, 4, 3e30, too_long)]
    else:               # (name, array of (ranges, poses), ...)
        good = (env.ranges, env.poses)
        cases = [("nan in the first scan", 0, 0, 5, np.nan, nan), ("nan in the last scan", 0, K - 1, 7, np.nan, nan),
                 ("range too long", 0, K // 2, 4, 3e30, too_long)]
    for name, i, s, j, v, verdict in cases:
        b = list(good)
        b[i] = b[i].copy()
        b[i][s, j] = v
        yield (name, tuple(b)) + verdict


def _expect_rejected(env, exc, status, text, fn):
    with pytest.raises(exc) as info:
        fn()
    if exc is env.lib.B2SlamError:
        assert info.value.status == status
    assert env.lib.lib().b2s_last_error().decode() == text


@pytest.fixture(params=CHUNKS)
def chunks(env, request):
    """Forces the pipeline depth of the call under test (0: automatic)."""
    L = env.lib.lib()
    assert L.b2s_tune(b"h2d_chunks", request.param) == 0
    try:
        yield request.param
    finally:
        L.b2s_tune(b"h2d_chunks", 0)


def _same_counts(m, h, ms):
    h1, m1 = m.counts()
    return np.array_equal(h1, h) and np.array_equal(m1, ms)


@pytest.mark.parametrize("entry", sorted(BLOCKING))
def test_blocking_call_applies_and_rolls_back(env, entry, chunks):
    fn, form = BLOCKING[entry]
    oh, om = env.want[form]
    pmap = env.corc.grid_finalize(oh, om)[1]
    m = env.b2slam.Mapping(G, G, RESO)
    pm = fn(env, m, _good(env, form))
    assert _same_counts(m, oh, om)
    assert np.array_equal(pm, pmap)
    for name, b, exc, status, text in _bad(env, form):
        _expect_rejected(env, exc, status, text, lambda: fn(env, m, b))
        assert _same_counts(m, oh, om), name
        assert np.array_equal(m._pmap8, pmap), name       # the map read back is that of the restored counts


@pytest.mark.parametrize("entry", sorted(STREAMED))
def test_streamed_step_applies_and_rolls_back(env, entry, chunks):
    fn, form = STREAMED[entry]
    oh, om = [a.copy() for a in env.want[form]]
    dh, dm = env.small[form]
    m = env.b2slam.Mapping(G, G, RESO)
    assert np.array_equal(fn(env, m, _good(env, form)).wait(), env.corc.grid_finalize(oh, om)[1])
    assert _same_counts(m, oh, om)
    for name, b, exc, status, text in _bad(env, form):
        t_bad = fn(env, m, b)
        t_ok = fn(env, m, _good(env, form, SMALL))           # submitted while the rejected step is in flight
        _expect_rejected(env, exc, status, text, t_bad.wait)
        t_ok.wait()
        oh += dh
        om += dm
        assert _same_counts(m, oh, om), name
