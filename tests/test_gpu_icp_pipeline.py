"""ICP's host-buffer pipeline (b2s_icp_process / _process_sequence / _odometry / _process_scans / _submit_*) at every
pipeline depth.

Every call, at the automatic chunk count and with b2s_tune("h2d_chunks", k) forcing k chunks, must give bit for bit
the transforms and iteration counts of process_batch on the explicit consecutive pairs at one chunk; the raw-range
calls those of process_batch on the laser_to_points clouds of their ranges.  A trajectory must equal that of the same
pose chain at one chunk."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K, N = 3000, 360        # float64 points: more than one automatic chunk for the pair and the point-sequence forms
KR = 4200               # raw ranges get more than one automatic chunk only from their floor of 4, at >= 4096 pairs
SECOND = 1200           # scans of the call submitted while the first one is in flight
SHORT = 5               # a stream with fewer pairs than 16 chunks
CHUNKS = (0, 1, 3, 16)  # 0: automatic
STATE = (0.5, -0.25, 0.1)


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, scan, synth
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.lib, e.icp = _lib, b2slam.ICP()
    e.xy = synth.room_sequence(9001, K, N)[0].astype(np.float64)
    e.src = np.ascontiguousarray(e.xy[1:, :, ::2])   # unequal sizes: 180 source points against 360 target points
    xy, _ = synth.room_sequence(9002, KR, N)
    ranges = np.hypot(xy[:, 0], xy[:, 1]).astype(np.float32)
    inf = ranges.copy()
    rng = np.random.Generator(np.random.PCG64(5))
    inf[rng.integers(0, KR, 40), rng.integers(0, N, 40)] = np.inf
    e.ranges = {None: ranges, 30.0: inf}
    L = _lib.lib()
    assert L.b2s_tune(b"h2d_chunks", 1) == 0
    try:
        e.want = {}
        for dt in (np.float32, np.float64):
            e.want["batch", dt] = e.icp.process_batch(e.xy[:-1].astype(dt), e.src.astype(dt)) + (None,)
        e.want["points"] = e.icp.process_batch(e.xy[:-1], e.xy[1:]) + (e.icp.odometry(e.xy, state=STATE)[0],)
        for clamp, r in e.ranges.items():
            clouds = np.stack([scan.laser_to_points(s, -math.pi, math.pi, clamp_inf_to=clamp)[:2] for s in r])
            e.want["raw", clamp] = (e.icp.process_batch(clouds[:-1], clouds[1:])
                                    + (e.icp.odometry(clouds, state=STATE)[0],))
    finally:
        L.b2s_tune(b"h2d_chunks", 0)
    return e


def _head(want, scans):
    """The wanted transforms and iteration counts of a call on the first `scans` scans (no trajectory)."""
    return want[0][:scans - 1], want[1][:scans - 1], None


# ----------------------------------------------------------------------------- calls
# Each takes env and returns [(T, iterations, trajectory or None, wanted (T, iterations, trajectory or None))].

def _batch(dt):
    def run(e):
        T, it = e.icp.process_batch(e.xy[:-1].astype(dt), e.src.astype(dt))
        return [(T, it, None, e.want["batch", dt])]
    return run


def _sequence(e):
    return [e.icp.process_sequence(e.xy) + (None, _head(e.want["points"], K))]


def _odometry(e):
    traj, T, it = e.icp.odometry(e.xy, state=STATE)
    return [(T, it, traj, e.want["points"])]


def _scans(clamp, state):
    def run(e):
        out = e.icp.process_scans(e.ranges[clamp], -math.pi, math.pi, clamp_inf_to=clamp,
                                  state=STATE if state else None)
        if state:
            return [(out[1], out[2], out[0], e.want["raw", clamp])]
        return [out + (None, _head(e.want["raw", clamp], KR))]
    return run


def _submit_sequence(e):
    t1 = e.icp.submit_sequence(e.xy)
    t2 = e.icp.submit_sequence(e.xy[:SECOND])
    T1, it1 = [a.copy() for a in t1.wait()]
    return [(T1, it1, None, _head(e.want["points"], K)), t2.wait() + (None, _head(e.want["points"], SECOND))]


def _submit_scans(e):
    t1 = e.icp.submit_scans(e.ranges[None], -math.pi, math.pi)
    t2 = e.icp.submit_scans(e.ranges[30.0][:SECOND], -math.pi, math.pi, clamp_inf_to=30.0)
    T1, it1 = [a.copy() for a in t1.wait()]
    return [(T1, it1, None, _head(e.want["raw", None], KR)), t2.wait() + (None, _head(e.want["raw", 30.0], SECOND))]


CALLS = {"process_batch_f32": _batch(np.float32), "process_batch_f64": _batch(np.float64),
         "process_sequence": _sequence, "odometry": _odometry,
         "process_scans": _scans(None, False), "process_scans_clamp": _scans(30.0, False),
         "process_scans_state": _scans(None, True), "process_scans_clamp_state": _scans(30.0, True),
         "submit_sequence": _submit_sequence, "submit_scans": _submit_scans}


@pytest.fixture(params=CHUNKS)
def chunks(env, request):
    """Forces the pipeline depth of the call under test (0: automatic)."""
    L = env.lib.lib()
    assert L.b2s_tune(b"h2d_chunks", request.param) == 0
    try:
        yield request.param
    finally:
        L.b2s_tune(b"h2d_chunks", 0)


def _same(got, want):
    return got.shape == want.shape and got.dtype == want.dtype and got.tobytes() == want.tobytes()


def _check(results):
    for i, (T, it, traj, (wT, wit, wtraj)) in enumerate(results):
        assert _same(it, wit), i
        assert _same(T, wT), i
        if wtraj is not None:
            assert _same(traj, wtraj), i


@pytest.mark.parametrize("call", sorted(CALLS))
def test_call_equals_the_pair_form_at_one_chunk(env, call, chunks):
    _check(CALLS[call](env))


def test_short_stream_at_sixteen_chunks(env):
    """16 forced chunks of a 5-scan stream: the depth is clamped to its 4 pairs."""
    e = env
    L = e.lib.lib()
    assert L.b2s_tune(b"h2d_chunks", 16) == 0
    try:
        points, raw = _head(e.want["points"], SHORT), _head(e.want["raw", 30.0], SHORT)
        results = [e.icp.process_batch(e.xy[:SHORT - 1], e.xy[1:SHORT]) + (None, points),
                   e.icp.process_sequence(e.xy[:SHORT]) + (None, points),
                   e.icp.odometry(e.xy[:SHORT], state=STATE)[1:] + (None, points),
                   e.icp.process_scans(e.ranges[30.0][:SHORT], -math.pi, math.pi, clamp_inf_to=30.0) + (None, raw),
                   e.icp.submit_sequence(e.xy[:SHORT]).wait() + (None, points)]
    finally:
        L.b2s_tune(b"h2d_chunks", 0)
    _check(results)
