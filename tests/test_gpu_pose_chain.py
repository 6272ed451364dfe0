"""pose_chain_kernel (b2s_pose_chain, csrc/b2s_next.cu) against the long-double chain of test_pose_chain_host.

The kernel splits the pairs over 1024 threads in segments of per = ceil(pairs / 1024) and joins them with three block
scans (yaw, x, y).  Every finite entry must lie within chain_bound(m = 2 per + C_DEVICE) of the reference, and every
entry must be of the reference's class (finite, NaN, +inf, -inf): entries stay below 1e300, so no finite sum overflows
and IEEE sums give the same class in any order.  Rows before a non-finite transform must be finite, as in the
sequential loop: a NaN or inf in a thread's own segment must not reach the offset it starts from.

Layer 1 calls b2s_pose_chain on torch tensors on a non-default stream, into a trajectory pre-filled with a NaN of a
payload the kernel never writes, so an unwritten row shows.  The host calls (scan.compose_odometry_gpu, ICP.odometry,
ICP.process_scans with a state) are held to the reference of the transforms they return."""
import math

import numpy as np
import pytest

from test_pose_chain_host import (IDENTITY_STARTS, SHAPES, START, SYNTHETIC, LD, chain_bound, check_chain, classes,
                                  device_m, reference_chain, rigid, segments, tiled)

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SENTINEL = 0x7FF8B2C50FF1CE00   # a quiet NaN with a payload no arithmetic produces
NONFINITE_PAIRS = (2047, 3072, 10 ** 6)   # per 2, 3 and 977
ENTRIES = {"T00": 0, "T10": 3, "T02": 2, "T12": 5}
BAD = {"nan": math.nan, "+inf": math.inf, "-inf": -math.inf}
HOST_MAX = 100003                          # the largest chain the host-buffer form runs here


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, scan, synth
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.lib, e.L, e.scan, e.synth = _lib, _lib.lib(), scan, synth
    e.icp = b2slam.ICP()
    e.stream = torch.cuda.Stream()
    xy, _ = synth.room_sequence(9001, 3074, 360)
    e.room = e.icp.process_batch(xy[:-1], xy[1:])[0]   # cfg-2: 3073 consecutive pairs
    return e


def device_chain(env, T, state):
    """b2s_pose_chain on env.stream.  T: (P, 9) float64 CUDA tensor or (P, 3, 3) array.  Returns (P + 1, 3) float64
    and checks that the kernel wrote every entry."""
    Td = T if torch.is_tensor(T) else torch.from_numpy(np.ascontiguousarray(T, dtype=np.float64).reshape(-1, 9)).cuda()
    P = Td.shape[0]
    traj = torch.full(((P + 1) * 3,), SENTINEL, dtype=torch.int64, device="cuda")
    s = env.stream
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        env.lib.check(env.L.b2s_pose_chain(Td.data_ptr() if P else None, P, float(state[0]), float(state[1]),
                                           float(state[2]), traj.data_ptr(), s.cuda_stream))
    s.synchronize()
    bits = traj.cpu().numpy()
    unwritten = np.flatnonzero(bits == SENTINEL)
    assert unwritten.size == 0, "%d entries never written, first in row %d" % (unwritten.size, unwritten[0] // 3)
    return bits.view(np.float64).reshape(P + 1, 3)


def _family(env, name, P):
    if name == "room":
        return tiled(env.room, P), START
    return SYNTHETIC[name](np.random.Generator(np.random.PCG64(P + 1)), P)


def _first_bad_pair(T):
    bad = np.flatnonzero(~np.isfinite(np.asarray(T).reshape(-1, 9)[:, list(ENTRIES.values())]).all(axis=1))
    return int(bad[0]) if bad.size else np.asarray(T).reshape(-1, 9).shape[0]


def check_nonfinite(got, T, ref, bound, what):
    """ref, bound: of the chain without its non-finite transforms.  Rows up to the first non-finite pair j are finite
    and within the bound; past it, every entry is of the class of the reference continued from row j over T[j:]."""
    j = _first_bad_pair(T)
    fin = np.isfinite(got[:j + 1]).all(axis=1)
    assert fin.all(), "%s: row %d is not finite, the first non-finite pair is %d" % (what, int(np.argmin(fin)), j)
    tail = reference_chain(T[j:], ref[j])[1:]
    check_chain(got, np.concatenate([ref[:j + 1], tail]),
                np.concatenate([bound[:j + 1], np.full(tail.shape, np.inf, dtype=LD)]), what)


# ----------------------------------------------------------------------------- finite chains at every segment shape

@pytest.mark.parametrize("P", SHAPES)
@pytest.mark.parametrize("name", ["room"] + sorted(SYNTHETIC))
def test_chain_within_bound(env, name, P):
    T, state = _family(env, name, P)
    ref, bound = reference_chain(T, state), chain_bound(T, state, device_m(P))
    got = device_chain(env, T, state)
    assert got[0].tobytes() == np.array(state, dtype=np.float64).tobytes()
    check_chain(got, ref, bound, "%s P=%d" % (name, P))
    if P <= HOST_MAX:
        check_chain(env.scan.compose_odometry_gpu(state, T), ref, bound, "compose_odometry_gpu %s P=%d" % (name, P))


@pytest.mark.parametrize("P", SHAPES)
def test_identity_transforms_keep_the_start(env, P):
    """Every row equals the start bit for bit (a +0.0 start stays +0.0)."""
    T = rigid(np.zeros(P), 0.0, 0.0)
    Td = torch.from_numpy(T.reshape(-1, 9)).cuda()
    for state in IDENTITY_STARTS:
        want = np.tile(np.array(state, dtype=np.float64), (P + 1, 1)).tobytes()
        assert device_chain(env, Td, state).tobytes() == want, state
        if P <= HOST_MAX:
            assert env.scan.compose_odometry_gpu(state, T).tobytes() == want, state


# ----------------------------------------------------------------------------- non-finite transforms and starts

def _placements(P):
    """(thread, pair): the first, a middle and the last pair of the segments of thread 0, a middle active thread and
    the last active thread."""
    per, lo, hi = segments(P)
    active = np.flatnonzero(hi > lo)
    out = []
    for t in (0, int(active[active.size // 2]), int(active[-1])):
        for j in sorted({int(lo[t]), int(lo[t] + (hi[t] - lo[t]) // 2), int(hi[t] - 1)}):
            out.append((t, j))
    return out


def check_one_bad_pair(got, clean, T, j, ref, what):
    """One non-finite value, in pair j.  Rows up to j are those of the same call without it (`clean`, held to the
    bound by the caller) and finite; rows j + 1 and j + 2 are of the classes of the reference continued from row j;
    every later row keeps the classes of row j + 2, because past one non-finite value each sum only adds finite terms
    to a non-finite one (a NaN yaw at row j + 1 makes x and y NaN from row j + 2)."""
    fin = np.isfinite(got[:j + 1]).all(axis=1)
    assert fin.all(), "%s: row %d is not finite, the first non-finite pair is %d" % (what, int(np.argmin(fin)), j)
    same = (got[:j + 1] == clean[:j + 1]).all(axis=1)
    assert same.all(), "%s: row %d differs from the chain without the non-finite value" % (what, int(np.argmin(same)))
    near = classes(reference_chain(T[j:j + 2], ref[j])[1:])
    want = np.concatenate([near, np.repeat(near[-1:], got.shape[0] - j - 1 - near.shape[0], axis=0)])
    bad = np.argwhere(classes(got[j + 1:]) != want)
    assert bad.size == 0, "%s: %d entries of another class than the reference's, first at row %d col %d: %r" % (
        what, bad.shape[0], j + 1 + bad[0][0], bad[0][1], got[j + 1 + bad[0][0]])


@pytest.mark.parametrize("P", NONFINITE_PAIRS)
def test_one_nonfinite_transform(env, P):
    """NaN, +inf and -inf in each of T00, T10, T02, T12, at the first, a middle and the last pair of a segment of the
    first, a middle and the last active thread."""
    T = tiled(env.room, P)
    ref, bound = reference_chain(T, START), chain_bound(T, START, device_m(P))
    Td = torch.from_numpy(T.reshape(-1, 9)).cuda()
    clean = {"device": device_chain(env, Td, START)}
    if P <= HOST_MAX:
        clean["host"] = env.scan.compose_odometry_gpu(START, T)
    for name, got in clean.items():
        check_chain(got, ref, bound, "%s P=%d without a non-finite value" % (name, P))
    per, lo, hi = segments(P)
    failed, cases = [], 0
    for t, j in _placements(P):
        assert lo[t] <= j < hi[t]                                    # the pair landed in the thread it is meant for
        for ename, e in ENTRIES.items():
            for vname, v in BAD.items():
                what = "P=%d thread %d pair %d (segment [%d, %d)) %s=%s" % (P, t, j, lo[t], hi[t], ename, vname)
                Tb = T.copy()
                Tb.reshape(-1, 9)[j, e] = v
                Td[j, e] = v
                try:
                    runs = {"device": device_chain(env, Td, START)}
                finally:
                    Td[j, e] = float(T.reshape(-1, 9)[j, e])
                if P <= HOST_MAX:
                    runs["host"] = env.scan.compose_odometry_gpu(START, Tb)
                for name, got in runs.items():
                    cases += 1
                    try:
                        check_one_bad_pair(got, clean[name], Tb, j, ref, "%s %s" % (name, what))
                    except AssertionError as err:
                        failed.append(str(err).splitlines()[0])
    assert not failed, "%d of %d cases:\n%s" % (len(failed), cases, "\n".join(failed))


@pytest.mark.parametrize("P", NONFINITE_PAIRS)
def test_two_nonfinite_translations(env, P):
    """+inf in one pair's T02 and -inf in a later segment's: the x sums meet inf - inf, NaN from there on."""
    T = tiled(env.room, P)
    ref, bound = reference_chain(T, START), chain_bound(T, START, device_m(P))
    per, lo, hi = segments(P)
    j1 = int(lo[1] + (hi[1] - lo[1]) // 2)
    cos = np.cos(ref[:-1, 2])
    later = [int(lo[t] + (hi[t] - lo[t]) // 2) for t in range(600, 1024) if hi[t] > lo[t]]
    j2 = next(j for j in later if np.sign(cos[j]) == np.sign(cos[j1]))   # same sign: +inf and -inf reach x
    Tb = T.copy()
    Tb[j1, 0, 2], Tb[j2, 0, 2] = np.inf, -np.inf
    tail = reference_chain(Tb[j1:], ref[j1])
    assert np.isnan(tail[j2 - j1 + 1:, 0]).all()
    check_nonfinite(device_chain(env, Tb, START), Tb, ref, bound, "P=%d pairs %d, %d" % (P, j1, j2))
    if P <= HOST_MAX:
        check_nonfinite(env.scan.compose_odometry_gpu(START, Tb), Tb, ref, bound, "host P=%d" % P)


@pytest.mark.parametrize("state", [(math.nan, -0.25, 0.1), (math.inf, -0.25, 0.1), (0.5, -math.inf, 0.1),
                                   (0.5, -0.25, math.nan), (0.5, -0.25, math.inf), (0.5, -0.25, -math.inf)],
                         ids=["x0_nan", "x0_inf", "y0_-inf", "th0_nan", "th0_inf", "th0_-inf"])
def test_nonfinite_start(env, state):
    for P in (1, 3072):
        T = tiled(env.room, P)
        ref, bound = reference_chain(T, state), chain_bound(T, state, device_m(P))
        got = device_chain(env, T, state)
        assert got[0].tobytes() == np.array(state, dtype=np.float64).tobytes()
        check_chain(got, ref, bound, "P=%d" % P)
        check_chain(env.scan.compose_odometry_gpu(state, T), ref, bound, "host P=%d" % P)


# ----------------------------------------------------------------------------- through the ICP's host calls

@pytest.fixture
def tuning(env):
    L = env.L
    yield L
    assert L.b2s_tune(b"h2d_chunks", 0) == 0


@pytest.mark.parametrize("chunks", (0, 1, 3, 16))
def test_odometry_chain_waits_for_every_chunk(env, tuning, chunks):
    """ICP.odometry at 3000 float64 scans (per 3): the trajectory is the chain of the transforms it returns, whichever
    of the two compute streams solved them.  The stream run backwards first leaves other transforms in the device
    buffer, so a chain that started before the last chunk was solved would not match."""
    K = 3000
    xy = env.synth.room_sequence(9001, K, 360)[0].astype(np.float64)
    assert tuning.b2s_tune(b"h2d_chunks", chunks) == 0
    env.icp.odometry(np.ascontiguousarray(xy[::-1]), state=START)
    traj, T, _ = env.icp.odometry(xy, state=START)
    assert segments(K - 1)[0] == 3 and np.isfinite(T).all()
    check_chain(traj, reference_chain(T, START), chain_bound(T, START, device_m(K - 1)), "chunks %d" % chunks)


def test_process_scans_chain_over_nonfinite_ranges(env):
    """process_scans without the inf clamp at 4200 scans (per 5): one NaN range and one +inf range, each in a scan
    whose pair as the source lands mid-segment, give non-finite transforms; the trajectory keeps the rows before
    them finite and continues like the reference."""
    K = 4200
    per, lo, hi = segments(K - 1)
    assert per == 5
    xy, _ = env.synth.room_sequence(9002, K, 360)
    ranges = np.hypot(xy[:, 0], xy[:, 1]).astype(np.float32)
    s_nan, s_inf = 5 * 300 + 2, 5 * 700 + 3                        # pairs 1501 and 3502: inside segments 300 and 700
    ranges[s_nan, 17] = np.nan
    ranges[s_inf, 200] = np.inf
    traj, T, _ = env.icp.process_scans(ranges, -math.pi, math.pi, clamp_inf_to=None, state=START)
    for s in (s_nan, s_inf):
        t = (s - 1) // per
        assert lo[t] < s - 1 < hi[t] - 1
        assert not np.isfinite(T[s - 1].reshape(9)[list(ENTRIES.values())]).all(), s
    clean = T.copy()
    clean[~np.isfinite(clean)] = 0.0
    check_nonfinite(traj, T, reference_chain(clean, START), chain_bound(clean, START, device_m(K - 1)), "process_scans")
