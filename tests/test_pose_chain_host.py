"""The odometry pose chain of [ICP]:185-190 / [LOC9]:79-83 on the host (no GPU): a long-double reference, a bound on
the rounding error of any float64 evaluation of the chain, and the segmentation of pose_chain_kernel
(csrc/b2s_next.cu).

The chain over transforms T_0 .. T_{P-1} from (x0, y0, th0) is
    th_k = th0 + sum_{i<k} atan2(T10_i, T00_i)
    x_k  = x0 + sum_{i<k} (cos th_i T02_i - sin th_i T12_i),   y_k = y0 + sum_{i<k} (sin th_i T02_i + cos th_i T12_i),
each step rotated by the yaw BEFORE it.  The sequential loop (scan.compose_odometry, pyref.compose_pose) and the
device's blocked scan add the same terms in different orders; both must lie within chain_bound of reference_chain.
The checks here hold the loop and the reference's own publishResult golden to the bound and show that the bound
rejects chains wrong by one step; tests/test_gpu_pose_chain.py holds the kernel to it and imports these helpers."""
import math

import numpy as np
import pytest

from conftest import load_golden

LD = np.longdouble
U = 2.0 ** -53                       # float64 unit roundoff
U_LD = float(np.finfo(LD).eps) / 2   # long double unit roundoff (2^-64 for x87 80-bit)
THREADS = 1024                       # CHAIN_THREADS: one CTA
# Additions any summand passes through on its way to a row of pose_chain_kernel, besides the 2 * per of the
# segments: 5 in the warp scan, 5 in the cross-warp scan, 1 joining the warp's offset to the lane's, 1 adding the start.
# (The segment partial and the in-segment steps are at most per each.)
C_DEVICE = 12
C_TERM = 8                           # cos / sin (2 ulp each), two products and the difference of one increment, in u
ATAN2_ULP = 2                        # CUDA's double atan2 bound; glibc's is tighter
TINY = 2.0 ** -1073                  # 2 ulp of a subnormal dth

# the pair counts the device checks run: per 1, 2, 3, 4, 32, 98 and 977, idle tail threads and warp edges
SHAPES = (0, 1, 2, 31, 32, 33, 1023, 1024, 1025, 2047, 2048, 2049, 3072, 3073, 32767, 100003, 10 ** 6)


def segments(pairs):
    """pose_chain_kernel's split of `pairs` over its threads: (per, lo (THREADS,), hi (THREADS,)); thread t owns the
    pairs [lo[t], hi[t]), an empty range for the idle threads at the tail."""
    per = -(-int(pairs) // THREADS)
    lo = np.minimum(pairs, np.arange(THREADS, dtype=np.int64) * per)
    return per, lo, np.minimum(pairs, lo + per)


def device_m(pairs):
    """Longest chain of float64 additions into a row of pose_chain_kernel: the segment partial, the two block scans,
    the start state and the steps inside the segment."""
    return 2 * segments(pairs)[0] + C_DEVICE


def sequential_m(pairs):
    """Per row k, the additions into row k of the sequential loop.  `x + cos(th) * T02 - sin(th) * T12` evaluates
    left to right, (x + a) - b: x passes through two additions per step and th through one, so m = 2k (0 at the
    start row, which is the state itself)."""
    return 2 * np.arange(int(pairs) + 1)


def rigid(dth, tx, ty):
    """(P, 3, 3) float64 transforms [[cos, -sin, tx], [sin, cos, ty], [0, 0, 1]], the form the ICP returns."""
    dth, tx, ty = np.broadcast_arrays(*(np.asarray(v, dtype=np.float64) for v in (dth, tx, ty)))
    T = np.zeros(dth.shape + (3, 3))
    T[..., 0, 0], T[..., 0, 1], T[..., 0, 2] = np.cos(dth), -np.sin(dth), tx
    T[..., 1, 0], T[..., 1, 1], T[..., 1, 2] = np.sin(dth), np.cos(dth), ty
    T[..., 2, 2] = 1.0
    return T


def _flat(T):
    return np.asarray(T, dtype=np.float64).reshape(-1, 9)


def _exclusive_cumsum(v):
    out = np.zeros(v.shape[0] + 1, dtype=v.dtype)
    np.cumsum(v, out=out[1:])
    return out


def reference_chain(T, state):
    """(P + 1, 3) long double x, y, th of the chain over the float64 transforms T (P, 3, 3) from `state` (float64 or
    long double), evaluated in long double and vectorised."""
    assert np.finfo(LD).nmant >= 63, "the reference needs at least the x87 80-bit long double"
    T = _flat(T).astype(LD)
    x0, y0, th0 = (LD(v) for v in state)
    with np.errstate(invalid="ignore", over="ignore"):
        th = th0 + _exclusive_cumsum(np.arctan2(T[:, 3], T[:, 0]))
        c, s = np.cos(th[:-1]), np.sin(th[:-1])
        x = x0 + _exclusive_cumsum(c * T[:, 2] - s * T[:, 5])
        y = y0 + _exclusive_cumsum(s * T[:, 2] + c * T[:, 5])
    return np.stack([x, y, th], axis=1)


def _error(T, state, m, u):
    gamma = m * u / (1 - m * u)
    with np.errstate(invalid="ignore", over="ignore"):
        dth = np.abs(np.arctan2(T[:, 3], T[:, 0]))
        t = np.abs(T[:, 2]) + np.abs(T[:, 5])
        e_th = gamma * (abs(state[2]) + _exclusive_cumsum(dth)) + _exclusive_cumsum(ATAN2_ULP * 2 * u * dth + TINY)
        steps = (1 + gamma) * _exclusive_cumsum((e_th[:-1] + C_TERM * u) * t)  # E_th(i): the yaw before step i
        e_x = gamma * (abs(state[0]) + _exclusive_cumsum(t)) + steps
        e_y = gamma * (abs(state[1]) + _exclusive_cumsum(t)) + steps
    return np.stack([e_x, e_y, e_th], axis=1)


def chain_bound(T, state, m):
    """(P + 1, 3) long double: for every row k and entry (x, y, th), the allowed |float64 result - reference_chain|
    of an evaluation in which every summand reaches row k through at most m (a scalar, or one value per row)
    float64 additions.

    A sum evaluated along any tree in which each summand passes through at most m roundings errs by at most
    gamma_m * sum |summands| (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., 4.2),
    gamma_m = m u / (1 - m u), u = 2^-53.

    Yaw: the summands are th0 and the computed dth_i, each within 2 ulp (<= 4 u |dth_i|) of atan2, so
        E_th(k) = gamma_m (|th0| + sum_{i<k} |dth_i|) + sum_{i<k} 2 ulp(dth_i).
    Position: the increment of step i is evaluated at the computed yaw th_i, off by at most E_th(i); cos and sin are
    1-Lipschitz, so that moves it by at most E_th(i) (|T02_i| + |T12_i|).  cos and sin (2 ulp each), the two products
    and the difference add at most c u (|T02_i| + |T12_i|), c = C_TERM.  The computed increments are then summed as
    above, and they exceed |T02_i| + |T12_i| by at most those errors:
        E_x(k) = gamma_m (|x0| + sum_{i<k} (|T02_i| + |T12_i|)) + (1 + gamma_m) sum_{i<k} (E_th(i) + c u)(|T02_i| + |T12_i|),
    and E_y(k) alike with |y0|.

    m is device_m(pairs) = 2 per + C_DEVICE for pose_chain_kernel and sequential_m(pairs) for the loop.  The same
    bound in long double (u = 2^-64) at m = k + 1, the additions of the reference's cumulative sums, is added: it is
    the reference's own distance from the exact chain.  Rows past a non-finite transform get a NaN or inf bound;
    their entries are compared by class."""
    T = _flat(T).astype(LD)
    state = [LD(v) for v in state]
    k = np.arange(T.shape[0] + 1)
    m = np.broadcast_to(np.asarray(m, dtype=LD), k.shape)
    return _error(T, state, m, LD(U)) + _error(T, state, (k + 1).astype(LD), LD(U_LD))


def classes(a):
    """0 finite, 1 NaN, 2 +inf, 3 -inf, elementwise."""
    a = np.asarray(a)
    return np.select([np.isfinite(a), np.isnan(a), a > 0], [0, 1, 2], 3)


def check_chain(got, ref, bound, what=""):
    """got (P + 1, 3) float64 against the reference: the same class in every entry, and every finite entry within
    the bound.  Returns the largest |error| / bound over the finite entries."""
    got = np.asarray(got)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    cg, cr = classes(got), classes(ref)
    bad = np.argwhere(cg != cr)
    assert bad.size == 0, "%s: %d entries of another class, first at row %d col %d: got %r, reference %r" % (
        what, bad.shape[0], bad[0][0], bad[0][1], got[tuple(bad[0])], ref[tuple(bad[0])])
    fin = cg == 0
    err = np.abs(got[fin].astype(LD) - ref[fin])
    over = err > bound[fin]
    if over.any():
        rows = np.argwhere(fin)[over]
        i = int(np.argmax(over))
        raise AssertionError("%s: %d finite entries outside the bound, first at row %d col %d: error %.3g, bound %.3g"
                             % (what, rows.shape[0], rows[0][0], rows[0][1], float(err[i]), float(bound[fin][i])))
    return float((err / np.maximum(bound[fin], LD(1e-300))).max()) if err.size else 0.0


# ----------------------------------------------------------------------------- families

START = (0.5, -0.25, 0.1)


def spinning(rng, P):
    """dth ~ N(0, 0.3): the yaw wanders to thousands of radians at 10^5 - 10^6 pairs."""
    return rigid(rng.normal(0, 0.3, P), rng.normal(0.05, 0.03, P), rng.normal(0, 0.03, P)), START


def rotations(rng, P):
    return rigid(rng.uniform(-math.pi, math.pi, P), 0.0, 0.0), START


def translations(rng, P):
    return rigid(0.0, rng.normal(0, 0.1, P), rng.normal(0, 0.1, P)), START


def large_start(rng, P):
    """|x0|, |y0|, |th0| ~ 1e4 with small steps."""
    return rigid(rng.normal(0, 0.02, P), rng.normal(0.05, 0.02, P), rng.normal(0, 0.02, P)), (1.25e4, -9.5e3, 1.1e4)


def tiled(base, P):
    """The first P transforms of `base` repeated."""
    return np.tile(base, (-(-P // base.shape[0]), 1, 1))[:P]


SYNTHETIC = {"spinning": spinning, "rotations": rotations, "translations": translations, "large_start": large_start}
IDENTITY_STARTS = ((0.0, 0.0, 0.0), (1.5, -2.25, 0.7), (-3.0e4, 7.0e-3, -2.5e3))


@pytest.fixture(scope="module")
def room():
    """cfg-2 room chain: the oracle's transforms of 512 consecutive pairs of room_sequence(9001)."""
    from b2slam import synth
    from oracle import corc
    xy, _ = synth.room_sequence(9001, 513, 360)
    T, _ = corc.icp_batch(xy[:-1], xy[1:], 30, 1e-3)
    return T


def _sequential(T, state):
    from b2slam import scan
    return scan.compose_odometry(state, T)


# ----------------------------------------------------------------------------- checks

def test_long_double_is_wide_enough():
    assert np.finfo(LD).nmant >= 63


def test_segments_are_the_kernels():
    for P in SHAPES:
        per, lo, hi = segments(P)
        assert per == (P + THREADS - 1) // THREADS and device_m(P) == 2 * per + C_DEVICE
        assert lo[0] == 0 and hi[-1] == P and np.array_equal(lo[1:], hi[:-1])  # consecutive, covering [0, P)
        assert (hi - lo <= per).all() and (hi >= lo).all()
        active = int((hi > lo).sum())
        assert active == -(-P // per) if P else active == 0
        assert (hi[:active] - lo[:active] == per)[:-1].all()                    # only the last active one is short
    assert [segments(P)[0] for P in (1, 1025, 2049, 3073, 32767, 100003, 10 ** 6)] == [1, 2, 3, 4, 32, 98, 977]
    per, lo, hi = segments(10 ** 6)
    assert int((hi > lo).sum()) == 1024 and hi[1023] - lo[1023] == 10 ** 6 - 1023 * 977
    per, lo, hi = segments(1000)
    assert int((hi > lo).sum()) == 1000                                          # 24 idle threads


def test_reference_is_the_loop_in_long_double():
    """reference_chain against a literal long-double loop of [ICP]:185-190 on a short chain."""
    rng = np.random.Generator(np.random.PCG64(11))
    T, state = spinning(rng, 300)
    ref = reference_chain(T, state)
    x, y, th = (LD(v) for v in state)
    for k in range(300):
        t = T[k].astype(LD)
        assert abs(ref[k, 0] - x) <= 1e-15 and abs(ref[k, 1] - y) <= 1e-15 and abs(ref[k, 2] - th) <= 1e-15, k
        x, y, th = (x + np.cos(th) * t[0, 2] - np.sin(th) * t[1, 2], y + np.sin(th) * t[0, 2] + np.cos(th) * t[1, 2],
                    th + np.arctan2(t[1, 0], t[0, 0]))


@pytest.mark.parametrize("P", (1, 2, 1000, 100000))
@pytest.mark.parametrize("family", sorted(SYNTHETIC) + ["room"])
def test_sequential_loop_within_bound(family, P, room):
    if family == "room":
        T, state = tiled(room, P), START
    else:
        T, state = SYNTHETIC[family](np.random.Generator(np.random.PCG64(P)), P)
    got = _sequential(T, state)
    check_chain(got, reference_chain(T, state), chain_bound(T, state, sequential_m(P)), family)
    if P <= 1000:                                                                 # the literal port, step by step
        from oracle import pyref
        st = tuple(state)
        for k in range(P):
            st = pyref.compose_pose(st, T[k])
            assert st == tuple(got[k + 1])


def test_identity_chain_keeps_the_start_exactly():
    for state in IDENTITY_STARTS:
        got = _sequential(rigid(np.zeros(1000), 0.0, 0.0), state)
        assert got.tobytes() == np.tile(np.array(state), (1001, 1)).tobytes(), state


def test_reference_publishResult_golden_within_bound():
    z = load_golden("next_rows.npz")
    T, state = z["chain_T"], tuple(z["chain_start"])
    check_chain(z["chain_traj"], reference_chain(T, state), chain_bound(T, state, sequential_m(T.shape[0])), "golden")


def _outside(wrong, ref, bound):
    with np.errstate(invalid="ignore"):
        return np.abs(np.asarray(wrong, dtype=LD) - ref) > bound


@pytest.mark.parametrize("P", (3072, 100003))
def test_bound_rejects_wrong_chains(P, room):
    """At the device's m for P pairs, the bound rejects the room chain with one pair's translation dropped, with each
    step rotated by the yaw after it, and with one yaw off by 1e-9 rad."""
    T, state = tiled(room, P), START
    ref, bound = reference_chain(T, state), chain_bound(T, state, device_m(P))
    j = P // 2 + 1
    dropped = T.copy()
    dropped[j, :2, 2] = 0.0
    assert _outside(reference_chain(dropped, state), ref, bound)[j + 1:, :2].any(axis=1).all()
    assert not _outside(reference_chain(dropped, state), ref, bound)[:j + 1].any()
    th = ref[:, 2]
    Tl = T.reshape(-1, 9).astype(LD)
    c, s = np.cos(th[1:]), np.sin(th[1:])
    after = np.stack([state[0] + _exclusive_cumsum(c * Tl[:, 2] - s * Tl[:, 5]),
                      state[1] + _exclusive_cumsum(s * Tl[:, 2] + c * Tl[:, 5]), th], axis=1)
    assert _outside(after, ref, bound)[1:, :2].any(axis=1).all()                   # every row after the first step
    off = ref.copy()
    off[j, 2] += LD(1e-9)
    assert _outside(off, ref, bound)[j, 2]
    assert not _outside(ref.astype(np.float64), ref, bound).any()
