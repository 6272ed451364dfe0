"""GPU parity of the float64 endpoint path: Mapping.update / update_batch and b2s_grid_raycast[_ws]_f64 fed the
UNROUNDED float64 coordinates the reference's callers pass ([SLAM]:89-90), against goldens produced by the reference
itself at three grid scales (tests/golden/mapping_f64.npz, oracle/make_golden.py: mapping_f64_golden) and against the
float64 oracle.  Cell indices and counts are bit-exact; no input is rounded to float32 anywhere in this file except
where the float32 fast path is the thing under test."""
import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, synth
    from oracle import corc, pyref
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.lib, e.dev, e.synth, e.corc, e.pyref = b2slam, _lib, devapi, synth, corc, pyref
    return e


# (grid_variant, grid_tile_layout) of every kernel arm; variant 6 with layout 1 is the default that Mapping runs
ARMS = ((1, 1), (2, 1), (3, 1), (4, 1), (5, 1), (6, 0), (6, 1))
DEFAULT_ARM = (6, 1)


def _select(env, arm):
    L = env.lib.lib()
    assert L.b2s_tune(b"grid_variant", arm[0]) == 0 and L.b2s_tune(b"grid_tile_layout", arm[1]) == 0


@pytest.fixture(autouse=True)
def _default_kernel(env):
    """Every test starts on the default kernel and leaves it selected, whether it passes or fails."""
    _select(env, DEFAULT_ARM)
    try:
        yield
    finally:
        _select(env, DEFAULT_ARM)


def _sparse_check(hit, miss, z, tag, w_hit=20.0, suffix=""):
    cells = z[tag + "_cells" + suffix]
    h, m = hit.reshape(-1), miss.reshape(-1)
    touched = np.flatnonzero((h != 0) | (m != 0))
    assert np.array_equal(touched, cells), "touched cells differ from the reference's"
    score = 0.01 * m[cells].astype(np.float64) + w_hit * h[cells].astype(np.float64)
    np.testing.assert_allclose(score, z[tag + "_score" + suffix], rtol=1e-12, atol=0)


@pytest.mark.parametrize("tag", ["g200", "g4096", "g16384"])
def test_layer1_float64_raycast_equals_reference(env, tag):
    """b2s_grid_raycast_ws_f64 / b2s_grid_raycast_f64 with the reference's literals (10, 10, 10) on the reference's own
    float64 inputs; every kernel variant, with and without the workspace."""
    z = load_golden("mapping_f64.npz")
    side = int(z[tag + "_side"])
    ox, oy, cx, cy = (torch.from_numpy(np.ascontiguousarray(z[tag + k])).cuda() for k in ("_ox", "_oy", "_cx", "_cy"))
    assert ox.dtype == torch.float64
    ws = env.dev.new_workspace(side, side)
    arms = ARMS if side <= 4096 else ((4, 1), (5, 1), (6, 0), (6, 1))
    for arm in arms:
        _select(env, arm)
        # without a workspace b2s_grid_raycast_ws_f64 runs variant 3 whatever is selected
        for workspace in (ws, None):
            hit, miss = env.dev.new_planes(side, side)
            cnt = torch.zeros(4, dtype=torch.int32, device="cuda")
            env.dev.grid_raycast(hit, miss, 10.0, 10.0, 10.0, ox, oy, cx, cy, counters=cnt, workspace=workspace)
            torch.cuda.synchronize()
            c = cnt.cpu().numpy()
            assert c[0] == 0 and c[1] == 0 and c[3] == 0 and c[2] == int(np.isinf(z[tag + "_ox"]).sum()), arm
            _sparse_check(hit.cpu().numpy(), miss.cpu().numpy(), z, tag)
            pm = torch.empty((side, side), dtype=torch.int8, device="cuda")
            env.dev.grid_finalize(hit, miss, pmap=pm)
            pmh = pm.cpu().numpy().reshape(-1)
            assert np.array_equal(pmh[z[tag + "_cells"]], z[tag + "_pmap"]), arm
            rest = np.ones(side * side, dtype=bool)
            rest[z[tag + "_cells"]] = False
            assert (pmh[rest] == 50).all(), arm
            del hit, miss, pm


@pytest.mark.parametrize("w_hit,suffix", [(20.0, ""), (4.0, "_w4")])
def test_mapping_update_on_unrounded_float64_equals_reference(env, w_hit, suffix):
    """The drop-in call itself, scan by scan, exactly as the reference was called when the golden was made."""
    z = load_golden("mapping_f64.npz")
    m = env.b2slam.Mapping(200, 200, 0.1, hit_weight=w_hit)
    for ox, oy, cx, cy in zip(z["g200_ox"], z["g200_oy"], z["g200_cx"], z["g200_cy"]):
        pm = m.update(ox, oy, float(cx), float(cy))
    hit, miss = m.counts()
    _sparse_check(hit, miss, z, "g200", w_hit, suffix)
    want = np.full(200 * 200, 50, dtype=np.int8)
    want[z["g200_cells" + suffix]] = z["g200_pmap" + suffix]
    amb = env.pyref.boundary_ambiguous(hit, miss, w_hit).reshape(-1)
    assert ((pm.reshape(-1).astype(np.int8) == want) | amb).all()
    if w_hit == 20.0:
        assert np.array_equal(pm.reshape(-1).astype(np.int8), want)
    # the batched call on the same float64 arrays gives the same planes
    mb = env.b2slam.Mapping(200, 200, 0.1, hit_weight=w_hit)
    mb.update_batch(z["g200_ox"], z["g200_oy"], z["g200_cx"], z["g200_cy"])
    hb, msb = mb.counts()
    assert np.array_equal(hb, hit) and np.array_equal(msb, miss)


def test_decimal_cell_boundaries_single_scan(env):
    """ADVICE r1: 77 of the 199 multiples of 0.1 m in [-9.9, 9.9] change cell when narrowed to float32
    (9.9 -> 198 in float64, 199 after narrowing).  The drop-in must give the float64 answer for every one."""
    ticks = np.round(np.arange(-9.9, 9.95, 0.1), 1)
    want_cells = np.array([int(10 * (t + 10)) for t in ticks])
    narrowed = np.array([int(10 * (float(np.float32(t)) + 10)) for t in ticks])
    assert int((want_cells != narrowed).sum()) > 50
    m = env.b2slam.Mapping(200, 200, 0.1)
    m.update(ticks, np.full_like(ticks, 5.05), 0.05, -5.05)      # endpoints on row y = 150, sensor at (100, 49)
    hit, _ = m.counts()
    got = np.flatnonzero(hit[:, 150])
    assert np.array_equal(got, np.unique(want_cells))
    assert int(hit.sum()) == len(ticks)


def test_update_batch_dispatches_on_dtype(env):
    """float64 arrays: bit-identical to the float64 oracle (= the reference); float32 arrays: the float32 fast path,
    identical to the oracle on the float32 values; and the two differ on these inputs, i.e. the test can tell."""
    G = 4096
    rng = np.random.Generator(np.random.PCG64(515))
    K, N = 48, 1080
    cx = rng.uniform(-90, 90, K)
    cy = rng.uniform(-90, 90, K)
    ang = np.linspace(-np.pi, np.pi, N)
    r = rng.uniform(0.2, 29.0, (K, N))
    ox = cx[:, None] + r * np.cos(ang)
    oy = cy[:, None] + r * np.sin(ang)
    ox[:, ::7] = np.round(ox[:, ::7] * 20) / 20          # multiples of the 5 cm cell size
    oy[:, ::5] = np.round(oy[:, ::5] * 20) / 20
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    res = {}
    for name, dt in (("f64", np.float64), ("f32", np.float32)):
        a = [np.ascontiguousarray(v, dtype=dt) for v in (ox, oy, cx, cy)]
        m = env.b2slam.Mapping(G, G, 0.05)
        pm = m.update_batch(*a).copy()
        hit, miss = m.counts()
        oh = np.zeros((G, G), dtype=np.int32)
        om = np.zeros((G, G), dtype=np.int32)
        env.corc.grid_raycast(oh, om, S, Hx, Hy, *a)
        assert np.array_equal(hit, oh) and np.array_equal(miss, om), name
        assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1]), name
        res[name] = (hit, miss)
    assert not (np.array_equal(res["f64"][0], res["f32"][0]) and np.array_equal(res["f64"][1], res["f32"][1]))


def test_float64_batch_rollback_and_errors(env):
    G = 512
    ox, oy, cx, cy = (a.astype(np.float64) + 1e-9 for a in env.synth.grid_scans(79, 3000, 360, half_extent_m=10.0))
    m = env.b2slam.Mapping(G, G, 0.05)
    m.update_batch(ox[:100], oy[:100], cx[:100], cy[:100])
    h0, m0 = m.counts()
    bad = oy.copy()
    bad[2900, 11] = np.nan
    with pytest.raises(ValueError):
        m.update_batch(ox, bad, cx, cy)
    bad[2900, 11] = np.inf
    with pytest.raises(OverflowError):
        m.update_batch(ox, bad, cx, cy)
    h1, m1 = m.counts()
    assert np.array_equal(h0, h1) and np.array_equal(m0, m1)


def test_cfg5_scale_float64_fuzz_has_zero_cell_differences(env):
    """16384 x 16384 @ 5 cm (cfg 5): random float64 poses / endpoints out to +-400 m, a third of them on exact
    multiples of the cell size, through Mapping.update_batch (float64) vs the float64 oracle: zero differences.
    Narrowed to float32 the same scans move cells (about 1e-4 per coordinate at this scale)."""
    G = 16384
    rng = np.random.Generator(np.random.PCG64(5005))
    K, N = 192, 1080
    cx = rng.uniform(-400, 400, K)
    cy = rng.uniform(-400, 400, K)
    ang = np.linspace(-np.pi, np.pi, N)
    r = rng.uniform(0.2, 30.0, (K, N))
    ox = cx[:, None] + r * np.cos(ang)
    oy = cy[:, None] + r * np.sin(ang)
    ox[:, ::3] = np.round(ox[:, ::3] * 20) / 20
    oy[:, 1::3] = np.round(oy[:, 1::3] * 20) / 20
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    m = env.b2slam.Mapping(G, G, 0.05)
    m.update_batch(ox, oy, cx, cy, want_pmap=False)
    hit, miss = m.counts()
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    visits = env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
    assert visits > 10_000_000
    diff = int((hit != oh).sum() + (miss != om).sum())
    assert diff == 0, "%d cells differ from the float64 oracle" % diff
    # what float32 narrowing would have done to these scans
    f = lambda v, H: np.trunc(S * (v + H))
    moved = int((f(ox, Hx) != f(ox.astype(np.float32).astype(np.float64), Hx)).sum()
                + (f(oy, Hy) != f(oy.astype(np.float32).astype(np.float64), Hy)).sum())
    assert moved > 100
    del m
