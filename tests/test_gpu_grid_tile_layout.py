"""The two CTA layouts of ray-cast variant 6 (b2s_tune "grid_tile_layout"): 0 = 1024 threads, one 32-beam unit per warp;
1 = 512 threads, two units per warp, longest paired with shortest.  Both must count exactly what variant 5 and
oracle.c count, with the same status counters."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, synth
    from oracle import corc
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.lib, e.dev, e.synth, e.corc = b2slam, _lib, devapi, synth, corc
    yield e
    _lib.lib().b2s_tune(b"grid_variant", 6)
    _lib.lib().b2s_tune(b"grid_tile_layout", 1)


ARMS = {"v5": (5, 1), "layout0": (6, 0), "layout1": (6, 1)}  # grid_variant, grid_tile_layout


def _cast(env, arm, G, arrays, Gy=None):
    """One ray-cast launch with a workspace; returns hit, miss, counters."""
    Gy = Gy or G
    variant, layout = ARMS[arm]
    assert env.lib.lib().b2s_tune(b"grid_variant", variant) == 0
    assert env.lib.lib().b2s_tune(b"grid_tile_layout", layout) == 0
    S, Hx, Hy = env.dev.grid_scale(G, Gy, 0.05)
    hit, miss = env.dev.new_planes(G, Gy)
    ws = env.dev.new_workspace(G, Gy)
    cnt = torch.zeros(4, dtype=torch.int32, device="cuda")
    env.dev.grid_raycast(hit, miss, S, Hx, Hy, *[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays],
                         counters=cnt, workspace=ws)
    torch.cuda.synchronize()
    return hit, miss, cnt


def _all_equal(env, G, arrays, Gy=None, oracle=True):
    """Variant 5 and both layouts: planes byte for byte and counters; and the planes against oracle.c."""
    out = {a: _cast(env, a, G, arrays, Gy) for a in ARMS}
    h5, m5, c5 = out["v5"]
    for a in ("layout0", "layout1"):
        h, m, c = out[a]
        assert torch.equal(h, h5) and torch.equal(m, m5), a
        assert c.tolist() == c5.tolist(), a
    if oracle:
        Gy = Gy or G
        oh = np.zeros((G, Gy), dtype=np.int32)
        om = np.zeros((G, Gy), dtype=np.int32)
        S, Hx, Hy = env.dev.grid_scale(G, Gy, 0.05)
        env.corc.grid_raycast(oh, om, S, Hx, Hy, *arrays)
        assert np.array_equal(h5.cpu().numpy(), oh) and np.array_equal(m5.cpu().numpy(), om)
    return out["layout1"]


def _scans_around(cx, cy, ang, r, dtype=np.float32):
    ox = cx[:, None].astype(np.float64) + r * np.cos(ang)
    oy = cy[:, None].astype(np.float64) + r * np.sin(ang)
    return ox.astype(dtype), oy.astype(dtype), cx.astype(dtype), cy.astype(dtype)


def _trajectory(K, N, r, seed=70):
    """A slow trajectory (consecutive scans a few cells apart) with ranges r (K, N): CTAs take the tile."""
    t = np.arange(K)
    cx, cy = -3.0 + 0.02 * t, 1.0 * np.sin(t / 80.0)
    phi = np.linspace(-np.pi, np.pi, N)[None, :] + 0.005 * t[:, None]
    return _scans_around(cx, cy, phi, r)


def test_grid_tile_layout_key_accepts_0_and_1_only():
    from b2slam import _lib
    L = _lib.lib()
    try:
        assert L.b2s_tune(b"grid_tile_layout", 0) == 0
        assert L.b2s_tune(b"grid_tile_layout", 1) == 0
        assert L.b2s_tune(b"grid_tile_layout", 2) == _lib.ERR_INVALID_ARG
        assert L.b2s_tune(b"grid_tile_layout", -1) == _lib.ERR_INVALID_ARG
    finally:
        L.b2s_tune(b"grid_tile_layout", 1)


@pytest.mark.gpu
def test_bench_launch_both_layouts_match_the_oracle(env):
    """The bench launch (seed 12001, 16 384 scans x 1080 beams into 4096^2 @ 5 cm), as float32 endpoints and as raw
    ranges + poses."""
    from b2slam import scan
    G, K, N = 4096, 16384, 1080
    host = env.synth.grid_scans(12001, K, N)
    h, m, _ = _all_equal(env, G, host)
    assert int(h.sum(dtype=torch.int64).item() + m.sum(dtype=torch.int64).item()) == 1767256201
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    ranges, poses = env.synth.grid_scan_ranges(12001, K, N)
    table, beams = scan.pose_table(poses), scan.beam_table(-math.pi, math.pi, N)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    env.corc.grid_raycast_ranges(oh, om, S, Hx, Hy, ranges, table, beams, 30.0)
    ws = env.dev.new_workspace(G, G)
    for layout in (0, 1):
        assert env.lib.lib().b2s_tune(b"grid_tile_layout", layout) == 0
        hit, miss = env.dev.new_planes(G, G)
        env.dev.grid_raycast_ranges(hit, miss, S, Hx, Hy, torch.from_numpy(ranges).cuda(),
                                    torch.from_numpy(table).cuda(), torch.from_numpy(beams).cuda(), 30.0, workspace=ws)
        assert np.array_equal(hit.cpu().numpy(), oh) and np.array_equal(miss.cpu().numpy(), om), layout


@pytest.mark.gpu
def test_layouts_on_float64_input(env):
    ox, oy, cx, cy = env.synth.grid_scans(12002, 512, 1080)
    rng = np.random.Generator(np.random.PCG64(71))
    ox = ox.astype(np.float64) + rng.uniform(-1e-3, 1e-3, ox.shape)
    oy = oy.astype(np.float64) + rng.uniform(-1e-3, 1e-3, oy.shape)
    cx, cy = cx.astype(np.float64), cy.astype(np.float64)
    ox[3, 5] = np.inf
    ox[40, 7] = np.nan
    oy[200, 9] = np.inf
    _, _, cnt = _all_equal(env, 4096, (ox, oy, cx, cy), oracle=False)
    assert sorted(cnt.tolist()) == [0, 1, 1, 1]


@pytest.mark.gpu
def test_layouts_on_random_scans(env):
    """Scans at random places with rays out of the grid: every CTA falls back."""
    rng = np.random.Generator(np.random.PCG64(72))
    K, N = 64, 360
    cx, cy = rng.uniform(-16, 16, K), rng.uniform(-16, 16, K)
    _all_equal(env, 512, _scans_around(cx, cy, rng.uniform(-np.pi, np.pi, (K, N)), rng.uniform(0.0, 30.0, (K, N))))


@pytest.mark.gpu
def test_layouts_on_a_trajectory_crossing_the_map_edge(env):
    G, K, N = 1024, 480, 1080
    t = np.arange(K)
    cx, cy = -20.0 + 0.1 * t, 3.0 * np.sin(t / 60.0)
    phi = np.linspace(-np.pi, np.pi, N)[None, :] + 0.01 * t[:, None]
    rng = np.random.Generator(np.random.PCG64(73))
    r = rng.uniform(3.0, 8.0, (K, 1)) + rng.uniform(0.5, 2.0, (K, 1)) * np.sin(3 * phi)
    _all_equal(env, G, _scans_around(cx, cy, phi, r))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 1), (3, 70), (40, 33), (97, 64)])
def test_layouts_on_tiny_grids(env, shape):
    xw, yw = shape
    rng = np.random.Generator(np.random.PCG64(74 + xw))
    K, N = 40, 100
    cx, cy = rng.uniform(-0.02 * xw, 0.02 * xw, K), rng.uniform(-0.02 * yw, 0.02 * yw, K)
    arrays = _scans_around(cx, cy, rng.uniform(-np.pi, np.pi, (K, N)), rng.uniform(0.0, 0.04 * max(xw, yw), (K, N)))
    _all_equal(env, xw, arrays, Gy=yw)


@pytest.mark.gpu
@pytest.mark.parametrize("centre", [0.0, 0.5 * np.pi, np.pi, -0.5 * np.pi, 0.25 * np.pi])
def test_layouts_on_steep_and_shallow_sectors(env, centre):
    K, N = 64, 256
    t = np.arange(K)
    cx, cy = 0.1 * t - 3.0, 0.05 * t
    phi = centre + np.linspace(-np.pi / 18, np.pi / 18, N)[None, :] + np.zeros((K, 1))
    _all_equal(env, 2048, _scans_around(cx, cy, phi, 9.5 + 0.5 * np.sin(7 * phi)))


@pytest.mark.gpu
def test_layouts_on_the_cfg5_shape(env):
    """16384^2 @ 5 cm, 8 scan streams ray-cast one after the other into one pair of planes."""
    G, streams, K, N = 16384, 8, 512, 1080
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    planes = {}
    for arm, (variant, layout) in ARMS.items():
        assert env.lib.lib().b2s_tune(b"grid_variant", variant) == 0
        assert env.lib.lib().b2s_tune(b"grid_tile_layout", layout) == 0
        hit, miss = env.dev.new_planes(G, G)
        ws = env.dev.new_workspace(G, G)
        for s in range(streams):
            one = [torch.from_numpy(a).cuda() for a in env.synth.grid_scans(5001 + s, K, N, half_extent_m=380.0)]
            env.dev.grid_raycast(hit, miss, S, Hx, Hy, *one, workspace=ws)
        torch.cuda.synchronize()
        planes[arm] = (hit, miss)
        del ws
    h5, m5 = planes["v5"]
    assert int(m5.sum(dtype=torch.int64).item()) > 0
    for arm in ("layout0", "layout1"):
        assert torch.equal(planes[arm][0], h5) and torch.equal(planes[arm][1], m5), arm


@pytest.mark.gpu
def test_layouts_on_ranges_alternating_short_and_long(env):
    """Ranges of 0.5 m and 10 m alternating by scan and by 32-beam unit: a CTA's units differ 20x in length, which is
    what layout 1 pairs up."""
    K, N = 256, 1080
    k, j = np.arange(K)[:, None], np.arange(N)[None, :]
    r = np.where((k + j // 32) % 2 == 0, 0.5, 10.0)
    _all_equal(env, 2048, _trajectory(K, N, r))


@pytest.mark.gpu
@pytest.mark.parametrize("K, N", [(37, 100), (16, 1080), (5, 33), (50, 64 + 1)])
def test_layouts_on_partial_ctas_and_units(env, K, N):
    """Scan counts that are not a multiple of 16 and beam counts that are not a multiple of 64 or 32."""
    k, j = np.arange(K)[:, None], np.arange(N)[None, :]
    _all_equal(env, 2048, _trajectory(K, N, 3.0 + 2.0 * np.sin(0.3 * k + 0.05 * j)))


@pytest.mark.gpu
def test_layouts_on_ctas_of_only_nan_or_inf_beams(env):
    """One CTA's beams all skipped (inf in ox), one CTA's all NaN: only status counts, next to CTAs that take the tile."""
    K, N = 64, 256
    ox, oy, cx, cy = _trajectory(K, N, 4.0 + np.zeros((K, N)))
    ox[0:16, 0:64] = np.inf
    oy[16:32, 64:128] = np.nan
    _, _, cnt = _all_equal(env, 2048, (ox, oy, cx, cy), oracle=False)
    assert sorted(cnt.tolist()) == [0, 0, 16 * 64, 16 * 64]
    ox[16:32, 64:128] = 1.0  # without the NaN CTA, the inf-only one against the oracle
    oy[16:32, 64:128] = 1.0
    _all_equal(env, 2048, (ox, oy, cx, cy))
