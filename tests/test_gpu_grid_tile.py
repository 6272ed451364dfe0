"""GPU parity of ray-cast variant 6 (consecutive scans counted in a shared-memory tile; variant 5 for CTAs whose box
does not fit or that hold a clipped ray) against oracle.c and against variant 5."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

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


def _variant(env, v):
    assert env.lib.lib().b2s_tune(b"grid_variant", v) == 0


def _cast(env, v, G, arrays, Gy=None, reso=0.05):
    """One ray-cast launch with a workspace under variant v; returns hit, miss, counters, workspace."""
    Gy = Gy or G
    _variant(env, v)
    S, Hx, Hy = env.dev.grid_scale(G, Gy, reso)
    hit, miss = env.dev.new_planes(G, Gy)
    ws = env.dev.new_workspace(G, Gy)
    cnt = torch.zeros(4, dtype=torch.int32, device="cuda")
    env.dev.grid_raycast(hit, miss, S, Hx, Hy, *[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays],
                         counters=cnt, workspace=ws)
    torch.cuda.synchronize()
    return hit, miss, cnt, ws


def _v6_equals_v5(env, G, arrays, Gy=None, reso=0.05):
    h5, m5, c5, _ = _cast(env, 5, G, arrays, Gy, reso)
    h6, m6, c6, _ = _cast(env, 6, G, arrays, Gy, reso)
    assert torch.equal(h5, h6) and torch.equal(m5, m6)
    assert c5.tolist() == c6.tolist()
    return h6, m6


def _scans_around(cx, cy, ang, r, dtype=np.float32):
    """Endpoints of beams at angles ang (K, N) and ranges r (K, N) from sensor positions cx, cy (K,)."""
    ox = cx[:, None].astype(np.float64) + r * np.cos(ang)
    oy = cy[:, None].astype(np.float64) + r * np.sin(ang)
    return ox.astype(dtype), oy.astype(dtype), cx.astype(dtype), cy.astype(dtype)


def test_bench_launch_v6_is_bit_identical_to_the_oracle(env):
    """The bench launch (seed 12001, 16 384 scans x 1080 beams into 4096^2 @ 5 cm) under variant 6: both planes bit for
    bit and the visit count, for world-frame endpoints and for raw ranges + poses."""
    from b2slam import scan
    G, K, N = 4096, 16384, 1080
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    host = env.synth.grid_scans(12001, K, N)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    assert env.corc.grid_raycast(oh, om, S, Hx, Hy, *host) == 1767256201
    hit, miss, cnt, ws = _cast(env, 6, G, host)
    assert int(hit.sum(dtype=torch.int64).item() + miss.sum(dtype=torch.int64).item()) == 1767256201
    assert np.array_equal(hit.cpu().numpy(), oh) and np.array_equal(miss.cpu().numpy(), om)
    assert cnt.tolist() == [0, 0, 0, 0]
    ranges, poses = env.synth.grid_scan_ranges(12001, K, N)
    table, beams = scan.pose_table(poses), scan.beam_table(-math.pi, math.pi, N)
    oh[:] = 0
    om[:] = 0
    env.corc.grid_raycast_ranges(oh, om, S, Hx, Hy, ranges, table, beams, 30.0)
    hit.zero_()
    miss.zero_()
    env.dev.grid_raycast_ranges(hit, miss, S, Hx, Hy, torch.from_numpy(ranges).cuda(), torch.from_numpy(table).cuda(),
                                torch.from_numpy(beams).cuda(), 30.0, workspace=ws)
    assert np.array_equal(hit.cpu().numpy(), oh) and np.array_equal(miss.cpu().numpy(), om)


def test_v6_equals_v5_on_independent_random_scans(env):
    """Scans at random places with rays out of the grid: every CTA falls back."""
    G = 512
    rng = np.random.Generator(np.random.PCG64(61))
    K, N = 64, 360
    cx, cy = rng.uniform(-16, 16, K), rng.uniform(-16, 16, K)
    arrays = _scans_around(cx, cy, rng.uniform(-np.pi, np.pi, (K, N)), rng.uniform(0.0, 30.0, (K, N)))
    h, m = _v6_equals_v5(env, G, arrays)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, *arrays)
    assert np.array_equal(h.cpu().numpy(), oh) and np.array_equal(m.cpu().numpy(), om)


def test_v6_equals_v5_on_a_trajectory_crossing_the_map_edge(env):
    """A trajectory that drives out of a small map: CTAs inside take the tile, those at the edge fall back."""
    G = 1024
    K, N = 480, 1080
    t = np.arange(K)
    cx = -20.0 + 0.1 * t            # from inside the +-25.6 m map to 2.4 m past its edge
    cy = 3.0 * np.sin(t / 60.0)
    phi = np.linspace(-np.pi, np.pi, N)[None, :] + 0.01 * t[:, None]
    rng = np.random.Generator(np.random.PCG64(62))
    r = rng.uniform(3.0, 8.0, (K, 1)) + rng.uniform(0.5, 2.0, (K, 1)) * np.sin(3 * phi)
    arrays = _scans_around(cx, cy, phi, r)
    h, m = _v6_equals_v5(env, G, arrays)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, *arrays)
    assert np.array_equal(h.cpu().numpy(), oh) and np.array_equal(m.cpu().numpy(), om)


@pytest.mark.parametrize("shape", [(1, 1), (3, 70), (40, 33), (97, 64)])
def test_v6_equals_v5_on_tiny_grids(env, shape):
    xw, yw = shape
    rng = np.random.Generator(np.random.PCG64(63 + xw))
    K, N = 40, 100
    cx = rng.uniform(-0.02 * xw, 0.02 * xw, K)
    cy = rng.uniform(-0.02 * yw, 0.02 * yw, K)
    arrays = _scans_around(cx, cy, rng.uniform(-np.pi, np.pi, (K, N)), rng.uniform(0.0, 0.04 * max(xw, yw), (K, N)))
    h, m = _v6_equals_v5(env, xw, arrays, Gy=yw)
    oh = np.zeros((xw, yw), dtype=np.int32)
    om = np.zeros((xw, yw), dtype=np.int32)
    S, Hx, Hy = env.dev.grid_scale(xw, yw, 0.05)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, *arrays)
    assert np.array_equal(h.cpu().numpy(), oh) and np.array_equal(m.cpu().numpy(), om)


@pytest.mark.parametrize("centre", [0.0, 0.5 * np.pi, np.pi, -0.5 * np.pi, 0.25 * np.pi])
def test_v6_equals_v5_on_steep_and_shallow_sectors(env, centre):
    """All beams in a 20-degree fan around one heading: shallow (x-major), steep (y-major), flipped, diagonal."""
    G = 2048
    K, N = 64, 256
    t = np.arange(K)
    cx, cy = 0.1 * t - 3.0, 0.05 * t
    phi = centre + np.linspace(-np.pi / 18, np.pi / 18, N)[None, :] + np.zeros((K, 1))
    r = 9.5 + 0.5 * np.sin(7 * phi)
    arrays = _scans_around(cx, cy, phi, r)
    h, m = _v6_equals_v5(env, G, arrays)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, *arrays)
    assert np.array_equal(h.cpu().numpy(), oh) and np.array_equal(m.cpu().numpy(), om)


def test_v6_equals_v5_on_float64_input(env):
    """IN_F64: unrounded float64 endpoints of the cfg-3 trajectory, and a few beams that int() rejects."""
    ox, oy, cx, cy = env.synth.grid_scans(12002, 512, 1080)
    rng = np.random.Generator(np.random.PCG64(64))
    ox = ox.astype(np.float64) + rng.uniform(-1e-3, 1e-3, ox.shape)
    oy = oy.astype(np.float64) + rng.uniform(-1e-3, 1e-3, oy.shape)
    cx, cy = cx.astype(np.float64), cy.astype(np.float64)
    ox[3, 5] = np.inf
    ox[40, 7] = np.nan
    oy[200, 9] = np.inf
    h, m = _v6_equals_v5(env, 4096, (ox, oy, cx, cy))
    _, _, cnt, _ = _cast(env, 6, 4096, (ox, oy, cx, cy))
    assert sorted(cnt.tolist()) == [0, 1, 1, 1]


def test_v6_batch_rolled_back_to_zero(env):
    """A batch applied chunk by chunk under variant 6 and rejected at its end comes back out exactly."""
    _variant(env, 6)
    G = 2048
    ox, oy, cx, cy = env.synth.grid_scans(65, 6000, 1080, half_extent_m=40.0)
    m = env.b2slam.Mapping(G, G, 0.05)
    bad = oy.copy()
    bad[5900, 100] = np.nan
    with pytest.raises(ValueError):
        m.update_batch(ox, bad, cx, cy)
    hit, miss = m.counts()
    assert not hit.any() and not miss.any()
    pm = m.update_batch(ox, oy, cx, cy)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
    hit, miss = m.counts()
    assert np.array_equal(hit, oh) and np.array_equal(miss, om)
    assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1])


@pytest.mark.parametrize("half", [40.0, 60.0])
def test_v6_dirty_map_covers_every_touched_cell(env, half):
    """After b2s_grid_clear_dirty the planes are all zero: the tiles marked by private and fallback CTAs cover every
    cell they counted (half = 60 m drives the trajectory off a 2048^2 map)."""
    G = 2048
    arrays = env.synth.grid_scans(66, 2048, 1080, half_extent_m=half)
    hit, miss, _, ws = _cast(env, 6, G, arrays)
    assert int(miss.sum(dtype=torch.int64).item()) > 0
    env.lib.check(env.lib.lib().b2s_grid_clear_dirty(hit.data_ptr(), miss.data_ptr(), G, G, ws.data_ptr(),
                                                     torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert not bool(hit.any().item()) and not bool(miss.any().item())


def test_cfg5_shape_v6_equals_single_pass_v5(env):
    """16384^2 @ 5 cm, 8 scan streams ray-cast one after the other into one pair of planes (the single-pass parity of
    bench.py's cfg 5): variant 6 equals variant 5 byte for byte."""
    G, streams, K, N = 16384, 8, 512, 1080
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    planes = {}
    for v in (5, 6):
        _variant(env, v)
        hit, miss = env.dev.new_planes(G, G)
        ws = env.dev.new_workspace(G, G)
        for s in range(streams):
            one = [torch.from_numpy(a).cuda() for a in env.synth.grid_scans(5001 + s, K, N, half_extent_m=380.0)]
            env.dev.grid_raycast(hit, miss, S, Hx, Hy, *one, workspace=ws)
        torch.cuda.synchronize()
        planes[v] = (hit, miss)
        del ws
    (h5, m5), (h6, m6) = planes[5], planes[6]
    assert int(m6.sum(dtype=torch.int64).item()) > 0
    assert torch.equal(h5, h6) and torch.equal(m5, m6)
