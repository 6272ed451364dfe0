"""GPU parity: occupancy-grid path (A4-A7) through the C ABI against the CPU oracle and the
golden vectors produced by the reference.  Integer counts and cell indices are bit-exact."""
import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi, synth
    from b2slam import bresenham as bres
    from oracle import corc, pyref
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.lib, e.dev, e.synth, e.bres, e.corc, e.pyref = b2slam, _lib, devapi, synth, bres, corc, pyref
    return e


# Every kernel arm as (grid_variant, grid_tile_layout).  The default, variant 6 with tile layout 1, is what Mapping,
# the streamed calls and bench.py run; a loop over ARMS checks it beside the older variants.  Variants 4-6 are given a
# workspace: b2s_grid_raycast_ws without one runs variant 3, whatever is selected.
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


def _variants(env):
    """Selects each arm in turn and yields (grid_variant, arm name); the fixture above puts the default back."""
    for arm in ARMS:
        _select(env, arm)
        yield arm[0], ("v6/layout%d" % arm[1] if arm[0] == 6 else "v%d" % arm[0])


# ----------------------------------------------------------------------------- bresenham (A7)

def test_bresenham_paths_equal_reference(env):
    z = load_golden("bresenham.npz")
    cells, offs = env.bres.paths(z["segs"])
    assert np.array_equal(offs, z["offsets"])
    assert np.array_equal(cells, z["cells"])


def test_bresenham_class_api(env):
    drawing = env.bres                         # mapping.py: `import bresenham as drawing`
    p = drawing.bresenham([0, 0], [10, 3]).path
    assert p == env.corc.bresenham([0, 0], [10, 3])
    assert drawing.bresenham([5, 5], [5, 5]).path == []
    assert drawing.bresenham([3, 9], [3, 2]).path == env.pyref.bresenham_cells([3, 9], [3, 2])


def test_bresenham_long_random_segments_vs_oracle(env):
    rng = np.random.Generator(np.random.PCG64(77))
    segs = rng.integers(-3000, 3000, size=(3000, 4)).astype(np.int32)
    cells, offs = env.bres.paths(segs)
    for i in rng.integers(0, len(segs), size=150):
        want = env.corc.bresenham(segs[i, :2], segs[i, 2:])
        got = [tuple(r) for r in cells[offs[i]:offs[i + 1]].tolist()]
        assert got == want


# ----------------------------------------------------------------------------- Mapping (A4-A6)

@pytest.mark.parametrize("tag,w_hit", [("w20", 20.0), ("w4", 4.0)])
def test_mapping_class_reproduces_reference_maps(env, tag, w_hit):
    z = load_golden("mapping.npz")
    for v, name in _variants(env):
        m = env.b2slam.Mapping(200, 200, 0.1, hit_weight=w_hit)
        assert m.pmap.shape == (200, 200) and (m.pmap == 50).all()
        for ox, oy, cx, cy in zip(z[tag + "_ox"], z[tag + "_oy"], z[tag + "_cx"], z[tag + "_cy"]):
            pm = m.update(ox.astype(np.float64), oy.astype(np.float64), float(cx), np.array([float(cy)]))
        hit, miss = m.counts()
        oh = np.zeros((200, 200), dtype=np.int32)
        om = np.zeros((200, 200), dtype=np.int32)
        env.corc.grid_raycast(oh, om, 10.0, 10.0, 10.0, z[tag + "_ox"], z[tag + "_oy"], z[tag + "_cx"], z[tag + "_cy"])
        assert np.array_equal(hit, oh) and np.array_equal(miss, om), name
        amb = env.pyref.boundary_ambiguous(hit, miss, w_hit)
        assert ((pm == z[tag + "_pmap"]) | amb).all()
        if w_hit == 20.0:
            assert np.array_equal(pm.astype(np.int8), z[tag + "_pmap"])
        assert pm.dtype == np.float64 and set(np.unique(pm)) <= {0.0, 50.0, 100.0}
        np.testing.assert_allclose(m.datamap, z[tag + "_datamap"], rtol=1e-5, atol=1e-6)  # fp32 score
        assert np.array_equal(m.occupancy(), pm.astype(np.int8))


def test_mapping_edge_cases(env):
    m = env.b2slam.Mapping(200, 200, 0.1)
    pm = m.update(np.array([]), np.array([]), 0.0, 0.0)            # empty scan
    assert (pm == 50).all()
    pm = m.update(np.array([np.inf, -np.inf]), np.array([0.0, 1.0]), 0.0, 0.0)  # skipped beams
    assert (pm == 50).all()
    pm = m.update(np.array([0.004]), np.array([0.003]), 0.0, 0.0)  # same cell: no update at all
    assert (pm == 50).all()
    with pytest.raises(ValueError):
        m.update(np.array([1.0, np.nan]), np.array([0.0, 0.0]), 0.0, 0.0)
    with pytest.raises(OverflowError):
        m.update(np.array([1.0]), np.array([np.inf]), 0.0, 0.0)
    with pytest.raises(ValueError):
        m.update(np.array([1.0]), np.array([1.0]), np.nan, 0.0)
    assert (m.counts()[0] == 0).all() and (m.counts()[1] == 0).all()  # nothing applied on error
    pm = m.update(np.array([30.0]), np.array([0.45]), 0.05, 0.05)  # endpoint outside: clipped, no hit
    hit, miss = m.counts()
    assert hit.sum() == 0 and miss.sum() == 100 and int((pm == 0).sum()) == 100 and (pm != 100).all()
    m.reset()
    assert (m.counts()[1] == 0).all() and (m.pmap == 50).all() and (m.occupancy() == 50).all()


def test_rejected_batch_is_rolled_back_exactly(env):
    """A batch with a NaN deep inside is applied chunk by chunk while it streams in; the error must
    leave the counts exactly as they were (the kernel takes the chunks back out with sign -1)."""
    G = 1024
    ox, oy, cx, cy = env.synth.grid_scans(77, 6000, 1080, half_extent_m=20.0)   # > 2 chunks
    m = env.b2slam.Mapping(G, G, 0.05)
    m.update_batch(ox[:500], oy[:500], cx[:500], cy[:500])
    h0, m0 = m.counts()
    bad = oy.copy()
    bad[5500, 17] = np.nan
    with pytest.raises(ValueError):
        m.update_batch(ox, bad, cx, cy)
    h1, m1 = m.counts()
    assert np.array_equal(h0, h1) and np.array_equal(m0, m1)
    bad[5500, 17] = np.inf
    with pytest.raises(OverflowError):
        m.update_batch(ox, bad, cx, cy)
    h1, m1 = m.counts()
    assert np.array_equal(h0, h1) and np.array_equal(m0, m1)
    pm = m.update_batch(ox, oy, cx, cy)                                       # and the good batch lands
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox[:500], oy[:500], cx[:500], cy[:500])
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
    h2, m2 = m.counts()
    assert np.array_equal(h2, oh) and np.array_equal(m2, om)
    assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1])


def test_mapping_threshold_stream(env):
    """1000 traversals stay free, the 1001st flips the cell (reference golden, [MAP]:47)."""
    z = load_golden("mapping.npz")
    m = env.b2slam.Mapping(200, 200, 0.1)
    ox = np.full((1000, 1), 1.05, dtype=np.float32)
    oy = np.full((1000, 1), 0.05, dtype=np.float32)
    c = np.full(1000, 0.05, dtype=np.float32)
    pm = m.update_batch(ox, oy, c, c)
    assert pm.dtype == np.int8 and pm[105, 100] == z["miss_stream_pmap"][0] == 0
    pm = m.update_batch(ox[:1], oy[:1], c[:1], c[:1])
    assert pm[105, 100] == z["miss_stream_pmap"][1] == 100


def test_non_square_grid_and_generalised_scale(env):
    S, Hx, Hy = env.dev.grid_scale(300, 180, 0.05)
    ox, oy, cx, cy = env.synth.grid_scans(31, 12, 360, half_extent_m=3.0)
    for v, name in _variants(env):
        m = env.b2slam.Mapping(300, 180, 0.05)
        m.update_batch(ox, oy, cx, cy)
        hit, miss = m.counts()
        oh = np.zeros((300, 180), dtype=np.int32)
        om = np.zeros((300, 180), dtype=np.int32)
        env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
        assert np.array_equal(hit, oh) and np.array_equal(miss, om)


# ----------------------------------------------------------------------------- cfg 3 (4096^2, 1080 beams)

def _device_scans(env, seed, K, N, half):
    ox, oy, cx, cy = env.synth.grid_scans(seed, K, N, half_extent_m=half)
    t = [torch.from_numpy(a).cuda() for a in (ox, oy, cx, cy)]
    return (ox, oy, cx, cy), t


def test_cfg3_counts_bit_exact_vs_oracle(env):
    G, reso, K, N = 4096, 0.05, 96, 1080
    S, Hx, Hy = env.dev.grid_scale(G, G, reso)
    assert (S, Hx, Hy) == (20.0, 102.4, 102.4)
    host, devt = _device_scans(env, 12001, K, N, 80.0)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    visits = env.corc.grid_raycast(oh, om, S, Hx, Hy, *host)
    for v, name in _variants(env):
        hit, miss = env.dev.new_planes(G, G)
        cnt = torch.zeros(4, dtype=torch.int32, device="cuda")
        ws = env.dev.new_workspace(G, G) if v >= 4 else None
        env.dev.grid_raycast(hit, miss, S, Hx, Hy, *devt, counters=cnt, workspace=ws)
        if ws is not None:  # the workspace comes back clean and is reusable
            torch.cuda.synchronize()
            assert int(ws[-G * G:].abs().sum().item()) == 0 and ws[:4].tolist() == [-2139062144] * 4
            assert int(ws[16:-G * G].sum().item()) > 0      # the dirty-tile map stays set until it is consumed
            env.dev.grid_raycast(hit, miss, S, Hx, Hy, *devt, workspace=ws)
            hit //= 2
            miss //= 2
        torch.cuda.synchronize()
        assert int(hit.sum().item() + miss.sum().item()) == visits
        assert np.array_equal(hit.cpu().numpy(), oh), name
        assert np.array_equal(miss.cpu().numpy(), om), name
        assert cnt.tolist() == [0, 0, 0, 0]
    pmap = torch.empty((G, G), dtype=torch.int8, device="cuda")
    score = torch.empty((G, G), dtype=torch.float32, device="cuda")
    env.dev.grid_finalize(hit, miss, pmap=pmap, datamap=score)
    osc, opm = env.corc.grid_finalize(oh, om)
    assert np.array_equal(pmap.cpu().numpy(), opm)
    np.testing.assert_allclose(score.cpu().numpy(), osc, rtol=1e-6, atol=0)
    ros = env.dev.grid_pack_ros(pmap).cpu().numpy()
    assert np.array_equal(ros, opm.T.reshape(-1))  # slam_ekf.py:270


def test_bench_launch_is_bit_identical_to_the_oracle(env):
    """THE launch bench.py times -- cfg 3, seed 12001, 16 384 scans x 1080 beams into 4096^2 @ 5 cm, 1.77 G cell
    visits -- against oracle.c on the same inputs: both int32 planes bit for bit, the visit count, the occupancy map.
    Both input forms (world-frame endpoints; raw ranges + poses through the fused-ingestion kernel)."""
    import math
    from b2slam import scan
    G, reso, K, N = 4096, 0.05, 16384, 1080
    S, Hx, Hy = env.dev.grid_scale(G, G, reso)
    host, devt = _device_scans(env, 12001, K, N, 80.0)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    visits = env.corc.grid_raycast(oh, om, S, Hx, Hy, *host)
    assert visits == 1767256201                     # the figure bench.py derives its algorithmic bytes from
    hit, miss = env.dev.new_planes(G, G)
    ws = env.dev.new_workspace(G, G)
    cnt = torch.zeros(4, dtype=torch.int32, device="cuda")
    env.dev.grid_raycast(hit, miss, S, Hx, Hy, *devt, counters=cnt, workspace=ws)
    assert np.array_equal(hit.cpu().numpy(), oh) and np.array_equal(miss.cpu().numpy(), om)
    assert int(cnt.sum().item()) == 0
    pm = torch.empty((G, G), dtype=torch.int8, device="cuda")
    env.dev.grid_finalize(hit, miss, pmap=pm)
    assert np.array_equal(pm.cpu().numpy(), env.corc.grid_finalize(oh, om)[1])
    # raw form of the same stream
    ranges, poses = env.synth.grid_scan_ranges(12001, K, N)
    oh[:] = 0
    om[:] = 0
    table, beams = scan.pose_table(poses), scan.beam_table(-math.pi, math.pi, N)
    env.corc.grid_raycast_ranges(oh, om, S, Hx, Hy, ranges, table, beams, 30.0)
    hit.zero_()
    miss.zero_()
    env.dev.grid_raycast_ranges(hit, miss, S, Hx, Hy, torch.from_numpy(ranges).cuda(), torch.from_numpy(table).cuda(),
                                torch.from_numpy(beams).cuda(), 30.0, workspace=ws)
    assert np.array_equal(hit.cpu().numpy(), oh) and np.array_equal(miss.cpu().numpy(), om)


def test_cfg3_full_size_properties(env):
    """Size-independent checks at the bench size: variants agree, sharded == single pass,
    update(A) + update(B) == update(A u B), visits == sum of per-beam path lengths in grid."""
    G, reso, K, N = 4096, 0.05, 4096, 1080
    S, Hx, Hy = env.dev.grid_scale(G, G, reso)
    _, devt = _device_scans(env, 12001, K, N, 80.0)
    ox, oy, cx, cy = devt
    _select(env, ARMS[0])
    h1, m1 = env.dev.new_planes(G, G)
    env.dev.grid_raycast(h1, m1, S, Hx, Hy, ox, oy, cx, cy)
    h2, m2 = env.dev.new_planes(G, G)
    ws = env.dev.new_workspace(G, G)
    for v, name in _variants(env):
        h2.zero_()
        m2.zero_()
        env.dev.grid_raycast(h2, m2, S, Hx, Hy, ox, oy, cx, cy, workspace=ws if v >= 4 else None)
        assert torch.equal(h1, h2) and torch.equal(m1, m2), name
    _select(env, DEFAULT_ARM)
    # every beam of this workload ends inside the grid -> exactly one hit per non-degenerate beam
    assert int(h2.sum().item()) <= K * N and int(h2.sum().item()) > 0.99 * K * N
    # 4 emulated ranks: private delta planes summed == single pass (integer sums commute)
    acc_h, acc_m = env.dev.new_planes(G, G)
    for r in range(4):
        lo, hi = r * K // 4, (r + 1) * K // 4
        dh, dm = env.dev.new_planes(G, G)
        env.dev.grid_raycast(dh, dm, S, Hx, Hy, ox[lo:hi].contiguous(), oy[lo:hi].contiguous(),
                             cx[lo:hi].contiguous(), cy[lo:hi].contiguous(), workspace=ws)
        acc_h += dh
        acc_m += dm
    assert torch.equal(acc_h, h2) and torch.equal(acc_m, m2)
    # accumulate in two calls on the same planes
    bh, bm = env.dev.new_planes(G, G)
    half = K // 2
    env.dev.grid_raycast(bh, bm, S, Hx, Hy, ox[:half].contiguous(), oy[:half].contiguous(),
                         cx[:half].contiguous(), cy[:half].contiguous())
    env.dev.grid_raycast(bh, bm, S, Hx, Hy, ox[half:].contiguous(), oy[half:].contiguous(),
                         cx[half:].contiguous(), cy[half:].contiguous())
    assert torch.equal(bh, h2) and torch.equal(bm, m2)


def test_clipping_out_of_grid_and_counters(env):
    """Sensor outside the grid, endpoints outside, rays crossing a corner; inf / NaN counters."""
    G = 512
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)   # +-12.8 m
    rng = np.random.Generator(np.random.PCG64(9))
    K, N = 40, 256
    cx = rng.uniform(-20, 20, K).astype(np.float32)
    cy = rng.uniform(-20, 20, K).astype(np.float32)
    ang = rng.uniform(-np.pi, np.pi, (K, N))
    r = rng.uniform(0.0, 30.0, (K, N))
    ox = (cx[:, None] + r * np.cos(ang)).astype(np.float32)
    oy = (cy[:, None] + r * np.sin(ang)).astype(np.float32)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
    assert om.sum() > 0
    for v, name in _variants(env):
        hit, miss = env.dev.new_planes(G, G)
        ws = env.dev.new_workspace(G, G) if v >= 4 else None
        env.dev.grid_raycast(hit, miss, S, Hx, Hy, *[torch.from_numpy(a).cuda() for a in (ox, oy, cx, cy)],
                             workspace=ws)
        assert np.array_equal(hit.cpu().numpy(), oh) and np.array_equal(miss.cpu().numpy(), om), name
    ox2 = ox.copy()
    oy2 = oy.copy()
    ox2[0, 0] = np.inf
    ox2[0, 1] = np.nan
    oy2[0, 2] = np.inf
    ox2[0, 3] = 3e30
    for ws in (None, env.dev.new_workspace(G, G)):
        hit, miss = env.dev.new_planes(G, G)
        cnt = torch.zeros(4, dtype=torch.int32, device="cuda")
        env.dev.grid_raycast(hit, miss, S, Hx, Hy, *[torch.from_numpy(a).cuda() for a in (ox2, oy2, cx, cy)],
                             counters=cnt, workspace=ws)
        assert cnt.tolist() == [1, 1, 1, 1]   # NaN, too long, inf-skipped, inf where int() overflows


def test_cfg5_shape_smoke(env):
    """16384^2 planes (1 GiB each): allocation, a few scans, finalize."""
    G = 16384
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    assert (Hx, Hy) == (409.6, 409.6)
    host, devt = _device_scans(env, 5001, 8, 1080, 300.0)
    hit, miss = env.dev.new_planes(G, G)
    env.dev.grid_raycast(hit, miss, S, Hx, Hy, *devt, workspace=env.dev.new_workspace(G, G))
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, *host)
    nz = np.nonzero(oh | om)
    assert np.array_equal(hit.cpu().numpy()[nz], oh[nz]) and np.array_equal(miss.cpu().numpy()[nz], om[nz])
    assert int(miss.sum().item()) == int(om.sum())


# ----------------------------------------------------------------------------- fused ingestion (SURVEY 8f-1)

def test_update_scans_reproduces_the_reference_node(env):
    """Raw ranges + poses through the fused kernel == the reference node's laserToNumpy + u2T.dot + update."""
    import math
    z = load_golden("ingestion.npz")
    m = env.b2slam.Mapping(200, 200, 0.1)
    pm = m.update_scans(z["ranges"], z["poses"], float(z["angle_min"]), float(z["angle_max"]))
    assert np.array_equal(pm, z["pmap"])
    np.testing.assert_allclose(m.datamap, z["datamap"], rtol=1e-5, atol=1e-6)
    hit, miss = m.counts()
    from b2slam import scan
    oh = np.zeros((200, 200), dtype=np.int32)
    om = np.zeros((200, 200), dtype=np.int32)
    env.corc.grid_raycast_ranges(oh, om, 10.0, 10.0, 10.0, z["ranges"], scan.pose_table(z["poses"]),
                                 scan.beam_table(-math.pi, math.pi, z["ranges"].shape[1]), 30.0)
    assert np.array_equal(hit, oh) and np.array_equal(miss, om)


def test_update_scans_cfg3_vs_oracle_and_errors(env):
    import math
    from b2slam import scan
    G, K, N = 4096, 300, 1080
    rng = np.random.Generator(np.random.PCG64(12001))
    ranges = env.synth.noisy(rng, env.synth.clean_ranges(rng, K, N)).astype(np.float32)
    ranges[5, 100:110] = np.inf                              # clamped to 30 m
    poses = np.stack([rng.uniform(-60, 60, K), rng.uniform(-60, 60, K), rng.uniform(-math.pi, math.pi, K)], axis=1)
    m = env.b2slam.Mapping(G, G, 0.05)
    pm = m.update_scans(ranges, poses, -math.pi, math.pi)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    env.corc.grid_raycast_ranges(oh, om, 20.0, 102.4, 102.4, ranges, scan.pose_table(poses),
                                 scan.beam_table(-math.pi, math.pi, N), 30.0)
    hit, miss = m.counts()
    assert np.array_equal(hit, oh) and np.array_equal(miss, om)
    assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1])
    bad = ranges.copy()
    bad[200, 3] = np.nan
    with pytest.raises(ValueError):
        m.update_scans(bad, poses, -math.pi, math.pi)
    h2, m2 = m.counts()
    assert np.array_equal(h2, oh) and np.array_equal(m2, om)   # rejected batch rolled back exactly
    # without the clamp an infinite range makes ox infinite (beam skipped) or oy infinite (OverflowError)
    with pytest.raises((OverflowError, ValueError)):
        m.update_scans(ranges, poses, -math.pi, math.pi, clamp_inf_to=None)
    h2, m2 = m.counts()
    assert np.array_equal(h2, oh) and np.array_equal(m2, om)


# ----------------------------------------------------------------------------- checkpoint (SURVEY 8f-3)

def test_checkpoint_roundtrip(env, tmp_path):
    ox, oy, cx, cy = env.synth.grid_scans(5, 40, 360, half_extent_m=8.0)
    m = env.b2slam.Mapping(400, 300, 0.05, hit_weight=4.0)
    m.update_batch(ox[:20], oy[:20], cx[:20], cy[:20])
    path = str(tmp_path / "map.npz")
    m.save(path)
    m2 = env.b2slam.Mapping.load(path)
    assert (m2.xw, m2.yw, m2.xyreso, m2.hit_weight) == (400, 300, 0.05, 4.0)
    assert all(np.array_equal(a, b) for a, b in zip(m.counts(), m2.counts()))
    assert np.array_equal(m.occupancy(), m2.occupancy())
    pa = m.update_batch(ox[20:], oy[20:], cx[20:], cy[20:]).copy()      # resumed map evolves identically
    pb = m2.update_batch(ox[20:], oy[20:], cx[20:], cy[20:]).copy()
    assert np.array_equal(pa, pb) and all(np.array_equal(a, b) for a, b in zip(m.counts(), m2.counts()))


# ----------------------------------------------------------------------------- randomised sweep

def test_random_grids_all_variants_vs_oracle(env):
    """Seeded fuzz: odd grid shapes (down to 1 x 1), resolutions, beam counts that are not warp multiples,
    sensors and endpoints inside / outside / far outside, degenerate beams -- every kernel variant, with and
    without workspace, must reproduce the oracle's counts bit for bit."""
    rng = np.random.Generator(np.random.PCG64(20251018))
    for trial in range(40):
        xw = int(rng.choice([1, 2, 3, 7, 31, 32, 33, 64, 100, 129, 257, 300]))
        yw = int(rng.choice([1, 2, 5, 16, 31, 33, 65, 128, 200, 255, 320]))
        reso = float(rng.choice([0.05, 0.1, 0.155, 0.25, 1.0]))
        K = int(rng.integers(1, 6))
        N = int(rng.choice([1, 2, 31, 32, 33, 100, 120, 257]))
        S, Hx, Hy = env.dev.grid_scale(xw, yw, reso)
        span = max(xw, yw) * reso
        cx = rng.uniform(-span, span, K).astype(np.float32)
        cy = rng.uniform(-span, span, K).astype(np.float32)
        ang = rng.uniform(-np.pi, np.pi, (K, N))
        r = rng.uniform(0.0, 2.5 * span, (K, N)) * rng.choice([0.0, 0.05, 1.0], size=(K, N), p=[0.05, 0.25, 0.7])
        ox = (cx[:, None] + r * np.cos(ang)).astype(np.float32)
        oy = (cy[:, None] + r * np.sin(ang)).astype(np.float32)
        if trial % 5 == 0:
            ox[0, 0] = np.inf
        oh = np.zeros((xw, yw), dtype=np.int32)
        om = np.zeros((xw, yw), dtype=np.int32)
        env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
        dev = [torch.from_numpy(a).cuda() for a in (ox, oy, cx, cy)]
        for v, name in _variants(env):
            hit, miss = env.dev.new_planes(xw, yw)
            ws = env.dev.new_workspace(xw, yw) if v >= 4 else None
            env.dev.grid_raycast(hit, miss, S, Hx, Hy, *dev, workspace=ws)
            ok = np.array_equal(hit.cpu().numpy(), oh) and np.array_equal(miss.cpu().numpy(), om)
            assert ok, "trial %d %s grid %dx%d reso %g K %d N %d" % (trial, name, xw, yw, reso, K, N)
        m = env.b2slam.Mapping(xw, yw, reso)
        pm = m.update_batch(ox, oy, cx, cy)
        assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1])


def test_single_scan_updates_patch_only_touched_tiles(env):
    """Mapping.update on a large map: incremental read-back must give exactly the full map, call after call,
    also when mixed with batched calls, errors and resets."""
    G = 2048
    ox, oy, cx, cy = env.synth.grid_scans(909, 30, 1080, half_extent_m=40.0)
    m = env.b2slam.Mapping(G, G, 0.05)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    live = None
    for k in range(12):
        pm = m.update(ox[k].astype(np.float64), oy[k].astype(np.float64), float(cx[k]), float(cy[k]))
        env.corc.grid_raycast(oh, om, S, Hx, Hy, ox[k][None], oy[k][None], cx[k:k + 1], cy[k:k + 1])
        assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1].astype(np.float64)), k
        if live is None:
            live = pm
        else:
            assert pm is live                  # the reference hands out its live array; so does update()
        if k == 5:                             # a rejected scan in between changes nothing
            with pytest.raises(ValueError):
                m.update(np.array([1.0, np.nan]), np.array([0.0, 0.0]), 0.0, 0.0)
        if k == 8:                             # a batched call in between: the mirror is rebuilt lazily
            m.update_batch(ox[20:25], oy[20:25], cx[20:25], cy[20:25])
            env.corc.grid_raycast(oh, om, S, Hx, Hy, ox[20:25], oy[20:25], cx[20:25], cy[20:25])
            live = None
    assert np.array_equal(m.occupancy(), env.corc.grid_finalize(oh, om)[1])
    m.reset()
    pm = m.update(ox[0].astype(np.float64), oy[0].astype(np.float64), float(cx[0]), float(cy[0]))
    oh[:] = 0
    om[:] = 0
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox[0][None], oy[0][None], cx[0:1], cy[0:1])
    assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1].astype(np.float64))


def test_layer1_validate_flags(env):
    """b2s_grid_validate: NaN -> flags[0], inf in oy / sensor position -> flags[1], inf in ox alone is legal."""
    L = env.lib.lib()
    ox, oy, cx, cy = env.synth.grid_scans(1, 4, 100, half_extent_m=5.0)

    def run(ox, oy, cx, cy):
        dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (ox, oy, cx, cy)]
        flags = torch.zeros(2, dtype=torch.int32, device="cuda")
        env.lib.check(L.b2s_grid_validate(dev[0].data_ptr(), dev[1].data_ptr(), dev[2].data_ptr(), dev[3].data_ptr(),
                                          ox.shape[0], ox.shape[1], flags.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream))
        return flags.tolist()

    assert run(ox, oy, cx, cy) == [0, 0]
    a = ox.copy(); a[1, 5] = np.inf
    assert run(a, oy, cx, cy) == [0, 0]
    b = oy.copy(); b[1, 5] = np.inf
    assert run(a, b, cx, cy) == [0, 0]          # the beam is skipped before oy is looked at ([MAP]:30)
    b = oy.copy(); b[2, 7] = np.inf
    assert run(ox, b, cx, cy) == [0, 1]
    a = ox.copy(); a[3, 99] = np.nan
    assert run(a, oy, cx, cy) == [1, 0]
    c = cx.copy(); c[0] = -np.inf
    assert run(ox, oy, c, cy) == [0, 1]


def test_streamed_mapping_calls_equal_blocking_calls(env):
    """Mapping.submit_scans / submit_batch + MapTicket.wait (b2s_mapping_submit* / b2s_mapping_wait), two steps in flight:
    every step's map equals the oracle's after that step, the counts at the end are the sum of all steps, a step the
    reference would raise on raises at ITS ticket and is taken back out exactly, and zero_first starts over."""
    import math
    from b2slam import scan
    G = 1024
    S, Hx, Hy = env.dev.grid_scale(G, G, 0.05)
    m = env.b2slam.Mapping(G, G, 0.05)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    beams = scan.beam_table(-math.pi, math.pi, 360)
    want, tickets = [], []
    for k in range(7):
        if k % 2:
            ox, oy, cx, cy = env.synth.grid_scans(400 + k, 96, 360, half_extent_m=20.0)
            tickets.append(m.submit_batch(ox, oy, cx, cy))
            env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
        else:
            ranges, poses = env.synth.grid_scan_ranges(400 + k, 96, 360, half_extent_m=20.0)
            tickets.append(m.submit_scans(ranges, poses, -math.pi, math.pi))
            env.corc.grid_raycast_ranges(oh, om, S, Hx, Hy, ranges, scan.pose_table(poses), beams, 30.0)
        want.append(env.corc.grid_finalize(oh, om)[1].copy())
        if k >= 1:
            assert np.array_equal(tickets[k - 1].wait(), want[k - 1]), "step %d" % (k - 1)
    assert np.array_equal(tickets[-1].wait(), want[-1])
    h, ms = m.counts()
    assert np.array_equal(h, oh) and np.array_equal(ms, om)
    # a bad step: raises at its own ticket, is rolled back exactly; the good step submitted behind it stays applied
    ox, oy, cx, cy = env.synth.grid_scans(999, 16, 360, half_extent_m=20.0)
    bad = oy.copy()
    bad[3, 5] = np.nan
    t_bad = m.submit_batch(ox, bad, cx, cy)
    t_ok = m.submit_batch(ox, oy, cx, cy)
    with pytest.raises(ValueError):
        t_bad.wait()
    t_ok.wait()
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
    h, ms = m.counts()
    assert np.array_equal(h, oh) and np.array_equal(ms, om)
    # the blocking call after streamed steps, and zero_first
    pm = m.update_batch(ox, oy, cx, cy)
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
    assert np.array_equal(pm, env.corc.grid_finalize(oh, om)[1])
    t = m.submit_batch(ox, oy, cx, cy, zero_first=True)
    oh[:] = 0
    om[:] = 0
    env.corc.grid_raycast(oh, om, S, Hx, Hy, ox, oy, cx, cy)
    assert np.array_equal(t.wait(), env.corc.grid_finalize(oh, om)[1])
    h, ms = m.counts()
    assert np.array_equal(h, oh) and np.array_equal(ms, om)
