"""Which code the default ray-cast (variant 6) runs for a given input, and parity on inputs built to reach each part.

A variant-6 CTA ray-casts 16 consecutive scans x one 64-beam sector.  It counts into its shared-memory tile only when no
live ray is clipped by the grid and the bounding box of the live beams' sensor and obstacle cells fits the tile,
w * (h | 1) <= 27 * 1024 words; every other CTA runs the variant-5 march.  `v6_routes` is a NumPy model of that
routing (csrc/b2s_grid.cu: beam_cells and the box pass of grid_raycast_v6).  It is a coverage tool, not an oracle:
the parity tests below assert through it that their inputs reach the paths they are about, and check the planes against
oracle.c and variant 5."""
import math

import numpy as np
import pytest

from conftest import load_golden

torch = pytest.importorskip("torch")

V6_SCANS, V6_SECTOR, V6_TILE_WORDS = 16, 64, 27 * 1024   # csrc/b2s_grid.cu
MAX_PATH_CELLS = 1 << 22                                  # include/b2slam.h B2S_MAX_PATH_CELLS
GRID_TILE = 64                                            # csrc/b2s_common.cuh
OK, NOOP, NAN, TOO_LONG, INF_SKIP, OVERFLOW = range(6)    # BeamStatus
ROUTES = ("tile", "clipped", "oversize", "empty")


# ----------------------------------------------------------------------------- the model

def fused_endpoints(ranges, pose4, beam_cs, clamp):
    """load_beam<IN_FUSED> in float64: the world-frame endpoints and sensor positions of raw ranges + poses."""
    r = np.asarray(ranges, dtype=np.float32).astype(np.float64)
    if clamp and clamp > 0:
        r = np.where(r == np.inf, clamp, r)
    px, py = beam_cs[None, :, 0] * r, beam_cs[None, :, 1] * r
    x, y, cw, sw = (pose4[:, k:k + 1] for k in range(4))
    with np.errstate(invalid="ignore"):
        ox = (cw * px + (-sw) * py) + x
        oy = (sw * px + cw * py) + y
    return ox, oy, np.broadcast_to(x, ox.shape), np.broadcast_to(y, ox.shape)


def beam_cells(xw, yw, S, Hx, Hy, ox, oy, cx, cy):
    """beam_cells for every beam: (status, sx, sy, hx, hy, span) arrays of the shape of ox.  Inputs are widened to
    float64 exactly (float32 -> float64), the cell is trunc(S * (v + H))."""
    ox, oy = np.asarray(ox, dtype=np.float64), np.asarray(oy, dtype=np.float64)
    cx = np.broadcast_to(np.asarray(cx, dtype=np.float64).reshape(-1, 1) if np.ndim(cx) == 1 else cx, ox.shape)
    cy = np.broadcast_to(np.asarray(cy, dtype=np.float64).reshape(-1, 1) if np.ndim(cy) == 1 else cy, ox.shape)
    st = np.full(ox.shape, OK, dtype=np.int8)
    with np.errstate(invalid="ignore", over="ignore"):
        dxo, dyo, dxc, dyc = (S * (v + H) for v, H in ((ox, Hx), (oy, Hy), (cx, Hx), (cy, Hy)))
        fin = np.isfinite(dxo) & np.isfinite(dyo) & np.isfinite(dxc) & np.isfinite(dyc)
        lim = 1073741824.0
        inlim = fin & (np.abs(dxo) < lim) & (np.abs(dyo) < lim) & (np.abs(dxc) < lim) & (np.abs(dyc) < lim)
        cell = [np.where(inlim, np.trunc(v), 0).astype(np.int64) for v in (dxc, dyc, dxo, dyo)]
    sx, sy, hx, hy = cell
    span = np.maximum(np.abs(hx - sx), np.abs(hy - sy))
    outside = (np.maximum(sx, hx) < 0) | (np.minimum(sx, hx) >= xw) | (np.maximum(sy, hy) < 0) | (np.minimum(sy, hy) >= yw)
    # the order of the kernel's tests: the first that applies wins
    st = np.where(span > MAX_PATH_CELLS, TOO_LONG, st)
    st = np.where(((sx == hx) & (sy == hy)) | outside, NOOP, st)
    st = np.where(~inlim, TOO_LONG, st)
    st = np.where(np.isinf(oy) | np.isinf(cx) | np.isinf(cy), OVERFLOW, st)
    st = np.where(np.isnan(ox) | np.isnan(oy) | np.isnan(cx) | np.isnan(cy), NAN, st)
    st = np.where(np.isinf(ox), INF_SKIP, st)
    return st, sx, sy, hx, hy, span


def v6_routes(xw, yw, S, Hx, Hy, ox, oy, cx, cy):
    """Route of every CTA of one variant-6 launch, in blockIdx order (scan group major, sector minor): an array of
    "tile", "clipped", "oversize" or "empty" (no live beam).  ox, oy (K, N); cx, cy (K,) or (K, N)."""
    st, sx, sy, hx, hy, _ = beam_cells(xw, yw, S, Hx, Hy, ox, oy, cx, cy)
    K, N = st.shape
    G, C = -(-K // V6_SCANS), -(-N // V6_SECTOR)

    def blocks(a, fill):
        p = np.full((G * V6_SCANS, C * V6_SECTOR), fill, dtype=a.dtype)
        p[:K, :N] = a
        return p.reshape(G, V6_SCANS, C, V6_SECTOR).transpose(0, 2, 1, 3).reshape(G * C, -1)

    live = blocks(st == OK, False)
    big, small = np.iinfo(np.int64).max, np.iinfo(np.int64).min
    lo_x = np.where(live, blocks(np.minimum(sx, hx), 0), big).min(axis=1)
    hi_x = np.where(live, blocks(np.maximum(sx, hx), 0), small).max(axis=1)
    lo_y = np.where(live, blocks(np.minimum(sy, hy), 0), big).min(axis=1)
    hi_y = np.where(live, blocks(np.maximum(sy, hy), 0), small).max(axis=1)
    empty = ~live.any(axis=1)
    clipped = ~empty & ((lo_x < 0) | (hi_x >= xw) | (lo_y < 0) | (hi_y >= yw))
    w, h = hi_x - lo_x + 1, hi_y - lo_y + 1
    oversize = ~empty & ~clipped & (w * (h | 1) > V6_TILE_WORDS)
    out = np.full(G * C, "tile", dtype=object)
    out[oversize] = "oversize"
    out[clipped] = "clipped"
    out[empty] = "empty"
    return out


def route_counts(routes):
    return {r: int((np.asarray(routes) == r).sum()) for r in ROUTES}


def v6_boxes(xw, yw, S, Hx, Hy, ox, oy, cx, cy):
    """(x0, x1, y0, y1) of every CTA's box (None for an empty CTA), blockIdx order."""
    st, sx, sy, hx, hy, _ = beam_cells(xw, yw, S, Hx, Hy, ox, oy, cx, cy)
    K, N = st.shape
    out = []
    for g in range(0, K, V6_SCANS):
        for b in range(0, N, V6_SECTOR):
            live = st[g:g + V6_SCANS, b:b + V6_SECTOR] == OK
            if not live.any():
                out.append(None)
                continue
            xs = np.concatenate([sx[g:g + V6_SCANS, b:b + V6_SECTOR][live], hx[g:g + V6_SCANS, b:b + V6_SECTOR][live]])
            ys = np.concatenate([sy[g:g + V6_SCANS, b:b + V6_SECTOR][live], hy[g:g + V6_SCANS, b:b + V6_SECTOR][live]])
            out.append((int(xs.min()), int(xs.max()), int(ys.min()), int(ys.max())))
    return out


# ----------------------------------------------------------------------------- inputs built cell by cell

RESO = 0.05


class Launch(object):
    """One launch described once and fed in the three input forms.  Sensor k sits at the centre of cell sc[k]; beam j of
    scan k ends at sc[k] + r[k, j] * d[j] (cells), i.e. the fused form with pose (x, y, cos 1, sin 0) and beam table d * RESO
    (so both endpoint forms get bit for bit what the fused kernel computes).  An infinite range takes the clamp."""

    def __init__(self, xw, yw, sc, d, r, clamp=1.0):
        self.xw, self.yw, self.clamp = xw, yw, clamp
        self.S, self.Hx, self.Hy = 1.0 / RESO, xw * RESO / 2.0, yw * RESO / 2.0
        sc = np.asarray(sc, dtype=np.float64)
        self.ranges = np.ascontiguousarray(r, dtype=np.float32)
        self.pose4 = np.stack([(sc[:, 0] + 0.5) * RESO - self.Hx, (sc[:, 1] + 0.5) * RESO - self.Hy,
                               np.ones(len(sc)), np.zeros(len(sc))], axis=1)
        self.beam_cs = np.ascontiguousarray(np.asarray(d, dtype=np.float64) * RESO)
        ox, oy, cx, cy = fused_endpoints(self.ranges, self.pose4, self.beam_cs, clamp)
        self.f64 = [np.ascontiguousarray(a) for a in (ox, oy, cx[:, 0], cy[:, 0])]

    def arrays(self, mode):
        return [a.astype(np.float32) for a in self.f64] if mode == "f32" else [a.copy() for a in self.f64]

    def routes(self, mode="f64", arrays=None):
        if mode == "fused":
            return v6_routes(self.xw, self.yw, self.S, self.Hx, self.Hy,
                             *fused_endpoints(self.ranges, self.pose4, self.beam_cs, self.clamp))
        return v6_routes(self.xw, self.yw, self.S, self.Hx, self.Hy, *(arrays or self.arrays(mode)))

    def boxes(self):
        return v6_boxes(self.xw, self.yw, self.S, self.Hx, self.Hy, *self.f64)


def fan(n, ax, ay):
    """n beam offsets (cells) round an ellipse of half-axes ax, ay; beams 0, n/4, n/2, 3n/4 reach the four extremes."""
    t = 2.0 * np.pi * np.arange(n) / n
    return np.stack([np.rint(ax * np.cos(t)), np.rint(ay * np.sin(t))], axis=1).astype(np.int64)


def capacity_launch(w, h):
    """16 scans x 64 beams, one CTA, whose box is exactly w x h cells: the sensor on the box's corner (bx, by), 32 beams
    to the far column, 32 to the far row."""
    bx, by = 37, 50
    ys = np.rint(np.linspace(0, h - 1, 32)).astype(np.int64)
    xs = np.rint(np.linspace(1, w - 1, 32)).astype(np.int64)
    d = np.concatenate([np.stack([np.full(32, w - 1), ys], 1), np.stack([xs, np.full(32, h - 1)], 1)])
    return Launch(w + 76, 333, np.tile([bx, by], (16, 1)), d, np.ones((16, 64)))


def edge_launch(xw, yw, a=50):
    """Four CTAs (64 scans x 64 beams) whose boxes (2a + 1 cells square) touch, without crossing, the corners of the
    grid: x = 0 and y = 0, x = xw - 1 and y = yw - 1, and the two mixed corners."""
    lo_x, hi_x, lo_y, hi_y = a, xw - 1 - a, a, yw - 1 - a
    corners = [(lo_x, lo_y), (hi_x, hi_y), (lo_x, hi_y), (hi_x, lo_y)]
    sc = np.repeat(np.array(corners), 16, axis=0)
    return Launch(xw, yw, sc, fan(64, a, a), np.ones((64, 64)))


def mixed_launch():
    """One launch on 1000 x 333 with a tile, a clipped, an oversize and an empty CTA, in that order."""
    xw, yw = 1000, 333
    sc = np.repeat(np.array([(500, 160), (20, 160), (700, 160), (300, 160)]), 16, axis=0)
    r = np.ones((64, 64))
    r[32:48] = 2.0          # 241 x 241 cells: does not fit
    r[48:64] = 0.0          # every endpoint in the sensor's cell: no live beam
    return Launch(xw, yw, sc, fan(64, 60, 60), r)


def slope_offsets():
    """Beam offsets (cells) with |minor| / span = k / q for every reduced fraction k / q, q <= 16, in all eight octants,
    plus the axis-aligned and 45-degree beams of span 1 and 2."""
    from math import gcd
    base = set()
    for q in range(1, 17):
        for k in range(0, q + 1):
            if gcd(k, q) == 1:
                span = q * max(1, 48 // q)
                base.add((span, k * span // q))
    base |= {(1, 0), (1, 1), (2, 0), (2, 1), (2, 2)}
    out = set()
    for a, b in base:
        for sx in (1, -1):
            for sy in (1, -1):
                out.add((sx * a, sy * b))
                out.add((sy * b, sx * a))
    return np.array(sorted(out), dtype=np.int64)


def slope_launch():
    d = slope_offsets()
    K = 16
    sc = np.stack([333 + np.arange(K), 160 - np.arange(K) // 2], axis=1)
    return Launch(1000, 333, sc, d, np.ones((K, len(d))))


def partial_launch(K, N):
    """K scans x N beams of a slowly moving sensor: CTAs with 1 or 15 scans, units with 1, 31 or 33 beams."""
    sc = np.stack([400 + np.arange(K), 150 + (np.arange(K) % 5)], axis=1)
    r = np.where((np.arange(K)[:, None] + np.arange(N)[None, :]) % 3 == 0, 0.5, 1.0)
    return Launch(1000, 333, sc, 2 * fan(N, 30, 20), r)


EDGE_LAUNCHES = {
    "cap_1024x27": lambda: capacity_launch(1024, 27),
    "cap_1024x26": lambda: capacity_launch(1024, 26),
    "cap_1025x27": lambda: capacity_launch(1025, 27),
    "cap_1024x28": lambda: capacity_launch(1024, 28),
    "cap_167x165": lambda: capacity_launch(167, 165),
    "cap_168x165": lambda: capacity_launch(168, 165),
    "edges_200x200": lambda: edge_launch(200, 200),
    "edges_333x1000": lambda: edge_launch(333, 1000),
    "edges_1000x333": lambda: edge_launch(1000, 333),
    "mixed": mixed_launch,
    "slopes": slope_launch,
    "partial_17x31": lambda: partial_launch(17, 31),
    "partial_15x63": lambda: partial_launch(15, 63),
    "partial_33x97": lambda: partial_launch(33, 97),
    "partial_31x129": lambda: partial_launch(31, 129),
}

# the model's route counts (tile, clipped, oversize, empty) that each launch is built to give
EDGE_ROUTES = {
    "cap_1024x27": (1, 0, 0, 0), "cap_1024x26": (1, 0, 0, 0), "cap_1025x27": (0, 0, 1, 0),
    "cap_1024x28": (0, 0, 1, 0), "cap_167x165": (1, 0, 0, 0), "cap_168x165": (0, 0, 1, 0),
    "edges_200x200": (4, 0, 0, 0), "edges_333x1000": (4, 0, 0, 0), "edges_1000x333": (4, 0, 0, 0),
    "mixed": (1, 1, 1, 1),
}


# ----------------------------------------------------------------------------- CPU checks of the model and the inputs

@pytest.mark.parametrize("w,h", [(1024, 27), (1024, 26), (1025, 27), (1024, 28), (167, 165), (168, 165)])
def test_capacity_launches_have_the_intended_box(w, h):
    L = capacity_launch(w, h)
    (x0, x1, y0, y1), = L.boxes()
    assert (x1 - x0 + 1, y1 - y0 + 1) == (w, h)
    assert x0 > 0 and x1 < L.xw - 1 and y0 > 0 and y1 < L.yw - 1
    fits = w * (h | 1) <= V6_TILE_WORDS
    assert list(L.routes("f32")) == list(L.routes("f64")) == list(L.routes("fused")) == ["tile" if fits else "oversize"]


@pytest.mark.parametrize("name", sorted(EDGE_ROUTES))
def test_edge_launches_route_as_intended(name):
    L = EDGE_LAUNCHES[name]()
    for mode in ("f32", "f64", "fused"):
        c = route_counts(L.routes(mode))
        assert tuple(c[r] for r in ROUTES) == EDGE_ROUTES[name], (name, mode, c)


@pytest.mark.parametrize("shape", [(200, 200), (333, 1000), (1000, 333)])
def test_edge_boxes_touch_the_grid_border(shape):
    xw, yw = shape
    boxes = edge_launch(xw, yw).boxes()
    assert boxes[0][0] == 0 and boxes[0][2] == 0 and boxes[1][1] == xw - 1 and boxes[1][3] == yw - 1
    assert boxes[2][0] == 0 and boxes[2][3] == yw - 1 and boxes[3][1] == xw - 1 and boxes[3][2] == 0


def test_slope_launch_hits_the_half_exactly_and_one_ulp_below():
    """The reference's recurrence on these beams lands on acc == 0.5 and on the double just below it, where the tile
    march's integer compare of the high word must still agree with acc >= 0.5."""
    d = slope_offsets()
    assert len(d) > 600 and {(1, 0), (0, -1), (1, 1), (-1, -1)} <= {tuple(v) for v in d}
    half, below = 0, 0
    for dx, dy in d:
        span = max(abs(dx), abs(dy))
        slope = min(abs(dx), abs(dy)) / float(span)
        acc = 0.0
        for _ in range(span):
            acc += slope
            half += acc == 0.5
            below += acc == np.nextafter(0.5, 0.0)
            if acc >= 0.5:
                acc -= 1.0
    assert half > 100 and below > 0
    c = route_counts(slope_launch().routes())
    assert c["tile"] >= 10 and c["tile"] == sum(c.values())


@pytest.mark.parametrize("K,N", [(17, 31), (15, 63), (33, 97), (31, 129)])
def test_partial_launches_reach_the_tile(K, N):
    L = partial_launch(K, N)
    routes = L.routes()
    assert len(routes) == (-(-K // 16)) * (-(-N // 64)) and (routes == "tile").all()


def test_model_statuses_follow_the_kernel_order():
    st, *_ = beam_cells(100, 100, 20.0, 2.5, 2.5,
                        np.array([[np.inf, np.nan, 1.0, 1e9, 3e5, 0.001, 100.0, 1.0, np.inf]]),
                        np.array([[np.nan, 0.0, np.inf, 0.0, 0.0, 0.001, 100.0, 1.0, np.inf]]),
                        np.array([0.0]), np.array([0.0]))
    # (100, 100) leaves the grid but its segment crosses it: live, and clipped
    assert st[0].tolist() == [INF_SKIP, NAN, OVERFLOW, TOO_LONG, TOO_LONG, NOOP, OK, OK, INF_SKIP]


# ----------------------------------------------------------------------------- GPU parity on the built inputs

@pytest.fixture(scope="module")
def env():
    import b2slam
    from b2slam import _lib, devapi
    from oracle import corc
    if _lib.device_count() <= 0:
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box")

    class E:
        pass
    e = E()
    e.b2slam, e.lib, e.dev, e.corc = b2slam, _lib, devapi, corc
    return e


ARMS = {"v5": (5, 1), "v6/layout0": (6, 0), "v6/layout1": (6, 1)}   # grid_variant, grid_tile_layout


def _select(env, arm):
    L = env.lib.lib()
    assert L.b2s_tune(b"grid_variant", arm[0]) == 0 and L.b2s_tune(b"grid_tile_layout", arm[1]) == 0


@pytest.fixture(autouse=True)
def _default_kernel(request):
    """GPU tests start on the default kernel and leave it selected, whether they pass or fail."""
    if request.node.get_closest_marker("gpu") is None:
        yield
        return
    e = request.getfixturevalue("env")
    _select(e, ARMS["v6/layout1"])
    try:
        yield
    finally:
        _select(e, ARMS["v6/layout1"])


def _cast(env, arm, L, mode, arrays=None):
    """One launch of L (with a workspace) under arm; returns hit, miss, counters as NumPy arrays."""
    _select(env, ARMS[arm])
    hit, miss = env.dev.new_planes(L.xw, L.yw)
    ws = env.dev.new_workspace(L.xw, L.yw)
    cnt = torch.zeros(4, dtype=torch.int32, device="cuda")
    if mode == "fused":
        env.dev.grid_raycast_ranges(hit, miss, L.S, L.Hx, L.Hy, *[torch.from_numpy(a).cuda() for a in
                                    (L.ranges, L.pose4, L.beam_cs)], L.clamp, counters=cnt, workspace=ws)
    else:
        env.dev.grid_raycast(hit, miss, L.S, L.Hx, L.Hy, *[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in
                             (arrays or L.arrays(mode))], counters=cnt, workspace=ws)
    torch.cuda.synchronize()
    return hit.cpu().numpy(), miss.cpu().numpy(), cnt.cpu().numpy()


def _oracle(env, L, mode, arrays=None):
    oh = np.zeros((L.xw, L.yw), dtype=np.int32)
    om = np.zeros((L.xw, L.yw), dtype=np.int32)
    if mode == "fused":
        env.corc.grid_raycast_ranges(oh, om, L.S, L.Hx, L.Hy, L.ranges, L.pose4, L.beam_cs, L.clamp)
    else:
        env.corc.grid_raycast(oh, om, L.S, L.Hx, L.Hy, *(arrays or L.arrays(mode)))
    return oh, om


def _check(env, L, mode, arrays=None, oracle=True):
    """Both variant-6 layouts against variant 5 (planes byte for byte, counters) and, with oracle, against oracle.c."""
    h5, m5, c5 = _cast(env, "v5", L, mode, arrays)
    if oracle:
        oh, om = _oracle(env, L, mode, arrays)
        assert np.array_equal(h5, oh) and np.array_equal(m5, om), mode
    for arm in ("v6/layout0", "v6/layout1"):
        h, m, c = _cast(env, arm, L, mode, arrays)
        if oracle:
            bad = np.argwhere((h != oh) | (m != om))
            assert len(bad) == 0, "%s %s: %d cells differ from oracle.c, first %s" % (mode, arm, len(bad), bad[:4])
        assert np.array_equal(h, h5) and np.array_equal(m, m5), (mode, arm)
        assert c.tolist() == c5.tolist(), (mode, arm)
    return h5, m5, c5


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(EDGE_LAUNCHES))
def test_tile_path_edges_match_oracle_and_v5(env, name):
    """Tile capacity, boxes on the grid's border, a mixed launch, exact slopes and partial CTAs, as float32 and float64
    endpoints and as raw ranges + poses (some of them infinite, taking the clamp)."""
    L = EDGE_LAUNCHES[name]()
    routes = L.routes()
    assert (routes == "tile").any() or name in ("cap_1025x27", "cap_1024x28", "cap_168x165")
    if name in ("mixed", "slopes") or name.startswith("partial"):
        r = L.ranges[:, ::7]
        r[r == 1.0] = np.inf             # the clamp (1.0) gives back the same endpoints
    for mode in ("f32", "f64", "fused"):
        assert list(L.routes(mode)) == list(routes), mode
        h, m, c = _check(env, L, mode)
        assert c.tolist() == [0, 0, 0, 0] and m.sum() > 0


@pytest.mark.gpu
def test_tile_ctas_holding_rejected_and_skipped_beams(env):
    """Tile CTAs that also hold NaN, inf-in-ox, inf-in-oy, too-long (coordinate and span) beams: planes and counters
    equal variant 5's, the counters are what the model says, and the other beams equal oracle.c."""
    L = mixed_launch()
    specials = [(1, 3), (2, 9), (5, 17), (9, 33), (14, 60)]   # (scan, beam) inside the tile CTA (scans 0-15)
    for mode in ("f32", "f64"):
        a = L.arrays(mode)
        ox, oy = a[0], a[1]
        ox[1, 3] = np.nan
        ox[2, 9] = np.inf
        oy[5, 17] = np.inf
        ox[9, 33] = 1e9                              # |S (v + H)| >= 2^30
        ox[14, 60] = 3e5                             # span > B2S_MAX_PATH_CELLS
        c = route_counts(L.routes(mode, a))
        assert (c["tile"], c["clipped"], c["oversize"], c["empty"]) == (1, 1, 1, 1)
        st = beam_cells(L.xw, L.yw, L.S, L.Hx, L.Hy, *a)[0]
        assert [int(st[s, b]) for s, b in specials] == [NAN, INF_SKIP, OVERFLOW, TOO_LONG, TOO_LONG]
        h5, m5, c5 = _check(env, L, mode, a, oracle=False)
        assert c5.tolist() == [1, 2, 1, 1]           # NaN, too long, inf-skipped, overflow
        clean = L.arrays(mode)
        for s, b in specials:
            clean[0][s, b] = np.inf                  # the same beams skipped: what oracle.c can count
        oh, om = _oracle(env, L, mode, clean)
        assert np.array_equal(h5, oh) and np.array_equal(m5, om), mode
    # raw ranges: NaN, too long, and -inf, which the clamp leaves alone (0 * inf in the pose product makes it NaN)
    L.ranges[1, 3] = np.nan
    L.ranges[9, 33] = 1e30
    L.ranges[14, 1] = -np.inf
    fused = fused_endpoints(L.ranges, L.pose4, L.beam_cs, L.clamp)
    assert route_counts(v6_routes(L.xw, L.yw, L.S, L.Hx, L.Hy, *fused))["tile"] == 1
    st = beam_cells(L.xw, L.yw, L.S, L.Hx, L.Hy, *fused)[0]
    _, _, c5 = _check(env, L, "fused", oracle=False)
    assert c5.tolist() == [int((st == k).sum()) for k in (NAN, TOO_LONG, INF_SKIP, OVERFLOW)] == [2, 1, 0, 0]


# ----------------------------------------------------------------------------- the reference's golden maps

def _golden_scans(name):
    """(label, xw, yw, S, H, [(ox, oy, cx, cy) per scan] as float64) of each golden the suite checks the grid with."""
    out = []
    z = load_golden("mapping.npz")
    for tag in ("w20", "w4"):
        out.append(("mapping_" + tag, [tuple(np.asarray(z[tag + k][s], dtype=np.float64).reshape(1, -1)
                                             for k in ("_ox", "_oy", "_cx", "_cy")) for s in range(8)]))
    z = load_golden("mapping_f64.npz")
    for tag in ("g200", "g4096", "g16384"):
        K = z[tag + "_ox"].shape[0]
        out.append((tag, [tuple(np.asarray(z[tag + k][s]).reshape(1, -1) for k in ("_ox", "_oy", "_cx", "_cy"))
                          for s in range(K)]))
    z = load_golden("ingestion.npz")
    from b2slam import scan
    ox, oy, cx, cy = fused_endpoints(z["ranges"], scan.pose_table(z["poses"]),
                                     scan.beam_table(-math.pi, math.pi, z["ranges"].shape[1]), 30.0)
    out.append(("ingestion", [(ox[s:s + 1], oy[s:s + 1], cx[s:s + 1, :1], cy[s:s + 1, :1]) for s in range(8)]))
    return dict(out)[name]


def _golden_counts(name, side, H, batch):
    scans = _golden_scans(name)
    if batch:
        scans = [tuple(np.concatenate([s[k] for s in scans]) for k in range(4))]
    c = {r: 0 for r in ROUTES}
    for ox, oy, cx, cy in scans:
        for r, n in route_counts(v6_routes(side, side, 10.0, H, H, ox, oy, cx.reshape(-1), cy.reshape(-1))).items():
            c[r] += n
    return tuple(c[r] for r in ROUTES)


# (golden, grid side, H, one launch for all scans?) -> model's (tile, clipped, oversize, empty) CTA counts over the calls.
# Batched, every golden falls back: at 0.1 m a 64-beam sector of 8 scans spans more than the tile, and at the golden's
# own size some ray leaves the grid.  Scan by scan (Mapping.update) the 120-beam goldens reach the tile; the 800^2 and
# 4700^2 companions move the same scans ~300 cells inside the grid.  g200's beams (to 69 m) overflow the tile at any size.
GOLDEN_ROUTES = {
    ("mapping_w20", 200, 10.0, True): (0, 2, 0, 0), ("mapping_w20", 200, 10.0, False): (4, 12, 0, 0),
    ("mapping_w4", 200, 10.0, True): (0, 2, 0, 0), ("mapping_w4", 200, 10.0, False): (4, 12, 0, 0),
    ("mapping_w20", 800, 40.0, True): (0, 0, 2, 0), ("mapping_w20", 800, 40.0, False): (8, 0, 8, 0),
    ("g200", 200, 10.0, True): (0, 3, 0, 0), ("g200", 200, 10.0, False): (0, 24, 0, 0),
    ("g200", 2000, 100.0, False): (0, 0, 24, 0),
    ("g4096", 4096, 10.0, True): (0, 4, 0, 0), ("g4096", 4700, 40.0, False): (6, 6, 12, 0),
    ("g16384", 16384, 10.0, True): (0, 4, 0, 0),
    ("ingestion", 200, 10.0, True): (0, 2, 0, 0), ("ingestion", 200, 10.0, False): (8, 8, 0, 0),
}


@pytest.mark.parametrize("key", sorted(GOLDEN_ROUTES), ids=lambda k: "%s-%d-%s" % (k[0], k[1], "batch" if k[3] else "scans"))
def test_golden_route_counts(key):
    assert _golden_counts(*key) == GOLDEN_ROUTES[key]


def _finalize(env, oh, om, w_hit=20.0):
    return env.corc.grid_finalize(oh, om, w_hit)[1]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("tag,w_hit", [("w20", 20.0), ("w4", 4.0)])
def test_mapping_golden_on_a_larger_grid_takes_the_tile(env, layout, tag, w_hit):
    """The scans of mapping.npz, scan by scan (8 tile CTAs) and batched, on an 800 x 800 map at the same 0.1 m: counts and
    map against oracle.c after every call."""
    assert _golden_counts("mapping_" + tag, 800, 40.0, False)[0] > 0
    _select(env, (6, layout))
    z = load_golden("mapping.npz")
    m = env.b2slam.Mapping(800, 800, 0.1, hit_weight=w_hit)
    oh = np.zeros((800, 800), dtype=np.int32)
    om = np.zeros((800, 800), dtype=np.int32)
    for ox, oy, cx, cy in zip(z[tag + "_ox"], z[tag + "_oy"], z[tag + "_cx"], z[tag + "_cy"]):
        pm = m.update(ox.astype(np.float64), oy.astype(np.float64), float(cx), float(cy))
        env.corc.grid_raycast(oh, om, 10.0, 40.0, 40.0, ox[None], oy[None], cx[None], cy[None])
        assert np.array_equal(pm, _finalize(env, oh, om, w_hit).astype(np.float64))
    hit, miss = m.counts()
    assert np.array_equal(hit, oh) and np.array_equal(miss, om)
    mb = env.b2slam.Mapping(800, 800, 0.1, hit_weight=w_hit)
    pb = mb.update_batch(z[tag + "_ox"], z[tag + "_oy"], z[tag + "_cx"], z[tag + "_cy"])
    assert np.array_equal(pb, _finalize(env, oh, om, w_hit)) and all(np.array_equal(a, b) for a, b in
                                                                     zip(mb.counts(), (oh, om)))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [0, 1])
def test_ingestion_golden_scan_by_scan(env, layout):
    """ingestion.npz through update_scans one scan at a time (8 tile CTAs) gives the reference's own map."""
    assert _golden_counts("ingestion", 200, 10.0, False)[0] > 0
    _select(env, (6, layout))
    z = load_golden("ingestion.npz")
    m = env.b2slam.Mapping(200, 200, 0.1)
    for s in range(z["ranges"].shape[0]):
        pm = m.update_scans(z["ranges"][s:s + 1], z["poses"][s:s + 1], float(z["angle_min"]), float(z["angle_max"]))
    assert np.array_equal(pm, z["pmap"])
    np.testing.assert_allclose(m.datamap, z["datamap"], rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [0, 1])
def test_float64_golden_on_a_larger_grid_takes_the_tile(env, layout):
    """g4096's float64 scans, one launch per scan, on 4700^2 with the offset moved from 10 m to 40 m (6 tile CTAs):
    both planes against the float64 oracle and against variant 5."""
    assert _golden_counts("g4096", 4700, 40.0, False)[0] > 0
    G = 4700
    planes = {}
    for arm in ((5, 1), (6, layout)):
        _select(env, arm)
        hit, miss = env.dev.new_planes(G, G)
        ws = env.dev.new_workspace(G, G)
        for ox, oy, cx, cy in _golden_scans("g4096"):
            env.dev.grid_raycast(hit, miss, 10.0, 40.0, 40.0, *[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in
                                 (ox, oy, cx.reshape(-1), cy.reshape(-1))], workspace=ws)
        torch.cuda.synchronize()
        planes[arm] = (hit.cpu().numpy(), miss.cpu().numpy())
        del hit, miss, ws
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    for ox, oy, cx, cy in _golden_scans("g4096"):
        env.corc.grid_raycast(oh, om, 10.0, 40.0, 40.0, ox, oy, cx.reshape(-1), cy.reshape(-1))
    for arm, (h, m) in planes.items():
        assert np.array_equal(h, oh) and np.array_equal(m, om), arm


# ----------------------------------------------------------------------------- incremental read-back on the default kernel

def _tiles_of(cells_mask, yw):
    x, y = np.nonzero(cells_mask)
    return set((x // GRID_TILE * (-(-yw // GRID_TILE)) + y // GRID_TILE).tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("xw,yw,reso", [(200, 200, 0.1), (1000, 333, 0.05)])
def test_update_scan_by_scan_patches_ragged_tiles(env, xw, yw, reso):
    """Mapping.update one scan at a time, on the reference's 200 x 200 map and on 1000 x 333: scans in the grid's
    corners (boxes in the ragged last tiles) take the tile, scans over the border fall back; after every call the
    host map equals the oracle's."""
    Hx, Hy = xw * reso / 2.0, yw * reso / 2.0
    spots = [(30, 30), (xw - 31, yw - 31), (xw - 31, 30), (30, yw - 31), (xw // 2, yw // 2), (xw - 5, yw // 2),
             (xw // 2, yw - 3), (xw - 20, yw - 20)]
    d = fan(128, 25, 25)
    m = env.b2slam.Mapping(xw, yw, reso)
    oh = np.zeros((xw, yw), dtype=np.int32)
    om = np.zeros((xw, yw), dtype=np.int32)
    seen = {r: 0 for r in ROUTES}
    for i, j in spots:
        cx, cy = np.array([(i + 0.5) * reso - Hx]), np.array([(j + 0.5) * reso - Hy])
        ox, oy = cx[:, None] + d[None, :, 0] * reso, cy[:, None] + d[None, :, 1] * reso
        for r, n in route_counts(v6_routes(xw, yw, 1.0 / reso, Hx, Hy, ox, oy, cx, cy)).items():
            seen[r] += n
        pm = m.update(ox[0], oy[0], float(cx[0]), float(cy[0]))
        env.corc.grid_raycast(oh, om, 1.0 / reso, Hx, Hy, ox, oy, cx, cy)
        assert np.array_equal(pm, _finalize(env, oh, om).astype(np.float64)), (i, j)
    assert seen["tile"] >= 8 and seen["clipped"] >= 4, seen
    assert np.array_equal(m.occupancy(), _finalize(env, oh, om))


def _incremental(env, m, arrays, cap):
    import ctypes
    f64 = arrays[0].dtype == np.float64
    a = [np.ascontiguousarray(v) for v in arrays]
    ids = np.full(max(cap, 1), -1, dtype=np.int32)
    count = ctypes.c_int(-2)
    fn = m._L.b2s_mapping_update_incremental_f64 if f64 else m._L.b2s_mapping_update_incremental
    env.lib.check(fn(m._h, *[env.lib.ptr(v) for v in a], a[0].shape[0], a[0].shape[1], env.lib.ptr(m._pmap8),
                     env.lib.ptr(ids), cap, ctypes.byref(count)))
    return count.value, ids


@pytest.mark.gpu
def test_incremental_batch_read_back(env):
    """b2s_mapping_update_incremental[_f64] with whole batches on 1000 x 333: the returned tile ids hold every tile whose
    map changed; with tiles_cap below the dirty count, tiles_count is -1 and the map is still patched."""
    xw, yw = 1000, 333
    m = env.b2slam.Mapping(xw, yw, RESO)
    oh = np.zeros((xw, yw), dtype=np.int32)
    om = np.zeros((xw, yw), dtype=np.int32)
    first = edge_launch(xw, yw)
    m.update_batch(*first.arrays("f64"))                  # a full read-back: the host map is current from here on
    env.corc.grid_raycast(oh, om, first.S, first.Hx, first.Hy, *first.arrays("f64"))
    for L, mode, cap in ((slope_launch(), "f64", 1024), (mixed_launch(), "f32", 3), (partial_launch(33, 97), "f32", 1024)):
        assert (L.routes(mode) == "tile").any()
        before = _finalize(env, oh, om)
        env.corc.grid_raycast(oh, om, L.S, L.Hx, L.Hy, *L.arrays(mode))
        after = _finalize(env, oh, om)
        count, ids = _incremental(env, m, L.arrays(mode), cap)
        assert np.array_equal(m._pmap8, after), mode
        changed = _tiles_of(before != after, yw)
        assert changed
        if cap < len(changed):
            assert count == -1
        else:
            assert count >= len(changed) and changed <= set(ids[:count].tolist())
            assert len(set(ids[:count].tolist())) == count


@pytest.mark.gpu
def test_incremental_read_back_beyond_the_pack_capacity(env):
    """More than 1024 dirty 64 x 64 tiles (3000^2 at 0.01 m, 2209 tiles): the whole map is read back instead."""
    G, reso = 3000, 0.01
    m = env.b2slam.Mapping(G, G, reso)
    H = G * reso / 2.0
    c = np.array([0.005])
    ang = np.linspace(-np.pi, np.pi, 1080, endpoint=False)
    ox, oy = c[:, None] + 14.0 * np.cos(ang)[None], c[:, None] + 14.0 * np.sin(ang)[None]
    small = (ox[:, :8] * 0.01, oy[:, :8] * 0.01, c, c)
    m.update_batch(*small)
    oh = np.zeros((G, G), dtype=np.int32)
    om = np.zeros((G, G), dtype=np.int32)
    env.corc.grid_raycast(oh, om, 1.0 / reso, H, H, *small)
    env.corc.grid_raycast(oh, om, 1.0 / reso, H, H, ox, oy, c, c)
    assert len(_tiles_of((oh != 0) | (om != 0), G)) > 1024
    count, _ = _incremental(env, m, (ox, oy, c, c), 1024)
    assert count == -1 and np.array_equal(m._pmap8, _finalize(env, oh, om))


# ----------------------------------------------------------------------------- finalize and ROS packing at odd sizes

@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(200, 200), (1, 1), (33, 70), (300, 180), (3, 3), (2, 3), (3, 5), (333, 7)])
def test_finalize_and_pack_ros_at_odd_shapes(env, shape):
    """grid_finalize (cells % 4 = 1, 2, 3 among these) against oracle.c for pmap and datamap, and grid_pack_ros against
    pmap.T.reshape(-1) ([SLAM]:270-271)."""
    xw, yw = shape
    rng = np.random.Generator(np.random.PCG64(xw * 1000 + yw))
    oh = rng.integers(0, 3, (xw, yw)).astype(np.int32)
    om = (rng.integers(0, 2000, (xw, yw)) * (rng.random((xw, yw)) < 0.7)).astype(np.int32)
    om.reshape(-1)[-1] = 1001                             # the last cell sits in the tail of a shape with cells % 4 != 0
    hit, miss = (torch.from_numpy(a).cuda() for a in (oh, om))
    pm = torch.full((xw, yw), 77, dtype=torch.int8, device="cuda")
    dm = torch.full((xw, yw), -1.0, dtype=torch.float32, device="cuda")
    env.dev.grid_finalize(hit, miss, datamap=dm, pmap=pm)
    score, want = env.corc.grid_finalize(oh, om)
    assert np.array_equal(pm.cpu().numpy(), want)
    assert np.array_equal(dm.cpu().numpy(), score.astype(np.float32))
    ros = env.dev.grid_pack_ros(pm).cpu().numpy()
    assert np.array_equal(ros, want.T.reshape(-1))
