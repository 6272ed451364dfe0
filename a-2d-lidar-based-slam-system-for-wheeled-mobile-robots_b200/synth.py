"""Seeded synthetic 2-D LiDAR workloads (SURVEY.md section 8d).  Host-side NumPy only.

This is input generation for tests and bench.py, not part of the hot path.  All
point coordinates are rounded to float32 ONCE here; the oracle and the CUDA path
both consume those float32 values (upcast exactly to float64 where needed), which
is what makes integer cell indices comparable bit for bit.

Scan model (mirrors the simulated sensor, W12 course_agv.gazebo:32-62): beam angles
linspace(-pi, pi, N); ranges r(phi) = r0 + a sin(k phi + psi), r0 ~ U[3, 8] m,
a ~ U[0.5, 2] m, k in {2..5}, plus N(0, 0.01^2) noise, clipped to [0.10, 30] m.
"""
import numpy as np

RANGE_MIN = 0.10
RANGE_MAX = 30.0
RANGE_SIGMA = 0.01


def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def beam_angles(n_beams):
    return np.linspace(-np.pi, np.pi, n_beams)


def clean_ranges(rng, count, n_beams):
    """(count, n_beams) noise-free range profiles."""
    phi = beam_angles(n_beams)[None, :]
    r0 = rng.uniform(3.0, 8.0, size=(count, 1))
    amp = rng.uniform(0.5, 2.0, size=(count, 1))
    k = rng.integers(2, 6, size=(count, 1)).astype(np.float64)
    psi = rng.uniform(0.0, 2.0 * np.pi, size=(count, 1))
    return r0 + amp * np.sin(k * phi + psi)


def noisy(rng, ranges):
    out = ranges + rng.normal(0.0, RANGE_SIGMA, size=ranges.shape)
    return np.clip(out, RANGE_MIN, RANGE_MAX)


def icp_pairs(seed, pairs, n_beams, max_trans=0.15, max_rot=0.08):
    """Independent scan pairs (cfg 1 with pairs=1 / seed 7001, cfg 4 with seed 4001+rank).

    Returns (tar, src, truth): tar, src float32 (pairs, 2, n_beams) x/y rows;
    truth float64 (pairs, 3) = (tx, ty, theta) of the SE(2) that moved target to source.
    """
    rng = _rng(seed)
    phi = beam_angles(n_beams)[None, :]
    base = clean_ranges(rng, pairs, n_beams)
    r_t = noisy(rng, base)
    r_s = noisy(rng, base)
    tx = rng.uniform(-max_trans, max_trans, size=(pairs, 1))
    ty = rng.uniform(-max_trans, max_trans, size=(pairs, 1))
    th = rng.uniform(-max_rot, max_rot, size=(pairs, 1))
    tar = np.stack([r_t * np.cos(phi), r_t * np.sin(phi)], axis=1)
    sx = r_s * np.cos(phi)
    sy = r_s * np.sin(phi)
    c, s = np.cos(th), np.sin(th)
    src = np.stack([c * sx - s * sy + tx, s * sx + c * sy + ty], axis=1)
    truth = np.concatenate([tx, ty, th], axis=1)
    return tar.astype(np.float32), src.astype(np.float32), truth


def homogeneous(xy):
    """(2, N) -> (3, N) float64 [x; y; 1], the layout ICP.process receives."""
    out = np.ones((3, xy.shape[1]))
    out[:2, :] = xy
    return out


# ------------------------------------------------------------------ cfg 2: room sequence

def _room_polygon(rng):
    """A fixed non-convex room: 12-gon with radius 6..11 m."""
    m = 12
    ang = np.sort(rng.uniform(0, 2 * np.pi, m))
    ang = (ang + np.linspace(0, 2 * np.pi, m, endpoint=False)) / 2.0
    rad = rng.uniform(6.0, 11.0, m)
    return np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=1)


def _raycast_polygon(poly, px, py, ang):
    """Distance from (px,py) along each angle to the nearest polygon edge. ang (K,N)."""
    a = poly
    b = np.roll(poly, -1, axis=0)
    dx = np.cos(ang)[..., None]
    dy = np.sin(ang)[..., None]
    ex = (b[:, 0] - a[:, 0])[None, None, :]
    ey = (b[:, 1] - a[:, 1])[None, None, :]
    ox = a[None, None, :, 0] - px[:, None, None]
    oy = a[None, None, :, 1] - py[:, None, None]
    den = dx * ey - dy * ex
    with np.errstate(divide="ignore", invalid="ignore"):
        t = (ox * ey - oy * ex) / den
        u = (ox * dy - oy * dx) / den
    ok = (np.abs(den) > 1e-12) & (t > 0) & (u >= 0) & (u <= 1)
    t = np.where(ok, t, np.inf)
    return t.min(axis=-1)


def _room_ranges(seed, scans, n_beams, chunk=512):
    """The room, trajectory and noisy float64 ranges (scans, n_beams) behind room_sequence."""
    rng = _rng(seed)
    poly = _room_polygon(rng)
    poses = np.zeros((scans, 3))
    x = y = 0.0
    th = rng.uniform(-np.pi, np.pi)
    w = 0.0
    for i in range(scans):
        poses[i] = (x, y, th)
        w = float(np.clip(0.9 * w + rng.normal(0, 0.01), -0.05, 0.05))
        step = rng.uniform(0.02, 0.1)
        nx, ny = x + step * np.cos(th), y + step * np.sin(th)
        if np.hypot(nx, ny) > 3.5:  # stay well inside the room: turn back toward the origin
            back = np.arctan2(-y, -x)
            d = (back - th + np.pi) % (2 * np.pi) - np.pi
            w = float(np.clip(d, -0.05, 0.05))
            nx, ny = x, y
        x, y = nx, ny
        th = th + w
    phi = beam_angles(n_beams)[None, :]
    r = np.empty((scans, n_beams))
    for s in range(0, scans, chunk):
        e = min(scans, s + chunk)
        ang = phi + poses[s:e, 2:3]
        r[s:e] = noisy(rng, np.minimum(_raycast_polygon(poly, poses[s:e, 0], poses[s:e, 1], ang), RANGE_MAX))
    return poly, r, poses, rng


def room_sequence(seed, scans, n_beams, chunk=512):
    """cfg 2: `scans` scans of one polygon room from a smooth trajectory (seed 9001).

    Steps are <= 0.1 m and <= 0.05 rad per scan.  Returns (xy float32 (scans, 2, n_beams)
    in the sensor frame, poses float64 (scans, 3)).
    """
    _, r, poses, _ = _room_ranges(seed, scans, n_beams, chunk)
    phi = beam_angles(n_beams)[None, :]
    out = np.empty((scans, 2, n_beams), dtype=np.float32)
    out[:, 0, :] = r * np.cos(phi)
    out[:, 1, :] = r * np.sin(phi)
    return out, poses


def _wall_cells(poly, reso, cells, half_width):
    """Centres (2, C) of the cells of a cells x cells map at `reso` m, centred on the origin, that lie within
    half_width of an edge of the polygon: the room rasterised into the obstacle list of a static map."""
    c = (np.arange(cells) + 0.5) * reso - cells * reso / 2.0
    keep = []
    for row in range(0, cells, 256):  # rows of the map in blocks: bounded memory on fine maps
        gx, gy = np.meshgrid(c[row:row + 256], c, indexing="ij")
        near = np.zeros(gx.shape, dtype=bool)
        for a, b in zip(poly, np.roll(poly, -1, axis=0)):
            e = b - a
            t = np.clip(((gx - a[0]) * e[0] + (gy - a[1]) * e[1]) / (e @ e), 0.0, 1.0)
            near |= np.hypot(gx - a[0] - t * e[0], gy - a[1] - t * e[1]) <= half_width
        keep.append(np.stack([gx[near], gy[near]]))
    return np.concatenate(keep, axis=1)


def room_map_observation(seed, scans, n_beams, pose_sigma=(0.03, 0.03, 0.02)):
    """The map observation of W9 localization ([LOC9]:152-157) on the cfg-2 room: a static map, the scans of
    room_sequence's trajectory and the EKF prior poses at which the map is observed.

    Returns a dict: ranges float32 (scans, n_beams) (beam angles linspace(-pi, pi, n_beams)), poses float64 (scans, 3)
    the true poses, prior float64 (scans, 3) the poses perturbed by N(0, pose_sigma) (m, m, rad), and two obstacle lists
    (2, C) of wall cell centres: obstacles_course on the course map's grid (129 x 129 cells at 0.155 m,
    course_agv_gazebo/config/map.yaml; walls 0.2 m either side) and obstacles_fine on a finer, larger one
    (2600 x 2600 cells at 0.01 m; walls 0.25 m either side), more than 2 * 10^5 cells.
    """
    poly, r, poses, rng = _room_ranges(seed, scans, n_beams)
    prior = poses + rng.normal(0.0, 1.0, size=poses.shape) * np.asarray(pose_sigma)
    return {"ranges": r.astype(np.float32), "poses": poses, "prior": prior,
            "obstacles_course": _wall_cells(poly, 0.155, 129, 0.2),
            "obstacles_fine": _wall_cells(poly, 0.01, 2600, 0.25)}


def _polygon_inside(poly, x, y):
    """Even-odd point-in-polygon test of the points (x, y)."""
    inside = np.zeros(x.shape, dtype=bool)
    for a, b in zip(poly, np.roll(poly, -1, axis=0)):
        crosses = (a[1] > y) != (b[1] > y)
        with np.errstate(divide="ignore", invalid="ignore"):
            xc = a[0] + (y - a[1]) * (b[0] - a[0]) / (b[1] - a[1])
        inside ^= crosses & (x < xc)
    return inside


def _polygon_wall_distance(poly, x, y):
    """Distance from the points (x, y) to the nearest edge of the polygon."""
    d = np.full(x.shape, np.inf)
    for a, b in zip(poly, np.roll(poly, -1, axis=0)):
        e = b - a
        t = np.clip(((x - a[0]) * e[0] + (y - a[1]) * e[1]) / (e @ e), 0.0, 1.0)
        d = np.minimum(d, np.hypot(x - a[0] - t * e[0], y - a[1] - t * e[1]))
    return d


def room_relocalization(seed, scans, n_beams, xy_step=0.5, yaw_step_deg=10):
    """Relocalization on the cfg-2 room: the scans and true poses of room_sequence's trajectory, the course obstacle
    map of room_map_observation, and a grid of candidate poses over the room's free interior that knows nothing of
    the trajectory.

    The candidates are the centres of the xy_step grid cells, aligned on the origin, whose centre lies inside the
    room at least 0.3 m from any wall, each at the yaws -pi + i * yaw_step_deg (i = 0 .. 360 / yaw_step_deg - 1),
    x-major, then y, then yaw.  With seed 9001 and the defaults that is 759 cells x 36 yaws = 27 324 candidates.

    Returns a dict: ranges float32 (scans, n_beams) (beam angles linspace(-pi, pi, n_beams)), poses float64
    (scans, 3) the true poses, obstacles_course (2, C), candidates float64 (H, 3), poly the room polygon (12, 2).
    """
    poly, r, poses, _ = _room_ranges(seed, scans, n_beams)
    lim = np.abs(poly).max()
    c = np.arange(-np.ceil(lim / xy_step), np.ceil(lim / xy_step) + 1) * xy_step
    gx, gy = np.meshgrid(c, c, indexing="ij")
    gx, gy = gx.ravel(), gy.ravel()
    keep = _polygon_inside(poly, gx, gy) & (_polygon_wall_distance(poly, gx, gy) >= 0.3)
    yaw_count = int(round(360.0 / yaw_step_deg))
    yaws = -np.pi + np.arange(yaw_count) * np.deg2rad(yaw_step_deg)
    xy = np.stack([gx[keep], gy[keep]], axis=1)
    cand = np.concatenate([np.repeat(xy, yaw_count, axis=0), np.tile(yaws, xy.shape[0])[:, None]], axis=1)
    return {"ranges": r.astype(np.float32), "poses": poses, "obstacles_course": _wall_cells(poly, 0.155, 129, 0.2),
            "candidates": np.ascontiguousarray(cand), "poly": poly}


# ------------------------------------------------------------------ cfg 3 / 5: grid streams

def grid_scan_ranges(seed, scans, n_beams, half_extent_m=80.0, step_m=0.1):
    """Raw form of the cfg 3 / cfg 5 streams: ranges float32 (scans, n_beams) and poses float64
    (scans, 3) = x, y, yaw -- what the node holds before laserToNumpy / u2T (slam_ekf.py:89)."""
    rng = _rng(seed)
    r = noisy(rng, clean_ranges(rng, scans, n_beams))
    turn = np.cumsum(rng.normal(0.0, 0.05, size=scans))
    th = rng.uniform(-np.pi, np.pi) + turn
    x = np.cumsum(step_m * np.cos(th)) + rng.uniform(-0.5, 0.5) * half_extent_m
    y = np.cumsum(step_m * np.sin(th)) + rng.uniform(-0.5, 0.5) * half_extent_m

    def reflect(v):
        span = 2.0 * half_extent_m
        v = np.mod(v + half_extent_m, 2.0 * span)
        v = np.where(v > span, 2.0 * span - v, v)
        return v - half_extent_m

    x = reflect(x)
    y = reflect(y)
    # positions and ranges are float32-representable so both input forms describe the same scans
    x = x.astype(np.float32).astype(np.float64)
    y = y.astype(np.float32).astype(np.float64)
    return r.astype(np.float32), np.stack([x, y, th], axis=1)


def grid_scans(seed, scans, n_beams, half_extent_m=80.0, step_m=0.1):
    """cfg 3 (seed 12001) / cfg 5 (seeds 5001..): world-frame beam endpoints from known poses.

    Poses follow a seeded random walk (heading noise, forward step `step_m`) reflected
    inside +-half_extent_m.  Returns ox, oy float32 (scans, n_beams) world-frame endpoints
    and cx, cy float32 (scans,) sensor positions.
    """
    r, poses = grid_scan_ranges(seed, scans, n_beams, half_extent_m, step_m)
    phi = beam_angles(n_beams)[None, :]
    x, y, th = poses[:, 0], poses[:, 1], poses[:, 2]
    ang = phi + th[:, None]
    ox = x[:, None] + r.astype(np.float64) * np.cos(ang)
    oy = y[:, None] + r.astype(np.float64) * np.sin(ang)
    return (ox.astype(np.float32), oy.astype(np.float32),
            x.astype(np.float32), y.astype(np.float32))
