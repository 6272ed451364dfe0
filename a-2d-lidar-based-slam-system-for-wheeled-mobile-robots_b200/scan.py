"""Host-side adjacent steps of the hot path (SURVEY.md section 8f): scan conversion, pose chain.

These are the tiny sequential pieces the ROS nodes run around ICP.process / Mapping.update;
they stay on the host in float64 exactly like the reference.
"""
import math

import numpy as np

MAX_LASER_RANGE = 30  # W12 slam_ekf.py:18


def laser_to_points(ranges, angle_min, angle_max, clamp_inf_to=None):
    """laserToNumpy: [ICP]:216-229 (clamp_inf_to=None) / W12 slam_ekf.py:115-123 (30 m clamp).

    Returns the (3, N) float64 homogeneous cloud [r cos a; r sin a; 1].
    """
    r = np.array(ranges, dtype=np.float64)
    if clamp_inf_to is not None:
        r[r == np.inf] = clamp_inf_to
    n = r.shape[0]
    a = np.linspace(angle_min, angle_max, n)
    pc = np.ones((3, n))
    pc[0, :] = np.cos(a) * r
    pc[1, :] = np.sin(a) * r
    return pc


def T2u(t):
    """W12 slam_ekf.py:125-128: 3x3 transform -> (dx, dy, dyaw) column."""
    return np.array([[t[0, 2], t[1, 2], math.atan2(t[1, 0], t[0, 0])]]).T


def u2T(u):
    """W12 slam_ekf.py:130-137: pose (x, y, yaw) -> 2x3 world transform."""
    x, y, w = (float(np.asarray(v).reshape(-1)[0]) for v in (u[0], u[1], u[2]))
    return np.array([[math.cos(w), -math.sin(w), x], [math.sin(w), math.cos(w), y]])


def compose_odometry(state, transforms):
    """Odometry chain, [ICP]:185-190 / W9 localization.py:79-83, over a (P,3,3) stack.

    Returns the (P+1, 3) trajectory starting at `state`.
    """
    out = np.empty((len(transforms) + 1, 3))
    x, y, th = (float(v) for v in state)
    out[0] = (x, y, th)
    for i, t in enumerate(transforms):
        dyaw = math.atan2(t[1, 0], t[0, 0])
        nx = x + math.cos(th) * t[0, 2] - math.sin(th) * t[1, 2]
        ny = y + math.sin(th) * t[0, 2] + math.cos(th) * t[1, 2]
        x, y, th = nx, ny, th + dyaw
        out[i + 1] = (x, y, th)
    return out


def beam_table(angle_min, angle_max, beams):
    """(beams, 2) float64 [cos a, sin a] of the beam angles, evaluated like laserToNumpy does
    (np.linspace, np.cos, np.sin: slam_ekf.py:121-122) -- the table b2s_grid_raycast_ranges consumes."""
    a = np.linspace(angle_min, angle_max, beams)
    return np.ascontiguousarray(np.stack([np.cos(a), np.sin(a)], axis=1))


def pose_table(poses):
    """(K, 4) float64 [x, y, cos yaw, sin yaw] from (K, 3) poses.  u2T (slam_ekf.py:130-137) uses
    math.cos / math.sin; np.cos / np.sin return the same doubles (checked in tests/test_host_logic.py)
    and are 12x faster on a 16k-scan batch."""
    poses = np.asarray(poses, dtype=np.float64).reshape(-1, 3)
    out = np.empty((poses.shape[0], 4))
    out[:, 0] = poses[:, 0]
    out[:, 1] = poses[:, 1]
    np.cos(poses[:, 2], out=out[:, 2])
    np.sin(poses[:, 2], out=out[:, 3])
    return out


def compose_odometry_gpu(state, transforms):
    """compose_odometry on the device (b2s_pose_chain): a parallel prefix instead of the sequential loop.

    Agrees with the loop to summation order.  Any summand of a row passes through at most m = 2 ceil(P / 1024) + 12
    float64 additions, so each entry is off the exact chain by at most gamma_m = m 2^-53 / (1 - m 2^-53) times the
    sum of its summands' magnitudes, plus the atan2 / cos / sin rounding carried through the yaw
    (tests/test_pose_chain_host.py: chain_bound).  A NaN or inf acts as in the loop: from a finite start, the rows
    before the first transform holding one stay finite, and every entry is finite, NaN, +inf or -inf as the loop's is."""
    from b2slam import _lib
    T = np.ascontiguousarray(transforms, dtype=np.float64).reshape(-1, 9)
    traj = np.empty((T.shape[0] + 1, 3))
    _lib.require_device()
    _lib.check(_lib.lib().b2s_pose_chain_host(_lib.ptr(T) if T.shape[0] else None, T.shape[0], float(state[0]),
                                              float(state[1]), float(state[2]), _lib.ptr(traj)))
    return traj


def virtual_scan(obstacle_xy, pose, angle_min, angle_increment, beams, far_range=100.0):
    """laserEstimation, W9 localization.py:128-150, on the device: obstacle_xy (2, C) world coordinates
    of the occupied map cells (self.obstacle), pose (x, y, yaw) -> ranges (beams,) float64."""
    from b2slam import _lib
    ox = np.ascontiguousarray(obstacle_xy[0], dtype=np.float64)
    oy = np.ascontiguousarray(obstacle_xy[1], dtype=np.float64)
    out = np.empty(int(beams))
    _lib.require_device()
    _lib.check(_lib.lib().b2s_virtual_scan_host(_lib.ptr(ox) if ox.size else None, _lib.ptr(oy) if oy.size else None,
                                                ox.shape[0], float(pose[0]), float(pose[1]), float(pose[2]),
                                                float(angle_min), float(angle_increment), int(beams),
                                                float(far_range), _lib.ptr(out)))
    return out
