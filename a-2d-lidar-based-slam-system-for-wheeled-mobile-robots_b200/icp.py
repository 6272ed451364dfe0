"""ICP scan matching on the GPU behind the reference's class API.

Drop-in for `from icp import ICP` (W9 / W12 course_agv_slam/scripts/icp.py): same method
names, argument order (TARGET first), shapes and float64 NumPy in/out.  All arithmetic runs
in the CUDA library (include/b2slam.h); nothing here computes a distance or a fit.
"""
import ctypes

import numpy as np

from b2slam import _lib


def _ros_param(name, default):
    """rospy.get_param when a ROS master is reachable, else the reference default."""
    try:
        import rospy  # noqa: F401  (absent outside ROS; the class must import without it)
        return rospy.get_param(name, default)
    except Exception:
        return default


class IcpTicket(object):
    """Handle of a stream submitted with ICP.submit_sequence / submit_scans."""

    def __init__(self, owner, ticket, T, iters, pairs):
        self._owner, self._ticket, self._T, self._iters, self._pairs = owner, ticket, T, iters, pairs

    def wait(self):
        """Block until the transforms are in host memory: (T (P,3,3) float64, iterations (P,) int32)."""
        _lib.check(self._owner._L.b2s_icp_wait(self._owner._h, self._ticket))
        P = self._pairs
        return self._T[:P].reshape(P, 3, 3), self._iters[:P]


class ICP(object):
    """[ICP]:10-36.  max_iter / dis_th / tolerance default to the reference's 30 / 5 / 0.001.

    `dis_th` is read but never used by the reference either ([ICP]:23).  Pass
    use_ros_params=True to look the values up on the ROS parameter server like the original.
    """

    def __init__(self, max_iter=30, dis_th=5, tolerance=0.001, use_ros_params=False, device=-1):
        if use_ros_params:
            max_iter = _ros_param('/icp/max_iter', max_iter)
            dis_th = _ros_param('/icp/dis_th', dis_th)
            tolerance = _ros_param('/icp/tolerance', tolerance)
        self.max_iter = int(max_iter)
        self.dis_th = dis_th
        self.tolerance = float(tolerance)
        self.isFirstScan = True
        self.src_pc = []
        self.tar_pc = []
        self.last_iterations = None
        self._L = _lib.lib()
        _lib.require_device()
        h = ctypes.c_void_p()
        _lib.check(self._L.b2s_icp_create(ctypes.byref(h), int(device)))
        self._h = h

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._L.b2s_icp_destroy(h)
            self._h = None

    # ------------------------------------------------------------------ reference methods

    def process(self, tar_pc, src_pc):
        """[ICP]:38-88.  tar_pc (3,M) / src_pc (3,N) (rows x, y, 1; only rows 0-1 are read).

        Returns the 3x3 float64 transform taking the source scan into the target frame.
        Inputs are not modified.
        """
        tar = np.ascontiguousarray(np.asarray(tar_pc, dtype=np.float64)[:2, :])
        src = np.ascontiguousarray(np.asarray(src_pc, dtype=np.float64)[:2, :])
        T, iters = self.process_batch(tar[None], src[None])
        self.last_iterations = int(iters[0])
        return T[0]

    def findNearest(self, src, tar):
        """[ICP]:90-114.  src (N,2), tar (M,2) -> (distances (N,), indices (N,) int)."""
        src = np.ascontiguousarray(src, dtype=np.float64).reshape(-1, 2)
        tar = np.ascontiguousarray(tar, dtype=np.float64).reshape(-1, 2)
        n, m = src.shape[0], tar.shape[0]
        dist = np.zeros(n)
        idx = np.zeros(n, dtype=np.int64)
        _lib.check(self._L.b2s_icp_find_nearest(self._h, _lib.ptr(src), n, _lib.ptr(tar), m,
                                                _lib.ptr(dist), _lib.ptr(idx)))
        return dist, idx

    def getTransform(self, src, tar):
        """[ICP]:149-179.  Row-matched src (N,2), tar (N,2) -> 3x3 T with tar ~= R src + t."""
        src = np.ascontiguousarray(src, dtype=np.float64).reshape(-1, 2)
        tar = np.ascontiguousarray(tar, dtype=np.float64).reshape(-1, 2)
        if src.shape != tar.shape:
            raise ValueError("getTransform needs row-matched clouds, got %s and %s"
                             % (src.shape, tar.shape))
        T = np.empty(9)
        _lib.check(self._L.b2s_icp_get_transform(self._h, _lib.ptr(src), _lib.ptr(tar),
                                                 src.shape[0], _lib.ptr(T)))
        return T.reshape(3, 3)

    def laserToNumpy(self, msg):
        """[ICP]:216-229 (no inf clamp in this copy of the reference)."""
        from b2slam import scan
        return scan.laser_to_points(msg.ranges, msg.angle_min, msg.angle_max)

    # ------------------------------------------------------------------ batched entry point

    def process_batch(self, tar, src, max_iter=None, tolerance=None):
        """ICP.process over P independent pairs in one launch.

        tar (P,2,M), src (P,2,N): x row / y row per pair, float64 (the reference dtype) or
        float32.  Returns (T (P,3,3) float64, iterations (P,) int32).
        """
        tar = np.asarray(tar)
        src = np.asarray(src)
        if tar.ndim != 3 or src.ndim != 3 or tar.shape[1] != 2 or src.shape[1] != 2 \
                or tar.shape[0] != src.shape[0]:
            raise ValueError("expected tar (P,2,M) and src (P,2,N), got %s and %s"
                             % (tar.shape, src.shape))
        f64 = not (tar.dtype == np.float32 and src.dtype == np.float32)
        dt = np.float64 if f64 else np.float32
        tar = np.ascontiguousarray(tar, dtype=dt)
        src = np.ascontiguousarray(src, dtype=dt)
        P, M, N = tar.shape[0], tar.shape[2], src.shape[2]
        T = np.empty((P, 9))
        iters = np.empty(P, dtype=np.int32)
        _lib.check(self._L.b2s_icp_process(
            self._h, _lib.ptr(tar), _lib.ptr(src), 1 if f64 else 0, P, N, M,
            self.max_iter if max_iter is None else int(max_iter),
            self.tolerance if tolerance is None else float(tolerance),
            _lib.ptr(T), _lib.ptr(iters)))
        return T.reshape(P, 3, 3), iters

    def process_sequence(self, scans, max_iter=None, tolerance=None):
        """LiDAR odometry over a scan stream, the loop of [LOC9]:159-168 / [SLAM]:109-113: pair k matches scan
        k + 1 (source) onto scan k (target), i.e. process_batch(scans[:-1], scans[1:]) bit for bit, but every scan
        crosses PCIe once instead of twice.

        scans (K,2,N) float64 or float32.  Returns (T (K-1,3,3) float64, iterations (K-1,) int32).
        """
        scans = np.asarray(scans)
        if scans.ndim != 3 or scans.shape[1] != 2:
            raise ValueError("expected scans (K,2,N), got %s" % (scans.shape,))
        f64 = scans.dtype != np.float32
        scans = np.ascontiguousarray(scans, dtype=np.float64 if f64 else np.float32)
        K, N = scans.shape[0], scans.shape[2]
        P = max(K - 1, 0)
        T = np.empty((P, 9))
        iters = np.empty(P, dtype=np.int32)
        if P > 0 and N == 0:
            raise ValueError("empty scans")
        if P > 0:
            _lib.check(self._L.b2s_icp_process_sequence(
                self._h, _lib.ptr(scans), 1 if f64 else 0, K, N,
                self.max_iter if max_iter is None else int(max_iter),
                self.tolerance if tolerance is None else float(tolerance),
                _lib.ptr(T), _lib.ptr(iters)))
        return T.reshape(P, 3, 3), iters

    # ------------------------------------------------------------------ streaming calls (two in flight)

    def _stream_out(self, pairs):
        """Page-locked result buffers of the next streamed call (two slots, re-allocated when the size grows)."""
        slots = getattr(self, "_stream_slots", None)
        if slots is None:
            slots = self._stream_slots = [None, None]
            self._stream_n = 0
            self._stream_keep = [None, None]
        k = self._stream_n % 2
        if slots[k] is None or slots[k][0].shape[0] < max(pairs, 1):
            slots[k] = (_lib.pinned_empty((max(pairs, 1), 9), np.float64), _lib.pinned_empty((max(pairs, 1),), np.int32))
        return k, slots[k]

    def submit_sequence(self, scans, max_iter=None, tolerance=None):
        """process_sequence without the wait (b2s_icp_submit_sequence): the uploads and solves are enqueued and an
        IcpTicket is returned at once; with two calls in flight the scans of the next stream cross PCIe while this one
        is being solved.  ticket.wait() -> (T (K-1,3,3), iterations (K-1,)), views of page-locked buffers that the
        second-next submit overwrites.  `scans` must stay untouched until then."""
        scans = np.asarray(scans)
        if scans.ndim != 3 or scans.shape[1] != 2 or scans.shape[2] < 1:
            raise ValueError("expected scans (K,2,N), got %s" % (scans.shape,))
        f64 = scans.dtype != np.float32
        scans = np.ascontiguousarray(scans, dtype=np.float64 if f64 else np.float32)
        K, N = scans.shape[0], scans.shape[2]
        P = max(K - 1, 0)
        k, (T, iters) = self._stream_out(P)
        t = ctypes.c_int(-1)
        _lib.check(self._L.b2s_icp_submit_sequence(
            self._h, _lib.ptr(scans), 1 if f64 else 0, K, N, self.max_iter if max_iter is None else int(max_iter),
            self.tolerance if tolerance is None else float(tolerance), _lib.ptr(T), _lib.ptr(iters), ctypes.byref(t)))
        self._stream_n += 1
        self._stream_keep[k] = scans
        return IcpTicket(self, t.value, T, iters, P)

    def submit_scans(self, ranges, angle_min, angle_max, clamp_inf_to=None, max_iter=None, tolerance=None):
        """process_scans (raw ranges, no pose chain) without the wait; see submit_sequence."""
        ranges = np.ascontiguousarray(ranges, dtype=np.float32)
        if ranges.ndim != 2 or ranges.shape[1] < 1:
            raise ValueError("expected ranges (K,N) with N >= 1, got %s" % (ranges.shape,))
        K, N = ranges.shape
        self._beam_table(angle_min, angle_max, N)
        P = max(K - 1, 0)
        k, (T, iters) = self._stream_out(P)
        t = ctypes.c_int(-1)
        _lib.check(self._L.b2s_icp_submit_scans(
            self._h, _lib.ptr(ranges), _lib.ptr(self._beam_cs), float(clamp_inf_to or 0.0), K, N,
            self.max_iter if max_iter is None else int(max_iter),
            self.tolerance if tolerance is None else float(tolerance), _lib.ptr(T), _lib.ptr(iters), ctypes.byref(t)))
        self._stream_n += 1
        self._stream_keep[k] = ranges
        return IcpTicket(self, t.value, T, iters, P)

    def odometry(self, scans, state=(0.0, 0.0, 0.0), max_iter=None, tolerance=None):
        """The LiDAR-odometry loop of localization.py:66-83 for a recorded stream: process_sequence(scans) followed
        by the pose chain `x += cos(th) T02 - sin(th) T12; y += sin(th) T02 + cos(th) T12; th += atan2(T10, T00)`
        ([ICP]:185-190), the chain as a parallel prefix on the device (scan.compose_odometry_gpu) without the
        transforms leaving it in between.

        Returns (trajectory (K,3) = x, y, yaw starting at `state`, T (K-1,3,3), iterations (K-1,)).
        """
        scans = np.asarray(scans)
        if scans.ndim != 3 or scans.shape[1] != 2 or scans.shape[0] < 1 or scans.shape[2] < 1:
            raise ValueError("expected scans (K,2,N) with K, N >= 1, got %s" % (scans.shape,))
        f64 = scans.dtype != np.float32
        scans = np.ascontiguousarray(scans, dtype=np.float64 if f64 else np.float32)
        K, N = scans.shape[0], scans.shape[2]
        traj = np.empty((K, 3))
        T = np.empty((K - 1, 9))
        iters = np.empty(K - 1, dtype=np.int32)
        _lib.check(self._L.b2s_icp_odometry(
            self._h, _lib.ptr(scans), 1 if f64 else 0, K, N,
            self.max_iter if max_iter is None else int(max_iter),
            self.tolerance if tolerance is None else float(tolerance),
            float(state[0]), float(state[1]), float(state[2]), _lib.ptr(traj),
            _lib.ptr(T) if K > 1 else None, _lib.ptr(iters) if K > 1 else None))
        return traj, T.reshape(K - 1, 3, 3), iters

    def _beam_table(self, angle_min, angle_max, N):
        from b2slam import scan
        key = (float(angle_min), float(angle_max), N)
        if getattr(self, "_beam_key", None) != key:
            self._beam_cs = scan.beam_table(angle_min, angle_max, N)
            self._beam_key = key
        return self._beam_cs

    # ------------------------------------------------------------------ map observation (W9 localization)

    def set_static_map(self, obstacle_xy):
        """The localization node's static map (self.obstacle): obstacle_xy (2, C) world coordinates of the occupied
        cell centres, as scan.virtual_scan takes them.  Uploaded once and kept on the device until replaced; C = 0
        clears it.  A NaN coordinate raises ValueError (the reference's int() raises on it) and clears the map."""
        obstacle_xy = np.asarray(obstacle_xy, dtype=np.float64)
        if obstacle_xy.ndim != 2 or obstacle_xy.shape[0] != 2:
            raise ValueError("expected obstacle_xy (2, C), got %s" % (obstacle_xy.shape,))
        ox = np.ascontiguousarray(obstacle_xy[0])
        oy = np.ascontiguousarray(obstacle_xy[1])
        C = ox.shape[0]
        _lib.check(self._L.b2s_icp_set_map(self._h, _lib.ptr(ox) if C else None, _lib.ptr(oy) if C else None, C))

    def map_observation(self, ranges, poses, angle_min, angle_max, angle_increment=None, clamp_inf_to=None,
                        far_range=100.0, max_iter=None, tolerance=None, return_virtual=False):
        """calc_map_observation ([LOC9]:152-157) for a recorded stream: for scan k the virtual scan of the static map
        (set_static_map) at poses[k] (laserEstimation, [LOC9]:128-150) is the target, laserToNumpy(ranges[k]) the
        source, T[k] = ICP.process(target, source).  Everything runs on the device: the same transforms as
        process_batch(stack(laser_to_points(virtual_k)[:2]), stack(laser_to_points(ranges_k, ...)[:2])), bit for bit.

        ranges (K,N) float32 (LaserScan.ranges), poses (K,3) = x, y, yaw.  The virtual scan bins with angle_increment
        (default (angle_max - angle_min) / (N - 1); pass the LaserScan's own field where it differs); both clouds
        take their beam angles from linspace(angle_min, angle_max, N) like laserToNumpy.  clamp_inf_to: the W12 inf
        clamp of the source.  Returns (T (K,3,3), iterations (K,)), and the virtual ranges (K,N) float64 with
        return_virtual=True.  A NaN pose raises ValueError like the reference's int().
        """
        ranges = np.ascontiguousarray(ranges, dtype=np.float32)
        if ranges.ndim != 2 or ranges.shape[1] < 1:
            raise ValueError("expected ranges (K,N) with N >= 1, got %s" % (ranges.shape,))
        K, N = ranges.shape
        poses = np.ascontiguousarray(poses, dtype=np.float64)
        if poses.shape != (K, 3):
            raise ValueError("expected poses (%d,3), got %s" % (K, poses.shape))
        if angle_increment is None:
            if N < 2:
                raise ValueError("a one-beam scan needs an explicit angle_increment")
            angle_increment = (float(angle_max) - float(angle_min)) / (N - 1)
        cs = self._beam_table(angle_min, angle_max, N)
        T = np.empty((K, 9))
        iters = np.empty(K, dtype=np.int32)
        virt = np.empty((K, N)) if return_virtual else None
        _lib.check(self._L.b2s_icp_map_observation(
            self._h, _lib.ptr(ranges), _lib.ptr(poses), _lib.ptr(cs), float(clamp_inf_to or 0.0), K, N,
            float(angle_min), float(angle_increment), float(far_range),
            self.max_iter if max_iter is None else int(max_iter),
            self.tolerance if tolerance is None else float(tolerance),
            _lib.ptr(T), _lib.ptr(iters), _lib.ptr(virt)))
        T = T.reshape(K, 3, 3)
        return (T, iters, virt) if return_virtual else (T, iters)

    def relocalize(self, ranges, candidates, angle_min, angle_max, angle_increment=None, clamp_inf_to=None,
                   far_range=100.0, max_iter=None, tolerance=None, return_T=False):
        """Relocalization in the static map (set_static_map) for a robot whose pose is unknown: at start-up, after the
        EKF has diverged, or where a recorded stream starts at an unknown place.  The map observation is run at every
        candidate pose and the best one is kept; the caller supplies the candidates (synth.room_relocalization shows
        one grid layout).

        ranges (K,N) float32, or (N,) for one scan; candidates (H,3) float64 x, y, yaw, shared by the K scans.
        Hypothesis (k, h) is map_observation(ranges[k:k+1], candidates[h:h+1], ...) bit for bit (T and iterations);
        the H virtual scans are built once per call.  score[k, h] is the reference's mean_error of the last iteration
        that ran ([ICP]:75-76): the mean matched distance before that iteration's move, unmatched (inf / NaN)
        distances counting 0.  best[k] is the h with the smallest score among the hypotheses whose score and T are
        finite, the lowest h on ties, or -1 when none is (then pose[k] is NaN).  pose[k] is the sensor pose in the map
        frame, candidates[best[k]] composed with T[k, best[k]] by the pose-chain step of [ICP]:185-190.

        Scans with +inf ranges need clamp_inf_to for meaningful scores: without it their inf points count as distance
        0 for every hypothesis.

        Returns (best (K,) int32, pose (K,3), score (K,H), iterations (K,H) int32), plus T (K,H,3,3) with
        return_T=True; for one (N,) scan the K axis is dropped.  Errors are those of map_observation: a NaN candidate
        raises ValueError like the reference's int(), before any device work.
        """
        ranges = np.asarray(ranges, dtype=np.float32)
        one = ranges.ndim == 1
        ranges = np.ascontiguousarray(ranges[None] if one else ranges)
        if ranges.ndim != 2 or ranges.shape[1] < 1:
            raise ValueError("expected ranges (K,N) or (N,) with N >= 1, got %s" % (ranges.shape,))
        K, N = ranges.shape
        candidates = np.ascontiguousarray(candidates, dtype=np.float64)
        if candidates.ndim != 2 or candidates.shape[1] != 3 or candidates.shape[0] < 1:
            raise ValueError("expected candidates (H,3) with H >= 1, got %s" % (candidates.shape,))
        H = candidates.shape[0]
        if angle_increment is None:
            if N < 2:
                raise ValueError("a one-beam scan needs an explicit angle_increment")
            angle_increment = (float(angle_max) - float(angle_min)) / (N - 1)
        cs = self._beam_table(angle_min, angle_max, N)
        best = np.empty(K, dtype=np.int32)
        pose = np.empty((K, 3))
        score = np.empty((K, H))
        iters = np.empty((K, H), dtype=np.int32)
        T = np.empty((K, H, 3, 3)) if return_T else None
        _lib.check(self._L.b2s_icp_relocalize(
            self._h, _lib.ptr(ranges), _lib.ptr(candidates), _lib.ptr(cs), float(clamp_inf_to or 0.0), K, H, N,
            float(angle_min), float(angle_increment), float(far_range),
            self.max_iter if max_iter is None else int(max_iter),
            self.tolerance if tolerance is None else float(tolerance),
            _lib.ptr(best), _lib.ptr(pose), _lib.ptr(score), _lib.ptr(iters), _lib.ptr(T)))
        out = (best, pose, score, iters) + ((T,) if return_T else ())
        return tuple(a[0] for a in out) if one else out

    def process_scans(self, ranges, angle_min, angle_max, clamp_inf_to=None, state=None, max_iter=None,
                      tolerance=None):
        """process_sequence / odometry fed with what the sensor delivers: ranges (K,N) float32 (LaserScan.ranges of
        K consecutive scans).  laserToNumpy -- [ICP]:216-229, or with clamp_inf_to (MAX_LASER_RANGE = 30) the W12
        form slam_ekf.py:115-123 -- runs inside the ICP kernel in float64, so 4 bytes per beam cross PCIe instead
        of the 16 of the reference's float64 points.  Same transforms as
        process_sequence(stack of laser_to_points(ranges[k])[:2]), bit for bit.

        Returns (T (K-1,3,3), iterations (K-1,)), or with state=(x, y, yaw) (trajectory (K,3), T, iterations).
        """
        ranges = np.ascontiguousarray(ranges, dtype=np.float32)
        if ranges.ndim != 2 or ranges.shape[1] < 1:
            raise ValueError("expected ranges (K,N) with N >= 1, got %s" % (ranges.shape,))
        K, N = ranges.shape
        self._beam_table(angle_min, angle_max, N)
        P = max(K - 1, 0)
        T = np.empty((P, 9))
        iters = np.empty(P, dtype=np.int32)
        traj = None
        st = None
        if state is not None:
            if K < 1:
                raise ValueError("a trajectory needs at least one scan")
            traj = np.empty((K, 3))
            st = np.array([float(state[0]), float(state[1]), float(state[2])])
        if K > 0:
            _lib.check(self._L.b2s_icp_process_scans(
                self._h, _lib.ptr(ranges), _lib.ptr(self._beam_cs), float(clamp_inf_to or 0.0), K, N,
                self.max_iter if max_iter is None else int(max_iter),
                self.tolerance if tolerance is None else float(tolerance),
                _lib.ptr(st) if st is not None else None, _lib.ptr(traj) if traj is not None else None,
                _lib.ptr(T), _lib.ptr(iters)))
        T = T.reshape(P, 3, 3)
        return (T, iters) if state is None else (traj, T, iters)
