"""ctypes front end for oracle/oracle.c (compiled CPU oracle).  TEST INFRASTRUCTURE ONLY."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liboracle.so")
_lib = None


def build(force=False):
    src = os.path.join(_HERE, "oracle.c")
    if force or not os.path.isfile(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(_SO):
            build()
        L = ctypes.CDLL(_SO)
        i32, i64, dbl, vp = ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p
        L.orc_nearest.argtypes = [vp, i32, vp, i32, vp, vp]
        L.orc_nearest.restype = None
        L.orc_rigid_fit.argtypes = [vp, vp, vp, i32, vp]
        L.orc_rigid_fit.restype = None
        L.orc_icp_batch.argtypes = [vp, vp, i32, i32, i32, i32, dbl, vp, vp]
        L.orc_icp_batch.restype = i32
        L.orc_icp_batch_err.argtypes = [vp, vp, i32, i32, i32, i32, dbl, vp, vp, vp]
        L.orc_icp_batch_err.restype = i32
        L.orc_bresenham.argtypes = [i64, i64, i64, i64, vp, i64]
        L.orc_bresenham.restype = i64
        L.orc_grid_raycast.argtypes = [vp, vp, i32, i32, dbl, dbl, dbl, vp, vp, vp, vp, i32, i32]
        L.orc_grid_raycast.restype = i64
        L.orc_grid_raycast_f64.argtypes = [vp, vp, i32, i32, dbl, dbl, dbl, vp, vp, vp, vp, i32, i32]
        L.orc_grid_raycast_f64.restype = i64
        L.orc_grid_raycast_ranges.argtypes = [vp, vp, i32, i32, dbl, dbl, dbl, vp, vp, vp, dbl, i32, i32]
        L.orc_grid_raycast_ranges.restype = i64
        L.orc_grid_finalize.argtypes = [vp, vp, i64, dbl, dbl, dbl, vp, vp]
        L.orc_grid_finalize.restype = None
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def nearest(src, tar):
    src = np.ascontiguousarray(src, dtype=np.float64)
    tar = np.ascontiguousarray(tar, dtype=np.float64)
    dist = np.empty(src.shape[0])
    idx = np.empty(src.shape[0], dtype=np.int32)
    lib().orc_nearest(_p(src), src.shape[0], _p(tar), tar.shape[0], _p(dist), _p(idx))
    return dist, idx


def rigid_fit(src, tar):
    src = np.ascontiguousarray(src, dtype=np.float64)
    tar = np.ascontiguousarray(tar, dtype=np.float64)
    T = np.empty(9)
    lib().orc_rigid_fit(_p(src), _p(tar), None, src.shape[0], _p(T))
    return T.reshape(3, 3)


def icp_batch(tar, src, max_iter=30, tol=1e-3, return_err=False):
    """tar (P,2,M), src (P,2,N) (x/y rows, any float dtype) -> (T (P,3,3), iters (P,)), and with return_err=True
    err (P,) as well: each pair's mean_error of its last iteration ([ICP]:75), 0 when none ran."""
    tar = np.ascontiguousarray(np.transpose(np.asarray(tar, dtype=np.float64), (0, 2, 1)))
    src = np.ascontiguousarray(np.transpose(np.asarray(src, dtype=np.float64), (0, 2, 1)))
    P, N, M = src.shape[0], src.shape[1], tar.shape[1]
    T = np.empty((P, 9))
    iters = np.empty(P, dtype=np.int32)
    if return_err:
        err = np.empty(P)
        rc = lib().orc_icp_batch_err(_p(tar), _p(src), P, N, M, int(max_iter), float(tol), _p(T), _p(iters), _p(err))
    else:
        rc = lib().orc_icp_batch(_p(tar), _p(src), P, N, M, int(max_iter), float(tol), _p(T),
                                 _p(iters))
    if rc != 0:
        raise ValueError("orc_icp_batch: bad arguments")
    return (T.reshape(P, 3, 3), iters, err) if return_err else (T.reshape(P, 3, 3), iters)


def bresenham(start, end):
    cap = max(abs(int(end[0]) - int(start[0])), abs(int(end[1]) - int(start[1]))) + 1
    out = np.empty((cap, 2), dtype=np.int32)
    n = lib().orc_bresenham(int(start[0]), int(start[1]), int(end[0]), int(end[1]), _p(out), cap)
    return [tuple(int(v) for v in row) for row in out[:n]]


def grid_raycast(hit, miss, cells_per_m, off_x, off_y, ox, oy, cx, cy):
    """In-place integer update of hit/miss int32 (xw,yw); ox, oy (K,N); cx, cy (K,). Returns visits.
    float32 arrays go through the float32 entry (upcast exactly); anything else is consumed as float64,
    like the reference consumes it ([MAP]:33-36)."""
    assert hit.dtype == np.int32 and miss.dtype == np.int32
    assert hit.flags.c_contiguous and miss.flags.c_contiguous
    if not all(np.asarray(a).dtype == np.float32 for a in (ox, oy, cx, cy)):
        ox = np.ascontiguousarray(np.atleast_2d(ox), dtype=np.float64)
        oy = np.ascontiguousarray(np.atleast_2d(oy), dtype=np.float64)
        cx = np.ascontiguousarray(np.atleast_1d(cx), dtype=np.float64)
        cy = np.ascontiguousarray(np.atleast_1d(cy), dtype=np.float64)
        K, N = ox.shape
        v = lib().orc_grid_raycast_f64(_p(hit), _p(miss), hit.shape[0], hit.shape[1], float(cells_per_m),
                                       float(off_x), float(off_y), _p(ox), _p(oy), _p(cx), _p(cy), K, N)
        if v < 0:
            raise ValueError("non-finite coordinate")
        return int(v)
    ox = np.ascontiguousarray(np.atleast_2d(ox), dtype=np.float32)
    oy = np.ascontiguousarray(np.atleast_2d(oy), dtype=np.float32)
    cx = np.ascontiguousarray(np.atleast_1d(cx), dtype=np.float32)
    cy = np.ascontiguousarray(np.atleast_1d(cy), dtype=np.float32)
    K, N = ox.shape
    v = lib().orc_grid_raycast(_p(hit), _p(miss), hit.shape[0], hit.shape[1], float(cells_per_m),
                               float(off_x), float(off_y), _p(ox), _p(oy), _p(cx), _p(cy), K, N)
    if v < 0:
        raise ValueError("non-finite coordinate")
    return int(v)


def grid_raycast_ranges(hit, miss, cells_per_m, off_x, off_y, ranges, pose4, beam_cs, clamp=30.0):
    """Raw scans: ranges (K,N) float32, pose4 (K,4) = x, y, cos yaw, sin yaw, beam_cs (N,2).  Returns visits."""
    ranges = np.ascontiguousarray(np.atleast_2d(ranges), dtype=np.float32)
    pose4 = np.ascontiguousarray(np.atleast_2d(pose4), dtype=np.float64)
    beam_cs = np.ascontiguousarray(beam_cs, dtype=np.float64)
    K, N = ranges.shape
    v = lib().orc_grid_raycast_ranges(_p(hit), _p(miss), hit.shape[0], hit.shape[1], float(cells_per_m),
                                      float(off_x), float(off_y), _p(ranges), _p(pose4), _p(beam_cs),
                                      float(clamp or 0.0), K, N)
    if v < 0:
        raise ValueError("non-finite coordinate")
    return int(v)


def grid_finalize(hit, miss, w_hit=20.0, w_miss=0.01, thresh=10.0):
    score = np.empty(hit.shape)
    pmap = np.empty(hit.shape, dtype=np.int8)
    lib().orc_grid_finalize(_p(hit), _p(miss), hit.size, w_hit, w_miss, thresh, _p(score), _p(pmap))
    return score, pmap
