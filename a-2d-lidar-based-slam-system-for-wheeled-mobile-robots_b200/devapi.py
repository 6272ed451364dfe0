"""Layer-1 C ABI on torch CUDA tensors: device pointers in, asynchronous on torch's current stream.

torch is plumbing here (device memory, streams, torch.distributed); every kernel is in
libb2slam.so.  Used by bench.py, the multi-GPU path (dist.py) and the parity tests.
"""
import torch

from b2slam import _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _chk(t, dtype, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise ValueError("%s must be a contiguous CUDA tensor of dtype %s" % (name, dtype))
    return t.data_ptr()


class _CudaView(object):
    """Minimal __cuda_array_interface__ carrier for memory torch did not allocate."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


_TYPESTR = {torch.int32: "<i4", torch.int8: "|i1", torch.float32: "<f4", torch.float64: "<f8", torch.uint8: "|u1"}


def tensor_from_ptr(ptr, shape, dtype, device=None):
    """A torch view of device memory owned by someone else (b2s_device_alloc, a peer's IPC mapping)."""
    dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
    return torch.as_tensor(_CudaView(ptr, shape, _TYPESTR[dtype]), device=dev)


def grid_scale(xw, yw, xyreso):
    """(cells_per_m, off_x, off_y) exactly as b2s_mapping_create derives them."""
    return 1.0 / xyreso, xw * xyreso / 2.0, yw * xyreso / 2.0


def new_planes(xw, yw, device=None):
    hit = torch.zeros((xw, yw), dtype=torch.int32, device=device or "cuda")
    miss = torch.zeros_like(hit)
    return hit, miss


def new_workspace(xw, yw, device=None):
    """Workspace for grid_raycast(..., workspace=): b2s_grid_workspace_bytes, initialised."""
    nbytes = _lib.lib().b2s_grid_workspace_bytes(int(xw), int(yw))
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=device or "cuda")
    _lib.check(_lib.lib().b2s_grid_workspace_init(ws.data_ptr(), int(xw), int(yw), _stream()))
    return ws


def grid_raycast(hit, miss, cells_per_m, off_x, off_y, ox, oy, cx, cy, counters=None, workspace=None):
    """b2s_grid_raycast_ws[_f64]: hit/miss int32 (xw,yw); ox, oy (K,N); cx, cy (K,), all float32 or all float64
    (float64 is what the reference's Mapping.update evaluates the cell transform on)."""
    xw, yw = hit.shape
    K, N = ox.shape
    dt = ox.dtype
    if dt not in (torch.float32, torch.float64):
        raise ValueError("ox must be float32 or float64")
    fn = _lib.lib().b2s_grid_raycast_ws if dt == torch.float32 else _lib.lib().b2s_grid_raycast_ws_f64
    rc = fn(
        _chk(hit, torch.int32, "hit"), _chk(miss, torch.int32, "miss"), xw, yw,
        float(cells_per_m), float(off_x), float(off_y),
        _chk(ox, dt, "ox"), _chk(oy, dt, "oy"),
        _chk(cx, dt, "cx"), _chk(cy, dt, "cy"), K, N,
        None if counters is None else _chk(counters, torch.int32, "counters"),
        None if workspace is None else _chk(workspace, torch.int32, "workspace"), _stream())
    _lib.check(rc)


def grid_raycast_ranges(hit, miss, cells_per_m, off_x, off_y, ranges, pose4, beam_cs, clamp_inf_to=30.0,
                        counters=None, workspace=None):
    """b2s_grid_raycast_ranges: ranges float32 (K,N), pose4 float64 (K,4), beam_cs float64 (N,2)."""
    xw, yw = hit.shape
    K, N = ranges.shape
    if workspace is None:
        raise ValueError("the fused-ingestion kernel needs a workspace (new_workspace)")
    rc = _lib.lib().b2s_grid_raycast_ranges(
        _chk(hit, torch.int32, "hit"), _chk(miss, torch.int32, "miss"), xw, yw,
        float(cells_per_m), float(off_x), float(off_y), _chk(ranges, torch.float32, "ranges"),
        _chk(pose4, torch.float64, "pose4"), _chk(beam_cs, torch.float64, "beam_cs"),
        float(clamp_inf_to or 0.0), K, N,
        None if counters is None else _chk(counters, torch.int32, "counters"),
        _chk(workspace, torch.int32, "workspace"), _stream())
    _lib.check(rc)


def grid_finalize(hit, miss, w_hit=20.0, w_miss=0.01, thresh=10.0, datamap=None, pmap=None):
    xw, yw = hit.shape
    rc = _lib.lib().b2s_grid_finalize(
        _chk(hit, torch.int32, "hit"), _chk(miss, torch.int32, "miss"), xw, yw, float(w_hit),
        float(w_miss), float(thresh),
        None if datamap is None else _chk(datamap, torch.float32, "datamap"),
        None if pmap is None else _chk(pmap, torch.int8, "pmap"), _stream())
    _lib.check(rc)


def grid_pack_ros(pmap, out=None):
    xw, yw = pmap.shape
    if out is None:
        out = torch.empty(xw * yw, dtype=torch.int8, device=pmap.device)
    _lib.check(_lib.lib().b2s_grid_pack_ros(_chk(pmap, torch.int8, "pmap"), xw, yw,
                                            _chk(out, torch.int8, "out"), _stream()))
    return out


def icp_batch(tar, src, max_iter=30, tol=1e-3, T_out=None, iters_out=None):
    """b2s_icp_batch_f32/f64: tar (P,2,M), src (P,2,N) float32 or float64 CUDA tensors."""
    P, _, M = tar.shape
    N = src.shape[2]
    if T_out is None:
        T_out = torch.empty((P, 3, 3), dtype=torch.float64, device=tar.device)
    if iters_out is None:
        iters_out = torch.empty(P, dtype=torch.int32, device=tar.device)
    fn = _lib.lib().b2s_icp_batch_f64 if tar.dtype == torch.float64 else _lib.lib().b2s_icp_batch_f32
    rc = fn(_chk(tar, tar.dtype, "tar"), _chk(src, tar.dtype, "src"), P, N, M, int(max_iter),
            float(tol), _chk(T_out, torch.float64, "T_out"), _chk(iters_out, torch.int32, "iters"),
            _stream())
    _lib.check(rc)
    return T_out, iters_out


def icp_batch_err(tar, src, max_iter=30, tol=1e-3, T_out=None, iters_out=None, err_out=None):
    """b2s_icp_batch_f64_err: icp_batch on float64 tar (P,2,M), src (P,2,N) that also returns each pair's mean_error
    of its last iteration ([ICP]:75-76) in err_out (P,) float64.  Returns (T_out, iters_out, err_out)."""
    P, _, M = tar.shape
    N = src.shape[2]
    if T_out is None:
        T_out = torch.empty((P, 3, 3), dtype=torch.float64, device=tar.device)
    if iters_out is None:
        iters_out = torch.empty(P, dtype=torch.int32, device=tar.device)
    if err_out is None:
        err_out = torch.empty(P, dtype=torch.float64, device=tar.device)
    rc = _lib.lib().b2s_icp_batch_f64_err(
        _chk(tar, torch.float64, "tar"), _chk(src, torch.float64, "src"), P, N, M, int(max_iter), float(tol),
        _chk(T_out, torch.float64, "T_out"), _chk(iters_out, torch.int32, "iters"), _chk(err_out, torch.float64, "err"),
        _stream())
    _lib.check(rc)
    return T_out, iters_out, err_out


def relocalize_select(score, T, candidates, best_out=None, pose_out=None):
    """b2s_relocalize_select: score (K,H) float64, T (K,H,3,3) float64, candidates (H,3) float64 CUDA tensors ->
    (best (K,) int32, pose (K,3) float64): per scan the lowest-index smallest score among the hypotheses whose score
    and T are finite (-1 and a NaN pose when none is), and candidates[best] composed with T[best] ([ICP]:185-190)."""
    K, H = score.shape
    for t, shape, name in ((T, (K, H, 3, 3), "T"), (candidates, (H, 3), "candidates")):
        if tuple(t.shape) != shape:
            raise ValueError("%s must have shape %s, got %s" % (name, shape, tuple(t.shape)))
    if best_out is None:
        best_out = torch.empty(K, dtype=torch.int32, device=score.device)
    if pose_out is None:
        pose_out = torch.empty((K, 3), dtype=torch.float64, device=score.device)
    rc = _lib.lib().b2s_relocalize_select(
        _chk(score, torch.float64, "score"), _chk(T, torch.float64, "T"), _chk(candidates, torch.float64, "candidates"),
        K, H, _chk(best_out, torch.int32, "best_out"), _chk(pose_out, torch.float64, "pose_out"), _stream())
    _lib.check(rc)
    return best_out, pose_out


def virtual_scan_batch(obs_x, obs_y, poses, angle_min, angle_increment, beams, far_range=100.0, beam_cs=None,
                       ranges=None, tar_xy=None):
    """b2s_virtual_scan_batch: laserEstimation for K poses at once.  obs_x, obs_y float64 (C,) obstacle cell centres,
    poses float64 (K,3) = x, y, yaw.  ranges (K,beams) float64 receives what scan.virtual_scan gives per pose;
    tar_xy (K,2,beams) float64 (needs beam_cs float64 (beams,2), scan.beam_table) receives their laserToNumpy points,
    the target layout of icp_batch.  Without either output, ranges is allocated.  Returns (ranges, tar_xy)."""
    K, C, beams = poses.shape[0], obs_x.shape[0], int(beams)
    if ranges is None and tar_xy is None:
        ranges = torch.empty((K, beams), dtype=torch.float64, device=poses.device)
    for t, shape, name in ((poses, (K, 3), "poses"), (obs_y, (C,), "obs_y"), (ranges, (K, beams), "ranges"),
                           (tar_xy, (K, 2, beams), "tar_xy"), (beam_cs, (beams, 2), "beam_cs")):
        if t is not None and tuple(t.shape) != shape:
            raise ValueError("%s must have shape %s, got %s" % (name, shape, tuple(t.shape)))
    rc = _lib.lib().b2s_virtual_scan_batch(
        _chk(obs_x, torch.float64, "obs_x"), _chk(obs_y, torch.float64, "obs_y"), C,
        _chk(poses, torch.float64, "poses"), K, float(angle_min), float(angle_increment), beams, float(far_range),
        None if beam_cs is None else _chk(beam_cs, torch.float64, "beam_cs"),
        None if ranges is None else _chk(ranges, torch.float64, "ranges"),
        None if tar_xy is None else _chk(tar_xy, torch.float64, "tar_xy"), _stream())
    _lib.check(rc)
    return ranges, tar_xy
