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


def relocalize_select(score, T, candidates, best_out=None, pose_out=None, kept=None):
    """b2s_relocalize_select: score (K,H) float64, T (K,H,3,3) float64, candidates (H,3) float64 CUDA tensors ->
    (best (K,) int32, pose (K,3) float64): per scan the lowest-index smallest score among the hypotheses whose score
    and T are finite (-1 and a NaN pose when none is), and candidates[best] composed with T[best] ([ICP]:185-190).

    With kept (K,M) int32 (relocalize_keep's survivors, ascending per row), b2s_relocalize_select_kept: score (K,M)
    and T (K,M,3,3) belong to candidates[kept[k, j]], and best is the original candidate index.  Every kept entry
    must lie in [0, C) for candidates (C,3): like the other device-layer calls this one stays asynchronous, so the
    entries are not checked here (relocalize_keep's output always satisfies it)."""
    K, H = score.shape
    want = ((T, (K, H, 3, 3), "T"),) + (((candidates, (H, 3), "candidates"),) if kept is None else
                                        ((kept, (K, H), "kept"),))
    for t, shape, name in want:
        if tuple(t.shape) != shape:
            raise ValueError("%s must have shape %s, got %s" % (name, shape, tuple(t.shape)))
    if candidates.dim() != 2 or candidates.shape[1] != 3:
        raise ValueError("candidates must have shape (C, 3), got %s" % (tuple(candidates.shape),))
    if best_out is None:
        best_out = torch.empty(K, dtype=torch.int32, device=score.device)
    if pose_out is None:
        pose_out = torch.empty((K, 3), dtype=torch.float64, device=score.device)
    common = (_chk(score, torch.float64, "score"), _chk(T, torch.float64, "T"),
              _chk(candidates, torch.float64, "candidates"))
    outs = (_chk(best_out, torch.int32, "best_out"), _chk(pose_out, torch.float64, "pose_out"), _stream())
    if kept is None:
        rc = _lib.lib().b2s_relocalize_select(*common, K, H, *outs)
    else:
        rc = _lib.lib().b2s_relocalize_select_kept(*common, _chk(kept, torch.int32, "kept"), K, H, *outs)
    _lib.check(rc)
    return best_out, pose_out


def relocalize_keep(score, T, keep, kept_out=None, keys=None):
    """b2s_relocalize_keep: score (K,H) float64 and T (K,H,3,3) float64 CUDA tensors (coarse solves) -> kept (K,M)
    int32, M = min(keep, H): per scan, in ascending h, the first M hypotheses of the order (score, h) over those whose
    score and T are finite (-0 == +0), followed by every other hypothesis by h.  keys: (K*H,) int64 scratch."""
    K, H = score.shape
    if tuple(T.shape) != (K, H, 3, 3):
        raise ValueError("T must have shape %s, got %s" % ((K, H, 3, 3), tuple(T.shape)))
    M = max(0, min(int(keep), H))
    if kept_out is None:
        kept_out = torch.empty((K, M), dtype=torch.int32, device=score.device)
    if keys is None:
        keys = torch.empty(K * H, dtype=torch.int64, device=score.device)
    if tuple(kept_out.shape) != (K, M) or keys.numel() < K * H:
        raise ValueError("kept_out must be (%d, %d) and keys hold %d words" % (K, M, K * H))
    rc = _lib.lib().b2s_relocalize_keep(
        _chk(score, torch.float64, "score"), _chk(T, torch.float64, "T"), K, H, max(0, min(int(keep), 0x7fffffff)),
        _chk(keys, torch.int64, "keys"), _chk(kept_out, torch.int32, "kept_out"), _stream())
    _lib.check(rc)
    return kept_out


def track_step(T, score, prior, pose, joint, finite, stage, odometry=None, next_prior=None):
    """b2s_track_step: one stage of pose tracking after that stage's solves.  T (H,3,3) and score (H,) float64 (icp_batch_err
    at the H priors), prior (H,3) float64; pose (H,3) float64 receives prior (+) T ([ICP]:185-190), joint (H,) float64
    the running score sum (started from 0.0 at stage 0) and finite (H,) int32 the running finiteness of score, T and
    pose.  With odometry (3,3) float64, next_prior (H,3) receives pose (+) odometry; both are None at the last stage."""
    H = score.shape[0]
    for t, shape, name in ((T, (H, 3, 3), "T"), (prior, (H, 3), "prior"), (pose, (H, 3), "pose"), (joint, (H,), "joint"),
                           (finite, (H,), "finite"), (odometry, (3, 3), "odometry"), (next_prior, (H, 3), "next_prior")):
        if t is not None and tuple(t.shape) != shape:
            raise ValueError("%s must have shape %s, got %s" % (name, shape, tuple(t.shape)))
    if (odometry is None) != (next_prior is None):
        raise ValueError("odometry and next_prior go together")
    rc = _lib.lib().b2s_track_step(
        _chk(T, torch.float64, "T"), _chk(score, torch.float64, "score"),
        None if odometry is None else _chk(odometry, torch.float64, "odometry"), H, int(stage),
        _chk(prior, torch.float64, "prior"), _chk(pose, torch.float64, "pose"),
        None if next_prior is None else _chk(next_prior, torch.float64, "next_prior"), _chk(joint, torch.float64, "joint"),
        _chk(finite, torch.int32, "finite"), _stream())
    _lib.check(rc)
    return pose


def track_select(joint, finite, best_out=None):
    """b2s_track_select: joint (H,) float64 and finite (H,) int32 CUDA tensors -> best (1,) int32, the lowest-index
    smallest joint score among the finite tracks, or -1."""
    H = joint.shape[0]
    if tuple(finite.shape) != (H,):
        raise ValueError("finite must have shape %s, got %s" % ((H,), tuple(finite.shape)))
    if best_out is None:
        best_out = torch.empty(1, dtype=torch.int32, device=joint.device)
    rc = _lib.lib().b2s_track_select(_chk(joint, torch.float64, "joint"), _chk(finite, torch.int32, "finite"), H,
                                     _chk(best_out, torch.int32, "best_out"), _stream())
    _lib.check(rc)
    return best_out


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
