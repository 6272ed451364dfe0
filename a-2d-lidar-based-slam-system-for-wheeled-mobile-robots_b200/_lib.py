"""ctypes binding of libb2slam.so (include/b2slam.h).  No torch types cross this boundary.

There is deliberately no CPU fallback: if the CUDA library is missing, or a compute call
finds no device, the caller gets an exception, never a silently slower answer.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2slam.so")

OK = 0
ERR_INVALID_ARG = -1
ERR_NONFINITE = -2
ERR_CUDA = -3
ERR_TOO_LONG = -4
ERR_NCCL = -5
ERR_NOMEM = -6
CNT_WORDS = 4

_vp, _i32, _i64, _dbl, _sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double,
                              ctypes.c_size_t)
_pp = ctypes.POINTER(ctypes.c_void_p)

# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "b2s_version": (_i32, []),
    "b2s_status_string": (ctypes.c_char_p, [_i32]),
    "b2s_last_error": (ctypes.c_char_p, []),
    "b2s_device_count": (_i32, [ctypes.POINTER(_i32)]),
    "b2s_tune": (_i32, [ctypes.c_char_p, _i32]),
    "b2s_measure_fp64_peak": (_i32, [ctypes.POINTER(_dbl)]),
    "b2s_icp_batch_f32": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _dbl, _vp, _vp, _vp]),
    "b2s_icp_batch_f64": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _dbl, _vp, _vp, _vp]),
    "b2s_icp_batch_f64_err": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _dbl, _vp, _vp, _vp, _vp]),
    "b2s_icp_dispatch": (_i32, [_i32, _i32, _i32, _i32, ctypes.POINTER(_i32), ctypes.POINTER(_i32), ctypes.POINTER(_i32)]),
    "b2s_icp_batch_ranges": (_i32, [_vp, _vp, _vp, _dbl, _i32, _i32, _i32, _dbl, _vp, _vp, _vp]),
    "b2s_nearest_f64": (_i32, [_vp, _i32, _vp, _i32, _vp, _vp, _vp]),
    "b2s_rigid_fit_f64": (_i32, [_vp, _vp, _i32, _vp, _vp]),
    "b2s_grid_raycast": (_i32, [_vp, _vp, _i32, _i32, _dbl, _dbl, _dbl, _vp, _vp, _vp, _vp,
                                _i32, _i32, _vp, _vp]),
    "b2s_grid_raycast_f64": (_i32, [_vp, _vp, _i32, _i32, _dbl, _dbl, _dbl, _vp, _vp, _vp, _vp,
                                    _i32, _i32, _vp, _vp]),
    "b2s_grid_workspace_bytes": (_sz, [_i32, _i32]),
    "b2s_grid_workspace_init": (_i32, [_vp, _i32, _i32, _vp]),
    "b2s_grid_raycast_ws": (_i32, [_vp, _vp, _i32, _i32, _dbl, _dbl, _dbl, _vp, _vp, _vp, _vp,
                                   _i32, _i32, _vp, _vp, _vp]),
    "b2s_grid_raycast_ws_f64": (_i32, [_vp, _vp, _i32, _i32, _dbl, _dbl, _dbl, _vp, _vp, _vp, _vp,
                                       _i32, _i32, _vp, _vp, _vp]),
    "b2s_grid_raycast_ranges": (_i32, [_vp, _vp, _i32, _i32, _dbl, _dbl, _dbl, _vp, _vp, _vp, _dbl,
                                       _i32, _i32, _vp, _vp, _vp]),
    "b2s_grid_validate": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "b2s_grid_validate_f64": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "b2s_grid_finalize": (_i32, [_vp, _vp, _i32, _i32, _dbl, _dbl, _dbl, _vp, _vp, _vp]),
    "b2s_grid_pack_ros": (_i32, [_vp, _i32, _i32, _vp, _vp]),
    "b2s_bresenham_paths": (_i32, [_vp, _i32, _vp, _vp, _vp]),
    "b2s_pose_chain": (_i32, [_vp, _i32, _dbl, _dbl, _dbl, _vp, _vp]),
    "b2s_pose_chain_host": (_i32, [_vp, _i32, _dbl, _dbl, _dbl, _vp]),
    "b2s_virtual_scan": (_i32, [_vp, _vp, _i32, _dbl, _dbl, _dbl, _dbl, _dbl, _i32, _dbl, _vp, _vp]),
    "b2s_virtual_scan_host": (_i32, [_vp, _vp, _i32, _dbl, _dbl, _dbl, _dbl, _dbl, _i32, _dbl, _vp]),
    "b2s_virtual_scan_batch": (_i32, [_vp, _vp, _i32, _vp, _i32, _dbl, _dbl, _i32, _dbl, _vp, _vp, _vp, _vp]),
    "b2s_relocalize_select": (_i32, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "b2s_relocalize_keep": (_i32, [_vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "b2s_relocalize_select_kept": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "b2s_grid_allreduce": (_i32, [_vp, _vp, _sz, _vp, _vp]),
    "b2s_grid_merge_p2p": (_i32, [_vp, _vp, _vp, _i32, _sz, _sz, _vp, _vp, _dbl, _dbl, _dbl, _vp]),
    "b2s_grid_merge_p2p_tiles": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _dbl, _dbl,
                                        _dbl, _vp]),
    "b2s_p2p_flag_bytes": (_sz, [_i32]),
    "b2s_p2p_dirty_stride": (_sz, [_i32, _i32]),
    "b2s_p2p_publish": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, ctypes.c_uint32, _vp]),
    "b2s_grid_merge_p2p_tiles_sync": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, ctypes.c_uint32, _i32, _i32, _i32, _i32,
                                             _vp, _vp, _dbl, _dbl, _dbl, _vp]),
    "b2s_p2p_wait_done": (_i32, [_vp, _i32, ctypes.c_uint32, _vp]),
    "b2s_p2p_status": (_i32, [_vp, _i32, ctypes.POINTER(_i32), ctypes.POINTER(_i64), _vp]),
    "b2s_grid_workspace_dirty": (_vp, [_vp]),
    "b2s_grid_tile_count": (_i32, [_i32, _i32, ctypes.POINTER(_i32), ctypes.POINTER(_i32)]),
    "b2s_grid_clear_dirty": (_i32, [_vp, _vp, _i32, _i32, _vp, _vp]),
    "b2s_device_alloc": (_i32, [_pp, _sz]),
    "b2s_device_free": (_i32, [_vp]),
    "b2s_ipc_export": (_i32, [_vp, _vp]),
    "b2s_ipc_open": (_i32, [_vp, _pp]),
    "b2s_ipc_close": (_i32, [_vp]),
    "b2s_nccl_unique_id": (_i32, [_vp]),
    "b2s_nccl_comm_init": (_i32, [_pp, _i32, _i32, _vp]),
    "b2s_nccl_comm_destroy": (_i32, [_vp]),
    "b2s_host_alloc": (_i32, [_pp, _sz]),
    "b2s_host_free": (_i32, [_vp]),
    "b2s_icp_create": (_i32, [_pp, _i32]),
    "b2s_icp_destroy": (_i32, [_vp]),
    "b2s_icp_process": (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _dbl, _vp, _vp]),
    "b2s_icp_process_sequence": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _dbl, _vp, _vp]),
    "b2s_icp_odometry": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _dbl, _dbl, _dbl, _dbl, _vp, _vp, _vp]),
    "b2s_icp_process_scans": (_i32, [_vp, _vp, _vp, _dbl, _i32, _i32, _i32, _dbl, _vp, _vp, _vp, _vp]),
    "b2s_icp_submit_sequence": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _dbl, _vp, _vp, ctypes.POINTER(_i32)]),
    "b2s_icp_submit_scans": (_i32, [_vp, _vp, _vp, _dbl, _i32, _i32, _i32, _dbl, _vp, _vp, ctypes.POINTER(_i32)]),
    "b2s_icp_wait": (_i32, [_vp, _i32]),
    "b2s_icp_set_map": (_i32, [_vp, _vp, _vp, _i32]),
    "b2s_icp_map_observation": (_i32, [_vp, _vp, _vp, _vp, _dbl, _i32, _i32, _dbl, _dbl, _dbl, _i32, _dbl, _vp, _vp,
                                       _vp]),
    "b2s_icp_relocalize": (_i32, [_vp, _vp, _vp, _vp, _dbl, _i32, _i32, _i32, _dbl, _dbl, _dbl, _i32, _dbl, _vp, _vp,
                                  _vp, _vp, _vp]),
    "b2s_icp_relocalize_keep": (_i32, [_vp, _vp, _vp, _vp, _dbl, _i32, _i32, _i32, _dbl, _dbl, _dbl, _i32, _dbl, _i32,
                                       _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2s_icp_find_nearest": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _vp]),
    "b2s_icp_get_transform": (_i32, [_vp, _vp, _vp, _i32, _vp]),
    "b2s_mapping_create": (_i32, [_pp, _i32, _i32, _dbl, _dbl, _dbl, _dbl, _i32]),
    "b2s_mapping_destroy": (_i32, [_vp]),
    "b2s_mapping_reset": (_i32, [_vp]),
    "b2s_mapping_update": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "b2s_mapping_update_f64": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "b2s_mapping_update_incremental_f64": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i32,
                                                  ctypes.POINTER(_i32)]),
    "b2s_mapping_update_incremental": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i32,
                                              ctypes.POINTER(_i32)]),
    "b2s_mapping_update_ranges": (_i32, [_vp, _vp, _vp, _vp, _dbl, _i32, _i32, _vp]),
    "b2s_mapping_update_scans": (_i32, [_vp, _vp, _vp, _vp, _dbl, _i32, _i32, _vp]),
    "b2s_mapping_submit": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, ctypes.POINTER(_i32)]),
    "b2s_mapping_submit_scans": (_i32, [_vp, _vp, _vp, _vp, _dbl, _i32, _i32, _i32, _vp, ctypes.POINTER(_i32)]),
    "b2s_mapping_wait": (_i32, [_vp, _i32]),
    "b2s_mapping_read": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "b2s_mapping_write": (_i32, [_vp, _vp, _vp]),
    "b2s_mapping_planes": (_i32, [_vp, _pp, _pp, _pp]),
    "b2s_bresenham_host": (_i32, [_vp, _i32, _vp, _vp]),
}

_lib = None


class B2SlamError(RuntimeError):
    def __init__(self, status, detail):
        RuntimeError.__init__(self, "b2slam status %d: %s" % (status, detail))
        self.status = status


def lib():
    """The loaded CUDA library; raises if it was not built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                "b2slam: %s is missing -- build it with `make -C %s/csrc` "
                "(there is no CPU fallback)" % (LIB_PATH, _HERE))
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    """Map a C status to the exception the reference would raise (SURVEY.md section 8b Errors)."""
    if status == OK:
        return
    detail = lib().b2s_last_error().decode("utf-8", "replace")
    if status == ERR_NONFINITE:
        # int(nan) -> ValueError, int(inf) -> OverflowError in [MAP]:33-36; both are ValueError-ish
        # to callers; keep the reference's two classes apart by message
        if "inf" in detail and "nan" not in detail.lower():
            raise OverflowError(detail)
        raise ValueError(detail or "non-finite coordinate")
    if status == ERR_INVALID_ARG:
        raise ValueError(detail or "invalid argument")
    if status == ERR_NOMEM:
        raise MemoryError(detail)
    raise B2SlamError(status, detail or lib().b2s_status_string(status).decode())


def ptr(a):
    """Address of a NumPy array's first element (or None)."""
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def device_count():
    n = ctypes.c_int(0)
    rc = lib().b2s_device_count(ctypes.byref(n))
    return n.value if rc == OK else 0


def require_device():
    if device_count() <= 0:
        raise B2SlamError(ERR_CUDA, "no CUDA device visible: b2slam has no CPU fallback")


def _free_pinned(address):
    try:
        lib().b2s_host_free(ctypes.c_void_p(address))
    except Exception:
        pass


def pinned_empty(shape, dtype):
    """NumPy array in page-locked memory (b2s_host_alloc); freed when the last view dies."""
    import weakref

    import numpy as np
    dtype = np.dtype(dtype)
    count = int(np.prod(shape))
    p = ctypes.c_void_p()
    check(lib().b2s_host_alloc(ctypes.byref(p), max(1, count * dtype.itemsize)))
    raw = (ctypes.c_char * max(1, count * dtype.itemsize)).from_address(p.value)
    weakref.finalize(raw, _free_pinned, p.value)
    return np.frombuffer(raw, dtype=dtype, count=count).reshape(shape)
