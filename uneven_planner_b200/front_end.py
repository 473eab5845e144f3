"""ctypes plumbing for the front-end entry points of libualm.so (SURVEY 8f-2): KinoAstar::plan for one (start, goal) pair and the
batch form (search + PlanManager's resampler) that produces the optimizer's inputs, on host threads (plan_batch) or on the GPU
(plan_batch_device, one warp per search)."""
import ctypes as C

import numpy as np

from . import _lib
from .problems import ProblemBatch

dp = C.POINTER(C.c_double)


def default_params():
    p = _lib.AstarParams()
    _lib.lib().ualm_astar_default_params(C.byref(p))
    return p


def resample_params(piece_len=0.3, yaw_piece_times=2.0, mean_vel=0.5, init_time_times=1.2, init_sig_vel=0.05):
    """plan_manager/* of run_hill.yaml:57-62"""
    return _lib.ResampleParams(piece_len, yaw_piece_times, mean_vel, init_time_times, init_sig_vel)


class MapView:
    """the ualm_astar_map_t of a UnevenMapData (keeps the arrays alive)"""

    def __init__(self, mapdata, min_cnormal=0.8, max_rho=0.05, use_cells64=True):
        self.mapdata = mapdata
        self.occ3, self.occ2 = mapdata.occupancy(min_cnormal, max_rho)
        self.geom = mapdata.geom
        u8 = C.POINTER(C.c_uint8)
        c64 = mapdata.cells64 if (use_cells64 and mapdata.cells64 is not None) else None
        self.c = _lib.AstarMap(C.pointer(self.geom), mapdata.cells.ctypes.data_as(C.POINTER(C.c_float)),
                               c64.ctypes.data_as(dp) if c64 is not None else None, self.occ3.ctypes.data_as(u8), self.occ2.ctypes.data_as(u8))


def plan(view, start, goal, params=None, max_pts=1 << 16):
    """KinoAstar::plan: (n, 3) polyline, empty when there is no path; also the number of closed nodes"""
    params = params or default_params()
    s = np.ascontiguousarray(start, dtype=np.float64); g = np.ascontiguousarray(goal, dtype=np.float64)
    buf = np.zeros((max_pts, 3))
    ex = C.c_int(0)
    n = _lib.lib().ualm_kino_astar_plan(C.byref(view.c), C.byref(params), s.ctypes.data_as(dp), g.ctypes.data_as(dp), buf.ctypes.data_as(dp), max_pts, C.byref(ex))
    if n < 0:
        raise RuntimeError(f"ualm_kino_astar_plan: {n}")
    return buf[:n].copy(), ex.value


def plan_det(view, start, goal, params=None, max_pts=1 << 16):
    """plan() with include/ualm_detmath.h's trigonometry instead of libm's (ualm_kino_astar_plan_det): what the device front-end
    computes, on the host.  For tests; the front-end's paths come from plan / plan_batch or plan_batch_device"""
    params = params or default_params()
    s = np.ascontiguousarray(start, dtype=np.float64); g = np.ascontiguousarray(goal, dtype=np.float64)
    buf = np.zeros((max_pts, 3))
    ex = C.c_int(0)
    n = _lib.lib().ualm_kino_astar_plan_det(C.byref(view.c), C.byref(params), s.ctypes.data_as(dp), g.ctypes.data_as(dp), buf.ctypes.data_as(dp), max_pts,
                                            C.byref(ex))
    if n < 0:
        raise RuntimeError(f"ualm_kino_astar_plan_det: {n}")
    return buf[:n].copy(), ex.value


def _packed_batch(starts, goals, N, M, bnd, T, ixy, iyaw, packed, k):
    nxy = int((2 * (N[:k].astype(np.int64) - 1)).sum()); nyaw = int((M[:k].astype(np.int64) - 1).sum())
    pb = ProblemBatch(N[:k].copy(), M[:k].copy(), bnd[:k].copy(), T[:k].copy(), ixy[:nxy].copy(), iyaw[:nyaw].copy())
    keep = packed >= 0
    pb.starts = starts[keep]; pb.goals = goals[keep]
    return pb


def plan_batch(view, starts, goals, params=None, rparams=None, nthreads=0):
    """(start, goal) pairs -> ProblemBatch of the pairs that have a path, the index of every pair in it (or -1), closed-node counts"""
    params = params or default_params()
    rparams = rparams or resample_params()
    starts = np.ascontiguousarray(starts, dtype=np.float64).reshape(-1, 3); goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(-1, 3)
    B = starts.shape[0]
    ip = C.POINTER(C.c_int32)
    N = np.zeros(B, np.int32); M = np.zeros(B, np.int32); bnd = np.zeros((B, 18)); T = np.zeros(B)
    ixy = np.zeros(2 * 63 * max(B, 1)); iyaw = np.zeros(127 * max(B, 1))
    packed = np.zeros(B, np.int32); nexp = np.zeros(B, np.int32)
    k = _lib.lib().ualm_front_end_batch(C.byref(view.c), C.byref(params), C.byref(rparams), B, starts.ctypes.data_as(dp), goals.ctypes.data_as(dp), nthreads,
                                        N.ctypes.data_as(ip), M.ctypes.data_as(ip), bnd.ctypes.data_as(dp), T.ctypes.data_as(dp), ixy.ctypes.data_as(dp), ixy.size,
                                        iyaw.ctypes.data_as(dp), iyaw.size, packed.ctypes.data_as(ip), nexp.ctypes.data_as(ip))
    if k < 0:
        raise RuntimeError(f"ualm_front_end_batch: {k}")
    return _packed_batch(starts, goals, N, M, bnd, T, ixy, iyaw, packed, k), packed, nexp


def plan_batch_device(opt, view, starts, goals, params=None, rparams=None, return_paths=False, timing=None):
    """plan_batch with the searches on opt's GPU (ualm_front_end_batch_device: one warp per search, bit-identical to plan_det; the
    resampler runs on the host).  Returns (ProblemBatch, packed, n_expanded[, paths]); paths: one (n, 3) polyline per pair, empty
    without a path.  timing: a dict that receives "search_ms", the search kernel's CUDA-event time"""
    from .api import _check
    params = params or default_params()
    rparams = rparams or resample_params()
    L = _lib.lib()
    up = getattr(opt, "_front_end_map", (None, None))       # upload the map once per view (and again when its grids were replaced)
    if up[0] is not view or up[1] is not view.c:
        _check(L.ualm_set_front_end_map(opt.h, C.byref(view.c)))
        opt._front_end_map = (view, view.c)
    starts = np.ascontiguousarray(starts, dtype=np.float64).reshape(-1, 3); goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(-1, 3)
    B = starts.shape[0]
    ip = C.POINTER(C.c_int32)
    N = np.zeros(B, np.int32); M = np.zeros(B, np.int32); bnd = np.zeros((B, 18)); T = np.zeros(B)
    ixy = np.zeros(2 * 63 * max(B, 1)); iyaw = np.zeros(127 * max(B, 1))
    packed = np.zeros(B, np.int32); nexp = np.zeros(B, np.int32)
    paths = off = None
    if return_paths:
        cap = L.ualm_front_end_path_cap(C.byref(params), C.byref(rparams))
        _check(min(cap, 0))
        paths = np.zeros((max(B * cap, 1), 3)); off = np.zeros(B + 1, np.int64)
    ms = C.c_float(0)
    k = L.ualm_front_end_batch_device(opt.h, C.byref(params), C.byref(rparams), B, starts.ctypes.data_as(dp), goals.ctypes.data_as(dp), N.ctypes.data_as(ip),
                                      M.ctypes.data_as(ip), bnd.ctypes.data_as(dp), T.ctypes.data_as(dp), ixy.ctypes.data_as(dp), ixy.size,
                                      iyaw.ctypes.data_as(dp), iyaw.size, packed.ctypes.data_as(ip), nexp.ctypes.data_as(ip),
                                      paths.ctypes.data_as(dp) if return_paths else None, paths.shape[0] if return_paths else 0,
                                      off.ctypes.data_as(C.POINTER(C.c_int64)) if return_paths else None, C.byref(ms))
    _check(min(k, 0))
    if timing is not None:
        timing["search_ms"] = ms.value
    pb = _packed_batch(starts, goals, N, M, bnd, T, ixy, iyaw, packed, k)
    if not return_paths:
        return pb, packed, nexp
    return pb, packed, nexp, [paths[off[b]:off[b + 1]].copy() for b in range(B)]
