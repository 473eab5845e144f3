"""ctypes binding of libualm.so (the C ABI declared in include/ualm.h).

The library is the product; this module only loads it and declares signatures.  There is no
Python/CPU fallback: if the shared library is missing the import raises, and compute entry points
return UALM_ENOCUDA (raised as RuntimeError) when no CUDA device is usable.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libualm.so")

UALM_OK, UALM_ENOCUDA, UALM_EINVAL, UALM_ESTATE, UALM_ELIMIT = 0, -1, -2, -3, -4


class Params(C.Structure):
    _fields_ = [(n, C.c_double) for n in
                ("rho_T", "rho_ter", "max_vel", "max_acc_lon", "max_acc_lat", "max_kap", "min_cxi", "max_sig")] + \
               [("use_scaling", C.c_int)] + \
               [(n, C.c_double) for n in ("rho", "beta", "gamma", "epsilon_con", "max_iter",
                                          "g_epsilon", "min_step", "inner_max_iter", "delta")] + \
               [("mem_size", C.c_int), ("past", C.c_int), ("int_K", C.c_int), ("gravity", C.c_double)]


class MapGeom(C.Structure):
    _fields_ = [("voxel_num", C.c_int * 3), ("origin", C.c_double * 3), ("max_boundary", C.c_double * 3),
                ("xy_resolution", C.c_double), ("yaw_resolution", C.c_double)]


class AstarParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("yaw_resolution", "lambda_heu", "weight_r2", "weight_so2", "weight_v_change", "weight_delta_change", "weight_sigma",
                                          "time_interval", "collision_interval", "oneshot_range", "wheel_base", "max_steer", "max_vel")]


class AstarMap(C.Structure):
    _fields_ = [("geom", C.POINTER(MapGeom)), ("cells", C.POINTER(C.c_float)), ("cells64", C.POINTER(C.c_double)), ("occ3", C.POINTER(C.c_uint8)),
                ("occ2", C.POINTER(C.c_uint8))]


class ResampleParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("piece_len", "yaw_piece_times", "mean_vel", "init_time_times", "init_sig_vel")]


class Result(C.Structure):
    _fields_ = [("ret_code", C.c_int32), ("outer_iters", C.c_int32), ("n_evals", C.c_int32),
                ("n_lbfgs_iters", C.c_int32), ("last_lbfgs_ret", C.c_int32), ("max_bound", C.c_int32), ("sum_bound", C.c_int32), ("reserved", C.c_int32),
                ("inner_cost", C.c_double), ("jerk_cost", C.c_double), ("total_T", C.c_double),
                ("res_h", C.c_double), ("res_g", C.c_double), ("scale_fx", C.c_double), ("rho_final", C.c_double),
                ("piece_T_xy", C.c_double), ("piece_T_yaw", C.c_double)]


_lib = None


def lib():
    """Load libualm.so (building is done by `python -m uneven_planner_b200.build` / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not built; run `python -m uneven_planner_b200.build` (nvcc, sm_100a)")
    L = C.CDLL(LIB_PATH)
    dp, ip, fp, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_float), C.c_void_p
    L.ualm_default_params.argtypes = [C.POINTER(Params)]
    L.ualm_default_params.restype = None
    L.ualm_map_geometry.argtypes = [C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(MapGeom)]
    L.ualm_map_geometry.restype = None
    L.ualm_map_build.argtypes = [fp, C.c_int64, C.POINTER(MapGeom), C.c_double, C.c_double, C.c_double, C.c_int,
                                 C.c_int, fp]
    L.ualm_map_occupancy.argtypes = [fp, C.POINTER(MapGeom), C.c_double, C.c_double, C.POINTER(C.c_uint8),
                                     C.POINTER(C.c_uint8)]
    L.ualm_dubins_path.argtypes = [dp, dp, C.c_double, C.c_double, dp, C.c_int]
    L.ualm_dubins_shot.argtypes = [dp, dp, C.c_double, C.c_double, dp, C.c_int, dp]
    L.ualm_astar_default_params.argtypes = [C.POINTER(AstarParams)]
    L.ualm_astar_default_params.restype = None
    L.ualm_kino_astar_plan.argtypes = [C.POINTER(AstarMap), C.POINTER(AstarParams), dp, dp, dp, C.c_int, C.POINTER(C.c_int)]
    L.ualm_kino_astar_plan_det.argtypes = [C.POINTER(AstarMap), C.POINTER(AstarParams), dp, dp, dp, C.c_int, C.POINTER(C.c_int)]
    L.ualm_front_end_batch.argtypes = [C.POINTER(AstarMap), C.POINTER(AstarParams), C.POINTER(ResampleParams), C.c_int, dp, dp, C.c_int, ip, ip, dp, dp, dp,
                                       C.c_longlong, dp, C.c_longlong, ip, ip]
    L.ualm_resample_path.argtypes = [dp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, dp, dp,
                                     C.c_int, dp, C.c_int, ip, ip, dp]
    L.ualm_map_preprocess_cloud.argtypes = [fp, C.c_int64, C.c_double, C.c_double, C.c_double, fp, C.c_int64]
    L.ualm_map_preprocess_cloud.restype = C.c_int64
    for name in ("ualm_map_build", "ualm_map_occupancy", "ualm_dubins_path", "ualm_resample_path"):
        getattr(L, name).restype = C.c_int
    # GPU entry points (present once the CUDA translation unit is linked in)
    if hasattr(L, "ualm_create"):
        L.ualm_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int]
        L.ualm_destroy.argtypes = [vp]
        L.ualm_last_error.argtypes = []
        L.ualm_last_error.restype = C.c_char_p
        L.ualm_set_stream.argtypes = [vp, vp]
        L.ualm_set_stream.restype = C.c_int
        L.ualm_set_params.argtypes = [vp, C.POINTER(Params)]
        L.ualm_set_map.argtypes = [vp, C.POINTER(MapGeom), fp]
        L.ualm_solve_batch.argtypes = [vp, C.c_int, ip, ip, dp, dp, dp, dp, C.POINTER(Result), dp, dp]
        L.ualm_upload.argtypes = [vp, C.c_int, ip, ip, dp, dp, dp, dp]
        L.ualm_solve_resident.argtypes = [vp]
        L.ualm_sync.argtypes = [vp]
        L.ualm_download.argtypes = [vp, C.POINTER(Result), dp, dp]
        L.ualm_last_solve_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
        L.ualm_pack_records_device.argtypes = [vp, vp, C.c_int]
        L.ualm_eval_batch.argtypes = [vp, dp, dp, dp, dp, dp, C.c_double, dp, dp, dp, dp, dp, dp]
        L.ualm_init_scaling_batch.argtypes = [vp, dp, dp]
        L.ualm_time_penalty_kernel.argtypes = [vp, C.c_int, C.POINTER(C.c_float), dp]
        L.ualm_profile.argtypes = [vp, C.c_int, C.POINTER(C.c_longlong)]
        L.ualm_map_build_device.argtypes = [vp, fp, C.c_int64, C.POINTER(MapGeom), C.c_double, C.c_double, C.c_double, C.c_int, fp, C.POINTER(C.c_float)]
        L.ualm_map_build_device.restype = C.c_int
        L.ualm_feasibility_batch.argtypes = [vp, C.c_double, dp]
        L.ualm_feasibility_batch.restype = C.c_int
        L.ualm_mpc_export_batch.argtypes = [vp, C.c_double] + [dp] * 9
        L.ualm_mpc_export_batch.restype = C.c_int
        L.ualm_profile.restype = C.c_int
        L.ualm_reset_stream.argtypes = [vp]
        L.ualm_set_map_f64.argtypes = [vp, C.POINTER(MapGeom), dp, C.c_int]
        L.ualm_max_lanes.argtypes = []
        L.ualm_select_lane.argtypes = [vp, C.c_int]
        L.ualm_submit_batch.argtypes = [vp, C.c_int, ip, ip, dp, dp, dp, dp, C.c_int, C.POINTER(C.c_int)]
        L.ualm_wait_batch.argtypes = [vp, C.c_int, C.POINTER(Result), dp, dp]
        L.ualm_mark_begin.argtypes = [vp]
        L.ualm_mark_end.argtypes = [vp, C.POINTER(C.c_float)]
        L.ualm_solve_batch_multi.argtypes = [C.POINTER(vp), C.c_int, C.c_int, ip, ip, dp, dp, dp, dp, C.POINTER(Result), dp, dp]
        L.ualm_pack_records_device_async.argtypes = [vp, vp, C.c_int]
        L.ualm_set_front_end_map.argtypes = [vp, C.POINTER(AstarMap)]
        L.ualm_front_end_batch_device.argtypes = [vp, C.POINTER(AstarParams), C.POINTER(ResampleParams), C.c_int, dp, dp, ip, ip, dp, dp, dp, C.c_longlong, dp,
                                                  C.c_longlong, ip, ip, dp, C.c_longlong, C.POINTER(C.c_int64), C.POINTER(C.c_float)]
        L.ualm_front_end_path_cap.argtypes = [C.POINTER(AstarParams), C.POINTER(ResampleParams)]
        for name in ("ualm_reset_stream", "ualm_set_map_f64", "ualm_max_lanes", "ualm_select_lane", "ualm_submit_batch", "ualm_wait_batch",
                     "ualm_mark_begin", "ualm_mark_end", "ualm_solve_batch_multi", "ualm_pack_records_device_async", "ualm_set_front_end_map",
                     "ualm_front_end_batch_device", "ualm_front_end_path_cap"):
            getattr(L, name).restype = C.c_int
        for name in ("ualm_create", "ualm_destroy", "ualm_set_params", "ualm_set_map", "ualm_solve_batch",
                     "ualm_upload", "ualm_solve_resident", "ualm_sync", "ualm_download", "ualm_last_solve_ms",
                     "ualm_pack_records_device", "ualm_eval_batch", "ualm_init_scaling_batch",
                     "ualm_time_penalty_kernel"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def default_params():
    p = Params()
    lib().ualm_default_params(C.byref(p))
    return p


def map_geometry(size_x=10.0, size_y=10.0, xy_res=0.05, yaw_res=0.1):
    g = MapGeom()
    lib().ualm_map_geometry(size_x, size_y, xy_res, yaw_res, C.byref(g))
    return g
