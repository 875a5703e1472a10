"""ctypes binding of the C-ABI library (include/f1l.h -> lib/libf1l.so).

There is no CPU fallback: if the CUDA library is missing or no GPU is visible, every entry point
raises.
"""
import ctypes as C
import os

import numpy as np

N_TERMS = 5
MAX_OPP = 16
MAX_M = 256
FLAG_VALID, FLAG_COLLIDE_OPP, FLAG_COLLIDE_MAP, FLAG_NO_CENTRE = 1, 2, 4, 8
CAR_HIT_MAP, CAR_HIT_CAR, CAR_NO_FEASIBLE = 1, 2, 4
MAX_GROUP = 1 + MAX_OPP
EVAL_LONE, EVAL_WEIGHTS = 1, 2   # f1l_debug_eval_choice flags

HERE = os.path.dirname(os.path.abspath(__file__))
# F1L_LIB selects another build of the same library (A/B builds of kernel variants)
LIB_PATH = os.environ.get("F1L_LIB") or os.path.join(HERE, "lib", "libf1l.so")

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int32)
_bp = C.POINTER(C.c_uint8)
_vp = C.c_void_p


class F1LError(RuntimeError):
    pass


class Config(C.Structure):
    """f1l_config (include/f1l.h)."""
    _fields_ = [("n_samples", C.c_int32), ("n_newton", C.c_int32), ("window", C.c_int32),
                ("n_shift", C.c_int32), ("n_cull", C.c_int32), ("literal_tracker", C.c_int32),
                ("use_goal_kappa", C.c_int32), ("generator", C.c_int32),
                ("prune_window", C.c_int32), ("collision_mode", C.c_int32),
                ("weights", C.c_double * N_TERMS), ("kappa_max", C.c_double),
                ("car_length", C.c_double), ("car_width", C.c_double),
                ("converge_tol", C.c_double), ("tracker_lookahead", C.c_double),
                ("wheelbase", C.c_double), ("max_reacquire", C.c_double)]


class PlanResult(C.Structure):
    """f1l_plan_result (include/f1l.h)."""
    _fields_ = [("steer", C.c_double), ("speed", C.c_double), ("best_idx", C.c_int32),
                ("no_feasible", C.c_int32), ("tracker_found", C.c_int32),
                ("n_candidates", C.c_int32), ("best_cost", C.c_float), ("reserved", C.c_int32),
                # float* / uint8_t* in the header; void* here so that plain addresses can be stored
                ("best_traj", _vp), ("costs", _vp), ("terms", _vp), ("flags", _vp),
                ("goals", _vp), ("params", _vp), ("states", _vp), ("headings", _vp),
                ("best_traj_map", _vp)]


class RolloutConfig(C.Structure):
    """f1l_rollout_config (include/f1l.h)."""
    _fields_ = [("dt", C.c_double), ("substeps", C.c_int32), ("group", C.c_int32),
                ("max_steer", C.c_double), ("max_accel", C.c_double), ("v_max", C.c_double)]


class FleetBuffers(C.Structure):
    """f1l_fleet (include/f1l.h): device pointers."""
    _fields_ = [("state", _vp), ("prev_theta", _vp), ("has_prev", _vp), ("status", _vp),
                ("progress", _vp), ("track_i", _vp), ("track_s", _vp)]


class RolloutTraceBuffers(C.Structure):
    """f1l_rollout_trace (include/f1l.h): device pointers, each nullable."""
    _fields_ = [("state", _vp), ("steer_speed", _vp), ("best_idx", _vp), ("status", _vp),
                ("progress", _vp)]


class Vehicle(C.Structure):
    """f1l_vehicle (include/f1l.h): the single-track model's parameters."""
    _fields_ = [(n, C.c_double) for n in ("mu", "C_Sf", "C_Sr", "lf", "lr", "h", "m", "I", "max_steer_vel",
                                          "v_switch", "v_kin")]


class BatchCall(C.Structure):
    """f1l_batch_call (include/f1l.h): every input and output of one batch call, host or device
    pointers; None for an absent array."""
    _fields_ = [("poses", _vp), ("opp", _vp), ("n_opp", _vp), ("n_scenarios", C.c_int32),
                ("max_opp", C.c_int32), ("prev_theta", _vp), ("has_prev", _vp),
                ("update_prev", C.c_int32), ("reserved", C.c_int32), ("weights", _vp),
                ("best_idx", _vp), ("best_cost", _vp), ("best_traj", _vp), ("costs", _vp),
                ("flags", _vp), ("steer_speed", _vp), ("terms", _vp)]


# Arrays the library uses in place: name -> (accepted dtypes, shape, direction).  Shapes name S
# scenarios or cars, K = max_opp, C candidates, M = n_samples, B poses.  INOUT is read and written
# in place (by a batch call only with update_prev).
IN, OUT, INOUT = "in", "out", "inout"

BATCH_FIELDS = {   # the pointer fields of f1l_batch_call
    "poses": (("float64",), ("S", 4), IN),
    "opp": (("float64",), ("S", "K", 3), IN),
    "n_opp": (("int32",), ("S",), IN),
    "prev_theta": (("float32",), ("S", "M"), INOUT),
    "has_prev": (("uint8", "bool"), ("S",), INOUT),
    "weights": (("float32",), ("S", N_TERMS), IN),
    "best_idx": (("int32",), ("S",), OUT),
    "best_cost": (("float32",), ("S",), OUT),
    "best_traj": (("float32",), ("S", "M", 4), OUT),
    "costs": (("float32",), ("S", "C"), OUT),
    "flags": (("uint8",), ("S", "C"), OUT),
    "steer_speed": (("float64",), ("S", 2), OUT),
    "terms": (("float32",), ("S", "C", N_TERMS), OUT),
}

FLEET_FIELDS = {   # f1l_fleet
    "state": (("float64",), ("S", 4), INOUT),
    "prev_theta": (("float32",), ("S", "M"), INOUT),
    "has_prev": (("uint8",), ("S",), INOUT),
    "status": (("uint8",), ("S",), INOUT),
    "progress": (("float64",), ("S",), INOUT),
    "track_i": (("int32",), ("S",), INOUT),
    "track_s": (("float64",), ("S",), INOUT),
}

ST_FIELDS = {   # the single-track fleet's array beside f1l_fleet (f1l_rollout_st_dev's dyn_dev)
    "dyn": (("float64",), ("S", 3), INOUT),
}

MOTION_FIELDS = {   # the opponent velocities beside a batch call (f1l_plan_batch_motion*)
    "opp_vel": (("float64",), ("S", "K", 2), IN),
}

PP_FIELDS = {   # the outputs of f1l_pure_pursuit_batch, in argument order
    "nearest": (("float64",), ("B", 4), OUT),
    "nearest_i": (("int32",), ("B",), OUT),
    "lookahead": (("float64",), ("B", 4), OUT),
    "lookahead_i": (("int32",), ("B",), OUT),
    "actuation": (("float64",), ("B", 2), OUT),
    "status": (("int32",), ("B",), OUT),
}


def shape_of(row, dims):
    """the shape of a field row with its sizes from `dims` (name -> size)"""
    return tuple([dims.get(d, d) for d in row[1]])


def zeros_or(a, row, dims):
    """`a`, or zeros of the row's shape and first dtype when `a` is None"""
    return np.zeros(shape_of(row, dims), row[0][0]) if a is None else a


def check_array(name, a, shape, dtypes, where, writes=False):
    """ValueError unless the library can use `a` in place: exactly this shape, one of `dtypes`, and
    for where="host" a C-contiguous numpy array (writeable if `writes`), else a contiguous CUDA
    tensor on device `where`."""
    if where == "host":
        if not (isinstance(a, np.ndarray) and a.dtype in dtypes and a.shape == shape
                and a.flags.c_contiguous and (a.flags.writeable or not writes)):
            raise ValueError("%s must be a %sC-contiguous %s numpy array %s"
                             % (name, "writeable " if writes else "", " / ".join(dtypes), list(shape)))
        return
    import torch
    if not (isinstance(a, torch.Tensor) and a.is_cuda and a.device.index == where
            and str(a.dtype)[6:] in dtypes and a.shape == shape and a.is_contiguous()):
        raise ValueError("%s must be a contiguous %s CUDA tensor %s on cuda:%d"
                         % (name, " / ".join(dtypes), list(shape), where))


def batch_call(arrays, where, dims, update_prev):
    """BatchCall of `arrays` (BATCH_FIELDS name -> array or None) with sizes `dims` (S, K, C, M),
    each given array checked against its row, on the host or device `where` (check_array)."""
    if arrays.get("prev_theta") is None and (arrays.get("has_prev") is not None or update_prev):
        raise ValueError("has_prev / update_prev need prev_theta")
    b = BatchCall(n_scenarios=dims["S"], max_opp=dims["K"], update_prev=int(bool(update_prev)))
    for name, a in arrays.items():
        if a is not None:
            row = BATCH_FIELDS[name]
            check_array(name, a, shape_of(row, dims), row[0], where,
                        row[2] == OUT or (row[2] == INOUT and update_prev))
            setattr(b, name, a.ctypes.data if where == "host" else a.data_ptr())
    return b


# name -> (restype, argtypes); must list every symbol include/f1l.h declares
SIGNATURES = {
    "f1l_default_config": (C.c_int, [C.POINTER(Config)]),
    "f1l_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.POINTER(Config)]),
    "f1l_destroy": (C.c_int, [_vp]),
    "f1l_strerror": (C.c_char_p, [C.c_int]),
    "f1l_set_config": (C.c_int, [_vp, C.POINTER(Config)]),
    "f1l_get_config": (C.c_int, [_vp, C.POINTER(Config)]),
    "f1l_device": (C.c_int, [_vp]),
    "f1l_last_cuda_error": (C.c_char_p, [_vp]),
    "f1l_set_track": (C.c_int, [_vp, _dp, C.c_int, C.c_int]),
    "f1l_set_grid": (C.c_int, [_vp, _bp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double]),
    "f1l_clear_grid": (C.c_int, [_vp]),
    "f1l_get_edt": (C.c_int, [_vp, _vp]),
    "f1l_set_goal_grid": (C.c_int, [_vp, _dp, C.c_int, _dp, C.c_int]),
    "f1l_get_lut_shape": (C.c_int, [_vp, _ip, _dp]),
    "f1l_get_lut": (C.c_int, [_vp, _fp]),
    "f1l_set_lut": (C.c_int, [_vp, _fp, _ip, _dp]),
    "f1l_set_prev_path": (C.c_int, [_vp, _fp, C.c_int]),
    "f1l_clear_prev_path": (C.c_int, [_vp]),
    "f1l_plan": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.POINTER(PlanResult)]),
    "f1l_plan_motion": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_double, C.c_int, C.POINTER(PlanResult)]),
    "f1l_plan_shard": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.POINTER(PlanResult)]),
    "f1l_plan_goals": (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, C.c_int, C.c_int,
                                 C.POINTER(PlanResult)]),
    "f1l_select_candidate": (C.c_int, [_vp, C.c_int, C.c_float, C.c_int, C.POINTER(PlanResult)]),
    "f1l_generate": (C.c_int, [_vp, _dp, C.c_int, _fp, _fp, _bp]),
    "f1l_plan_batch_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp,
                                     _vp, _vp, _vp]),
    "f1l_plan_batch": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp,
                                 _vp]),
    "f1l_plan_batch_prev_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "f1l_plan_batch_prev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int,
                                      _vp, _vp, _vp, _vp, _vp, _vp]),
    "f1l_plan_batch_call_dev": (C.c_int, [_vp, C.POINTER(BatchCall), _vp]),
    "f1l_plan_batch_call": (C.c_int, [_vp, C.POINTER(BatchCall)]),
    "f1l_plan_batch_motion_dev": (C.c_int, [_vp, C.POINTER(BatchCall), _vp, C.c_double, _vp]),
    "f1l_plan_batch_motion": (C.c_int, [_vp, C.POINTER(BatchCall), _vp, C.c_double]),
    "f1l_default_rollout_config": (C.c_int, [C.POINTER(RolloutConfig)]),
    "f1l_rollout_dev": (C.c_int, [_vp, C.POINTER(RolloutConfig), C.POINTER(FleetBuffers), C.c_int,
                                  C.c_int, C.POINTER(RolloutTraceBuffers), _vp]),
    "f1l_rollout_weights_dev": (C.c_int, [_vp, C.POINTER(RolloutConfig), C.POINTER(FleetBuffers), _vp,
                                          C.c_int, C.c_int, C.POINTER(RolloutTraceBuffers), _vp]),
    "f1l_default_vehicle": (C.c_int, [C.POINTER(Vehicle)]),
    "f1l_rollout_st_dev": (C.c_int, [_vp, C.POINTER(RolloutConfig), C.POINTER(Vehicle), C.POINTER(FleetBuffers),
                                     _vp, _vp, C.c_int, C.c_int, C.POINTER(RolloutTraceBuffers), _vp, _vp]),
    "f1l_rollout_predict_dev": (C.c_int, [_vp, C.POINTER(RolloutConfig), C.POINTER(Vehicle),
                                          C.POINTER(FleetBuffers), _vp, _vp, C.c_double, C.c_int, C.c_int,
                                          C.POINTER(RolloutTraceBuffers), _vp, _vp]),
    "f1l_pure_pursuit_batch_dev": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _vp, _vp, _vp,
                                             _vp, _vp, _vp]),
    "f1l_pure_pursuit_batch": (C.c_int, [_vp, _vp, C.c_int, C.c_double, _vp, _vp, _vp, _vp, _vp,
                                         _vp]),
    "f1l_front_axle_batch_dev": (C.c_int, [_vp, _vp, C.c_int, C.c_double, C.c_double, _vp, _vp, _vp]),
    "f1l_front_axle_batch": (C.c_int, [_vp, _vp, C.c_int, C.c_double, C.c_double, _vp, _vp]),
    "f1l_intersect_point_batch": (C.c_int, [_vp, _dp, _dp, C.c_int, C.c_double, C.c_int, _dp,
                                            _ip]),
    "f1l_get_actuation_batch": (C.c_int, [_vp, _dp, C.c_int, C.c_double, _dp]),
    "f1l_set_stats": (C.c_int, [_vp, C.c_int]),
    "f1l_get_stats": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.c_int]),
    "f1l_last_eval_shape": (C.c_int, [_vp, _ip, C.c_int]),
    "f1l_plan_rows": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(PlanResult)]),
    "f1l_xchg_export": (C.c_int, [_vp, _vp, C.c_int]),
    "f1l_xchg_attach": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "f1l_xchg_detach": (C.c_int, [_vp]),
    "f1l_launch_count": (C.c_int64, [_vp]),
    "f1l_set_graph": (C.c_int, [_vp, C.c_int]),
    "f1l_set_timing": (C.c_int, [_vp, C.c_int]),
    "f1l_last_kernel_ms": (C.c_int, [_vp, _fp, _fp, _fp]),
    "f1l_mean_kernel_ms": (C.c_int, [_vp, _fp, _fp, _fp, C.POINTER(C.c_int)]),
    "f1l_bind_host_numa": (C.c_int, [C.c_int]),
    "f1l_measure_peaks": (C.c_int, [_vp, _dp, _dp]),
    "f1l_measure_peaks_ex": (C.c_int, [_vp, _dp, C.c_int]),
    "f1l_debug_query_ctx": (C.c_int, [_vp, _fp, _ip]),
    "f1l_debug_motion_ctx": (C.c_int, [_vp, _fp, C.c_int]),
    "f1l_debug_eval_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _ip, C.c_int]),
    "f1l_debug_eval_choice": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _ip, C.c_int]),
    "f1l_debug_eval_builds": (C.c_int, [_ip, C.c_int]),
    "f1l_debug_pp_parts": (C.c_int, [C.c_int, C.c_int, C.c_int]),
}

_lib = None


def lib():
    """Loads libf1l.so (once).  Fails loudly: there is no fallback implementation."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise F1LError(
                "CUDA library %s is missing; build it with `python -m f1tenth_planning_b200.build` "
                "(or __graft_entry__.build()).  There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code, handle=None):
    if code == 0:
        return
    L = lib()
    msg = L.f1l_strerror(code).decode()
    if handle is not None and code == -3:
        msg += ": " + L.f1l_last_cuda_error(handle).decode()
    raise F1LError("f1l error %d: %s" % (code, msg))


def default_config():
    cfg = Config()
    check(lib().f1l_default_config(C.byref(cfg)))
    return cfg
