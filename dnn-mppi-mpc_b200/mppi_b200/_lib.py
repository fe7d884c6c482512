"""ctypes binding of libmppi_b200.so (include/mppi_b200.h).  No CPU fallback: importing
the engine without the built library, or creating a handle without a CUDA device, fails."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPPI_B200_LIB", os.path.join(_HERE, "libmppi_b200.so"))   # override: kernel A/B builds

MPPI_ABI_VERSION = 3
MODEL = {"diffdrive": 0, "bicycle": 1, "diffdrive_mlp": 2}
COST_MODE = {"last": 0, "sum": 1}
WAYPOINT_MODE = {"strict": 0, "frozen": 1}
FILTER = {"diffdrive": 0, "racecar": 1}
COLLISION = {"none": 0, "circle": 1, "footprint": 2}
COST_KIND = {"path": 0, "goal": 1, "target_soft": 2}
MAX_T, MAX_WINDOW, MAX_OBSTACLES = 128, 256, 16


class MppiConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "abi_version", "device", "model", "K", "T", "n_robots", "window", "cost_mode",
        "waypoint_mode", "filter_kind", "yaw_wrap", "collision", "K_global", "k_offset", "clamp_nominal", "cost_kind")] + [
        ("dt", C.c_double), ("wheel_base", C.c_double), ("u_max", C.c_double * 2),
        ("param_exploration", C.c_double), ("param_lambda", C.c_double), ("param_alpha", C.c_double),
        ("temperature", C.c_double), ("sigma", C.c_double * 4), ("stage_w", C.c_double * 4),
        ("term_w", C.c_double * 4), ("margin", C.c_double), ("robot_radius", C.c_double),
        ("vehicle_l", C.c_double), ("vehicle_w", C.c_double), ("goal", C.c_double * 4),
        ("ctrl_w", C.c_double * 2), ("soft_obs_weight", C.c_double), ("soft_obs_safety", C.c_double)]


class MppiTimings(C.Structure):
    _fields_ = [("last_step_ms", C.c_float), ("last_rollout_ms", C.c_float), ("last_update_ms", C.c_float),
                ("last_passes", C.c_int32), ("launches", C.c_int32)]


class MppiStats(C.Structure):
    _fields_ = [("rho", C.c_float), ("eta", C.c_float), ("ess", C.c_float),
                ("min_collisions", C.c_int32), ("idx", C.c_int32), ("u_first", C.c_float * 2)]


class MppiError(RuntimeError):
    pass


# every symbol include/mppi_b200.h declares: (restype, argtypes)
_H = C.c_void_p
_PD, _PF, _PI = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_int32)
SYMBOLS = {
    "mppi_create": (C.c_int, [C.POINTER(MppiConfig), C.POINTER(_H)]),
    "mppi_destroy": (C.c_int, [_H]),
    "mppi_default_config": (None, [C.POINTER(MppiConfig)]),
    "mppi_strerror": (C.c_char_p, [C.c_int]),
    "mppi_last_error": (C.c_char_p, [_H]),
    "mppi_set_stream": (C.c_int, [_H, C.c_void_p]),
    "mppi_synchronize": (C.c_int, [_H]),
    "mppi_set_ref_path": (C.c_int, [_H, _PD, C.c_int32, C.c_int32]),
    "mppi_set_ref_paths_spline": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int32, C.c_double, C.c_int32]),
    "mppi_get_ref_path": (C.c_int, [_H, C.c_int32, _PF, C.c_int32, _PI]),
    "mppi_set_obstacles": (C.c_int, [_H, _PD, C.c_int32]),
    "mppi_set_goal": (C.c_int, [_H, _PD, C.c_int32]),
    "mppi_set_moving_obstacles": (C.c_int, [_H, _PD, _PD, C.c_int32]),
    "mppi_set_robot_obstacles": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "mppi_set_robot_goals": (C.c_int, [_H, C.c_void_p, C.c_int32]),
    "mppi_set_nominal": (C.c_int, [_H, _PF]),
    "mppi_get_nominal": (C.c_int, [_H, _PF]),
    "mppi_set_waypoint_idx": (C.c_int, [_H, _PI]),
    "mppi_get_waypoint_idx": (C.c_int, [_H, _PI]),
    "mppi_set_mlp": (C.c_int, [_H, C.POINTER(_PF), C.POINTER(_PF)]),
    "mppi_set_mlp_ex": (C.c_int, [_H, C.c_int32, C.c_int32, C.POINTER(_PF), C.POINTER(_PF), _PD, _PD, _PD, _PD]),
    "mppi_step": (C.c_int, [_H, _PD, C.c_void_p, C.c_uint64, C.c_uint64, _PF, _PF]),
    "mppi_step_async": (C.c_int, [_H, _PD, C.c_void_p, C.c_uint64, C.c_uint64]),
    "mppi_rollout_costs": (C.c_int, [_H, _PD, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mppi_reduce_update": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, _PF, _PF, _PF]),
    "mppi_generate_noise": (C.c_int, [_H, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mppi_generate_noise_robot": (C.c_int, [_H, C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p]),
    "mppi_get_trajectories": (C.c_int, [_H, _PD, C.c_void_p, C.c_uint64, C.c_uint64, _PF, C.c_void_p]),
    "mppi_set_keep_costs": (C.c_int, [_H, C.c_int32]),
    "mppi_get_top_trajectories": (C.c_int, [_H, _PD, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int32, C.c_int32, _PF,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "mppi_get_stats": (C.c_int, [_H, C.POINTER(MppiStats)]),
    "mppi_run_closed_loop": (C.c_int, [_H, _PD, C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, _PF, _PF]),
    "mppi_step_batched": (C.c_int, [_H, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mppi_comm_get_unique_id": (C.c_int, [C.c_void_p]),
    "mppi_comm_init": (C.c_int, [_H, C.c_void_p, C.c_int32, C.c_int32]),
    "mppi_comm_p2p_export": (C.c_int, [_H, C.c_int32, C.c_void_p]),
    "mppi_comm_p2p_open": (C.c_int, [_H, C.c_void_p, C.c_int32, C.c_int32]),
    "mppi_comm_p2p_barrier": (C.c_int, [_H]),
    "mppi_comm_p2p_trace": (C.c_int, [_H, C.POINTER(C.c_uint64)]),
    "mppi_set_trace": (C.c_int, [_H, C.c_int32]),
    "mppi_get_trace": (C.c_int, [_H, C.POINTER(C.c_uint64), C.c_int32, _PI]),
    "mppi_debug_check_guards": (C.c_int, [_H]),
    "mppi_set_timing": (C.c_int, [_H, C.c_int32]),
    "mppi_get_timings": (C.c_int, [_H, C.POINTER(MppiTimings)]),
    "mppi_abi_version": (C.c_int, []),
    "mppi_probe_fp32_peak": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "mppi_probe_tanh": (C.c_int, [C.c_int32, _PF, _PF, C.c_int32]),
    "mppi_mlp_schedule_cut": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
}

_lib = None


def load():
    """Loads libmppi_b200.so and types every entry point.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MppiError("libmppi_b200.so is not built (%s): run __graft_entry__.build() or "
                        "`make -C dnn-mppi-mpc_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.mppi_abi_version() != MPPI_ABI_VERSION:
        raise MppiError("libmppi_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(lib, handle, status, what):
    if status != 0:
        detail = lib.mppi_last_error(handle).decode() if handle else ""
        raise MppiError("%s failed: %s %s" % (what, lib.mppi_strerror(status).decode(), detail))
