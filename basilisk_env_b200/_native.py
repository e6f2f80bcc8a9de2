"""ctypes binding of the C ABI in include/bskenv.h (libbskenv.so, hand-written CUDA for sm_100a).

There is deliberately no fallback: if the library is missing or no CUDA device is present the
product path raises."""
import ctypes as C
import os

from . import build as _build

_LIB = None


class Config(C.Structure):
    """Mirror of `bskenv_config` (include/bskenv.h)."""
    _fields_ = [("abi_version", C.c_int32), ("reserved0", C.c_int32),
                ("dynRate", C.c_double), ("fswRate", C.c_double), ("step_duration", C.c_double),
                ("mass", C.c_double), ("width", C.c_double), ("depth", C.c_double), ("height", C.c_double),
                ("planetRadius", C.c_double), ("baseDensity", C.c_double), ("scaleHeight", C.c_double),
                ("disturbance_magnitude", C.c_double),
                ("nHat_B", C.c_double * 3), ("panelArea", C.c_double), ("panelEfficiency", C.c_double),
                ("powerDraw", C.c_double), ("storageCapacity", C.c_double),
                ("sigma_R0N", C.c_double * 3), ("K", C.c_double), ("Ki", C.c_double), ("P", C.c_double),
                ("hs_min", C.c_double), ("thrMinFireTime", C.c_double),
                ("thrForceSign", C.c_int32), ("maxCounterValue", C.c_int32),
                ("max_length", C.c_int32), ("auto_reset", C.c_int32),
                ("wheel_limit_rpm", C.c_double), ("power_max", C.c_double), ("failure_penalty", C.c_double),
                ("use_j2", C.c_int32), ("hill_cel_pun", C.c_int32), ("rw_set", C.c_int32), ("precision", C.c_int32),
                ("reserved", C.c_int32 * 6)]


class OpNavConfig(C.Structure):
    """Mirror of `bskenv_opnav_config` (include/bskenv.h)."""
    _fields_ = [("abi_version", C.c_int32), ("reserved0", C.c_int32),
                ("dynRate", C.c_double), ("fswRate", C.c_double), ("step_duration_min", C.c_double),
                ("max_length", C.c_int32), ("numModes", C.c_int32), ("auto_reset", C.c_int32), ("nav_noise", C.c_int32),
                ("camera_reenable", C.c_int32), ("sample_orbit", C.c_int32),
                ("pixel_noise_std", C.c_double), ("circle_unc", C.c_double), ("reward_mult", C.c_double),
                ("noise_seed", C.c_uint64), ("reserved", C.c_int32 * 8)]


OPNAV_EXPORTS = ["bskenv_opnav_default_config", "bskenv_opnav_create", "bskenv_opnav_destroy", "bskenv_opnav_last_error",
                 "bskenv_opnav_num_envs", "bskenv_opnav_reset_seeded", "bskenv_opnav_reset_ics", "bskenv_opnav_reset_init",
                 "bskenv_opnav_get_ics", "bskenv_opnav_step", "bskenv_opnav_step_host", "bskenv_opnav_state_dims",
                 "bskenv_opnav_get_state", "bskenv_opnav_set_state", "bskenv_opnav_state_field",
                 "bskenv_opnav_episode_stats", "bskenv_opnav_launch_count", "bskenv_opnav_flops_per_step",
                 "bskenv_opnav_set_ephemeris", "bskenv_opnav_step_info", "bskenv_opnav_set_ic_pool", "bskenv_opnav_get_ic_rows"]

EXPORTS = ["bskenv_abi_version", "bskenv_default_config", "bskenv_create", "bskenv_destroy", "bskenv_last_error",
           "bskenv_num_envs", "bskenv_reset_seeded", "bskenv_reset_ics", "bskenv_reset_init", "bskenv_get_ics",
           "bskenv_step", "bskenv_step_host", "bskenv_state_dims", "bskenv_get_state", "bskenv_set_state",
           "bskenv_state_field", "bskenv_episode_stats", "bskenv_launch_count", "bskenv_fp64_peak",
           "bskenv_flops_per_step", "bskenv_set_ephemeris", "bskenv_set_gravity_degree2", "bskenv_step_info",
           "bskenv_step_host_async", "bskenv_step_host_wait", "bskenv_alloc_host", "bskenv_free_host", "bskenv_kernel_name",
           "bskenv_set_organisation", "bskenv_set_param_pool", "bskenv_get_env_params", "bskenv_set_ic_pool",
           "bskenv_get_ic_rows"]


def lib_path():
    return _build.LIB


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the environment step)")
    L = C.CDLL(path)
    vp, i64, u64, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32
    L.bskenv_abi_version.restype = C.c_int
    L.bskenv_default_config.argtypes = [C.POINTER(Config)]
    L.bskenv_create.argtypes = [C.POINTER(Config), C.c_int, i64, i64, C.POINTER(vp)]
    L.bskenv_destroy.argtypes = [vp]
    L.bskenv_last_error.restype = C.c_char_p
    L.bskenv_last_error.argtypes = [vp]
    L.bskenv_num_envs.restype = i64
    L.bskenv_num_envs.argtypes = [vp]
    L.bskenv_reset_seeded.argtypes = [vp, u64, vp, vp, vp]
    L.bskenv_reset_ics.argtypes = [vp, vp, vp, vp, vp]
    L.bskenv_reset_init.argtypes = [vp, vp, vp, vp]
    L.bskenv_get_ics.argtypes = [vp, vp, vp]
    L.bskenv_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.bskenv_step_host.argtypes = [vp, vp, vp, vp, vp, vp]
    L.bskenv_step_info.argtypes = [vp] * 10
    L.bskenv_step_host_async.argtypes = [vp] * 9
    L.bskenv_step_host_wait.argtypes = [vp]
    L.bskenv_alloc_host.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.bskenv_free_host.argtypes = [vp]
    L.bskenv_state_dims.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.bskenv_get_state.argtypes = [vp, vp, vp, vp]
    L.bskenv_set_state.argtypes = [vp, vp, vp, vp]
    L.bskenv_state_field.argtypes = [C.c_char_p, C.POINTER(i32)]
    L.bskenv_episode_stats.argtypes = [vp, vp]
    L.bskenv_launch_count.restype = i64
    L.bskenv_launch_count.argtypes = [vp]
    L.bskenv_kernel_name.restype = C.c_char_p
    L.bskenv_kernel_name.argtypes = [vp]
    L.bskenv_set_organisation.argtypes = [vp, C.c_int]
    L.bskenv_set_param_pool.argtypes = [vp, C.c_int, vp, C.c_int]
    L.bskenv_get_env_params.argtypes = [vp, vp, vp, vp]
    L.bskenv_set_ic_pool.argtypes = [vp, C.c_int, vp, C.c_int]
    L.bskenv_get_ic_rows.argtypes = [vp, vp, vp]
    L.bskenv_fp64_peak.argtypes = [C.c_int, C.c_double, C.POINTER(C.c_double)]
    L.bskenv_flops_per_step.restype = C.c_double
    L.bskenv_flops_per_step.argtypes = [vp]
    L.bskenv_set_ephemeris.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, vp]
    L.bskenv_set_gravity_degree2.argtypes = [vp, C.c_int, vp]
    L.bskenv_opnav_default_config.argtypes = [C.POINTER(OpNavConfig)]
    L.bskenv_opnav_create.argtypes = [C.POINTER(OpNavConfig), C.c_int, i64, i64, C.POINTER(vp)]
    L.bskenv_opnav_destroy.argtypes = [vp]
    L.bskenv_opnav_last_error.restype = C.c_char_p
    L.bskenv_opnav_last_error.argtypes = [vp]
    L.bskenv_opnav_num_envs.restype = i64
    L.bskenv_opnav_num_envs.argtypes = [vp]
    L.bskenv_opnav_reset_seeded.argtypes = [vp, u64, vp, vp, vp]
    L.bskenv_opnav_reset_ics.argtypes = [vp, vp, vp, vp, vp]
    L.bskenv_opnav_reset_init.argtypes = [vp, vp, vp, vp]
    L.bskenv_opnav_get_ics.argtypes = [vp, vp, vp]
    L.bskenv_opnav_step.argtypes = [vp] * 9
    L.bskenv_opnav_step_host.argtypes = [vp] * 7
    L.bskenv_opnav_step_info.argtypes = [vp] * 11
    L.bskenv_opnav_state_dims.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.bskenv_opnav_get_state.argtypes = [vp, vp, vp, vp]
    L.bskenv_opnav_set_state.argtypes = [vp, vp, vp, vp]
    L.bskenv_opnav_state_field.argtypes = [C.c_char_p, C.POINTER(i32)]
    L.bskenv_opnav_episode_stats.argtypes = [vp, vp]
    L.bskenv_opnav_launch_count.restype = i64
    L.bskenv_opnav_launch_count.argtypes = [vp]
    L.bskenv_opnav_flops_per_step.restype = C.c_double
    L.bskenv_opnav_flops_per_step.argtypes = [vp]
    L.bskenv_opnav_set_ephemeris.argtypes = [vp, C.c_double, C.c_double, C.c_int, C.c_int, vp]
    L.bskenv_opnav_set_ic_pool.argtypes = [vp, C.c_int, vp, C.c_int]
    L.bskenv_opnav_get_ic_rows.argtypes = [vp, vp, vp]
    if L.bskenv_abi_version() != 1:
        raise RuntimeError("libbskenv.so ABI version mismatch")
    _LIB = L
    return L


def default_config(**overrides):
    cfg = Config()
    lib().bskenv_default_config(C.byref(cfg))
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise AttributeError(f"bskenv_config has no field {k!r}")
        if isinstance(v, (list, tuple)):
            v = (C.c_double * len(v))(*v)
        setattr(cfg, k, v)
    return cfg


def state_field(name):
    is_int = C.c_int32(0)
    idx = lib().bskenv_state_field(name.encode(), C.byref(is_int))
    if idx < 0:
        raise KeyError(name)
    return idx, bool(is_int.value)


def opnav_default_config(**overrides):
    cfg = OpNavConfig()
    lib().bskenv_opnav_default_config(C.byref(cfg))
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise AttributeError(f"bskenv_opnav_config has no field {k!r}")
        setattr(cfg, k, v)
    return cfg


def opnav_state_field(name):
    is_int = C.c_int32(0)
    idx = lib().bskenv_opnav_state_field(name.encode(), C.byref(is_int))
    if idx < 0:
        raise KeyError(name)
    return idx, bool(is_int.value)
