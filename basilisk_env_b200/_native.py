"""ctypes binding of the C ABI in include/bskenv.h (libbskenv.so, hand-written CUDA for sm_100a).

There is deliberately no fallback: if the library is missing or no CUDA device is present the
product path raises."""
import ctypes as C
import os
import types

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


# C ABI prefix of each batch -> its configuration struct
BATCHES = {"bskenv_": Config, "bskenv_opnav_": OpNavConfig}

OPNAV_EXPORTS = ["bskenv_opnav_default_config", "bskenv_opnav_create", "bskenv_opnav_destroy", "bskenv_opnav_last_error",
                 "bskenv_opnav_num_envs", "bskenv_opnav_reset_seeded", "bskenv_opnav_reset_ics", "bskenv_opnav_reset_init",
                 "bskenv_opnav_get_ics", "bskenv_opnav_step", "bskenv_opnav_step_host", "bskenv_opnav_state_dims",
                 "bskenv_opnav_get_state", "bskenv_opnav_set_state", "bskenv_opnav_state_field",
                 "bskenv_opnav_episode_stats", "bskenv_opnav_launch_count", "bskenv_opnav_flops_per_step",
                 "bskenv_opnav_set_ephemeris", "bskenv_opnav_step_info", "bskenv_opnav_set_ic_pool", "bskenv_opnav_get_ic_rows",
                 "bskenv_opnav_snapshot_width", "bskenv_opnav_snapshot", "bskenv_opnav_restore"]

EXPORTS = ["bskenv_abi_version", "bskenv_default_config", "bskenv_create", "bskenv_destroy", "bskenv_last_error",
           "bskenv_num_envs", "bskenv_reset_seeded", "bskenv_reset_ics", "bskenv_reset_init", "bskenv_get_ics",
           "bskenv_step", "bskenv_step_host", "bskenv_state_dims", "bskenv_get_state", "bskenv_set_state",
           "bskenv_state_field", "bskenv_episode_stats", "bskenv_launch_count", "bskenv_fp64_peak",
           "bskenv_flops_per_step", "bskenv_set_ephemeris", "bskenv_set_gravity_degree2", "bskenv_step_info",
           "bskenv_step_host_async", "bskenv_step_host_wait", "bskenv_alloc_host", "bskenv_free_host", "bskenv_kernel_name",
           "bskenv_set_organisation", "bskenv_set_param_pool", "bskenv_get_env_params", "bskenv_set_ic_pool",
           "bskenv_get_ic_rows", "bskenv_snapshot_width", "bskenv_snapshot", "bskenv_restore"]


def _shared_signatures(cfg):
    """(restype, argtypes) of the entry points both batches export under their prefix; cfg = the batch's config struct."""
    vp, i64, u64, i32, ci = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32, C.c_int
    return {"default_config": (None, [C.POINTER(cfg)]), "create": (ci, [C.POINTER(cfg), ci, i64, i64, C.POINTER(vp)]),
            "destroy": (ci, [vp]), "last_error": (C.c_char_p, [vp]), "num_envs": (i64, [vp]),
            "reset_seeded": (ci, [vp, u64, vp, vp, vp]), "reset_ics": (ci, [vp] * 5), "reset_init": (ci, [vp] * 4),
            "get_ics": (ci, [vp] * 3), "state_dims": (ci, [vp, C.POINTER(i32), C.POINTER(i32)]),
            "get_state": (ci, [vp] * 4), "set_state": (ci, [vp] * 4), "state_field": (ci, [C.c_char_p, C.POINTER(i32)]),
            "episode_stats": (ci, [vp, vp]), "launch_count": (i64, [vp]), "flops_per_step": (C.c_double, [vp]),
            "set_ic_pool": (ci, [vp, ci, vp, ci]), "get_ic_rows": (ci, [vp] * 3),
            "snapshot_width": (ci, [vp]), "snapshot": (ci, [vp, i64, vp, vp, vp]), "restore": (ci, [vp, i64, vp, vp, vp, vp])}


def batch_abi(prefix):
    """The shared entry points of one batch ("bskenv_" or "bskenv_opnav_"), by their names without the prefix."""
    L = lib()
    return types.SimpleNamespace(**{name: getattr(L, prefix + name) for name in _shared_signatures(Config)})


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
    vp, ci = C.c_void_p, C.c_int
    for prefix, cfg in BATCHES.items():
        for name, (res, args) in _shared_signatures(cfg).items():
            f = getattr(L, prefix + name)
            f.restype, f.argtypes = res, args
    L.bskenv_abi_version.restype = ci
    L.bskenv_step.argtypes = [vp] * 8
    L.bskenv_step_host.argtypes = [vp] * 6
    L.bskenv_step_info.argtypes = [vp] * 10
    L.bskenv_step_host_async.argtypes = [vp] * 9
    L.bskenv_step_host_wait.argtypes = [vp]
    L.bskenv_alloc_host.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.bskenv_free_host.argtypes = [vp]
    L.bskenv_kernel_name.restype = C.c_char_p
    L.bskenv_kernel_name.argtypes = [vp]
    L.bskenv_set_organisation.argtypes = [vp, ci]
    L.bskenv_set_param_pool.argtypes = [vp, ci, vp, ci]
    L.bskenv_get_env_params.argtypes = [vp, vp, vp, vp]
    L.bskenv_fp64_peak.argtypes = [ci, C.c_double, C.POINTER(C.c_double)]
    L.bskenv_set_ephemeris.argtypes = [vp, ci, C.c_double, C.c_double, ci, ci, vp]
    L.bskenv_set_gravity_degree2.argtypes = [vp, ci, vp]
    L.bskenv_opnav_step.argtypes = [vp] * 9
    L.bskenv_opnav_step_host.argtypes = [vp] * 7
    L.bskenv_opnav_step_info.argtypes = [vp] * 11
    L.bskenv_opnav_set_ephemeris.argtypes = [vp, C.c_double, C.c_double, ci, ci, vp]
    if L.bskenv_abi_version() != 1:
        raise RuntimeError("libbskenv.so ABI version mismatch")
    _LIB = L
    return L


def batch_config(prefix, **overrides):
    cfg = BATCHES[prefix]()
    getattr(lib(), prefix + "default_config")(C.byref(cfg))
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise AttributeError(f"{prefix}config has no field {k!r}")
        if isinstance(v, (list, tuple)):
            v = (C.c_double * len(v))(*v)
        setattr(cfg, k, v)
    return cfg


def batch_state_field(prefix, name):
    is_int = C.c_int32(0)
    idx = getattr(lib(), prefix + "state_field")(name.encode(), C.byref(is_int))
    if idx < 0:
        raise KeyError(name)
    return idx, bool(is_int.value)


def default_config(**overrides):
    return batch_config("bskenv_", **overrides)


def state_field(name):
    return batch_state_field("bskenv_", name)


def opnav_default_config(**overrides):
    return batch_config("bskenv_opnav_", **overrides)


def opnav_state_field(name):
    return batch_state_field("bskenv_opnav_", name)
