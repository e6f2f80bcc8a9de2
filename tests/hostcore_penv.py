"""TEST INFRASTRUCTURE: ctypes binding of tests/hostcore/hostcore_penv.cpp, the device core compiled for the host with the
per-env parameter policy of the parameter-pool kernel (g++ -ffp-contract=off, as tests/hostcore_binding.py)."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.hostcore_binding import default_config

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcore")
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "libhostcore_penv.so")
    deps = [os.path.join(_HERE, "hostcore_penv.cpp")] + [os.path.join(_ROOT, "basilisk_env_b200", "csrc", f)
                                                         for f in ("leo_core.cuh", "leo_params.h", "leo_host.h", "leo_f32.cuh")]
    deps.append(os.path.join(_ROOT, "include", "bskenv.h"))
    if force or not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=c++17", "-Wno-unknown-pragmas",
                               "-o", so, deps[0]])
    return so


def lib():
    global _LIB
    if _LIB is None:
        from basilisk_env_b200._native import Config
        L = C.CDLL(build())
        vp = C.c_void_p
        L.hcp_create.restype = vp
        L.hcp_create.argtypes = [C.POINTER(Config), C.c_int64]
        L.hcp_destroy.argtypes = [vp]
        L.hcp_error.restype = C.c_char_p
        L.hcp_error.argtypes = [vp]
        L.hcp_set_env_params.argtypes = [vp, vp]
        L.hcp_reset_ics.argtypes = [vp, vp, vp]
        L.hcp_step.argtypes = [vp, C.c_int] + [vp] * 5
        L.hcp_get_state.argtypes = [vp, vp, vp]
        L.hcp_dims.argtypes = [C.POINTER(C.c_int)] * 3
        L.hcp_pool_row.restype = C.c_int64
        L.hcp_pool_row.argtypes = [C.c_int64, C.c_int, C.c_uint64, C.c_int64, C.c_int64]
        _LIB = L
    return _LIB


def pool_row(n_rows, assign, seed, global_env, episode):
    """The library's pool-row selection (leo::pool_row); assign 0 = by index, 1 = per episode."""
    return int(lib().hcp_pool_row(int(n_rows), int(assign), int(seed) & (2**64 - 1), int(global_env), int(episode)))


class HostCorePenv:
    """n envs of the reference configuration; `per_env` picks the per-env policy or the batch-global core."""

    def __init__(self, n, **kw):
        self.L = lib()
        self.n = n
        self.cfg = default_config(**kw)
        self.h = self.L.hcp_create(C.byref(self.cfg), n)
        assert self.h, "hcp_create rejected the configuration"
        nd, ni, npd = C.c_int(), C.c_int(), C.c_int()
        self.L.hcp_dims(C.byref(nd), C.byref(ni), C.byref(npd))
        self.nd, self.ni = nd.value, ni.value

    def __del__(self):
        if getattr(self, "h", None):
            self.L.hcp_destroy(self.h)
            self.h = None

    def set_env_params(self, raw):
        raw = np.ascontiguousarray(raw, dtype=np.float64)
        assert raw.shape == (self.n, 14)
        if self.L.hcp_set_env_params(self.h, raw.ctypes.data) != 0:
            raise ValueError(self.L.hcp_error(self.h).decode())

    def reset_ics(self, rows):
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        obs = np.zeros((self.n, 5))
        self.L.hcp_reset_ics(self.h, rows.ctypes.data, obs.ctypes.data)
        return obs

    def step(self, actions, per_env=True):
        a = np.ascontiguousarray(actions, dtype=np.int32)
        obs = np.zeros((self.n, 5)); rew = np.zeros(self.n)
        done = np.zeros(self.n, np.uint8); reason = np.zeros(self.n, np.uint8)
        self.L.hcp_step(self.h, int(per_env), a.ctypes.data, obs.ctypes.data, rew.ctypes.data, done.ctypes.data, reason.ctypes.data)
        return obs, rew, done.astype(bool), reason.astype(np.int32)

    def state(self):
        S = np.zeros((self.nd, self.n)); I = np.zeros((self.ni, self.n), np.int64)
        self.L.hcp_get_state(self.h, S.ctypes.data, I.ctypes.data)
        return S, I
