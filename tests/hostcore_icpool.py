"""TEST INFRASTRUCTURE: ctypes binding of tests/hostcore/hostcore_icpool.cpp, the initial-condition pool pieces of the device
core compiled for the host (g++ -ffp-contract=off, as tests/hostcore_binding.py)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcore")
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "libhostcore_icpool.so")
    deps = [os.path.join(_HERE, "hostcore_icpool.cpp")] + [os.path.join(_ROOT, "basilisk_env_b200", "csrc", f)
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
        i64, u64 = C.c_int64, C.c_uint64
        L.hci_ic_pool_row.restype = i64
        L.hci_ic_pool_row.argtypes = [i64, C.c_int, u64, i64, i64, i64]
        L.hci_param_pool_row.restype = i64
        L.hci_param_pool_row.argtypes = [i64, C.c_int, u64, i64, i64]
        L.hci_sample_ic.argtypes = [C.POINTER(Config), u64, i64, i64, C.c_void_p]
        L.hci_ic_row_check.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int]
        _LIB = L
    return _LIB


def ic_pool_row(n_rows, assign, seed, global_env, episode, param_row=-1):
    """The library's IC-pool row selection (leo::ic_pool_row); assign 0 = by index, 1 = per episode, 2 = parameter row."""
    return int(lib().hci_ic_pool_row(int(n_rows), int(assign), int(seed) & (2**64 - 1), int(global_env), int(episode),
                                     int(param_row)))


def param_pool_row(n_rows, assign, seed, global_env, episode):
    return int(lib().hci_param_pool_row(int(n_rows), int(assign), int(seed) & (2**64 - 1), int(global_env), int(episode)))


def sample_ic(cfg, seed, global_env, episode):
    out = np.zeros(19)
    assert lib().hci_sample_ic(C.byref(cfg), int(seed) & (2**64 - 1), int(global_env), int(episode), out.ctypes.data) == 0
    return out


def ic_row_check(row):
    """"" for a row the library accepts, else its message."""
    row = np.ascontiguousarray(row, dtype=np.float64)
    buf = C.create_string_buffer(256)
    rc = lib().hci_ic_row_check(row.ctypes.data, row.size, buf, 256)
    return "" if rc == 0 else buf.value.decode()
