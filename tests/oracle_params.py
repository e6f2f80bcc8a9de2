"""TEST INFRASTRUCTURE: the CPU oracle with per-sim spacecraft parameters (tests/oracle_params/oracle_params.c, which
includes oracle/bsk_oracle.c unchanged and adds orc_leo_set_params / orc_env_reset_params).  The reference for the
per-env parameter pools of the library (LeoPowerAttVecEnv.set_param_pool)."""
import ctypes as C
import os
import subprocess

import numpy as np

from basilisk_env_b200.initial_conditions import PARAM_KEYS
from oracle import oracle as orc

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_params")
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIB = None
PARAM_DIM = 14
# the reference's values (simulators/leoPowerAttitudeSimulator.py:129-190) in BSKENV_PARAM_DIM order
DEFAULT_ROW = np.array([330, 1.38, 1.04, 1.58, 1.22, 8e3, 2e-4, 0.2 * 0.3, 0.20, -5.0, 20.0 * 3600., 7, 35, 4.])


def dispersed_pool(k, seed):
    """k Monte Carlo rows around the reference spacecraft: mass +-20 %, dimensions +-10 %, baseDensity x0.5..2 (log-uniform),
    scaleHeight +-10 %, disturbance, power system and gains +-20 %."""
    rng = np.random.RandomState(seed)
    rel = np.array([0.2, 0.1, 0.1, 0.1, 0.0, 0.1, 0.2, 0.2, 0.2, 0.2, 0.2, 0.2, 0.2, 0.2])
    rows = DEFAULT_ROW * (1.0 + rel * rng.uniform(-1.0, 1.0, size=(k, PARAM_DIM)))
    rows[:, 4] = DEFAULT_ROW[4] * 2.0 ** rng.uniform(-1.0, 1.0, size=k)
    return rows


def build(force=False):
    so = os.path.join(_HERE, "liboracle_params.so")
    deps = [os.path.join(_HERE, "oracle_params.c")] + [os.path.join(_ROOT, "oracle", f) for f in ("bsk_oracle.c", "bsk_oracle.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-std=c99", "-shared", "-o", so, deps[0], "-lm"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = orc._bind(C.CDLL(build()))
        dp = C.POINTER(C.c_double)
        L.orc_leo_set_params.argtypes = [C.c_void_p, dp]
        L.orc_env_reset_params.argtypes = [C.c_void_p, C.POINTER(orc.LeoIC), dp, dp]
        _LIB = L
    return _LIB


class LeoEnvParams(orc.LeoEnv):
    """One oracle env whose sim is rebuilt with its own parameter row at every reset."""

    def __init__(self, params, cfg=None, max_length=None):
        super().__init__(cfg, max_length, L=lib())
        self.params = np.ascontiguousarray(params, dtype=np.float64).reshape(PARAM_DIM)

    def reset(self, ic):
        ic = ic if isinstance(ic, orc.LeoIC) else (orc.ic_from_dict(ic) if isinstance(ic, dict) else orc.ic_from_row(ic))
        ob = np.zeros(5)
        self._L.orc_env_reset_params(self._h, C.byref(ic), orc._p(self.params), orc._p(ob))
        return ob


class LeoEnvBatchParams:
    """n oracle envs, env i built with ic_rows[i] and params[i] ([n, 14] in BSKENV_PARAM_DIM order)."""

    def __init__(self, ic_rows, params, cfg=None, max_length=None):
        self.envs = [LeoEnvParams(p, cfg, max_length) for p in np.asarray(params, dtype=np.float64)]
        self.obs0 = np.stack([e.reset(r) for e, r in zip(self.envs, ic_rows)])

    def step(self, actions):
        outs = [e.step(a) for e, a in zip(self.envs, actions)]
        return (np.stack([o[0] for o in outs]), np.array([o[1] for o in outs]), np.array([o[2] for o in outs], dtype=bool),
                np.array([o[3] for o in outs], dtype=np.int32))

    def states(self):
        return [e.state() for e in self.envs]
