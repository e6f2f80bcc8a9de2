"""ctypes binding of the CPU oracle (oracle/bsk_oracle.c).

TEST INFRASTRUCTURE ONLY -- PARITY UNPINNED (Basilisk is not available; see bsk_oracle.h).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
Also holds the numpy restatement of the reference's initial-condition sampling
(/root/reference/basilisk_env/simulators/leoPowerAttitudeSimulator.py:119-193 and its helpers).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class LeoIC(C.Structure):
    _fields_ = [("rN", C.c_double * 3), ("vN", C.c_double * 3), ("sigma_init", C.c_double * 3),
                ("omega_init", C.c_double * 3), ("disturbance_vector", C.c_double * 3),
                ("wheelSpeeds_rpm", C.c_double * 3), ("storedCharge_Init", C.c_double)]


class LeoCfg(C.Structure):
    _fields_ = [("dynRate", C.c_double), ("fswRate", C.c_double), ("step_duration", C.c_double),
                ("use_j2", C.c_int), ("hill_cel_pun", C.c_int), ("rw_set", C.c_int), ("grav_pfix", C.c_int),
                ("reserved", C.c_int * 4)]


class LeoState(C.Structure):
    _fields_ = [("r_BN_N", C.c_double * 3), ("v_BN_N", C.c_double * 3), ("sigma_BN", C.c_double * 3),
                ("omega_BN_B", C.c_double * 3), ("Omega", C.c_double * 4), ("u_current", C.c_double * 4),
                ("storedCharge", C.c_double), ("shadowFactor", C.c_double), ("density", C.c_double),
                ("sigma_BR", C.c_double * 3), ("omega_BR_B", C.c_double * 3), ("sigma_RN", C.c_double * 3),
                ("Lr", C.c_double * 3), ("thrOnCmd", C.c_double * 8), ("thrOnTimeRemaining", C.c_double * 8),
                ("deltaH", C.c_double * 3), ("sun_r", C.c_double * 3), ("sun_v", C.c_double * 3),
                ("mrp_switch_count", C.c_int64), ("thr_fire_count", C.c_int64 * 8),
                ("thr_factor_mask", C.c_int32), ("dump_counter", C.c_int32), ("init_request", C.c_int32),
                ("task_mask", C.c_int32), ("sim_nanos", C.c_uint64)]


class EnvOut(C.Structure):
    _fields_ = [("ob", C.c_double * 5), ("reward", C.c_double), ("done", C.c_int), ("reason", C.c_int)]


def build(force=False):
    so = os.path.join(_HERE, "libbsk_oracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("bsk_oracle.c", "bsk_oracle.h", "opnav_oracle.c", "opnav_oracle.h", "Makefile")]
    if force or not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(f) for f in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def build_fast():
    """The same sources as an optimised host build (-O3 -march=native, contraction allowed): bench.py's second CPU
    baseline.  -march=native ties the binary to the CPU it was compiled on, so it is built where it runs.  It goes to a
    per-user temporary directory, not into the tree (the benchmark may run from a read-only checkout), under a name
    derived from that CPU's model and flags and from the sources."""
    import hashlib
    import tempfile
    try:
        info = open("/proc/cpuinfo").read()
        key = "".join(l for l in info.splitlines()[:40] if l.startswith(("model name", "flags")))
    except OSError:
        key = "unknown"
    h = hashlib.sha1(key.encode())
    for f in ("bsk_oracle.c", "bsk_oracle.h", "opnav_oracle.c", "opnav_oracle.h"):
        with open(os.path.join(_HERE, f), "rb") as fh:
            h.update(fh.read())
    d = os.path.join(tempfile.gettempdir(), f"bskenv_oracle_fast_{os.getuid()}")
    os.makedirs(d, mode=0o700, exist_ok=True)
    so = os.path.join(d, f"libbsk_oracle_fast_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call(["gcc", "-O3", "-march=native", "-fPIC", "-fopenmp", "-std=c99", "-shared", "-o", tmp,
                               os.path.join(_HERE, "bsk_oracle.c"), os.path.join(_HERE, "opnav_oracle.c"), "-lm"])
        os.replace(tmp, so)
    return so


FAST_FLAGS = "-O3 -march=native"
PARITY_FLAGS = "-O2 -ffp-contract=off"
_FAST = None


def fast_lib():
    global _FAST
    if _FAST is None:
        _FAST = _bind(C.CDLL(build_fast()))
    return _FAST


def lib():
    global _LIB
    if _LIB is None:
        _LIB = _bind(C.CDLL(build()))
    return _LIB


def _bind(L):
    if True:
        L.orc_leo_default_cfg.argtypes = [C.POINTER(LeoCfg)]
        L.orc_leo_create.restype = C.c_void_p
        L.orc_leo_create.argtypes = [C.POINTER(LeoIC), C.POINTER(LeoCfg)]
        L.orc_leo_destroy.argtypes = [C.c_void_p]
        L.orc_leo_run_sim.restype = C.c_int
        L.orc_leo_run_sim.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
        L.orc_leo_initial_obs.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.orc_leo_get_state.argtypes = [C.c_void_p, C.POINTER(LeoState)]
        L.orc_env_create.restype = C.c_void_p
        L.orc_env_create.argtypes = [C.POINTER(LeoCfg)]
        L.orc_env_destroy.argtypes = [C.c_void_p]
        L.orc_env_reset.argtypes = [C.c_void_p, C.POINTER(LeoIC), C.POINTER(C.c_double)]
        L.orc_env_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(EnvOut)]
        L.orc_env_sim.restype = C.c_void_p
        L.orc_env_sim.argtypes = [C.c_void_p]
        L.orc_env_set_max_length.argtypes = [C.c_void_p, C.c_int]
        L.orc_env_episode.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.orc_env_step_batch.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_int), C.POINTER(EnvOut), C.c_int]
        L.orc_max_threads.restype = C.c_int
        L.orc_elem2rv.argtypes = [C.c_double] * 7 + [C.POINTER(C.c_double)] * 2
        L.orc_sun_ephemeris.argtypes = [C.c_double] + [C.POINTER(C.c_double)] * 3
        dp = C.POINTER(C.c_double)
        L.orc_set_ephemeris.argtypes = [C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, dp]
        L.orc_eph_eval.argtypes = [C.c_int, C.c_double, dp, dp]
        L.orc_set_gravity_coeffs.argtypes = [dp]
        L.orc_earth_orientation.argtypes = [C.c_double, dp, dp]
        L.orc_grav_degree2_pfix.argtypes = [C.c_double, C.c_double, dp, dp, dp]
        L.orc_eclipse_shadow.restype = C.c_double
        L.orc_eclipse_shadow.argtypes = [C.POINTER(C.c_double)] * 3 + [C.c_double]
        L.orc_MRP2C.argtypes = [C.POINTER(C.c_double)] * 2
        L.orc_C2MRP.argtypes = [C.POINTER(C.c_double)] * 2
        L.orc_subMRP.argtypes = [C.POINTER(C.c_double)] * 3
        L.orc_addMRP.argtypes = [C.POINTER(C.c_double)] * 3
        L.orc_thr_force_mapping.argtypes = [C.POINTER(C.c_double)] * 3
    return L


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def default_cfg(**kw):
    cfg = LeoCfg()
    lib().orc_leo_default_cfg(C.byref(cfg))
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


# --------------------------------------------------------------------------------------------------
# IC sampling: numpy restatement of the reference's draw order (SURVEY 8a R3):
#   leo_orbit.sampled_400km  (initial_conditions/leo_orbit.py:25-39): e, i, Omega, omega, f
#   sc_attitudes.random_tumble (initial_conditions/sc_attitudes.py:3-13): sigma(3), omega(3)
#   set_ICs (simulators/leoPowerAttitudeSimulator.py:152,155,167): N(0,1)^3, U(-800,800)^3, U(8,20)*3600
#   balancedHR16Triad(useRandom=True) (actuatorPrimatives.py:18): 3 discarded U(-800,800)
# --------------------------------------------------------------------------------------------------
MU_EARTH = 0.3986004415e15
D2R = np.pi / 180.0


def elem2rv(mu, a, e, i, Omega, omega, f):
    r = np.zeros(3)
    v = np.zeros(3)
    lib().orc_elem2rv(mu, a, e, i, Omega, omega, f, _p(r), _p(v))
    return r, v


def sample_ic_dict(rng=None):
    """Draws one IC set from numpy's (legacy, global by default) RNG in the reference's order."""
    R = np.random if rng is None else rng
    a = 6371 * 1000.0 + 500. * 1000
    e = R.uniform(0, 0.05, 1)
    i = R.uniform(-90 * D2R, 90 * D2R, 1)
    Omega = R.uniform(0 * D2R, 360 * D2R, 1)
    omega = R.uniform(0 * D2R, 360 * D2R, 1)
    f = R.uniform(0 * D2R, 360 * D2R, 1)
    rN, vN = elem2rv(MU_EARTH, a, float(e[0]), float(i[0]), float(Omega[0]), float(omega[0]), float(f[0]))
    sigma = R.uniform(0, 1.0, [3, ])
    omega_bn = R.uniform(-0.00001, 0.00001, [3, ])
    dist = R.standard_normal(3)
    wheels = R.uniform(-800, 800, 3)
    charge = R.uniform(8. * 3600., 20. * 3600., 1)[0]
    R.uniform(-800, 800, 3)  # discarded by balancedHR16Triad
    return dict(oe=dict(a=a, e=float(e[0]), i=float(i[0]), Omega=float(Omega[0]), omega=float(omega[0]), f=float(f[0])),
                rN=rN, vN=vN, sigma_init=sigma, omega_init=omega_bn, disturbance_vector=dist,
                wheelSpeeds=wheels, storedCharge_Init=float(charge))


def ic_from_dict(d):
    ic = LeoIC()
    for k_c, k_d in (("rN", "rN"), ("vN", "vN"), ("sigma_init", "sigma_init"), ("omega_init", "omega_init"),
                     ("disturbance_vector", "disturbance_vector"), ("wheelSpeeds_rpm", "wheelSpeeds")):
        arr = np.asarray(d[k_d], dtype=np.float64).reshape(3)
        setattr(ic, k_c, (C.c_double * 3)(*arr))
    ic.storedCharge_Init = float(d["storedCharge_Init"])
    return ic


def ic_from_row(row):
    """row: 19 doubles [r3 v3 sigma3 omega3 dist3 wheels_rpm3 charge] (the C-ABI's IC layout)."""
    row = np.asarray(row, dtype=np.float64)
    return ic_from_dict(dict(rN=row[0:3], vN=row[3:6], sigma_init=row[6:9], omega_init=row[9:12],
                             disturbance_vector=row[12:15], wheelSpeeds=row[15:18], storedCharge_Init=row[18]))


def ic_to_row(d):
    return np.concatenate([np.asarray(d["rN"], float).reshape(3), np.asarray(d["vN"], float).reshape(3),
                           np.asarray(d["sigma_init"], float).reshape(3), np.asarray(d["omega_init"], float).reshape(3),
                           np.asarray(d["disturbance_vector"], float).reshape(3),
                           np.asarray(d["wheelSpeeds"], float).reshape(3), [float(d["storedCharge_Init"])]])


class LeoSim:
    """One scalar oracle sim == one LEOPowerAttitudeSimulator(0.1, 1.0, 180., ics)."""

    def __init__(self, ic, cfg=None):
        self._L = lib()
        self.cfg = cfg if cfg is not None else default_cfg()
        self.ic = ic if isinstance(ic, LeoIC) else (ic_from_dict(ic) if isinstance(ic, dict) else ic_from_row(ic))
        self._h = self._L.orc_leo_create(C.byref(self.ic), C.byref(self.cfg))

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.orc_leo_destroy(self._h)
            self._h = None

    def initial_obs(self):
        o = np.zeros(5)
        self._L.orc_leo_initial_obs(self._h, _p(o))
        return o

    def run_sim(self, action):
        o = np.zeros(5)
        over = self._L.orc_leo_run_sim(self._h, int(action), _p(o))
        return o, bool(over)

    def state(self):
        st = LeoState()
        self._L.orc_leo_get_state(self._h, C.byref(st))
        return st


class LeoEnv:
    """Oracle restatement of leoPowerAttEnv.reset/step for one env."""

    def __init__(self, cfg=None, max_length=None, L=None):
        self._L = L if L is not None else lib()
        self.cfg = cfg if cfg is not None else default_cfg()
        self._h = self._L.orc_env_create(C.byref(self.cfg))
        if max_length is not None:
            self._L.orc_env_set_max_length(self._h, int(max_length))

    def episode(self):
        """(reward_total, curr_step) as the reference puts them into info['episode'] (ENV:130-136)."""
        r, l = C.c_double(0.0), C.c_int(0)
        self._L.orc_env_episode(self._h, C.byref(r), C.byref(l))
        return r.value, l.value

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.orc_env_destroy(self._h)
            self._h = None

    def reset(self, ic):
        ic = ic if isinstance(ic, LeoIC) else (ic_from_dict(ic) if isinstance(ic, dict) else ic_from_row(ic))
        ob = np.zeros(5)
        self._L.orc_env_reset(self._h, C.byref(ic), _p(ob))
        return ob

    def step(self, action):
        out = EnvOut()
        self._L.orc_env_step(self._h, int(action), C.byref(out))
        return np.array(out.ob[:]), out.reward, bool(out.done), out.reason

    def state(self):
        st = LeoState()
        self._L.orc_leo_get_state(self._L.orc_env_sim(self._h), C.byref(st))
        return st


class LeoEnvBatch:
    """n independent oracle envs stepped with OpenMP over envs (the CPU baseline)."""

    def __init__(self, ic_rows, cfg=None, max_length=None, L=None):
        self._L = L if L is not None else lib()
        self.cfg = cfg if cfg is not None else default_cfg()
        self.n = len(ic_rows)
        self.envs = [LeoEnv(self.cfg, max_length, self._L) for _ in range(self.n)]
        self.obs0 = np.stack([e.reset(r) for e, r in zip(self.envs, ic_rows)])
        self._handles = (C.c_void_p * self.n)(*[e._h for e in self.envs])
        self._outs = (EnvOut * self.n)()

    def step(self, actions, nthreads=0):
        acts = (C.c_int * self.n)(*[int(a) for a in actions])
        self._L.orc_env_step_batch(self._handles, self.n, acts, self._outs, int(nthreads))
        ob = np.array([o.ob[:] for o in self._outs])
        rew = np.array([o.reward for o in self._outs])
        done = np.array([o.done for o in self._outs], dtype=bool)
        reason = np.array([o.reason for o in self._outs], dtype=np.int32)
        return ob, rew, done, reason


# ---- SURVEY 8(f)-4: ephemeris tables and planet-fixed degree-2 field (process-global settings of the oracle) ----
GGM03S_CBAR = np.array([-4.8416537173459064e-04, -2.0661550900e-10, 1.3844138138e-09, 2.4393836573e-06, -1.4002737040e-06])


def set_ephemeris(kind, table):
    """kind 0: Sun position rel. Earth [m]; 1: Earth RA, DEC, W [rad].  table: object with t0, seg_len, coef[nseg,3,ncoef]; None unloads."""
    if table is None:
        assert lib().orc_set_ephemeris(kind, 0.0, 0.0, 0, 0, None) == 0
        return
    coef = np.ascontiguousarray(table.coef, dtype=np.float64)
    assert lib().orc_set_ephemeris(kind, float(table.t0), float(table.seg_len), coef.shape[0], coef.shape[2], _p(coef)) == 0


def eph_eval(kind, t):
    v, r = np.zeros(3), np.zeros(3)
    assert lib().orc_eph_eval(kind, float(t), _p(v), _p(r)) == 0
    return v, r


def set_gravity_coeffs(cbar=None):
    c = np.ascontiguousarray(GGM03S_CBAR if cbar is None else cbar, dtype=np.float64)
    lib().orc_set_gravity_coeffs(_p(c))


def earth_orientation(t):
    P, Pd = np.zeros((3, 3)), np.zeros((3, 3))
    lib().orc_earth_orientation(float(t), _p(P), _p(Pd))
    return P, Pd


def grav_degree2_pfix(cbar, pos, mu=MU_EARTH, req=6378136.6):
    c = np.ascontiguousarray(cbar, dtype=np.float64); r = np.ascontiguousarray(pos, dtype=np.float64); a = np.zeros(3)
    lib().orc_grav_degree2_pfix(mu, req, _p(c), _p(r), _p(a))
    return a


def max_threads():
    return lib().orc_max_threads()
