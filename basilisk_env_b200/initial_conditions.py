"""Host-side initial-condition sampling in the reference's draw order ("legacy-stream" mode).

The reference samples every episode's initial conditions from numpy's GLOBAL legacy RNG
(SURVEY.md quirk Q8) in this order:
  1. `leo_orbit.sampled_400km()`   /root/reference/basilisk_env/simulators/initial_conditions/leo_orbit.py:25-39
       e, i, Omega, omega, f  -- five `uniform(lo, hi, 1)` draws, then `orbitalMotion.elem2rv`
  2. `sc_attitudes.random_tumble(maxSpinRate=1e-5)`   .../initial_conditions/sc_attitudes.py:3-13
       sigma ~ U(0,1)^3, omega ~ U(-1e-5, 1e-5)^3
  3. `set_ICs` dict literal   /root/reference/basilisk_env/simulators/leoPowerAttitudeSimulator.py:152,155,167
       disturbance_vector ~ N(0,1)^3, wheelSpeeds ~ U(-800,800)^3 RPM, storedCharge_Init ~ U(8,20) Wh
  4. `balancedHR16Triad(useRandom=True)`   .../dynamics/effectorPrimatives/actuatorPrimatives.py:18
       three U(-800,800) draws that are thrown away (the wheel speeds are overwritten at :303-305)
so `np.random.seed(s); env.reset()` here consumes the global stream exactly like the reference would.

The vectorised environment does NOT use this module on its hot path: it samples on the device with a
counter-based generator keyed by (seed, global env index, episode) -- same distributions, different
stream (csrc/leo_core.cuh `sample_ic`)."""
import numpy as np

D2R = np.pi / 180.0                    # Basilisk macros.D2R
RPM = 0.10471975511965977              # Basilisk macros.RPM  (2*pi/60)
MU_EARTH = 0.3986004415E+15            # leo_orbit.py:30
REQ_EARTH = 6378.1366                  # Basilisk orbitalMotion.REQ_EARTH [km]
IC_DIM = 19                            # include/bskenv.h BSKENV_IC_DIM


class ClassicElements:
    """Stand-in for Basilisk `orbitalMotion.ClassicElements` (a, e, i, Omega, omega, f)."""

    def __init__(self, a=0.0, e=0.0, i=0.0, Omega=0.0, omega=0.0, f=0.0):
        self.a, self.e, self.i, self.Omega, self.omega, self.f = a, e, i, Omega, omega, f


def elem2rv(mu, elements):
    """Classical elements -> inertial position/velocity (Basilisk `orbitalMotion.elem2rv`, the
    non-rectilinear branch, which is the only one `sampled_400km` can reach: a > 0, e < 1)."""
    a, e, i = float(elements.a), float(np.ravel(elements.e)[0]), float(np.ravel(elements.i)[0])
    AN, AP, f = float(np.ravel(elements.Omega)[0]), float(np.ravel(elements.omega)[0]), float(np.ravel(elements.f)[0])
    if not (a > 0.0 and 0.0 <= e < 1.0):
        raise ValueError("elem2rv: only bound, non-rectilinear orbits are on the reference path")
    p = a * (1.0 - e * e)
    r = p / (1.0 + e * np.cos(f))
    theta = AP + f
    rVec = np.zeros(3)
    rVec[0] = r * (np.cos(theta) * np.cos(AN) - np.cos(i) * np.sin(theta) * np.sin(AN))
    rVec[1] = r * (np.cos(theta) * np.sin(AN) + np.cos(i) * np.sin(theta) * np.cos(AN))
    rVec[2] = r * (np.sin(theta) * np.sin(i))
    h = np.sqrt(mu * p)
    vVec = np.zeros(3)
    vVec[0] = -mu / h * (np.cos(AN) * (e * np.sin(AP) + np.sin(theta)) + np.cos(i) * (e * np.cos(AP) + np.cos(theta)) * np.sin(AN))
    vVec[1] = -mu / h * (np.sin(AN) * (e * np.sin(AP) + np.sin(theta)) - np.cos(i) * (e * np.cos(AP) + np.cos(theta)) * np.cos(AN))
    vVec[2] = mu / h * (e * np.cos(AP) + np.cos(theta)) * np.sin(i)
    return rVec, vVec


def sampled_400km(rng=None):
    """leo_orbit.py:25-39.  (The name says 400 km; the code uses 6371 km + 500 km -- quirk Q11.)"""
    R = np.random if rng is None else rng
    oe = ClassicElements()
    oe.a = 6371 * 1000.0 + 500. * 1000
    oe.e = R.uniform(0, 0.05, 1)
    oe.i = R.uniform(-90 * D2R, 90 * D2R, 1)
    oe.Omega = R.uniform(0 * D2R, 360 * D2R, 1)
    oe.omega = R.uniform(0 * D2R, 360 * D2R, 1)
    oe.f = R.uniform(0 * D2R, 360 * D2R, 1)
    rN, vN = elem2rv(MU_EARTH, oe)
    return oe, rN, vN


def inclined_circular_300km():
    """leo_orbit.py:6-23 (not used by the reference env, kept for API parity): circular, i = 45 deg, 300 km."""
    oe = ClassicElements(a=6371 * 1000.0 + 300. * 1000, e=0.0, i=45.0 * D2R, Omega=0.0 * D2R, omega=0.0 * D2R, f=0.0 * D2R)
    rN, vN = elem2rv(MU_EARTH, oe)
    return oe, rN, vN


def static_inertial():
    """sc_attitudes.py:15-23 (not used by the reference env): zero MRP, zero body rate."""
    return np.zeros([3, ]), np.zeros([3, ])


def random_tumble(maxSpinRate=0.001, rng=None):
    """sc_attitudes.py:3-13."""
    R = np.random if rng is None else rng
    sigma_bn = R.uniform(0, 1.0, [3, ])
    omega_bn = R.uniform(-maxSpinRate, maxSpinRate, [3, ])
    return sigma_bn, omega_bn


def set_ICs(rng=None):
    """The `initial_conditions` dict of LEOPowerAttitudeSimulator.set_ICs (SIM:119-193), same keys."""
    R = np.random if rng is None else rng
    oe, rN, vN = sampled_400km(rng)
    sigma_init, omega_init = random_tumble(maxSpinRate=0.00001, rng=rng)
    ic = {
        "mass": 330,
        "oe": oe, "rN": rN, "vN": vN,
        "width": 1.38, "depth": 1.04, "height": 1.58,
        "sigma_init": sigma_init, "omega_init": omega_init,
        "planetRadius": REQ_EARTH * 1000., "baseDensity": 1.22, "scaleHeight": 8e3,
        "disturbance_magnitude": 2e-4,
        "disturbance_vector": R.standard_normal(3),
        "wheelSpeeds": R.uniform(-800, 800, 3),
        "nHat_B": np.array([0, -1, 0]), "panelArea": 0.2 * 0.3, "panelEfficiency": 0.20,
        "powerDraw": -5.0,
        "storageCapacity": 20.0 * 3600.,
        "storedCharge_Init": R.uniform(8. * 3600., 20. * 3600., 1)[0],
        "sigma_R0N": [1, 0, 0],
        "controlAxes_B": [1, 0, 0, 0, 1, 0, 0, 0, 1],
        "K": 7, "Ki": -1.0, "P": 35,
        "hs_min": 4.,
        "thrForceSign": 1,
        "maxCounterValue": 4, "thrMinFireTime": 0.002,
    }
    return ic


def consume_wheel_factory_draws(rng=None):
    """`balancedHR16Triad(useRandom=True, randomBounds=(-800,800))` draws three wheel speeds that
    set_dynamics immediately overwrites (SIM:301-305); the draws still advance the global stream."""
    R = np.random if rng is None else rng
    R.uniform(-800, 800, 3)


def ic_row(ic):
    """The 19 per-environment numbers of an `initial_conditions` dict in the C ABI's layout
    (include/bskenv.h BSKENV_IC_DIM): rN vN sigma_init omega_init disturbance_vector wheelSpeeds[RPM] storedCharge_Init."""
    return np.concatenate([np.asarray(ic["rN"], dtype=np.float64).reshape(3),
                           np.asarray(ic["vN"], dtype=np.float64).reshape(3),
                           np.asarray(ic["sigma_init"], dtype=np.float64).reshape(3),
                           np.asarray(ic["omega_init"], dtype=np.float64).reshape(3),
                           np.asarray(ic["disturbance_vector"], dtype=np.float64).reshape(3),
                           np.asarray(ic["wheelSpeeds"], dtype=np.float64).reshape(3),
                           np.asarray([ic["storedCharge_Init"]], dtype=np.float64)])


# keys of the initial_conditions dict that are batch-global configuration in the C ABI
# (bskenv_config); "controlAxes_B" must stay the identity and "mass".."height" set the inertia.
CONFIG_KEYS = ("mass", "width", "depth", "height", "planetRadius", "baseDensity", "scaleHeight",
               "disturbance_magnitude", "nHat_B", "panelArea", "panelEfficiency", "powerDraw",
               "storageCapacity", "sigma_R0N", "K", "Ki", "P", "hs_min", "thrForceSign",
               "maxCounterValue", "thrMinFireTime")


# keys of the initial_conditions dict that may differ from env to env through a parameter pool
# (LeoPowerAttVecEnv.set_param_pool, include/bskenv.h bskenv_set_param_pool), in the C ABI's row order (BSKENV_PARAM_DIM)
PARAM_KEYS = ("mass", "width", "depth", "height", "baseDensity", "scaleHeight", "disturbance_magnitude", "panelArea",
              "panelEfficiency", "powerDraw", "storageCapacity", "K", "P", "hs_min")


def scenario_rows(scenarios, config):
    """A scenario table from full reference `initial_conditions` dicts (the shape `set_ICs()` returns): (IC rows [K, 19],
    parameter rows [K, 14] in PARAM_KEYS order) for `LeoPowerAttVecEnv.set_scenario_pool`.
    config : the batch's configuration, a mapping of CONFIG_KEYS -> value; a PARAM_KEYS entry a dict leaves out takes its
        value from here.  A batch-global key (CONFIG_KEYS minus PARAM_KEYS) must equal it: ValueError names the key and the
        scenario index otherwise."""
    scenarios = list(scenarios)
    if not scenarios:
        raise ValueError("a scenario pool needs at least one scenario")
    ics, params = [], []
    for j, ic in enumerate(scenarios):
        for k in CONFIG_KEYS:
            if k in PARAM_KEYS or ic.get(k) is None:
                continue
            want = np.ravel(np.asarray(config[k], dtype=np.float64))
            got = np.ravel(np.asarray(ic[k], dtype=np.float64))
            if got.shape != want.shape or not np.array_equal(got, want):
                raise ValueError(f"scenario {j}: {k!r} = {got.tolist()} differs from the batch configuration {want.tolist()} "
                                 "(only the parameter-pool keys initial_conditions.PARAM_KEYS may differ per env)")
        axes = ic.get("controlAxes_B")
        if axes is not None and list(np.ravel(axes)) != [1, 0, 0, 0, 1, 0, 0, 0, 1]:
            raise ValueError(f"scenario {j}: controlAxes_B other than the identity is not on the reference path")
        ics.append(ic_row(ic))
        params.append([float(ic[k]) if ic.get(k) is not None else float(config[k]) for k in PARAM_KEYS])
    return np.stack(ics), np.asarray(params, dtype=np.float64)


def config_overrides(ic):
    """bskenv_config overrides carried by an `initial_conditions` dict."""
    out = {}
    for k in CONFIG_KEYS:
        if k in ic and ic[k] is not None:
            v = ic[k]
            out[k] = [float(x) for x in np.ravel(v)] if k in ("nHat_B", "sigma_R0N") else v
    axes = ic.get("controlAxes_B")
    if axes is not None and list(np.ravel(axes)) != [1, 0, 0, 0, 1, 0, 0, 0, 1]:
        raise ValueError("controlAxes_B other than the identity is not on the reference path")
    return out
