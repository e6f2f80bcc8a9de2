"""opNav environment: the dynamics half of the reference's opNav env plus a synthetic nav measurement
and the relative-OD filter, stepped by ONE CUDA launch per decision interval (no Vizard rendering).

Mirrors
  * `opNavEnv` (/root/reference/basilisk_env/envs/opNavEnvironment.py:11-177): Box(4,1) observations,
    Discrete(2) actions, 40 steps of 50 minutes, 4-tuple step return, `info` keys
    `full_states` / `obs` / `episode{r,l}`;
  * `scenario_OpNav` (/root/reference/basilisk_env/simulators/opNavSimulator.py:96-317):
    `run_sim(action) -> (obs(4,1), sim_states(12,1), sim_over)`, `.obs`, `.sim_states`, `.simTime`,
    `.modeCounter`, `close_gracefully()`;
over the C ABI `bskenv_opnav_*` of include/bskenv.h.  torch supplies device memory and streams only.
There is no CPU path: constructing any of these without a CUDA device raises."""
import ctypes as C

import numpy as np
import torch

from . import _native
from . import spaces
from .vec_env import BskEnvError, all_reduce_stats

OBS_DIM, DEBUG_DIM, IC_DIM = 4, 12, 12
DONE_MAXLEN, DONE_MODES = 1, 2
STAT_NAMES = ("return_sum", "length_sum", "episodes", "max_length_ends", "mode_limit_ends", "env_steps",
              "measurement_updates", "rejected_filter_updates")
MU_MARS = 4.2828371901284001E+13
D2R = np.pi / 180.0


def elem2rv(mu, a, e, i, Omega, omega, f):
    """orbitalMotion.elem2rv (non-rectilinear branch), as used at opNavSimulator.py:181."""
    p = a * (1.0 - e * e)
    r = p / (1.0 + e * np.cos(f))
    th = omega + f
    h = np.sqrt(mu * p)
    rN = np.array([r * (np.cos(th) * np.cos(Omega) - np.cos(i) * np.sin(th) * np.sin(Omega)),
                   r * (np.cos(th) * np.sin(Omega) + np.cos(i) * np.sin(th) * np.cos(Omega)),
                   r * (np.sin(th) * np.sin(i))])
    vN = np.array([-mu / h * (np.cos(Omega) * (e * np.sin(omega) + np.sin(th)) + np.cos(i) * (e * np.cos(omega) + np.cos(th)) * np.sin(Omega)),
                   -mu / h * (np.sin(Omega) * (e * np.sin(omega) + np.sin(th)) - np.cos(i) * (e * np.cos(omega) + np.cos(th)) * np.cos(Omega)),
                   mu / h * (e * np.cos(omega) + np.cos(th)) * np.sin(i)])
    return rN, vN


def configure_initial_conditions(rng=None):
    """One IC row [rN vN rError vError] drawn as `scenario_OpNav.configure_initial_conditions` draws it
    (opNavSimulator.py:163-189): fixed orbit, then uniform(100000,-100000,3) and uniform(1000,-1000,3) from
    numpy's global legacy stream."""
    R = np.random if rng is None else rng
    rN, vN = elem2rv(MU_MARS, 18000 * 1E3, 0.6, 10 * D2R, 25. * D2R, 190. * D2R, 80. * D2R)
    rError = R.uniform(100000, -100000, 3)
    vError = R.uniform(1000, -1000, 3)
    return np.concatenate([rN, vN, rError, vError])


class OpNavVecEnv:
    """N opNav environments on one GPU (see LeoPowerAttVecEnv for the conventions).

    **config : overrides of `bskenv_opnav_config` fields (include/bskenv.h), e.g. camera_reenable=1."""

    def __init__(self, num_envs, device=0, first_env_index=0, seed=0, auto_reset=False, **config):
        if not torch.cuda.is_available():
            raise BskEnvError("OpNavVecEnv needs a CUDA device: the environment step has no CPU path")
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if self.device.type != "cuda":
            raise BskEnvError("OpNavVecEnv needs a CUDA device: the environment step has no CPU path")
        self.num_envs = int(num_envs)
        self.first_env_index = int(first_env_index)
        self.seed_value = int(seed)
        self._L = _native.lib()
        config.setdefault("noise_seed", self.seed_value & (2**64 - 1))
        self.cfg = _native.opnav_default_config(auto_reset=int(bool(auto_reset)), **config)
        self.auto_reset = bool(auto_reset)
        h = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = self._L.bskenv_opnav_create(C.byref(self.cfg), dev_index, self.num_envs, self.first_env_index, C.byref(h))
        if rc != 0:
            raise BskEnvError(f"bskenv_opnav_create failed ({rc}): {self._L.bskenv_opnav_last_error(None).decode()}")
        self._h = h
        n = self.num_envs
        with torch.cuda.device(self.device):
            self.obs = torch.zeros((n, OBS_DIM), dtype=torch.float64, device=self.device)
            self.term_obs = torch.zeros((n, OBS_DIM), dtype=torch.float64, device=self.device)
            self.debug = torch.zeros((n, DEBUG_DIM), dtype=torch.float64, device=self.device)
            self.reward = torch.zeros(n, dtype=torch.float64, device=self.device)
            self.done = torch.zeros(n, dtype=torch.uint8, device=self.device)
            self.done_reason = torch.zeros(n, dtype=torch.uint8, device=self.device)
            self.episode_r = torch.zeros(n, dtype=torch.float64, device=self.device)
            self.episode_l = torch.zeros(n, dtype=torch.int64, device=self.device)
        self.observation_space = spaces.Box(-1e16, 1e16, shape=(OBS_DIM, 1))
        self.action_space = spaces.Discrete(2)
        self.max_length = int(self.cfg.max_length)
        self.step_duration = float(self.cfg.step_duration_min)
        nd, ni = C.c_int32(), C.c_int32()
        self._L.bskenv_opnav_state_dims(self._h, C.byref(nd), C.byref(ni))
        self.n_double_fields, self.n_int_fields = nd.value, ni.value

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.bskenv_opnav_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise BskEnvError(f"{what} failed ({rc}): {self._L.bskenv_opnav_last_error(self._h).decode()}")

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _mask_ptr(self, mask):
        if mask is None:
            return None, None
        m = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()
        if m.numel() != self.num_envs:
            raise ValueError("mask must have one entry per env")
        return m, C.c_void_p(m.data_ptr())

    def set_ephemeris(self, table):
        """SURVEY 8(f)-4: Sun position relative to the Mars barycentre [m] from a Chebyshev table
        (`basilisk_env_b200.ephemeris.ChebTable`; None = back to the analytic series).  Set before reset."""
        if table is None:
            self._check(self._L.bskenv_opnav_set_ephemeris(self._h, 0.0, 0.0, 0, 0, None), "set_ephemeris")
            return
        coef = np.ascontiguousarray(table.coef, dtype=np.float64)
        self._check(self._L.bskenv_opnav_set_ephemeris(self._h, float(table.t0), float(table.seg_len), coef.shape[0],
                                                       coef.shape[2], coef.ctypes.data), "set_ephemeris")

    def set_ic_pool(self, ics, assign="per_episode"):
        """Load a pool of initial conditions [K, 12] (rN vN rError vError) that `reset()` and the auto-reset of `step` draw
        from instead of the built-in sampler (include/bskenv.h: bskenv_opnav_set_ic_pool); None unloads it.
        assign : "per_episode" (row drawn per (seed, global env index, episode)) or "by_index" (global env index mod K)."""
        if ics is None:
            self._check(self._L.bskenv_opnav_set_ic_pool(self._h, 0, None, 0), "bskenv_opnav_set_ic_pool")
            return
        rows = ics.detach().cpu().numpy() if torch.is_tensor(ics) else ics
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        if rows.ndim != 2 or rows.shape[1] != IC_DIM or rows.shape[0] == 0:
            raise ValueError(f"ics must have shape (K, {IC_DIM}) with K > 0")
        self._check(self._L.bskenv_opnav_set_ic_pool(self._h, rows.shape[0], rows.ctypes.data, IC_ASSIGN[assign]),
                    "bskenv_opnav_set_ic_pool")

    def ic_rows(self):
        """The IC-pool row each env's current episode started from (int32 [N]; -1 = sampled or explicit ICs)."""
        row = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        self._check(self._L.bskenv_opnav_get_ic_rows(self._h, C.c_void_p(row.data_ptr()), self._stream()),
                    "bskenv_opnav_get_ic_rows")
        return row

    def reset(self, seed=None, mask=None):
        """Sample fresh initial conditions on the device; returns the initial observation [N,4] (zeros)."""
        if seed is not None:
            self.seed_value = int(seed)
        keep, mp = self._mask_ptr(mask)
        self._check(self._L.bskenv_opnav_reset_seeded(self._h, C.c_uint64(self.seed_value & (2**64 - 1)), mp,
                                                      C.c_void_p(self.obs.data_ptr()), self._stream()),
                    "bskenv_opnav_reset_seeded")
        del keep
        return self.obs

    def reset_ics(self, ics, mask=None):
        """Reset from explicit initial conditions: [N,12] rows [rN vN rError vError]."""
        t = torch.as_tensor(np.asarray(ics, dtype=np.float64) if not torch.is_tensor(ics) else ics)
        t = t.to(device=self.device, dtype=torch.float64).contiguous()
        if tuple(t.shape) != (self.num_envs, IC_DIM):
            raise ValueError(f"ics must have shape ({self.num_envs}, {IC_DIM})")
        keep, mp = self._mask_ptr(mask)
        self._check(self._L.bskenv_opnav_reset_ics(self._h, C.c_void_p(t.data_ptr()), mp, C.c_void_p(self.obs.data_ptr()),
                                                   self._stream()), "bskenv_opnav_reset_ics")
        torch.cuda.current_stream(self.device).synchronize()
        del keep
        return self.obs

    def reset_init(self, mask=None):
        keep, mp = self._mask_ptr(mask)
        self._check(self._L.bskenv_opnav_reset_init(self._h, mp, C.c_void_p(self.obs.data_ptr()), self._stream()),
                    "bskenv_opnav_reset_init")
        del keep
        return self.obs

    def initial_conditions(self):
        out = torch.empty((self.num_envs, IC_DIM), dtype=torch.float64, device=self.device)
        self._check(self._L.bskenv_opnav_get_ics(self._h, C.c_void_p(out.data_ptr()), self._stream()), "bskenv_opnav_get_ics")
        return out

    def step(self, actions):
        """actions: int32 CUDA tensor [N] (0 OpNav pointing + imaging / 1 sun-safe pointing).  Returns device tensors
        (obs [N,4], reward [N], done [N] u8, info) without synchronising."""
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions, dtype=np.int32))
        a = actions.to(device=self.device, dtype=torch.int32).contiguous()
        if a.numel() != self.num_envs:
            raise ValueError("one action per env")
        self._check(self._L.bskenv_opnav_step_info(self._h, C.c_void_p(a.data_ptr()), C.c_void_p(self.obs.data_ptr()),
                                                   C.c_void_p(self.reward.data_ptr()), C.c_void_p(self.done.data_ptr()),
                                                   C.c_void_p(self.done_reason.data_ptr()), C.c_void_p(self.debug.data_ptr()),
                                                   C.c_void_p(self.term_obs.data_ptr()), C.c_void_p(self.episode_r.data_ptr()),
                                                   C.c_void_p(self.episode_l.data_ptr()), self._stream()), "bskenv_opnav_step_info")
        self._last_actions = a
        # episode_r / episode_l: the reference's info['episode'] = {'r', 'l'} (opNavEnvironment.py:106-109) where done is set
        info = {"done_reason": self.done_reason, "terminal_obs": self.term_obs, "full_states": self.debug,
                "episode_r": self.episode_r, "episode_l": self.episode_l}
        return self.obs, self.reward, self.done, info

    def host_buffers(self):
        """Page-locked, device-mapped numpy buffers for `step_host`: (actions int32 [N], (obs [N,4], reward [N], done u8 [N],
        done_reason u8 [N], full_states [N,12])).  The second kernel of the step writes them in place (zero-copy over PCIe);
        ordinary numpy arrays work too, through staging and one memcpy each."""
        n = self.num_envs
        pin = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()     # noqa: E731
        return pin(n, torch.int32), (pin((n, OBS_DIM), torch.float64), pin(n, torch.float64), pin(n, torch.uint8),
                                     pin(n, torch.uint8), pin((n, DEBUG_DIM), torch.float64))

    def step_host(self, actions, out=None):
        """Host-buffer step: numpy int32 [N] in, numpy (obs, reward, done, done_reason, full_states) out."""
        a = actions if (isinstance(actions, np.ndarray) and actions.dtype == np.int32 and actions.flags.c_contiguous) \
            else np.ascontiguousarray(actions, dtype=np.int32)
        if a.size != self.num_envs:
            raise ValueError("one action per env")
        if out is None:
            out = (np.empty((self.num_envs, OBS_DIM)), np.empty(self.num_envs), np.empty(self.num_envs, np.uint8),
                   np.empty(self.num_envs, np.uint8), np.empty((self.num_envs, DEBUG_DIM)))
        obs, rew, done, reason, dbg = out
        self._check(self._L.bskenv_opnav_step_host(self._h, a.ctypes.data, obs.ctypes.data, rew.ctypes.data, done.ctypes.data,
                                                   reason.ctypes.data, dbg.ctypes.data if dbg is not None else None),
                    "bskenv_opnav_step_host")
        return obs, rew, done, reason, dbg

    def get_state(self):
        d = torch.empty((self.n_double_fields, self.num_envs), dtype=torch.float64, device=self.device)
        i = torch.empty((self.n_int_fields, self.num_envs), dtype=torch.int64, device=self.device)
        self._check(self._L.bskenv_opnav_get_state(self._h, C.c_void_p(d.data_ptr()), C.c_void_p(i.data_ptr()),
                                                   self._stream()), "bskenv_opnav_get_state")
        return d, i

    def set_state(self, dstate, istate):
        d = dstate.to(device=self.device, dtype=torch.float64).contiguous()
        i = istate.to(device=self.device, dtype=torch.int64).contiguous()
        if tuple(d.shape) != (self.n_double_fields, self.num_envs) or tuple(i.shape) != (self.n_int_fields, self.num_envs):
            raise ValueError("state blocks have the wrong shape")
        self._check(self._L.bskenv_opnav_set_state(self._h, C.c_void_p(d.data_ptr()), C.c_void_p(i.data_ptr()),
                                                   self._stream()), "bskenv_opnav_set_state")
        torch.cuda.current_stream(self.device).synchronize()

    def field(self, name, state=None):
        idx, is_int = _native.opnav_state_field(name)
        d, i = state if state is not None else self.get_state()
        return (i if is_int else d)[idx:idx + _FIELD_WIDTH.get(name, 1)]

    def episode_stats(self, all_reduce=False):
        buf = np.zeros(8)
        self._check(self._L.bskenv_opnav_episode_stats(self._h, buf.ctypes.data), "bskenv_opnav_episode_stats")
        if all_reduce:
            buf = all_reduce_stats(buf, self.device)
        return dict(zip(STAT_NAMES, (float(x) for x in buf)))

    def launch_count(self):
        return int(self._L.bskenv_opnav_launch_count(self._h))

    def flops_per_step(self):
        return float(self._L.bskenv_opnav_flops_per_step(self._h))


IC_ASSIGN = {"by_index": 0, "per_episode": 1}
_FIELD_WIDTH = {"r_BN_N": 3, "v_BN_N": 3, "sigma_BN": 3, "omega_BN_B": 3, "Omega": 4, "reactionwheel_cmds": 4,
                "navErrors": 15, "sun_point_data": 3, "filter_state": 6, "filter_sBar": 21, "sim_obs": 4, "sim_states": 12}


class scenario_OpNav:
    """One opNav simulation == one env of a 1-env CUDA batch (opNavSimulator.py:96-317)."""

    def __init__(self, dynRate, fswRate, step_duration, device=0, initial_conditions=None, **config):
        self.fswRate, self.dynRate, self.step_duration = fswRate, dynRate, step_duration
        self.filterUse = "relOD"
        row = configure_initial_conditions() if initial_conditions is None else np.asarray(initial_conditions, dtype=np.float64)
        self.initial_conditions = row
        config.setdefault("noise_seed", int(np.random.randint(0, 2**31 - 1)))
        config.setdefault("max_length", 2**31 - 1)          # episode bookkeeping lives in opNavEnv; keep the simulator free-running
        self._vec = OpNavVecEnv(1, device=device, dynRate=float(dynRate), fswRate=float(fswRate),
                                step_duration_min=float(step_duration), **config)
        self._vec.reset_ics(row[None, :])
        self.simTime = 0.0
        self.numModes = int(self._vec.cfg.numModes)
        self.modeCounter = 0
        self.obs = np.zeros([4, 1])
        self.sim_states = np.zeros([12, 1])
        self.sim_over = False
        self.modeRequest = 'OpNavOD'
        self._reward = 0.0

    def run_sim(self, action):
        """Mode switch, advance step_duration minutes, sample (opNavSimulator.py:225-299)."""
        self.modeCounter += 1
        code = {"0": 0, "1": 1}.get(str(action), -1)        # str(action) decoding as at :237, :249
        obs, rew, done, reason, dbg = self._vec.step_host(np.array([code], dtype=np.int32))
        self.simTime += self.step_duration
        self.obs = obs[0].reshape(4, 1).copy()
        self.sim_states = dbg[0].reshape(12, 1).copy()
        self.sim_over = bool(reason[0] & DONE_MODES)
        self._reward = float(rew[0])
        return self.obs, self.sim_states, self.sim_over

    def close_gracefully(self):
        if self._vec is not None:
            self._vec.close()
            self._vec = None


_GymEnv = spaces.gym_env_base()


class opNavEnv(_GymEnv):
    """OpNav scenario (opNavEnvironment.py:11-177): decide when to image Mars and when to point at the Sun."""

    def __init__(self, device=0, **config):
        self.__version__ = "0.0.2"
        self.max_length = int(40)
        self.sim_init = 0
        self.simulator = None
        self.reward_total = 0
        self.step_duration = 50.
        self.reward_mult = 1.
        self.observation_space = spaces.Box(-1e16, 1e16, shape=(4, 1))
        self.obs = np.zeros([4, ])
        self.debug_states = np.zeros([12, ])
        self.action_space = spaces.Discrete(2)
        self.curr_episode = -1
        self.action_episode_memory = []
        self.curr_step = 0
        self.episode_over = False
        self._device, self._config = device, dict(config)

    def _seed(self):
        np.random.seed()
        return

    def _new_simulator(self):
        return scenario_OpNav(1., 1., self.step_duration, device=self._device, **self._config)

    def step(self, action):
        if not self.action_episode_memory:
            raise BskEnvError("step() called before reset()")
        if self.sim_init == 0:
            self.simulator = self._new_simulator()
            self.sim_init = 1
        if self.curr_step >= self.max_length:
            self.episode_over = True
        self._take_action(action)
        reward = self._get_reward()
        self.reward_total += reward
        ob = self._get_state()
        if self.sim_over:
            self.episode_over = True
        if self.episode_over:
            info = {'episode': {'r': self.reward_total, 'l': self.curr_step}, 'full_states': self.debug_states, 'obs': ob}
            self.simulator.close_gracefully()
            self.sim_init = 0
        else:
            info = {'full_states': self.debug_states, 'obs': ob}
        self.curr_step += 1
        return ob, reward, self.episode_over, info

    def _take_action(self, action):
        self.action_episode_memory[self.curr_episode].append(action)
        self.obs, self.debug_states, self.sim_over = self.simulator.run_sim(action)

    def _get_reward(self):
        """opNavEnvironment.py:139-152 (the fused step evaluates the same expression on the device; it is repeated
        here on the sampled states so that a non-integer action compares as in the reference)."""
        reward = 0
        real = np.array([self.debug_states[3], self.debug_states[4], self.debug_states[5]]).reshape(3)
        nav = np.array([self.debug_states[0], self.debug_states[1], self.debug_states[2]]).reshape(3)
        nav = nav - real
        nav *= 1. / np.linalg.norm(real)
        if self.action_episode_memory[self.curr_episode][-1] == 1:
            reward = np.linalg.norm(self.reward_mult / (1. + np.linalg.norm(nav) ** 2.0))
        return reward

    def reset(self):
        self.action_episode_memory.append([])
        self.episode_over = False
        self.curr_step = 0
        self.reward_total = 0
        if self.simulator is not None:
            self.simulator.close_gracefully()
        self.simulator = self._new_simulator()
        self.sim_init = 1
        return self.simulator.obs

    def _render(self, mode='human', close=False):
        return

    def _get_state(self):
        return self.simulator.obs

    def close(self):
        if self.simulator is not None:
            self.simulator.close_gracefully()
