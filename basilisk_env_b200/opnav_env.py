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

from . import spaces
from .vec_env import BatchVecEnv, BskEnvError

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


class OpNavVecEnv(BatchVecEnv):
    """N opNav environments on one GPU (see LeoPowerAttVecEnv for the conventions).

    **config : overrides of `bskenv_opnav_config` fields (include/bskenv.h), e.g. camera_reenable=1."""
    _abi = "bskenv_opnav_"
    OBS_DIM, IC_DIM, STAT_NAMES = OBS_DIM, IC_DIM, STAT_NAMES
    IC_ASSIGN = {"by_index": 0, "per_episode": 1}
    FIELD_WIDTH = {"r_BN_N": 3, "v_BN_N": 3, "sigma_BN": 3, "omega_BN_B": 3, "Omega": 4, "reactionwheel_cmds": 4,
                   "navErrors": 15, "sun_point_data": 3, "filter_state": 6, "filter_sBar": 21, "sim_obs": 4, "sim_states": 12}

    def __init__(self, num_envs, device=0, first_env_index=0, seed=0, auto_reset=False, **config):
        config.setdefault("noise_seed", int(seed) & (2**64 - 1))
        super().__init__(num_envs, device, first_env_index, seed, auto_reset, config)
        with torch.cuda.device(self.device):
            self.debug = torch.zeros((self.num_envs, DEBUG_DIM), dtype=torch.float64, device=self.device)
        self.action_space = spaces.Discrete(2)
        self.step_duration = float(self.cfg.step_duration_min)

    def set_ephemeris(self, table):
        """SURVEY 8(f)-4: Sun position relative to the Mars barycentre [m] from a Chebyshev table
        (`basilisk_env_b200.ephemeris.ChebTable`; None = back to the analytic series).  Set before reset."""
        if table is None:
            self._check(self._L.bskenv_opnav_set_ephemeris(self._h, 0.0, 0.0, 0, 0, None), "set_ephemeris")
            return
        coef = np.ascontiguousarray(table.coef, dtype=np.float64)
        self._check(self._L.bskenv_opnav_set_ephemeris(self._h, float(table.t0), float(table.seg_len), coef.shape[0],
                                                       coef.shape[2], coef.ctypes.data), "set_ephemeris")

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
