"""Vectorised LEO power/attitude environment: N independent spacecraft stepped by ONE CUDA launch.

This is the batched form of `leoPowerAttEnv.step/reset/reset_init`
(/root/reference/basilisk_env/envs/leoPowerAttitudeEnvironment.py:65-216) over the C ABI of
include/bskenv.h.  torch supplies device memory and streams only; all arithmetic is in
csrc/bskenv.cu.  There is no CPU path: constructing the class without a CUDA device raises."""
import ctypes as C

import numpy as np
import torch

from . import _native
from . import spaces
from .initial_conditions import CONFIG_KEYS, PARAM_KEYS, ic_row, scenario_rows

DONE_MAXLEN, DONE_WHEEL, DONE_POWER, DONE_DECAY = 1, 2, 4, 8
OBS_DIM, IC_DIM = 5, 19
STAT_NAMES = ("return_sum", "length_sum", "episodes", "wheel_failures", "power_failures", "orbit_decays",
              "max_length_ends", "env_steps")
ORGANISATIONS = {"auto": 0, "thread": 1, "split": 2, "thread_index": 3}
PARAM_ASSIGN = {"by_index": 0, "per_episode": 1}
IC_ASSIGN = {"by_index": 0, "per_episode": 1, "param_row": 2}
_FIELD_WIDTH = {"r_BN_N": 3, "v_BN_N": 3, "sigma_BN": 3, "omega_BN_B": 3, "Omega": 4, "u_current": 4,
                "extTorquePntB_B": 3, "att_guidance": 12, "att_reference": 9, "commandedControlTorque": 3,
                "rwTorqueCommand": 4, "wheelDeltaH": 3, "ThrustOnCmd": 8, "thrOnTimeRemaining": 8, "OnTimeRequest": 8,
                "sim_obs": 5, "fireCounter": 8}


class BskEnvError(RuntimeError):
    pass


def shard_range(num_envs_total, rank, world_size):
    """Env index range [lo, hi) owned by `rank`: contiguous blocks, remainder to the low ranks."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(int(num_envs_total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class BatchVecEnv:
    """What the LEO and the opNav batch share: one handle of the batch's C ABI (`_abi`: the prefix of its entry points), the
    device output buffers, resets, the IC pool, the persistent state and the episode statistics.  A subclass sets the class
    attributes below, `action_space` and `step_duration`, and adds its step."""
    _abi = ""                   # "bskenv_" or "bskenv_opnav_"
    OBS_DIM = IC_DIM = 0
    IC_ASSIGN = {}
    STAT_NAMES = ()
    FIELD_WIDTH = {}

    def __init__(self, num_envs, device, first_env_index, seed, auto_reset, config):
        if not torch.cuda.is_available():
            raise BskEnvError(f"{type(self).__name__} needs a CUDA device: the environment step has no CPU path")
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if self.device.type != "cuda":
            raise BskEnvError(f"{type(self).__name__} needs a CUDA device: the environment step has no CPU path")
        self.num_envs = int(num_envs)
        self.first_env_index = int(first_env_index)
        self.seed_value = int(seed)
        self._L = _native.lib()
        self._f = _native.batch_abi(self._abi)
        self.cfg = _native.batch_config(self._abi, auto_reset=int(bool(auto_reset)), **config)
        self.auto_reset = bool(auto_reset)
        h = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = self._f.create(C.byref(self.cfg), dev_index, self.num_envs, self.first_env_index, C.byref(h))
        if rc != 0:
            raise BskEnvError(f"{self._f.create.__name__} failed ({rc}): {self._f.last_error(None).decode()}")
        self._h = h
        n = self.num_envs
        with torch.cuda.device(self.device):
            self.obs = torch.zeros((n, self.OBS_DIM), dtype=torch.float64, device=self.device)
            self.term_obs = torch.zeros((n, self.OBS_DIM), dtype=torch.float64, device=self.device)
            self.reward = torch.zeros(n, dtype=torch.float64, device=self.device)
            self.done = torch.zeros(n, dtype=torch.uint8, device=self.device)
            self.done_reason = torch.zeros(n, dtype=torch.uint8, device=self.device)
            # per env: the reference's reward_total and curr_step, the `info['episode']` record where done
            self.episode_r = torch.zeros(n, dtype=torch.float64, device=self.device)
            self.episode_l = torch.zeros(n, dtype=torch.int64, device=self.device)
        self.observation_space = spaces.Box(-1e16, 1e16, shape=(self.OBS_DIM, 1))
        self.max_length = int(self.cfg.max_length)
        nd, ni = C.c_int32(), C.c_int32()
        self._f.state_dims(self._h, C.byref(nd), C.byref(ni))
        self.n_double_fields, self.n_int_fields = nd.value, ni.value

    # ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._f.destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise BskEnvError(f"{what} failed ({rc}): {self._f.last_error(self._h).decode()}")

    def _call(self, fn, *args):
        self._check(fn(*args), fn.__name__)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _mask_ptr(self, mask):
        if mask is None:
            return None, None
        m = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()
        if m.numel() != self.num_envs:
            raise ValueError("mask must have one entry per env")
        return m, C.c_void_p(m.data_ptr())

    # ------------------------------------------------------------------------------------------
    def set_ic_pool(self, ics, assign="per_episode"):
        """Load a pool of initial conditions [K, IC_DIM] that `reset()` and the auto-reset of `step` draw from instead of the
        built-in sampler (include/bskenv.h: bskenv_set_ic_pool); None unloads it.
        assign : "per_episode" (row drawn per (seed, global env index, episode)) or "by_index" (global env index mod K)."""
        if ics is None:
            self._call(self._f.set_ic_pool, self._h, 0, None, 0)
            return
        rows = ics.detach().cpu().numpy() if torch.is_tensor(ics) else ics
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        if rows.ndim != 2 or rows.shape[1] != self.IC_DIM or rows.shape[0] == 0:
            raise ValueError(f"ics must have shape (K, {self.IC_DIM}) with K > 0")
        self._call(self._f.set_ic_pool, self._h, rows.shape[0], rows.ctypes.data, self.IC_ASSIGN[assign])

    def ic_rows(self):
        """The IC-pool row each env's current episode started from (int32 [N]; -1 = sampled or explicit ICs)."""
        row = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        self._call(self._f.get_ic_rows, self._h, C.c_void_p(row.data_ptr()), self._stream())
        return row

    def reset(self, seed=None, mask=None):
        """Sample fresh initial conditions on the device (or draw them from the IC pool) and return the initial
        observation [N, OBS_DIM]."""
        if seed is not None:
            self.seed_value = int(seed)
        keep, mp = self._mask_ptr(mask)
        self._call(self._f.reset_seeded, self._h, C.c_uint64(self.seed_value & (2**64 - 1)), mp, C.c_void_p(self.obs.data_ptr()),
                   self._stream())
        del keep
        return self.obs

    def reset_ics(self, ics, mask=None):
        """Reset from explicit initial conditions: [N, IC_DIM] rows."""
        t = torch.as_tensor(np.asarray(ics, dtype=np.float64) if not torch.is_tensor(ics) else ics)
        t = t.to(device=self.device, dtype=torch.float64).contiguous()
        if tuple(t.shape) != (self.num_envs, self.IC_DIM):
            raise ValueError(f"ics must have shape ({self.num_envs}, {self.IC_DIM})")
        keep, mp = self._mask_ptr(mask)
        self._call(self._f.reset_ics, self._h, C.c_void_p(t.data_ptr()), mp, C.c_void_p(self.obs.data_ptr()), self._stream())
        torch.cuda.current_stream(self.device).synchronize()   # `t` may be a temporary
        del keep
        return self.obs

    def reset_init(self, mask=None):
        """Rebuild every (masked) env from its stored initial conditions."""
        keep, mp = self._mask_ptr(mask)
        self._call(self._f.reset_init, self._h, mp, C.c_void_p(self.obs.data_ptr()), self._stream())
        del keep
        return self.obs

    def initial_conditions(self):
        out = torch.empty((self.num_envs, self.IC_DIM), dtype=torch.float64, device=self.device)
        self._call(self._f.get_ics, self._h, C.c_void_p(out.data_ptr()), self._stream())
        return out

    # ------------------------------------------------------------------------------------------
    def get_state(self):
        """Whole persistent state (a checkpoint): (double [n_double_fields, N], int64 [n_int_fields, N])."""
        d = torch.empty((self.n_double_fields, self.num_envs), dtype=torch.float64, device=self.device)
        i = torch.empty((self.n_int_fields, self.num_envs), dtype=torch.int64, device=self.device)
        self._call(self._f.get_state, self._h, C.c_void_p(d.data_ptr()), C.c_void_p(i.data_ptr()), self._stream())
        return d, i

    def set_state(self, dstate, istate):
        d = dstate.to(device=self.device, dtype=torch.float64).contiguous()
        i = istate.to(device=self.device, dtype=torch.int64).contiguous()
        if tuple(d.shape) != (self.n_double_fields, self.num_envs) or tuple(i.shape) != (self.n_int_fields, self.num_envs):
            raise ValueError("state blocks have the wrong shape")
        self._call(self._f.set_state, self._h, C.c_void_p(d.data_ptr()), C.c_void_p(i.data_ptr()), self._stream())
        torch.cuda.current_stream(self.device).synchronize()

    def _env_index(self, envs):
        if envs is None:
            return None, None
        idx = torch.as_tensor(envs).to(device=self.device, dtype=torch.int64).reshape(-1).contiguous()
        return idx, C.c_void_p(idx.data_ptr())

    def snapshot(self, envs=None):
        """Per-env state records (include/bskenv.h: bskenv_snapshot): float64 [m, W] on this handle's device, one row per env
        of `envs` (indices, None = every env in index order).  A record holds everything a step or a reset reads of its env and
        can be restored into any env of any handle with the same configuration (`restore`)."""
        idx, ip = self._env_index(envs)
        m = self.num_envs if idx is None else idx.numel()
        rec = torch.empty((m, int(self._f.snapshot_width(self._h))), dtype=torch.float64, device=self.device)
        self._call(self._f.snapshot, self._h, m, ip, C.c_void_p(rec.data_ptr()), self._stream())
        self._snap_keep = idx           # keep alive until the gather has consumed it
        return rec

    def restore(self, records, envs=None):
        """Write records [m, W] (from `snapshot` of this or another handle; `.to(self.device)` moves them) into the envs `envs`
        (indices, None = every env in index order) and return `obs`, in which each restored env's row is the observation its
        source returned last.  Waits for the current stream (the records are checked on the device first)."""
        idx, ip = self._env_index(envs)
        r = records.to(device=self.device, dtype=torch.float64).contiguous()
        m = self.num_envs if idx is None else idx.numel()
        if tuple(r.shape) != (m, int(self._f.snapshot_width(self._h))):
            raise ValueError(f"records must have shape ({m}, {int(self._f.snapshot_width(self._h))})")
        self._call(self._f.restore, self._h, m, ip, C.c_void_p(r.data_ptr()), C.c_void_p(self.obs.data_ptr()), self._stream())
        self._snap_keep = (r, idx)      # keep alive until the scatter has consumed them
        return self.obs

    def field(self, name, state=None):
        """Named slice of the state, e.g. field("r_BN_N") -> [3, N]."""
        idx, is_int = _native.batch_state_field(self._abi, name)
        d, i = state if state is not None else self.get_state()
        return (i if is_int else d)[idx:idx + self.FIELD_WIDTH.get(name, 1)]

    def episode_stats(self, all_reduce=False):
        """Episode statistics of this shard since the last call (dict of floats).  With `all_reduce`
        the eight numbers are summed over the process group -- the only collective of the design."""
        buf = np.zeros(8)
        self._call(self._f.episode_stats, self._h, buf.ctypes.data)
        if all_reduce:
            buf = all_reduce_stats(buf, self.device)
        return dict(zip(self.STAT_NAMES, (float(x) for x in buf)))

    def launch_count(self):
        return int(self._f.launch_count(self._h))

    def flops_per_step(self):
        return float(self._f.flops_per_step(self._h))


class LeoPowerAttVecEnv(BatchVecEnv):
    """N environments on one GPU.

    Parameters
    ----------
    num_envs : envs owned by THIS process (one process per GPU).
    device : CUDA device index or torch.device.
    first_env_index : global index of local env 0; random streams are keyed by the global index so
        results do not depend on how the envs are sharded across GPUs.
    seed : base seed of the device-side IC sampler.
    auto_reset : re-sample ICs inside the step launch for envs that finish (VecEnv convention: the
        returned obs is the first of the new episode, `info["terminal_obs"]` the last of the old).
    organisation : "auto" | "thread" | "split": work organisation of the step kernel (see `set_organisation`).
    **config : overrides of `bskenv_config` fields (include/bskenv.h), e.g. step_duration=60.
    """
    _abi = "bskenv_"
    OBS_DIM, IC_DIM, IC_ASSIGN, STAT_NAMES, FIELD_WIDTH = OBS_DIM, IC_DIM, IC_ASSIGN, STAT_NAMES, _FIELD_WIDTH

    def __init__(self, num_envs, device=0, first_env_index=0, seed=0, auto_reset=False, organisation="auto", **config):
        super().__init__(num_envs, device, first_env_index, seed, auto_reset, config)
        self.action_space = spaces.Discrete(3)
        self.step_duration = float(self.cfg.step_duration)
        if organisation != "auto":
            self.set_organisation(organisation)

    # ------------------------------------------------------------------------------------------
    # ---- SURVEY 8(f)-4: ephemeris tables and the planet-fixed degree-2 field (set before reset) ----
    def set_ephemeris(self, kind, table):
        """Load a Chebyshev ephemeris table (`basilisk_env_b200.ephemeris.ChebTable`, or None to go back to the analytic
        model).  kind: "sun" (Sun position relative to Earth [m]) or "orientation" (Earth RA, DEC, W [rad])."""
        k = {"sun": 0, "orientation": 1}[kind]
        if table is None:
            self._check(self._L.bskenv_set_ephemeris(self._h, k, 0.0, 0.0, 0, 0, None), "set_ephemeris")
            return
        coef = np.ascontiguousarray(table.coef, dtype=np.float64)
        nseg, three, ncoef = coef.shape
        assert three == 3
        self._check(self._L.bskenv_set_ephemeris(self._h, k, float(table.t0), float(table.seg_len), nseg, ncoef,
                                                 coef.ctypes.data), "set_ephemeris")

    def set_gravity_degree2(self, enable=True, cbar=None):
        """Earth's degree-2 field (normalised C20, C21, S21, C22, S22; None = built-in GGM03S-class values) evaluated in
        the planet-fixed frame with the orientation Euler-stepped from the last SPICE message."""
        ptr = None
        if cbar is not None:
            cbar = np.ascontiguousarray(cbar, dtype=np.float64)
            assert cbar.shape == (5,)
            ptr = cbar.ctypes.data
        self._check(self._L.bskenv_set_gravity_degree2(self._h, int(bool(enable)), ptr), "set_gravity_degree2")

    def set_param_pool(self, pool, assign="per_episode"):
        """Load a pool of spacecraft parameter sets (Monte Carlo dispersions / domain randomisation): each env runs one row
        for a whole episode, picked at its next reset (include/bskenv.h: bskenv_set_param_pool).
        pool : dict of `initial_conditions.PARAM_KEYS` -> arrays [K] (missing keys take the configuration's value), or an
            array [K, 14] in PARAM_KEYS order; None unloads the pool.
        assign : "per_episode" (row drawn per (seed, global env index, episode)) or "by_index" (row = global env index
            mod K: with K = the global env count, an explicit per-env table)."""
        if pool is None:
            self._check(self._L.bskenv_set_param_pool(self._h, 0, None, 0), "bskenv_set_param_pool")
            return
        if isinstance(pool, dict):
            unknown = set(pool) - set(PARAM_KEYS)
            if unknown:
                raise KeyError(f"not per-env parameters: {sorted(unknown)} (see initial_conditions.PARAM_KEYS)")
            cols = {k: np.ravel(np.asarray(v, dtype=np.float64)) for k, v in pool.items()}
            sizes = {len(v) for v in cols.values()}
            if len(sizes) != 1:
                raise ValueError("every pool column needs the same length")
            k = sizes.pop()
            rows = np.stack([cols[key] if key in cols else np.full(k, float(getattr(self.cfg, key))) for key in PARAM_KEYS], axis=1)
        else:
            rows = np.asarray(pool.cpu().numpy() if torch.is_tensor(pool) else pool, dtype=np.float64)
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        if rows.ndim != 2 or rows.shape[1] != len(PARAM_KEYS) or rows.shape[0] == 0:
            raise ValueError(f"pool must have shape (K, {len(PARAM_KEYS)}) with K > 0")
        self._check(self._L.bskenv_set_param_pool(self._h, rows.shape[0], rows.ctypes.data, PARAM_ASSIGN[assign]),
                    "bskenv_set_param_pool")

    def env_params(self):
        """The spacecraft parameters every env runs with: (dict of PARAM_KEYS -> [N] f64 tensors, pool row [N] int32,
        -1 = the batch configuration)."""
        p = torch.empty((self.num_envs, len(PARAM_KEYS)), dtype=torch.float64, device=self.device)
        row = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        self._check(self._L.bskenv_get_env_params(self._h, C.c_void_p(p.data_ptr()), C.c_void_p(row.data_ptr()), self._stream()),
                    "bskenv_get_env_params")
        return {k: p[:, j] for j, k in enumerate(PARAM_KEYS)}, row

    def set_ic_pool(self, ics, assign="per_episode"):
        """Load a pool of initial conditions that resets draw from instead of the built-in sampler -- `reset()` and the
        auto-reset of `step` alike (include/bskenv.h: bskenv_set_ic_pool).
        ics : array or tensor [K, 19] (see initial_conditions.ic_row), a sequence of reference `initial_conditions` dicts, or
            None to unload the pool.
        assign : "per_episode" (row drawn per (seed, global env index, episode)), "by_index" (row = global env index mod K)
            or "param_row" (row = the env's parameter-pool row: a scenario table, see `set_scenario_pool`)."""
        if ics is not None and not torch.is_tensor(ics) and len(ics) and isinstance(ics[0], dict):
            ics = np.stack([ic_row(ic) for ic in ics])
        super().set_ic_pool(ics, assign)

    def set_scenario_pool(self, scenarios, assign="per_episode"):
        """Load K full reference `initial_conditions` dicts (the shape `initial_conditions.set_ICs()` returns) as a scenario
        table: their PARAM_KEYS become the parameter pool (assigned by `assign`), their initial conditions an IC pool paired
        with it ("param_row"), so that every episode runs one (initial conditions, parameters) pair -- the batched form of
        K reference simulators, each built from its own dict.  A batch-global key that differs from this handle's
        configuration raises ValueError.  None unloads both pools."""
        self.set_ic_pool(None)
        if scenarios is None:
            self.set_param_pool(None)
            return
        config = {k: list(getattr(self.cfg, k)) if k in ("nHat_B", "sigma_R0N") else getattr(self.cfg, k) for k in CONFIG_KEYS}
        ics, params = scenario_rows(scenarios, config)
        self.set_param_pool(params, assign=assign)
        self.set_ic_pool(ics, assign="param_row")

    def step(self, actions):
        """actions: int32 CUDA tensor [N] (0 nadir / 1 sun / 2 desat).  Returns device tensors
        (obs [N,5] f64, reward [N] f64, done [N] u8, info) without synchronising."""
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions, dtype=np.int32))
        a = actions.to(device=self.device, dtype=torch.int32).contiguous()
        if a.numel() != self.num_envs:
            raise ValueError("one action per env")
        self._check(self._L.bskenv_step_info(self._h, C.c_void_p(a.data_ptr()), C.c_void_p(self.obs.data_ptr()),
                                             C.c_void_p(self.reward.data_ptr()), C.c_void_p(self.done.data_ptr()),
                                             C.c_void_p(self.done_reason.data_ptr()), C.c_void_p(self.term_obs.data_ptr()),
                                             C.c_void_p(self.episode_r.data_ptr()), C.c_void_p(self.episode_l.data_ptr()),
                                             self._stream()), "bskenv_step_info")
        self._last_actions = a          # keep alive until the launch has consumed it
        # episode_r / episode_l: the reference's info['episode'] = {'r', 'l'} (ENV:130-136) for the envs with done set
        info = {"done_reason": self.done_reason, "terminal_obs": self.term_obs, "episode_r": self.episode_r,
                "episode_l": self.episode_l}
        return self.obs, self.reward, self.done, info

    def host_buffers(self, episode=False):
        """Page-locked, device-mapped numpy buffers for `step_host`: (actions int32 [N], (obs [N,5], reward [N], done u8 [N],
        done_reason u8 [N][, episode_r f64 [N], episode_l i64 [N]])).  The step kernel reads / writes them in place
        (zero-copy over PCIe); ordinary numpy arrays work too, through staging and one memcpy each.  With `episode` the
        tuple also carries the per-env episode record and terminal_obs [N,5] (rows of finished envs only)."""
        n = self.num_envs
        pin = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()     # noqa: E731
        out = [pin((n, OBS_DIM), torch.float64), pin(n, torch.float64), pin(n, torch.uint8), pin(n, torch.uint8)]
        if episode:
            out += [pin(n, torch.float64), pin(n, torch.int64), pin((n, OBS_DIM), torch.float64)]
        return pin(n, torch.int32), tuple(out)

    def step_host_async(self, actions, out=None):
        """Queue one host-buffer step and return; `step_host_wait()` delivers the results.  `out` as returned by
        `host_buffers()` (4 arrays, or 7 with the per-env episode record and the terminal observations)."""
        a = actions if (isinstance(actions, np.ndarray) and actions.dtype == np.int32 and actions.flags.c_contiguous) \
            else np.ascontiguousarray(actions, dtype=np.int32)
        if a.size != self.num_envs:
            raise ValueError("one action per env")
        if out is None:
            out = (np.empty((self.num_envs, OBS_DIM)), np.empty(self.num_envs), np.empty(self.num_envs, np.uint8),
                   np.empty(self.num_envs, np.uint8))
        ep_r = out[4].ctypes.data if len(out) > 4 else None
        ep_l = out[5].ctypes.data if len(out) > 4 else None
        term = out[6].ctypes.data if len(out) > 6 else None
        self._check(self._L.bskenv_step_host_async(self._h, a.ctypes.data, out[0].ctypes.data, out[1].ctypes.data,
                                                   out[2].ctypes.data, out[3].ctypes.data, term, ep_r, ep_l),
                    "bskenv_step_host_async")
        self._host_pending = (a, out)       # keep the buffers alive while the launch is in flight
        return out

    def step_host_wait(self):
        self._check(self._L.bskenv_step_host_wait(self._h), "bskenv_step_host_wait")
        pend, self._host_pending = getattr(self, "_host_pending", None), None
        return pend[1] if pend else None

    def step_host(self, actions, out=None):
        """Host-buffer step (the plugin path a CPU-side RL trainer calls): numpy int32 [N] in, numpy
        (obs, reward, done, done_reason[, episode_r, episode_l]) out; the transfers and the synchronisation happen inside
        the C calls."""
        self.step_host_async(actions, out)
        return self.step_host_wait()

    def kernel_name(self):
        """The step-kernel instantiation the last step launched (as ncu lists it)."""
        return self._L.bskenv_kernel_name(self._h).decode()

    def set_organisation(self, organisation):
        """Work organisation of the step kernel (include/bskenv.h: bskenv_set_organisation): "auto" (by batch size), "thread"
        (one thread per env; large batches bucketed by action), "split" (two warps per group of 32 envs: the small-batch
        organisation) or "thread_index" (one thread per env, lanes in index order: no bucketing).  Same arithmetic."""
        org = ORGANISATIONS[organisation] if isinstance(organisation, str) else int(organisation)
        self._check(self._L.bskenv_set_organisation(self._h, org), "bskenv_set_organisation")


def all_reduce_stats(buf, device=None):
    """Sum the 8 episode statistics over the default process group (NCCL on GPUs, gloo on CPU)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return np.asarray(buf, dtype=np.float64)
    backend = dist.get_backend()
    t = torch.as_tensor(np.asarray(buf, dtype=np.float64))
    if backend == "nccl":
        t = t.to(device if device is not None else torch.device("cuda", torch.cuda.current_device()))
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t.cpu().numpy()


def fp64_peak_tflops(device=0, seconds=0.5):
    """DFMA-chain microbenchmark (bskenv_fp64_peak): the FP64 roofline denominator."""
    out = C.c_double(0.0)
    rc = _native.lib().bskenv_fp64_peak(int(device), float(seconds), C.byref(out))
    if rc != 0:
        raise BskEnvError(f"bskenv_fp64_peak failed ({rc})")
    return out.value
