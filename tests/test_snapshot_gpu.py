"""Per-env state snapshots on the GPU (BatchVecEnv.snapshot / restore; include/bskenv.h: bskenv_snapshot / bskenv_restore and
the opNav pair): round trips through auto-resets and pools, fan-out of one env into several, moves between handles (same
global index, other organisation, another device), opNav clones across indices with the noise off, the observation a
restore returns, and the refusals.  "Bit-identical" is torch.equal on every step output (terminal_obs in the rows of the
envs that finished: the step writes no others) and, at the end, on the state,
the stored ICs, the IC-pool rows and (LEO) the parameters."""
import ctypes as C
import struct

import numpy as np
import pytest

from tests.test_ic_pool_gpu import leo_pool

pytestmark = pytest.mark.gpu

OUTS = ("obs", "reward", "done", "done_reason", "terminal_obs", "episode_r", "episode_l")
SIZES = [4096, 60001]


def _leo(n, **kw):
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    return LeoPowerAttVecEnv(n, **{"device": 0, **kw})


def _opnav(n, **kw):
    from basilisk_env_b200.opnav_env import OpNavVecEnv
    return OpNavVecEnv(n, **{"device": 0, "step_duration_min": 5.0, **kw})


def _acts(steps, n, hi, seed, device="cuda"):
    import torch
    g = torch.Generator("cuda").manual_seed(seed)
    return torch.randint(0, hi, (steps, n), dtype=torch.int32, device="cuda", generator=g).to(device)


def _step(env, a):
    """The outputs of one interval; terminal_obs only in the rows of the envs that finished (the step writes no others)"""
    import torch
    o, r, d, info = env.step(a)
    term = torch.where(d.bool()[:, None], info["terminal_obs"], torch.zeros_like(info["terminal_obs"]))
    return [x.clone() for x in (o, r, d, info["done_reason"], term, info["episode_r"], info["episode_l"])]


def _end(env):
    """State, stored ICs, IC-pool rows and (LEO) parameters and parameter rows"""
    d, i = env.get_state()
    out = [d, i, env.initial_conditions(), env.ic_rows()]
    if hasattr(env, "env_params"):
        p, row = env.env_params()
        out += list(p.values()) + [row]
    return [x.clone() for x in out]


def _same(xs, ys, what):
    import torch
    for k, (x, y) in enumerate(zip(xs, ys)):
        assert torch.equal(x.cpu(), y.cpu()), f"{what}: item {k}"


def _scenario(env, k=29, seed=3):
    rng = np.random.RandomState(seed)
    env.set_param_pool({"mass": rng.uniform(250.0, 420.0, k), "panelArea": rng.uniform(0.5, 1.5, k),
                        "storageCapacity": rng.uniform(30.0, 60.0, k) * 3600.0}, assign="per_episode")
    env.set_ic_pool(leo_pool(k, seed), assign="param_row")


# ---- 1. round trip -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["leo", "leo_scenario", "opnav"])
@pytest.mark.parametrize("n", SIZES)
def test_round_trip(kind, n):
    k, steps = 3, 8
    if kind == "opnav":
        env, hi = _opnav(n, seed=11, auto_reset=True, max_length=3), 2
    else:
        env, hi = _leo(n, seed=11, auto_reset=True, max_length=3), 3
        if kind == "leo_scenario":
            _scenario(env)
    env.reset()
    acts = _acts(k + steps, n, hi, 5)
    for t in range(k):
        env.step(acts[t])
    rec = env.snapshot()
    ref = [_step(env, acts[t]) for t in range(k, k + steps)]
    ref_end = _end(env)
    assert any(bool(r[2].any()) for r in ref), "no auto-reset in the window"
    env.restore(rec)
    for j, t in enumerate(range(k, k + steps)):
        _same(_step(env, acts[t]), ref[j], f"{kind} n={n} interval {t}")
    _same(_end(env), ref_end, f"{kind} n={n} end")
    if kind == "leo_scenario":
        assert bool((env.ic_rows() >= 0).all()) and bool((env.env_params()[1] >= 0).all())
    env.close()


# ---- 2. fan-out ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
def test_fan_out(n):
    """One env's record in three envs, each with its own action: each follows the source env taking that action."""
    import torch
    k, steps, src, dst = 2, 5, 7, [n - 1, n // 2, 100]
    acts = _acts(k + steps, n, 3, 9)
    env = _leo(n, seed=4, max_length=5)
    env.reset()
    for t in range(k):
        env.step(acts[t])
    last_obs = env.obs[src].clone()
    full = env.snapshot()
    rec = env.snapshot([src])
    obs = env.restore(rec.repeat(3, 1), envs=dst)
    for e in dst:
        assert torch.equal(obs[e], last_obs)
    fan = []
    for t in range(k, k + steps):
        a = acts[t].clone()
        a[dst] = torch.tensor([0, 1, 2], dtype=torch.int32, device=a.device)
        fan.append(_step(env, a))
    ref = _leo(n, seed=4, max_length=5)
    ref.reset()
    for action, e in zip((0, 1, 2), dst):
        ref.restore(full)
        finished = False
        for j, t in enumerate(range(k, k + steps)):
            a = acts[t].clone()
            a[src] = action
            r = _step(ref, a)
            for q, (x, y) in enumerate(zip(fan[j], r)):
                assert torch.equal(x[e], y[src]), f"action {action} interval {t} {OUTS[q]}"
            if bool(r[2][src]):
                finished = True
                break
        assert finished or j == steps - 1
    env.close(); ref.close()


# ---- 3. cross-handle, same global index --------------------------------------------------------------------------------
@pytest.mark.parametrize("where", ["same_device", "second_device"])
def test_cross_handle_same_global_index(where):
    import torch
    if where == "second_device" and torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device")
    dev_b = 1 if where == "second_device" else 0
    k, steps = 3, 12
    acts = _acts(k + steps, 4096, 3, 21)
    a = _leo(4096, seed=8, auto_reset=True, max_length=3)
    b = _leo(1024, device=dev_b, first_env_index=1024, seed=8, auto_reset=True, max_length=3)
    a.reset(); b.reset()
    for t in range(k):
        a.step(acts[t])
        b.step(acts[k + t, :1024].to(b.device))             # b elsewhere: its own actions
    rec = a.snapshot(torch.arange(1024, 2048)).cpu()
    b.restore(rec.to(b.device))
    resets = 0
    for t in range(k, k + steps):
        ra = _step(a, acts[t])
        rb = _step(b, acts[t, 1024:2048].to(b.device))
        _same(rb, [x[1024:2048] for x in ra], f"interval {t}")
        resets += int(rb[2].sum())
    assert resets > 1024
    ea, eb = _end(a), _end(b)
    _same(eb[:2], [x[:, 1024:2048] for x in ea[:2]], "state")
    _same(eb[2:], [x[1024:2048] for x in ea[2:]], "ics / rows / params")
    a.close(); b.close()


# ---- 4. across organisations -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4096, 4001])
def test_split_to_thread(n):
    k, steps = 2, 8
    acts = _acts(k + steps, n, 3, 31)
    a = _leo(n, seed=6, auto_reset=True, max_length=3, organisation="split")
    b = _leo(n, seed=6, auto_reset=True, max_length=3, organisation="thread")
    a.reset(); b.reset()
    for t in range(k):
        a.step(acts[t])
    b.restore(a.snapshot())
    for t in range(k, k + steps):
        _same(_step(b, acts[t]), _step(a, acts[t]), f"interval {t}")
    assert a.kernel_name().startswith("leo_split_kernel") and b.kernel_name().startswith("leo_step_kernel")
    _same(_end(b), _end(a), "end")
    a.close(); b.close()


# ---- 5. opNav across indices, noise off -----------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
def test_opnav_clone_across_indices(n):
    import torch
    k, steps, m = 2, 4, n // 3
    env = _opnav(n, seed=2, nav_noise=0, pixel_noise_std=0.0, max_length=10)
    env.reset()
    acts = _acts(k + steps, n, 2, 41)
    for t in range(k):
        env.step(acts[t])
    g = torch.Generator().manual_seed(n)
    src = torch.randperm(n, generator=g)[:m]
    dst = torch.randperm(n, generator=g)
    dst = dst[~torch.isin(dst, src)][:m]
    env.restore(env.snapshot(src), envs=dst)
    src, dst = src.cuda(), dst.cuda()
    live = torch.ones(m, dtype=torch.bool, device="cuda")
    for t in range(k, k + steps):
        a = acts[t].clone()
        a[dst] = a[src]
        r = _step(env, a)
        for q, x in enumerate(r):
            assert torch.equal(x[dst][live], x[src][live]), f"interval {t} {OUTS[q]}"
        live &= ~r[2][src].bool()
    assert bool(live.any())
    env.close()


# ---- 6. observation -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["leo", "opnav"])
@pytest.mark.parametrize("n", SIZES)
def test_restore_returns_the_last_observation(kind, n):
    import torch
    mk, hi = (_leo, 3) if kind == "leo" else (_opnav, 2)
    env = mk(n, seed=13, auto_reset=True, max_length=1)
    other = mk(n, seed=13, auto_reset=True, max_length=1)
    other.reset()
    acts = _acts(4, n, hi, 51)
    obs0 = env.reset().clone()                                   # fresh from reset
    rec0 = env.snapshot()
    env.step(acts[0])
    env.reset(mask=torch.arange(n, device="cuda") % 3 == 0)      # a third back at curr_step 0: not done at the next step
    obs1, _, done1, _ = env.step(acts[1])                        # mid-episode (done = 0) and just auto-reset (done = 1)
    obs1, done1 = obs1.clone(), done1.clone().bool()
    assert bool(done1.any()) and bool((~done1).any())
    rec1 = env.snapshot()
    env.step(acts[2])
    assert torch.equal(env.restore(rec1), obs1)
    assert torch.equal(other.restore(rec0), obs0)
    if kind == "opnav":
        assert not bool(obs0.any())
    idx = torch.arange(0, n, 7)
    other.obs.fill_(-1.0)
    out = other.restore(rec1[idx], envs=idx)
    assert torch.equal(out[idx.cuda()], obs1[idx.cuda()])
    keep = torch.ones(n, dtype=torch.bool, device="cuda")
    keep[idx.cuda()] = False
    assert bool((out[keep] == -1.0).all())
    env.close(); other.close()


# ---- 7. refusals ------------------------------------------------------------------------------------------------------
def _fnv(cfg, names):
    h = 14695981039346656037
    for name in names:
        v = getattr(cfg, name)
        vals = list(v) if hasattr(v, "__len__") else [v]
        ctype = dict(type(cfg)._fields_)[name]
        base = ctype._type_ if isinstance(getattr(ctype, "_type_", None), type) else ctype     # element type of an array
        fmt = "<d" if base is C.c_double else "<i"
        for x in vals:
            for byte in struct.pack(fmt, x):
                h = ((h ^ byte) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


LEO_FP_FIELDS = ("abi_version", "dynRate", "fswRate", "step_duration", "mass", "width", "depth", "height", "planetRadius",
                 "baseDensity", "scaleHeight", "disturbance_magnitude", "nHat_B", "panelArea", "panelEfficiency", "powerDraw",
                 "storageCapacity", "sigma_R0N", "K", "Ki", "P", "hs_min", "thrMinFireTime", "thrForceSign", "maxCounterValue",
                 "max_length", "wheel_limit_rpm", "power_max", "failure_penalty", "use_j2", "hill_cel_pun", "rw_set", "precision")
OPNAV_FP_FIELDS = ("abi_version", "dynRate", "fswRate", "step_duration_min", "max_length", "numModes", "nav_noise",
                   "camera_reenable", "sample_orbit", "pixel_noise_std", "circle_unc", "reward_mult")


def _words(rec, col):
    return rec[:, col].contiguous().view(__import__("torch").int64)


def test_record_header():
    import torch
    a = _leo(64, first_env_index=500, seed=1)
    a.reset()
    rec = a.snapshot(torch.tensor([3, 0, 63]))
    assert rec.shape == (3, 172)
    assert _words(rec, 0).tolist() == [1 << 16 | 1] * 3 and _words(rec, 1).tolist() == [172] * 3
    assert _words(rec, 3).tolist() == [503, 500, 563]
    assert (_words(rec, 2).cpu().numpy().astype(np.uint64) == np.uint64(_fnv(a.cfg, LEO_FP_FIELDS))).all()
    assert _words(rec, 171).tolist() == [-1] * 3 and rec[:, 134 + 22].tolist() == [-1.0] * 3
    d, i = a.get_state()
    assert torch.equal(rec[:, 4:93], d[:, [3, 0, 63]].T) and torch.equal(_words(rec, slice(93, 115)), i[:, [3, 0, 63]].T)
    assert torch.equal(rec[:, 115:134], a.initial_conditions()[[3, 0, 63]])
    b = _leo(64, seed=1, auto_reset=True)                       # auto_reset is handle policy: same fingerprint
    assert _words(b.snapshot(), 2)[0] == _words(rec, 2)[0]
    o = _opnav(32, noise_seed=99)
    o.reset()
    orec = o.snapshot()
    assert orec.shape == (32, 114) and _words(orec, 0)[0] == 2 << 16 | 1
    assert np.uint64(_words(orec, 2)[0].item() & 0xFFFFFFFFFFFFFFFF) == np.uint64(_fnv(o.cfg, OPNAV_FP_FIELDS))
    for env in (a, b, o):
        env.close()


def _refused(env, fn, *args, match):
    from basilisk_env_b200.vec_env import BskEnvError
    before = _end(env)
    with pytest.raises(BskEnvError) as err:
        fn(*args)
    assert match in str(err.value), str(err.value)
    _same(_end(env), before, f"after refusal '{match}'")
    return str(err.value)


def test_refusals():
    import torch
    n = 4096
    a = _leo(n, seed=3)
    a.reset()
    a.step(_acts(1, n, 3, 1)[0])
    rec = a.snapshot()
    state0 = [x.clone() for x in a.get_state()]
    idx = torch.tensor([0, 1, 2, 3])
    part = a.snapshot(idx)
    bad = part.clone()
    bad[2, 0] = torch.tensor([2 << 16 | 1], dtype=torch.int64).view(torch.float64)[0]         # an opNav header
    _refused(a, a.restore, bad, idx, match="record 2: not a record of this batch kind")
    bad = part.clone()
    bad[1, 0] = torch.tensor([1 << 16 | 2], dtype=torch.int64).view(torch.float64)[0]         # another format version
    _refused(a, a.restore, bad, idx, match="record 1: not a record of this batch kind and format version")
    bad = part.clone()
    bad[3, 1] = torch.tensor([171], dtype=torch.int64).view(torch.float64)[0]
    _refused(a, a.restore, bad, idx, match="record 3: record width differs")
    other = _leo(n, seed=3, mass=331.0)
    other.reset()
    _refused(a, a.restore, other.snapshot(idx), idx, match="record 0: configuration fingerprint differs")
    _refused(a, a.restore, part, torch.tensor([0, 1, n, 3]), match="record 2: env index outside [0, n)")
    _refused(a, a.restore, part, torch.tensor([0, 1, -1, 3]), match="record 2: env index outside")
    _refused(a, a.restore, part, torch.tensor([5, 7, 5, 9]), match="record 2: env index named twice")
    _refused(a, a.restore, part, torch.tensor([5, 7, 9, 7]), match="record 3: env index named twice")
    _refused(a, a.snapshot, torch.tensor([0, n + 5]), match="record 1: env index outside [0, n)")
    pooled = _leo(n, seed=3)
    _scenario(pooled)
    pooled.reset()
    _refused(a, a.restore, pooled.snapshot(idx), idx, match="record 0: carries a parameter-pool row and no parameter pool is loaded")
    # null records, and the whole batch without indices but m != n (straight through the C ABI)
    before = _end(a)
    assert a._f.restore(a._h, n, None, None, None, a._stream()) == -1
    assert a._f.restore(a._h, 4, None, C.c_void_p(part.data_ptr()), None, a._stream()) == -1
    assert a._f.snapshot(a._h, 4, None, C.c_void_p(part.data_ptr()), a._stream()) == -1
    assert a._f.restore(a._h, 0, C.c_void_p(idx.cuda().data_ptr()), C.c_void_p(part.data_ptr()), None, a._stream()) == -1
    _same(_end(a), before, "after null / size refusals")
    # a host-buffer step in flight
    a.step_host_async(np.zeros(n, np.int32))
    try:
        with pytest.raises(Exception, match="host-buffer step is in flight"):
            a.restore(rec)
    finally:
        a.step_host_wait()
    # a LEO record given to the opNav batch
    o = _opnav(n)
    o.reset()
    before = _end(o)
    oidx = torch.tensor([0], device="cuda")
    assert o._f.restore(o._h, 1, C.c_void_p(oidx.data_ptr()), C.c_void_p(rec.data_ptr()), None, o._stream()) == -1
    assert "record 0: not a record of this batch kind" in o._f.last_error(o._h).decode()
    _same(_end(o), before, "opNav after a LEO record")
    # after all that (the host-buffer step moved the envs on), a restore still works
    a.restore(rec)
    _same(_end(a)[:2], state0, "restore after refusals")
    for env in (a, other, pooled, o):
        env.close()
