"""Initial-condition pools on the GPU (LeoPowerAttVecEnv.set_ic_pool / set_scenario_pool, OpNavVecEnv.set_ic_pool; include/
bskenv.h bskenv_set_ic_pool): the auto-reset through the reset kernel against a masked reset, pool rows against explicit ICs,
oracle parity, organisations and configurations, the assignment modes, no change without a pool, the host-buffer paths and
the refusals."""
import numpy as np
import pytest

from tests import parity

pytestmark = pytest.mark.gpu

OUTS = ("obs", "reward", "done", "done_reason", "terminal_obs", "episode_r", "episode_l")


# Philox4x32-10 (Salmon et al., SC'11), restated independently of the library
def _philox(c, k):
    c, k = [int(x) & 0xFFFFFFFF for x in c], [int(x) & 0xFFFFFFFF for x in k]
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, ((p0 >> 32) ^ c[3] ^ k[1]) & 0xFFFFFFFF, p0 & 0xFFFFFFFF]
        k = [(k[0] + 0x9E3779B9) & 0xFFFFFFFF, (k[1] + 0xBB67AE85) & 0xFFFFFFFF]
    return c


def ic_per_episode_row(n_rows, seed, global_env, episode):
    """The documented BSKENV_ICS_PER_EPISODE selection: one Philox4x32-10 block at counter (global env, episode, 0xFFFFFFFE),
    key = seed; row = (word1:word0) mod n_rows."""
    o = _philox([global_env, global_env >> 32, episode, 0xFFFFFFFE], [seed, seed >> 32])
    return ((o[1] << 32) | o[0]) % n_rows


def leo_pool(k, seed):
    """K reference dicts' initial conditions with a dispersed tumble rate, wheel speeds and charge."""
    from basilisk_env_b200 import initial_conditions as icm
    rng = np.random.RandomState(seed)
    rows = np.stack([icm.ic_row(icm.set_ICs(rng)) for _ in range(k)])
    rows[:, 9:12] *= rng.uniform(1.0, 100.0, (k, 1))
    rows[:, 15:18] = rng.uniform(-2000.0, 2000.0, (k, 3))
    rows[:, 18] = rng.uniform(4.0, 20.0, k) * 3600.0
    return rows


def opnav_pool(k, seed):
    """K opNav rows on dispersed orbits (the element ranges of opNavSimulator.py:166-171) with the reference filter error."""
    from basilisk_env_b200 import opnav_env as on
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(k):
        rN, vN = on.elem2rv(on.MU_MARS, rng.uniform(17000e3, 22000e3), rng.uniform(0, 0.6), rng.uniform(-20, 20) * on.D2R,
                            rng.uniform(0, 360) * on.D2R, rng.uniform(0, 360) * on.D2R, rng.uniform(0, 360) * on.D2R)
        out.append(np.concatenate([rN, vN, rng.uniform(-1e5, 1e5, 3), rng.uniform(-1e3, 1e3, 3)]))
    return np.stack(out)


def _leo(n, **kw):
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    return LeoPowerAttVecEnv(n, device=0, **kw)


def _opnav(n, **kw):
    from basilisk_env_b200.opnav_env import OpNavVecEnv
    return OpNavVecEnv(n, device=0, **kw)


def _step(env, a):
    o, r, d, info = env.step(a)
    return [x.clone() for x in (o, r, d, info["done_reason"], info["terminal_obs"], info["episode_r"], info["episode_l"])]


def _same_stats(a, b):
    assert {k: v for k, v in a.items() if k != "return_sum"} == {k: v for k, v in b.items() if k != "return_sum"}
    assert abs(a["return_sum"] - b["return_sum"]) <= 1e-12 * max(1.0, abs(a["return_sum"]))


def _acts(steps, n, hi, seed):
    import torch
    g = torch.Generator("cuda").manual_seed(seed)
    return torch.randint(0, hi, (steps, n), dtype=torch.int32, device="cuda", generator=g)


# ---- 1. auto-reset == masked reset ------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["leo", "opnav_noise", "opnav_truth"])
@pytest.mark.parametrize("n", [4096, 60001])
def test_auto_reset_equals_masked_reset(kind, n):
    import torch
    steps, seed = 20, 23
    if kind == "leo":
        pool, mk, kw, hi = leo_pool(37, 1), _leo, dict(max_length=6), 3
    else:
        pool, mk, kw, hi = opnav_pool(29, 2), _opnav, dict(max_length=6, nav_noise=int(kind == "opnav_noise")), 2
    acts = _acts(steps, n, hi, 3)
    a, b = mk(n, seed=seed, auto_reset=True, **kw), mk(n, seed=seed, auto_reset=False, **kw)
    for env in (a, b):
        env.set_ic_pool(pool, assign="per_episode")
        env.reset()
    for t in range(steps):
        ra = _step(a, acts[t])
        rb = _step(b, acts[t])
        b.reset(seed=seed, mask=b.done)
        rb[0] = b.obs.clone()
        for k, (x, y) in enumerate(zip(ra, rb)):
            assert torch.equal(x, y), f"interval {t} {OUTS[k]}"
        assert torch.equal(a.ic_rows(), b.ic_rows()), t
        assert torch.equal(a.initial_conditions(), b.initial_conditions()), t
    Sa, Ia = a.get_state()
    Sb, Ib = b.get_state()
    assert torch.equal(Sa, Sb) and torch.equal(Ia, Ib)
    _same_stats(a.episode_stats(), b.episode_stats())
    assert bool((a.ic_rows() >= 0).all())
    for env in (a, b):
        env.close()


# ---- 2. pool rows == explicit ICs ------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["leo", "opnav"])
def test_pool_rows_equal_explicit_ics(kind):
    """An env that auto-resets from row r continues bit for bit as an env that reset_ics put at row r (opNav without
    navigation and pixel noise: both noise streams are keyed by the episode, which reset_ics does not advance)."""
    import torch
    n, seed = 4096, 5
    if kind == "leo":
        pool, mk, kw, hi, ep_name = leo_pool(53, 7), _leo, dict(max_length=4), 3, "episode"
        from basilisk_env_b200 import _native
        ep_field = _native.state_field(ep_name)[0]
    else:
        pool, mk, kw, hi = opnav_pool(31, 8), _opnav, dict(max_length=4, nav_noise=0, pixel_noise_std=0.0), 2
        from basilisk_env_b200 import _native
        ep_field = _native.opnav_state_field("episode")[0]
    acts = _acts(12, n, hi, 9)
    a = mk(n, seed=seed, auto_reset=True, **kw)
    a.set_ic_pool(pool, assign="per_episode")
    a.reset()
    t = 0
    while True:
        a.step(acts[t]); t += 1
        fresh = a.done.clone().bool()
        if int(fresh.sum()) > n // 2:
            break
        assert t < 8
    rows = a.ic_rows()
    assert bool((rows >= 0).all())
    want = torch.as_tensor(pool, device="cuda")[rows.long()]
    assert torch.equal(a.initial_conditions()[fresh], want[fresh])
    b = mk(n, seed=seed, auto_reset=True, **kw)
    b.reset_ics(want)
    assert bool((b.ic_rows() == -1).all())
    Sa, Ia = a.get_state(); Sb, Ib = b.get_state()
    keep = torch.ones(Ia.shape[0], dtype=torch.bool); keep[ep_field] = False
    assert torch.equal(Sa[:, fresh], Sb[:, fresh]) and torch.equal(Ia[keep][:, fresh], Ib[keep][:, fresh])
    live = fresh.clone()
    for s in range(2):
        ra, rb = _step(a, acts[t + s]), _step(b, acts[t + s])
        for k in (1, 2, 3, 5, 6):
            assert torch.equal(ra[k][live], rb[k][live]), f"{OUTS[k]} {s}"
        live &= ~a.done.bool()
        assert torch.equal(ra[0][live], rb[0][live])
        Sa, Ia = a.get_state(); Sb, Ib = b.get_state()
        assert torch.equal(Sa[:, live], Sb[:, live]) and torch.equal(Ia[keep][:, live], Ib[keep][:, live])
    assert int(live.sum()) > 0
    a.close(); b.close()


# ---- 3. oracle parity -------------------------------------------------------------------------------------------------
def _perigee_altitude(rows):
    mu = 3.986004415e14
    r, v = rows[:, 0:3], rows[:, 3:6]
    a = -mu / (2.0 * (0.5 * (v * v).sum(1) - mu / np.linalg.norm(r, axis=1)))
    h = np.cross(r, v)
    ecc = np.sqrt(np.maximum(0.0, 1.0 - (h * h).sum(1) / (mu * a)))
    return a * (1.0 - ecc) - 6378136.6


@pytest.mark.parametrize("scenario", [False, True])
def test_auto_reset_from_pool_matches_the_oracle(orc, scenario):
    """64 LEO envs auto-reset from a dispersed IC pool (perigee above 200 km, as in test_param_pool_gpu.py) and run on
    against the oracle started from their rows.  With `scenario` the pool is paired with a dispersed parameter pool
    (param_row, per-env kernel) and the oracle gets each env's parameters too."""
    import torch
    n, steps = 64, 6
    rows = parity.sample_rows(orc, 4 * n, seed=61)
    pool = rows[_perigee_altitude(rows) > 200e3][:48]
    assert len(pool) == 48
    env = _leo(n, seed=3, auto_reset=True, max_length=8)
    if scenario:
        from tests import oracle_params as orp
        orp.lib()
        params = orp.dispersed_pool(48, seed=62)
        env.set_param_pool(params, assign="per_episode")
        env.set_ic_pool(pool, assign="param_row")
    else:
        env.set_ic_pool(pool, assign="per_episode")
    env.reset()
    env.step(torch.zeros(n, dtype=torch.int32, device="cuda"))
    env.reset(mask=torch.ones(n, dtype=torch.uint8, device="cuda"))     # every env from a pool row
    r = env.ic_rows().cpu().numpy()
    if scenario:
        assert np.array_equal(r, env.env_params()[1].cpu().numpy())
        ora = orp.LeoEnvBatchParams(pool[r], params[r], max_length=8)
        assert env.kernel_name().startswith("leo_step_penv_kernel")
    else:
        ora = orc.LeoEnvBatch(pool[r], max_length=8)
    np.testing.assert_allclose(env.obs.cpu().numpy(), ora.obs0, rtol=1e-14, atol=0)
    acts = (np.arange(n)[None, :] + np.arange(steps)[:, None]) % 3
    alive = np.ones(n, bool)            # an env that fails early is auto-reset on the GPU only: compared up to its end
    for t in range(steps):
        o, rw, d, info = env.step(torch.as_tensor(acts[t], dtype=torch.int32, device="cuda"))
        o, rw, d, why = o.cpu().numpy(), rw.cpu().numpy(), d.cpu().numpy(), info["done_reason"].cpu().numpy()
        S, I = (x.cpu().numpy() for x in env.get_state())
        o_ob, o_rew, o_done, o_reason = ora.step(acts[t])
        for e, st in enumerate(e_.state() for e_ in ora.envs):
            if not alive[e]:
                continue
            where = f"interval {t} env {e}"
            assert bool(d[e]) == o_done[e] and why[e] == o_reason[e], where
            assert abs(rw[e] - o_rew[e]) <= 1e-12, where
            if d[e]:
                alive[e] = False
                continue
            parity.compare_obs(o[e], o_ob[e], where)
            parity.compare_state(st, S[:, e], I[:, e], where)
    assert alive.sum() >= n // 2
    env.close()


# ---- 4. organisations and configurations ------------------------------------------------------------------------------
def _org_run(n, org, pool, acts, **kw):
    env = _leo(n, seed=31, auto_reset=True, organisation=org, max_length=3, **kw)
    env.set_ic_pool(pool, assign="per_episode")
    env.reset()
    outs = [_step(env, a) for a in acts]
    res = (outs, env.get_state(), env.ic_rows().clone(), env.initial_conditions().clone(), env.kernel_name())
    env.close()
    return res


def _same_runs(a, b):
    import torch
    for t in range(len(a[0])):
        for k, (x, y) in enumerate(zip(a[0][t], b[0][t])):
            assert torch.equal(x, y), f"interval {t} {OUTS[k]}"
    assert torch.equal(a[1][0], b[1][0]) and torch.equal(a[1][1], b[1][1])
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])


def test_organisations_and_configurations():
    import torch
    n = 4096
    pool = leo_pool(41, 11)
    acts = _acts(7, n, 3, 12)
    runs = {org: _org_run(n, org, pool, acts) for org in ("thread", "thread_index", "split")}
    assert runs["split"][4].startswith("leo_split_kernel") and runs["thread"][4].startswith("leo_step_kernel")
    _same_runs(runs["thread"], runs["thread_index"])
    _same_runs(runs["thread"], runs["split"])
    stress = {org: _org_run(n, org, pool, acts, rw_set=1, use_j2=1) for org in ("thread", "split")}
    assert stress["split"][4] == "leo_split_kernel<4,1,false>"
    _same_runs(stress["thread"], stress["split"])
    mixed = _org_run(n, "auto", pool, acts, precision=1)
    rows, ics = mixed[2], mixed[3]
    assert bool((rows >= 0).all()) and ",true," in mixed[4]
    assert torch.equal(ics, torch.as_tensor(pool, device="cuda")[rows.long()])


# ---- 5. assignment ----------------------------------------------------------------------------------------------------
def test_by_index_and_per_episode_sharding():
    import torch
    n, k0, m, K, seed, steps = 600, 200, 150, 7, 99, 5
    pool = leo_pool(K, 13)
    env = _leo(n, seed=seed, first_env_index=1000)
    env.set_ic_pool(pool, assign="by_index")
    env.reset()
    assert env.ic_rows().cpu().tolist() == [(1000 + e) % K for e in range(n)]
    acts = _acts(steps, n, 3, 14)
    big, shard = _leo(n, seed=seed, auto_reset=True, max_length=2), _leo(m, first_env_index=k0, seed=seed, auto_reset=True, max_length=2)
    from basilisk_env_b200 import _native
    ep_field = _native.state_field("episode")[0]
    for e in (big, shard):
        e.set_ic_pool(pool, assign="per_episode")
        e.reset()
    for t in range(steps + 1):
        ep = big.get_state()[1][ep_field].cpu().numpy()
        rows = big.ic_rows()
        assert rows.cpu().tolist() == [ic_per_episode_row(K, seed, e, int(ep[e])) for e in range(n)], t
        assert torch.equal(shard.ic_rows(), rows[k0:k0 + m])
        assert torch.equal(shard.initial_conditions(), big.initial_conditions()[k0:k0 + m])
        if t < steps:
            big.step(acts[t]); shard.step(acts[t, k0:k0 + m])
    for e in (env, big, shard):
        e.close()


def test_param_row_pairs_the_pools_and_scenarios_round_trip():
    import torch
    from basilisk_env_b200 import initial_conditions as icm
    n, K = 500, 9
    rng = np.random.RandomState(15)
    dicts = [icm.set_ICs(rng) for _ in range(K)]
    for j, d in enumerate(dicts):
        d["mass"] = 300.0 + 5 * j
        d["storageCapacity"] = (14.0 + j) * 3600.
        d["storedCharge_Init"] = min(d["storedCharge_Init"], d["storageCapacity"])
    env = _leo(n, seed=4, auto_reset=True, max_length=2)
    env.set_scenario_pool(dicts, assign="per_episode")
    env.reset()
    acts = _acts(6, n, 3, 16)
    for t in range(7):
        rows = env.ic_rows()
        params, prow = env.env_params()
        assert torch.equal(rows, prow), t
        r = rows.cpu().numpy()
        want = np.stack([icm.ic_row(dicts[j]) for j in r])
        np.testing.assert_array_equal(env.initial_conditions().cpu().numpy(), want)
        np.testing.assert_array_equal(params["mass"].cpu().numpy(), [dicts[j]["mass"] for j in r])
        np.testing.assert_array_equal(params["storageCapacity"].cpu().numpy(), [dicts[j]["storageCapacity"] for j in r])
        if t < 6:
            env.step(acts[t])
    assert len(set(r.tolist())) > 1
    bad = [dict(d) for d in dicts]
    bad[3]["Ki"] = -2.0
    with pytest.raises(ValueError, match="scenario 3: 'Ki'"):
        env.set_scenario_pool(bad)
    env.close()


# ---- 6. no behaviour change without a pool ---------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4096, 60001])
def test_unloaded_pool_changes_nothing(n):
    import torch
    acts = _acts(8, n, 3, 17)
    res, launches = [], []
    for mode in ("never", "unloaded", "loaded"):
        env = _leo(n, seed=8, auto_reset=True, max_length=3)
        if mode != "never":
            env.set_ic_pool(leo_pool(5, 18), assign="by_index")
        if mode == "unloaded":
            env.set_ic_pool(None)
        env.reset()
        c0 = env.launch_count()
        outs = [_step(env, a) for a in acts]
        launches.append(env.launch_count() - c0)
        res.append((outs, env.get_state(), env.episode_stats(), env.kernel_name(), env.ic_rows().clone()))
        env.close()
    a, b, c = res
    for t in range(len(acts)):
        for k, (x, y) in enumerate(zip(a[0][t], b[0][t])):
            assert torch.equal(x, y), f"interval {t} {OUTS[k]}"
    assert torch.equal(a[1][0], b[1][0]) and torch.equal(a[1][1], b[1][1])
    _same_stats(a[2], b[2])
    assert a[3] == b[3] == c[3]
    assert launches[0] == launches[1] and launches[2] == launches[0] + len(acts)
    assert bool((a[4] == -1).all()) and bool((b[4] == -1).all()) and bool((c[4] >= 0).all())


def test_unload_after_use_reports_sampled_episodes():
    """After an unload, envs that the in-kernel auto-reset restarted report -1; the others keep their row."""
    n = 256
    env = _leo(n, seed=2, auto_reset=True, max_length=2)
    env.set_ic_pool(leo_pool(4, 19), assign="by_index")
    env.reset()
    assert env.ic_rows().cpu().tolist() == [e % 4 for e in range(n)]
    env.set_ic_pool(None)
    acts = _acts(4, n, 3, 20)
    finished = np.zeros(n, bool)
    for t in range(4):
        env.step(acts[t])
        finished |= env.done.cpu().numpy().astype(bool)
    rows = env.ic_rows().cpu().numpy()
    assert finished.any()
    assert (rows[finished] == -1).all() and (rows[~finished] == np.arange(n)[~finished] % 4).all()
    env.close()


# ---- 7. host-buffer paths ----------------------------------------------------------------------------------------------
def test_host_buffer_paths_with_a_pool():
    import torch
    n, steps = 4096, 6
    pool = leo_pool(23, 21)
    acts = _acts(steps, n, 3, 22)
    envs = []
    for _ in range(4):
        env = _leo(n, seed=6, auto_reset=True, max_length=2)
        env.set_ic_pool(pool)
        env.reset()
        envs.append(env)
    dev, pinned, pageable, asy = envs
    a_pin, out_pin = pinned.host_buffers(episode=True)
    out_pg = tuple(np.empty_like(x) for x in out_pin)
    a_sp, out_sp = asy.host_buffers(episode=True)
    for t in range(steps):
        d = _step(dev, acts[t])
        np.copyto(a_pin, acts[t].cpu().numpy())
        pinned.step_host(a_pin, out_pin)
        pageable.step_host(acts[t].cpu().numpy(), out_pg)
        np.copyto(a_sp, acts[t].cpu().numpy())
        asy.step_host_async(a_sp, out_sp)
        asy.step_host_wait()
        want = [x.cpu().numpy() for x in d]
        for out in (out_pin, out_pg, out_sp):
            got = [out[0], out[1], out[2], out[3], out[6], out[4], out[5]]
            done = want[2].astype(bool)
            for k in range(7):
                w, g = want[k], got[k]
                if k == 4:             # terminal_obs: rows of finished envs only
                    w, g = w[done], g[done]
                np.testing.assert_array_equal(g, w, err_msg=f"interval {t} {OUTS[k]}")
    rows = dev.ic_rows()
    for env in envs:
        assert torch.equal(env.ic_rows(), rows)
    for env in envs:
        env.close()


def test_sb_vec_env_reaches_the_pool():
    import torch
    from basilisk_env_b200.sb_vec_env import LeoPowerAttSBVecEnv
    n = 300
    pool = leo_pool(11, 24)
    sb = LeoPowerAttSBVecEnv(n, seed=12, max_length=2)
    sb.env_method("set_ic_pool", pool, assign="per_episode")
    sb.reset()
    seen = 0
    for t in range(4):
        obs, rew, dones, infos = sb.step(np.zeros(n, np.int64))
        if dones.any():
            rows = sb.vec.ic_rows()
            ref = _leo(n)
            ref.reset_ics(torch.as_tensor(pool, device="cuda")[rows.long()])
            first = ref.obs.cpu().numpy()
            ref.close()
            for e in np.flatnonzero(dones):
                assert "terminal_observation" in infos[e] and "episode" in infos[e]
                np.testing.assert_array_equal(obs[e, :, 0], first[e])
                assert not np.array_equal(infos[e]["terminal_observation"][:, 0], first[e])
            seen += int(dones.sum())
    assert seen >= n
    sb.close()


# ---- 8. refusals ------------------------------------------------------------------------------------------------------
def test_refusals():
    from basilisk_env_b200.vec_env import BskEnvError
    env = _leo(64, auto_reset=True)
    pool = leo_pool(6, 25)
    bad = pool.copy(); bad[4, 7] = np.nan
    with pytest.raises(BskEnvError, match="row 4: non-finite"):
        env.set_ic_pool(bad)
    bad = pool.copy(); bad[2, :3] = 0.0
    with pytest.raises(BskEnvError, match="row 2: zero position"):
        env.set_ic_pool(bad)
    rows = np.ascontiguousarray(pool)
    assert env._L.bskenv_set_ic_pool(env._h, 6, rows.ctypes.data, 7) == -1
    assert "unknown assignment mode" in env._L.bskenv_last_error(env._h).decode()
    with pytest.raises(BskEnvError, match="same row count"):
        env.set_ic_pool(pool, assign="param_row")
    from tests import oracle_params as orp
    orp.lib()
    env.set_param_pool(orp.dispersed_pool(5, seed=1))
    with pytest.raises(BskEnvError, match="same row count"):
        env.set_ic_pool(pool, assign="param_row")
    env.set_param_pool(orp.dispersed_pool(6, seed=1))
    env.set_ic_pool(pool, assign="param_row")
    env.set_param_pool(orp.dispersed_pool(6, seed=2))               # same row count: allowed
    for change in (orp.dispersed_pool(5, seed=1), None):
        with pytest.raises(BskEnvError, match="paired"):
            env.set_param_pool(change)
    env.reset()
    a, out = env.host_buffers()
    env.step_host_async(a, out)
    with pytest.raises(BskEnvError, match="host-buffer step is in flight"):
        env.set_ic_pool(pool, assign="by_index")
    env.step_host_wait()
    env.set_ic_pool(None)
    env.set_param_pool(None)
    env.close()
    on = _opnav(64)
    with pytest.raises(BskEnvError, match="unknown assignment mode"):
        on._check(on._L.bskenv_opnav_set_ic_pool(on._h, 2, np.ascontiguousarray(opnav_pool(2, 1)).ctypes.data, 2),
                  "bskenv_opnav_set_ic_pool")
    bad = opnav_pool(3, 2); bad[1, 11] = np.inf
    with pytest.raises(BskEnvError, match="row 1: non-finite"):
        on.set_ic_pool(bad)
    on.close()
