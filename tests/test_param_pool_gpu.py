"""Per-env spacecraft parameters on the GPU (LeoPowerAttVecEnv.set_param_pool, include/bskenv.h bskenv_set_param_pool):
identity of a one-row default pool with the batch-global kernels, parity of dispersed rows with the oracle, the row
assignment, lane-order independence, and the refused configurations."""
import numpy as np
import pytest

from tests import parity

pytestmark = pytest.mark.gpu


def _vec(n, **kw):
    from basilisk_env_b200.vec_env import LeoPowerAttVecEnv
    return LeoPowerAttVecEnv(n, device=0, **kw)


@pytest.fixture(scope="module")
def orp():
    from tests import oracle_params
    oracle_params.lib()
    return oracle_params


def _same_stats(a, b):
    """Episode statistics: the counts exactly; the sum of returns is accumulated with floating-point atomics in whatever order
    the warps finish, so it agrees to rounding only."""
    assert {k: v for k, v in a.items() if k != "return_sum"} == {k: v for k, v in b.items() if k != "return_sum"}
    assert abs(a["return_sum"] - b["return_sum"]) <= 1e-12 * max(1.0, abs(a["return_sum"]))


def _run(env, acts):
    outs = []
    for a in acts:
        o, r, d, info = env.step(a)
        outs.append([x.clone() for x in (o, r, d, info["done_reason"], info["terminal_obs"], info["episode_r"], info["episode_l"])])
    S, I = env.get_state()
    return outs, S.clone(), I.clone(), env.episode_stats(), env.kernel_name()


@pytest.mark.parametrize("n", [4096, 60001])
def test_default_row_pool_is_bit_identical(bsk, orp, n):
    """A pool of one row equal to the configuration: every output, the full state and the episode statistics are those of
    the handle without a pool, over 20 intervals with in-kernel auto-reset (60001 envs: queued, action-bucketed path)."""
    import torch
    steps = 20
    g = torch.Generator("cuda").manual_seed(7)
    acts = torch.randint(0, 3, (steps, n), dtype=torch.int32, device="cuda", generator=g)
    res = []
    for pool in (None, orp.DEFAULT_ROW[None, :]):
        env = _vec(n, seed=5, auto_reset=True, max_length=6)
        if pool is not None:
            env.set_param_pool(pool, assign="per_episode")
        env.reset()
        res.append(_run(env, acts))
        if pool is not None:
            params, row = env.env_params()
            assert bool((row == 0).all())
            for j, k in enumerate(orp.PARAM_KEYS):
                assert bool((params[k] == float(orp.DEFAULT_ROW[j])).all()), k
        env.close()
    a, b = res
    assert b[4].startswith("leo_step_penv_kernel<3,0,true,") and not a[4].startswith("leo_step_penv")
    for t in range(steps):
        for k, (x, y) in enumerate(zip(a[0][t], b[0][t])):
            assert torch.equal(x, y), f"interval {t} output {k}"
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    _same_stats(a[3], b[3])
    assert a[3]["episodes"] >= n


def test_dispersed_by_index_pool_matches_the_oracle(bsk, orc, orp):
    """256 envs, row e = env e of a dispersed BY_INDEX pool, scripted actions 0 / 1 / 2, eight intervals: every env against
    the oracle built with its own row.  Orbits with a perigee above 200 km: below it the drag torque (up to twice the
    reference density here) amplifies rounding differences of the attitude by ~100x per interval, the regime that
    tests/test_gpu_round2.py bounds separately."""
    import torch
    n, steps = 256, 8
    rows = parity.sample_rows(orc, 2 * n, seed=71)
    rows = rows[_perigee_altitude(rows) > 200e3][:n]
    assert len(rows) == n
    params = orp.dispersed_pool(n, seed=72)
    env = _vec(n)
    env.set_param_pool(params, assign="by_index")
    ob = env.reset_ics(rows).cpu().numpy()
    ora = orp.LeoEnvBatchParams(rows, params)
    np.testing.assert_allclose(ob, ora.obs0, rtol=1e-14, atol=0)     # reset obs: norms, FMA-contracted on the GPU
    got, row = env.env_params()
    assert row.cpu().tolist() == list(range(n))
    np.testing.assert_array_equal(np.stack([got[k].cpu().numpy() for k in orp.PARAM_KEYS], axis=1), params)
    acts = (np.arange(n)[None, :] + np.arange(steps)[:, None]) % 3
    for t in range(steps):
        o, r, d, info = env.step(torch.as_tensor(acts[t], dtype=torch.int32, device="cuda"))
        o, r, d, why = o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy(), info["done_reason"].cpu().numpy()
        S, I = (x.cpu().numpy() for x in env.get_state())
        o_ob, o_rew, o_done, o_reason = ora.step(acts[t])
        for e, st in enumerate(ora.states()):
            where = f"interval {t} env {e} action {acts[t, e]}"
            parity.compare_obs(o[e], o_ob[e], where)
            assert bool(d[e]) == o_done[e] and why[e] == o_reason[e], where
            assert abs(r[e] - o_rew[e]) <= 1e-12, where
            parity.compare_state(st, S[:, e], I[:, e], where)
    assert env.kernel_name().startswith("leo_step_penv_kernel")
    env.close()


def _perigee_altitude(rows):
    mu = 3.986004415e14
    r, v = rows[:, 0:3], rows[:, 3:6]
    a = -mu / (2.0 * (0.5 * (v * v).sum(1) - mu / np.linalg.norm(r, axis=1)))
    h = np.cross(r, v)
    ecc = np.sqrt(np.maximum(0.0, 1.0 - (h * h).sum(1) / (mu * a)))
    return a * (1.0 - ecc) - 6378136.6


# Philox4x32-10 (Salmon et al., SC'11), restated independently of the library
def _philox(c, k):
    c, k = [int(x) & 0xFFFFFFFF for x in c], [int(x) & 0xFFFFFFFF for x in k]
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, ((p0 >> 32) ^ c[3] ^ k[1]) & 0xFFFFFFFF, p0 & 0xFFFFFFFF]
        k = [(k[0] + 0x9E3779B9) & 0xFFFFFFFF, (k[1] + 0xBB67AE85) & 0xFFFFFFFF]
    return c


def per_episode_row(n_rows, seed, global_env, episode):
    """The documented PER_EPISODE selection (include/bskenv.h): one Philox4x32-10 block at counter (global env, episode,
    0xFFFFFFFF), key = seed; row = (word1:word0) mod n_rows."""
    o = _philox([global_env, global_env >> 32, episode, 0xFFFFFFFF], [seed, seed >> 32])
    return ((o[1] << 32) | o[0]) % n_rows


def test_per_episode_assignment_sharding_and_ics(bsk, orp):
    """PER_EPISODE with auto-reset: the rows are the documented selection of (seed, global env, episode), the same for a
    shard at first_env_index = k as for the matching slice of a larger handle; the initial conditions are bit-identical to
    a run without a pool; reset_init keeps every env's row."""
    import torch
    n, k0, m, K, seed, steps = 600, 200, 150, 7, 99, 7
    pool = orp.dispersed_pool(K, seed=3)
    g = torch.Generator("cuda").manual_seed(1)
    acts = torch.randint(0, 3, (steps, n), dtype=torch.int32, device="cuda", generator=g)
    big, shard, plain = (_vec(n, seed=seed, auto_reset=True, max_length=2), _vec(m, first_env_index=k0, seed=seed, auto_reset=True, max_length=2),
                         _vec(n, seed=seed, auto_reset=True, max_length=2))
    big.set_param_pool(pool); shard.set_param_pool(pool)
    for env in (big, shard, plain):
        env.reset()
    from basilisk_env_b200 import _native
    ep_field = _native.state_field("episode")[0]
    for t in range(steps + 1):
        params, row = big.env_params()
        sp, srow = shard.env_params()
        ep = big.get_state()[1][ep_field].cpu().numpy()
        want = [per_episode_row(K, seed, e, int(ep[e])) for e in range(n)]
        assert row.cpu().tolist() == want, f"interval {t}"
        assert torch.equal(srow, row[k0:k0 + m])
        for j, key in enumerate(orp.PARAM_KEYS):
            np.testing.assert_array_equal(params[key].cpu().numpy(), pool[np.array(want), j])
            assert torch.equal(sp[key], params[key][k0:k0 + m])
        # the IC stream is that of the run without a pool: equal wherever the env is in the same episode in both runs (the
        # dispersed parameters may end an episode early by a wheel or power failure)
        same = torch.as_tensor(ep == plain.get_state()[1][ep_field].cpu().numpy())
        assert bool(same.all()) if t == 0 else float(same.double().mean()) > 0.9, f"interval {t}"
        ics_b, ics_p = big.initial_conditions().cpu(), plain.initial_conditions().cpu()
        assert torch.equal(ics_b[same], ics_p[same]), f"interval {t}"
        assert torch.equal(shard.initial_conditions().cpu(), ics_b[k0:k0 + m])
        if t < steps:
            for env, a in ((big, acts[t]), (shard, acts[t, k0:k0 + m]), (plain, acts[t])):
                env.step(a)
    assert len(set(want)) == K
    before = big.env_params()
    big.reset_init()
    after = big.env_params()
    assert torch.equal(before[1], after[1]) and all(torch.equal(before[0][k], after[0][k]) for k in orp.PARAM_KEYS)
    for env in (big, shard, plain):
        env.close()


def test_pool_lane_orders_are_bit_identical(bsk, orp):
    """With a pool, the action-bucketed lanes and lanes in index order give the same bits (60001 envs, auto-reset)."""
    import torch
    n, steps = 60001, 6
    g = torch.Generator("cuda").manual_seed(11)
    acts = torch.randint(0, 3, (steps, n), dtype=torch.int32, device="cuda", generator=g)
    acts[3] = 2
    res = {}
    for org in ("thread", "thread_index"):
        env = _vec(n, seed=17, auto_reset=True, organisation=org, max_length=3)
        env.set_param_pool(orp.dispersed_pool(33, seed=2), assign="per_episode")
        env.reset()
        res[org] = _run(env, acts) + (env.env_params()[1].clone(),)
        env.close()
    a, b = res["thread"], res["thread_index"]
    assert a[4] == b[4] and a[4].startswith("leo_step_penv_kernel")
    for t in range(steps):
        for x, y in zip(a[0][t], b[0][t]):
            assert torch.equal(x, y), t
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[5], b[5])
    _same_stats(a[3], b[3])


def test_refused_configurations_and_unload(bsk, orp):
    import ctypes as C
    from basilisk_env_b200.vec_env import BskEnvError
    pool = orp.dispersed_pool(4, seed=0)
    for cfg in (dict(rw_set=1, use_j2=1), dict(precision=1)):
        env = _vec(64, **cfg)
        with pytest.raises(BskEnvError, match="per-env parameters"):
            env.set_param_pool(pool)
        env.close()
    env = _vec(64)
    env.set_gravity_degree2(True)
    with pytest.raises(BskEnvError, match="degree-2"):
        env.set_param_pool(pool)
    env.set_gravity_degree2(False)
    env.set_organisation("split")
    with pytest.raises(BskEnvError, match="split"):
        env.set_param_pool(pool)
    env.set_organisation("auto")
    env.set_param_pool(pool)
    with pytest.raises(BskEnvError, match="split"):
        env.set_organisation("split")
    with pytest.raises(BskEnvError, match="parameter pool"):
        env.set_gravity_degree2(True)
    bad = pool.copy(); bad[2, 0] = -1.0
    with pytest.raises(BskEnvError, match="row 2"):
        env.set_param_pool(bad)
    rows = np.ascontiguousarray(pool)
    assert env._L.bskenv_set_param_pool(env._h, 4, rows.ctypes.data, 5) == -1
    assert "assignment mode" in env._L.bskenv_last_error(env._h).decode()
    env.reset(seed=3)
    env.step(np.zeros(64, np.int32))
    assert env.kernel_name().startswith("leo_step_penv_kernel")
    env.set_param_pool(None)
    env.reset(seed=3)
    env.step(np.zeros(64, np.int32))
    assert env.kernel_name().startswith("leo_step_kernel") or env.kernel_name().startswith("leo_split_kernel")
    params, row = env.env_params()
    assert bool((row == -1).all()) and float(params["mass"][0]) == 330.0
    env.close()


def test_dict_pool_fills_missing_keys_from_the_configuration(bsk):
    """A pool given as a dict of reference keys: the keys it leaves out take the handle's configuration values."""
    env = _vec(70, storageCapacity=10.0 * 3600.)
    env.set_param_pool({"mass": [300.0, 360.0], "K": [6.0, 8.0]}, assign="by_index")
    env.reset(seed=1)
    params, row = env.env_params()
    assert row.cpu().tolist() == [e % 2 for e in range(70)]
    assert params["mass"].cpu().tolist() == [300.0 if e % 2 == 0 else 360.0 for e in range(70)]
    assert params["K"].cpu().tolist() == [6.0 if e % 2 == 0 else 8.0 for e in range(70)]
    assert bool((params["storageCapacity"] == 36000.0).all()) and bool((params["width"] == 1.38).all())
    with pytest.raises(KeyError):
        env.set_param_pool({"Ki": [-1.0]})
    env.close()
