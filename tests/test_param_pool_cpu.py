"""CPU suite of the per-env spacecraft parameters (bskenv_set_param_pool): the per-env policy of the device core, compiled
for the host, against the batch-global core (bit for bit) and against the oracle with each env's parameter set; the C ABI
declarations; and the registers / spills of the batch-global step kernels, which the per-env kernel must leave alone."""
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from tests import parity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hcp():
    from tests import hostcore_penv
    hostcore_penv.lib()
    return hostcore_penv


@pytest.fixture(scope="module")
def orp():
    from tests import oracle_params
    oracle_params.lib()
    return oracle_params


def test_default_row_is_bit_identical_to_the_batch_core(orc, hcp, orp):
    """A parameter block holding the configuration's own values: the per-env core computes exactly what the batch-global
    core computes, over several intervals with all three actions (desat included)."""
    n = 8
    rows = parity.sample_rows(orc, n, seed=21)
    rng = np.random.RandomState(4)
    acts = rng.randint(0, 3, size=(7, n))
    acts[1] = 2
    a, b = hcp.HostCorePenv(n), hcp.HostCorePenv(n)
    a.set_env_params(np.tile(orp.DEFAULT_ROW, (n, 1)))
    np.testing.assert_array_equal(a.reset_ics(rows), b.reset_ics(rows))
    for t in range(len(acts)):
        ra = a.step(acts[t], per_env=True)
        rb = b.step(acts[t], per_env=False)
        for x, y in zip(ra, rb):
            np.testing.assert_array_equal(x, y, err_msg=f"interval {t}")
        Sa, Ia = a.state()
        Sb, Ib = b.state()
        np.testing.assert_array_equal(Sa, Sb)
        np.testing.assert_array_equal(Ia, Ib)


def test_dispersed_rows_match_the_oracle(orc, hcp, orp):
    """32 envs, each with its own mass, dimensions, atmosphere, power system, gains and disturbance magnitude: the per-env
    core against the oracle built with the same dict values (tests/parity.py tolerances), every action."""
    n = 32
    rows = parity.sample_rows(orc, n, seed=33)
    params = orp.dispersed_pool(n, seed=5)
    rng = np.random.RandomState(9)
    acts = rng.randint(0, 3, size=(5, n))
    acts[0, : n // 3] = 2
    hc = hcp.HostCorePenv(n)
    hc.set_env_params(params)
    ob_h = hc.reset_ics(rows)
    ora = orp.LeoEnvBatchParams(rows, params)
    np.testing.assert_array_equal(ob_h, ora.obs0)
    worst = {}
    for t in range(len(acts)):
        obs, rew, done, reason = hc.step(acts[t])
        o_ob, o_rew, o_done, o_reason = ora.step(acts[t])
        S, I = hc.state()
        for e, st in enumerate(ora.states()):
            where = f"interval {t} env {e} action {acts[t, e]}"
            parity.compare_obs(obs[e], o_ob[e], where)
            assert done[e] == o_done[e] and reason[e] == o_reason[e], where
            assert abs(rew[e] - o_rew[e]) <= 1e-12, where
            for k, v in parity.compare_state(st, S[:, e], I[:, e], where).items():
                worst[k] = max(worst.get(k, 0.0), v)
    assert max(worst.values()) <= parity.RTOL


def test_dispersion_reaches_the_dynamics(orc, hcp, orp):
    """The dispersed rows are not a no-op: the same ICs under the batch configuration end up elsewhere."""
    n = 8
    rows = parity.sample_rows(orc, n, seed=3)
    a, b = hcp.HostCorePenv(n), hcp.HostCorePenv(n)
    a.set_env_params(orp.dispersed_pool(n, seed=1))
    a.reset_ics(rows); b.reset_ics(rows)
    acts = np.zeros(n, np.int32)
    a.step(acts); b.step(acts, per_env=False)
    Sa, _ = a.state()
    Sb, _ = b.state()
    assert np.all(np.any(Sa != Sb, axis=0))


@pytest.mark.parametrize("col, value", [(0, 0.0), (1, -1.0), (3, 0.0), (5, 0.0), (10, -3600.0), (11, np.nan)])
def test_invalid_rows_are_refused(hcp, orp, col, value):
    hc = hcp.HostCorePenv(2)
    raw = np.tile(orp.DEFAULT_ROW, (2, 1))
    raw[1, col] = value
    with pytest.raises(ValueError):
        hc.set_env_params(raw)


def test_pool_row_selection(hcp):
    """BY_INDEX is the global index mod K; PER_EPISODE depends on (seed, global env, episode) only -- so a shard starting at
    first_env_index = k sees the rows of the matching slice -- and spreads over every row."""
    assert [hcp.pool_row(5, 0, 0, g, 1) for g in range(12)] == [g % 5 for g in range(12)]
    k = 64
    draws = np.array([[hcp.pool_row(k, 1, 17, g, ep) for g in range(400)] for ep in (1, 2)])
    assert draws.min() >= 0 and draws.max() < k
    assert len(np.unique(draws)) == k                                       # 800 draws cover all 64 rows
    assert np.mean(draws[0] == draws[1]) < 0.1                              # a new episode draws anew
    assert hcp.pool_row(k, 1, 17, 123, 2) == draws[1, 123]
    assert any(hcp.pool_row(k, 1, 18, g, 1) != draws[0, g] for g in range(50))   # keyed by the seed


def test_param_keys_match_the_abi():
    """initial_conditions.PARAM_KEYS, bskenv.h (BSKENV_PARAM_DIM, the assignment modes, the prototypes) and _native agree."""
    from basilisk_env_b200 import _native
    from basilisk_env_b200.initial_conditions import PARAM_KEYS, CONFIG_KEYS
    hdr = open(os.path.join(ROOT, "include", "bskenv.h")).read()
    assert int(re.search(r"#define BSKENV_PARAM_DIM (\d+)", hdr).group(1)) == len(PARAM_KEYS) == 14
    assert int(re.search(r"#define BSKENV_PARAMS_BY_INDEX (\d+)", hdr).group(1)) == 0
    assert int(re.search(r"#define BSKENV_PARAMS_PER_EPISODE (\d+)", hdr).group(1)) == 1
    assert set(PARAM_KEYS) <= set(CONFIG_KEYS)
    assert all(k in dict(_native.Config._fields_) for k in PARAM_KEYS)
    for fn, nargs in (("bskenv_set_param_pool", 4), ("bskenv_get_env_params", 4)):
        m = re.search(r"\bint " + fn + r"\(([^;]*)\);", hdr, re.S)
        assert m, fn
        assert len(re.sub(r"/\*.*?\*/", "", m.group(1)).split(",")) == nargs, fn
        assert fn in _native.EXPORTS
    order = re.search(r"A row is\s+\* BSKENV_PARAM_DIM doubles.*?order:\s*\*(.*?)\n \* Everything", hdr, re.S).group(1)
    assert [k.strip() for k in order.replace("*", "").split(",")] == list(PARAM_KEYS)


def _entries(ptxas_log):
    """-Xptxas -v figures of each step / split kernel entry, keyed by its template arguments."""
    out, full, cur, fn = {}, None, None, None
    for line in ptxas_log.splitlines():
        m = re.search(r"Compiling entry function '(\S+)' for", line)
        if m:
            full = m.group(1)
            k = re.search(r"\d+(leo_\w+_kernelI.*?EE)v", full)
            cur = k.group(1) if k else None
            continue
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur and fn == full:
            out.setdefault(cur, {}).update(zip(("stack", "spill_stores", "spill_loads"), map(int, m.groups())))
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            out.setdefault(cur, {})["registers"] = int(m.group(1))
    return out


def test_batch_global_step_kernels_keep_registers_and_spills(tmp_path):
    """Every batch-global step / split kernel compiles to the registers, stack frame and spill bytes it had before the
    per-env kernel existed (tests/golden/ptxas_leo_step_kernels.json), and the per-env kernel stays at the throughput
    organisation's 168 registers."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    from basilisk_env_b200 import build
    csrc = os.path.join(ROOT, "basilisk_env_b200", "csrc")
    r = subprocess.run([nvcc] + build.NVCC_FLAGS + ["-Xptxas", "-v", "-c", "-o", str(tmp_path / "bskenv.o"),
                                                    os.path.join(csrc, "bskenv.cu")], cwd=csrc, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    got = _entries(r.stderr + r.stdout)
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "ptxas_leo_step_kernels.json")))["kernels"]
    for k, v in want.items():
        assert got.get(k) == v, f"{k}: {got.get(k)} != {v}"
    penv = [v for k, v in got.items() if k.startswith("leo_step_penv_kernel")]
    assert len(penv) == 2 and all(v["registers"] == 168 for v in penv)
