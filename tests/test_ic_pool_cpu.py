"""CPU suite of the initial-condition pools (bskenv_set_ic_pool / bskenv_opnav_set_ic_pool): the C ABI declarations and
exports, the row selection and the row validation of the device core compiled for the host, and the conversion of reference
scenario dicts into (IC rows, parameter rows)."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hci():
    from tests import hostcore_icpool
    hostcore_icpool.lib()
    return hostcore_icpool


def test_header_declarations_and_exports():
    from basilisk_env_b200 import _native
    hdr = open(os.path.join(ROOT, "include", "bskenv.h")).read()
    for name, val in (("BSKENV_ICS_BY_INDEX", 0), ("BSKENV_ICS_PER_EPISODE", 1), ("BSKENV_ICS_PARAM_ROW", 2)):
        assert int(re.search(r"#define " + name + r" (\d+)", hdr).group(1)) == val
    for fn, nargs, exports in (("bskenv_set_ic_pool", 4, _native.EXPORTS), ("bskenv_get_ic_rows", 3, _native.EXPORTS),
                               ("bskenv_opnav_set_ic_pool", 4, _native.OPNAV_EXPORTS),
                               ("bskenv_opnav_get_ic_rows", 3, _native.OPNAV_EXPORTS)):
        m = re.search(r"\bint " + fn + r"\(([^;]*)\);", hdr, re.S)
        assert m, fn
        assert len(re.sub(r"/\*.*?\*/", "", m.group(1)).split(",")) == nargs, fn
        assert fn in exports, fn
    assert int(re.search(r"#define BSKENV_ABI_VERSION (\d+)", hdr).group(1)) == 1


def test_by_index_and_param_row_selection(hci):
    assert [hci.ic_pool_row(5, 0, 3, g, 1) for g in range(13)] == [g % 5 for g in range(13)]
    assert [hci.ic_pool_row(7, 2, 3, g, 4, param_row=g % 7) for g in range(20)] == [g % 7 for g in range(20)]


def test_per_episode_selection_has_its_own_stream(hci):
    """PER_EPISODE depends on (seed, global env, episode) only, covers every row, and is a different sequence from the
    parameter pool's PER_EPISODE rows for the same keys (its own Philox counter word)."""
    k = 64
    ic = np.array([[hci.ic_pool_row(k, 1, 17, g, ep) for g in range(400)] for ep in (1, 2)])
    par = np.array([[hci.param_pool_row(k, 1, 17, g, ep) for g in range(400)] for ep in (1, 2)])
    assert ic.min() >= 0 and ic.max() < k and len(np.unique(ic)) == k
    assert np.mean(ic == par) < 0.1                                         # not the parameter stream
    assert np.mean(ic[0] == ic[1]) < 0.1                                    # a new episode draws anew
    assert hci.ic_pool_row(k, 1, 17, 123, 2) == ic[1, 123]                  # a function of the keys: shards agree
    assert any(hci.ic_pool_row(k, 1, 18, g, 1) != ic[0, g] for g in range(50))
    from tests.test_ic_pool_gpu import ic_per_episode_row                  # the documented selection, restated
    assert [ic_per_episode_row(k, 17, g, 2) for g in range(400)] == ic[1].tolist()


# SHA-256 of the ICs the sampler drew for global envs 0..5, seed 41, episodes 1 and 2 ([12][19] float64) before the IC
# pools existed
_SAMPLE_IC_DIGEST = "6858bb241556290e3492e502221b1fcbce64fa1c7276c983e343207bf1aa92e7"


def test_sample_ic_is_unchanged(hci):
    """The built-in sampler the IC pool stands in for draws exactly what it drew before, bit for bit."""
    import hashlib
    from tests.hostcore_binding import default_config
    cfg = default_config()
    got = np.stack([hci.sample_ic(cfg, 41, e, ep) for ep in (1, 2) for e in range(6)])
    assert hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == _SAMPLE_IC_DIGEST
    assert got[0, 18] == pytest.approx(3.74781820e+04)


@pytest.mark.parametrize("dim", [19, 12])
def test_row_validation(hci, dim):
    row = np.arange(1.0, dim + 1.0)
    assert hci.ic_row_check(row) == ""
    for bad in (np.nan, np.inf, -np.inf):
        r = row.copy(); r[dim - 1] = bad
        assert "non-finite" in hci.ic_row_check(r) and str(dim - 1) in hci.ic_row_check(r)
    r = row.copy(); r[:3] = 0.0
    assert "zero position" in hci.ic_row_check(r)


def _config():
    from tests.hostcore_binding import default_config
    from basilisk_env_b200.initial_conditions import CONFIG_KEYS
    cfg = default_config()
    return {k: list(getattr(cfg, k)) if k in ("nHat_B", "sigma_R0N") else getattr(cfg, k) for k in CONFIG_KEYS}


def test_scenario_rows_from_reference_dicts():
    from basilisk_env_b200 import initial_conditions as icm
    rng = np.random.RandomState(3)
    dicts = [icm.set_ICs(rng) for _ in range(5)]
    for j, d in enumerate(dicts):
        d["mass"] = 300.0 + 10 * j
        d["K"] = 6.0 + j
    del dicts[4]["hs_min"]                                           # a missing parameter key takes the configuration's value
    ics, params = icm.scenario_rows(dicts, _config())
    assert ics.shape == (5, 19) and params.shape == (5, 14)
    for j, d in enumerate(dicts):
        np.testing.assert_array_equal(ics[j], icm.ic_row(d))
    assert params[:, icm.PARAM_KEYS.index("mass")].tolist() == [300.0, 310.0, 320.0, 330.0, 340.0]
    assert params[:, icm.PARAM_KEYS.index("K")].tolist() == [6.0, 7.0, 8.0, 9.0, 10.0]
    assert params[4, icm.PARAM_KEYS.index("hs_min")] == _config()["hs_min"]
    assert params[0, icm.PARAM_KEYS.index("storageCapacity")] == 20.0 * 3600.


@pytest.mark.parametrize("key, value", [("Ki", -2.0), ("planetRadius", 6.4e6), ("nHat_B", [0, 1, 0]), ("maxCounterValue", 5)])
def test_scenario_rows_refuse_a_differing_batch_global_key(key, value):
    from basilisk_env_b200 import initial_conditions as icm
    rng = np.random.RandomState(4)
    dicts = [icm.set_ICs(rng) for _ in range(3)]
    icm.scenario_rows(dicts, _config())
    dicts[2][key] = value
    with pytest.raises(ValueError, match=rf"scenario 2: '{key}'"):
        icm.scenario_rows(dicts, _config())
