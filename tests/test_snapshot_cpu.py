"""CPU suite of the per-env state snapshots (include/bskenv.h: bskenv_snapshot / bskenv_restore and the opNav pair): the C ABI
declarations and exports, the record width of each batch kind, the refusal of null handles, and the documented record layout
against the state, parameter and IC dimensions of the device core."""
import ctypes as C
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "basilisk_env_b200", "csrc")
FUNCS = (("snapshot_width", 1), ("snapshot", 5), ("restore", 6))


def _header():
    return open(os.path.join(ROOT, "include", "bskenv.h")).read()


def _define(hdr, name):
    return int(re.search(r"#define " + name + r" (-?\d+)", hdr).group(1))


def test_header_declarations_and_exports():
    from basilisk_env_b200 import _native
    hdr = _header()
    for prefix, exports in (("bskenv_", _native.EXPORTS), ("bskenv_opnav_", _native.OPNAV_EXPORTS)):
        for name, nargs in FUNCS:
            fn = prefix + name
            m = re.search(r"\bint " + fn + r"\(([^;]*)\);", hdr, re.S)
            assert m, fn
            assert len(re.sub(r"/\*.*?\*/", "", m.group(1)).split(",")) == nargs, fn
            assert fn in exports, fn
    assert _define(hdr, "BSKENV_ABI_VERSION") == 1


def test_snapshot_width_needs_no_device():
    from basilisk_env_b200 import _native
    L, hdr = _native.lib(), _header()
    assert L.bskenv_snapshot_width(None) == _define(hdr, "BSKENV_SNAPSHOT_W") == 172
    assert L.bskenv_opnav_snapshot_width(None) == _define(hdr, "BSKENV_OPNAV_SNAPSHOT_W") == 114
    assert _native.batch_abi("bskenv_").snapshot_width(None) == 172
    assert _native.batch_abi("bskenv_opnav_").snapshot_width(None) == 114


def test_null_handle_is_refused():
    from basilisk_env_b200 import _native
    buf = (C.c_double * 172)()
    for prefix in ("bskenv_", "bskenv_opnav_"):
        f = _native.batch_abi(prefix)
        assert f.snapshot(None, 1, None, C.cast(buf, C.c_void_p), None) == -1, prefix
        assert f.restore(None, 1, None, C.cast(buf, C.c_void_p), None, None) == -1, prefix


def test_layout_agrees_with_the_device_core(tmp_path):
    """The offsets documented in bskenv.h follow from the field counts the kernels are compiled with (the .cu files also
    static_assert them)."""
    src = tmp_path / "dims.cpp"
    src.write_text('#include <stdio.h>\n#include "bskenv.h"\n#include "leo_params.h"\n#include "opnav_params.h"\n'
                   'int main(void){printf("%d %d %d %d %d %d %d %d\\n", (int)LEO_ND, (int)LEO_NI, (int)LEO_NPD, (int)PE_ROW,'
                   '(int)OPNAV_ND, (int)OPNAV_NI, (int)OPNAV_IC_DIM, (int)BSKENV_IC_DIM);return 0;}\n')
    exe = tmp_path / "dims"
    subprocess.check_call(["g++", "-I", os.path.join(ROOT, "include"), "-I", CSRC, "-o", str(exe), str(src)])
    nd, ni, npd, pe_row, ond, oni, oic, lic = (int(x) for x in subprocess.check_output([str(exe)]).split())
    assert (nd, ni, npd, ond, oni, oic, lic) == (89, 22, 37, 83, 14, 12, 19)
    hdr = _header()
    g = lambda name: _define(hdr, name)   # noqa: E731
    assert g("BSKENV_SNAP_S") == 4
    assert g("BSKENV_SNAP_I") == g("BSKENV_SNAP_S") + nd
    assert g("BSKENV_SNAP_ICS") == g("BSKENV_SNAP_I") + ni
    assert g("BSKENV_SNAP_PARAMS") == g("BSKENV_SNAP_ICS") + lic
    assert g("BSKENV_SNAP_ICROW") == g("BSKENV_SNAP_PARAMS") + npd
    assert g("BSKENV_SNAPSHOT_W") == g("BSKENV_SNAP_ICROW") + 1
    assert g("BSKENV_OPNAV_SNAP_S") == 4
    assert g("BSKENV_OPNAV_SNAP_I") == g("BSKENV_OPNAV_SNAP_S") + ond
    assert g("BSKENV_OPNAV_SNAP_ICS") == g("BSKENV_OPNAV_SNAP_I") + oni
    assert g("BSKENV_OPNAV_SNAP_ICROW") == g("BSKENV_OPNAV_SNAP_ICS") + oic
    assert g("BSKENV_OPNAV_SNAPSHOT_W") == g("BSKENV_OPNAV_SNAP_ICROW") + 1
    assert "BSKENV_SNAP_PARAMS + 22" in hdr and pe_row == 22     # the pool-row word named in the layout table
    assert (g("BSKENV_SNAPSHOT_KIND_LEO"), g("BSKENV_SNAPSHOT_KIND_OPNAV"), g("BSKENV_SNAPSHOT_VERSION")) == (1, 2, 1)
