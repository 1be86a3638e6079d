"""CPU-side check of the final-destination ABI: macm_final_out and the final_* members of macm_rollout_out in
include/macm.h against their ctypes mirrors, and the ABI version the Python host expects."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _members(hdr, struct):
    body = hdr[hdr.index("typedef struct %s {" % struct):hdr.index("} %s;" % struct)]
    return re.findall(r"^\s*(?:float|int32_t|uint8_t)\*\s+(\w+);", body, re.M)


def test_final_structs_match_header():
    from gym_macm import _lib
    hdr = open(os.path.join(ROOT, "include", "macm.h")).read()
    assert _members(hdr, "macm_final_out") == [f[0] for f in _lib.MacmFinalOut._fields_] == list(_lib.FINAL_NAMES)
    ro = _members(hdr, "macm_rollout_out")
    assert ro[-4:] == ["final_" + n for n in _lib.FINAL_NAMES]
    assert ro == [f[0] for f in _lib.MacmRolloutOut._fields_]
    assert int(re.search(r"#define MACM_ABI_VERSION (\d+)", hdr).group(1)) == _lib.ABI_VERSION
    assert re.search(r"\bint macm_bind_final\(macm_sim\* sim, const macm_final_out\* f\);", hdr)
    assert "macm_bind_final" in _lib.EXPORTS


def test_keep_final_is_opt_in():
    from gym_macm.settings import combatSettings, flockSettings
    assert flockSettings().keep_final is False and combatSettings().keep_final is False
    assert flockSettings(keep_final=True, auto_reset=True).keep_final is True
