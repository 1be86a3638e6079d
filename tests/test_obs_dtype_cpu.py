"""CPU-side checks of the `obs_dtype` setting: the header's enum and the Python constants agree, macm_create refuses
an unknown element type before it looks for a device, the settings names map to the enum, and the drop-in
classes (which hand out the reference's float observations) refuse a 16-bit type."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    from gym_macm import _lib
    return _lib


def test_header_enum_matches_lib():
    from gym_macm import _lib
    hdr = open(os.path.join(ROOT, "include", "macm.h")).read()
    m = re.search(r"enum \{ MACM_OBS_F32 = (\d+), MACM_OBS_F16 = (\d+), MACM_OBS_BF16 = (\d+) \};", hdr)
    assert m, "MACM_OBS_* enum not found"
    assert tuple(int(x) for x in m.groups()) == (_lib.OBS_F32, _lib.OBS_F16, _lib.OBS_BF16)
    assert _lib.OBS_DTYPE == {"float32": 0, "float16": 1, "bfloat16": 2}
    assert re.search(r"int32_t obs_dtype;", hdr) and "reserved0" not in hdr
    assert [f[0] for f in _lib.MacmParams._fields_][-1] == "obs_dtype"


_NO_DEVICE = r"""
import ctypes as C
from gym_macm import _lib as built
L = built.lib()
h = C.c_void_p()
for kind in (built.FLOCK, built.TDM):
    p = built.default_params(kind)
    assert p.obs_dtype == 0
    for bad in (3, -1, 1 << 20):
        p.obs_dtype = bad
        assert L.macm_create(C.byref(h), C.byref(p), 0) == -1 and not h, bad
    for ok in (0, 1, 2):   # valid: the missing device is what fails
        p.obs_dtype = ok
        assert L.macm_create(C.byref(h), C.byref(p), 0) == -2 and not h, ok
"""


def test_create_refuses_unknown_obs_dtype_without_device(built):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="",
               PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "gym-macm_b200")]))
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr


def test_settings_names_map_to_the_enum(built):
    from gym_macm.batched import flock_params, tdm_params
    from gym_macm.settings import combatSettings, flockSettings
    assert flockSettings().obs_dtype == "float32" and combatSettings().obs_dtype == "float32"
    for name, code in (("float32", 0), ("float16", 1), ("bfloat16", 2)):
        assert flock_params(flockSettings(obs_dtype=name), 4, 8, 1).obs_dtype == code
        assert tdm_params(combatSettings(obs_dtype=name), 4, 8).obs_dtype == code
    for bad in ("float64", "fp16", "half", None):
        with pytest.raises(ValueError):
            flock_params(flockSettings(obs_dtype=bad), 4, 8, 1)
        with pytest.raises(ValueError):
            tdm_params(combatSettings(obs_dtype=bad), 4, 8)


@pytest.mark.parametrize("env_id", ["gym_macm:cm-flock-v0", "gym_macm:cm-tdm-v0"])
@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_drop_in_classes_refuse_16_bit(env_id, dtype):
    import gym_macm
    with pytest.raises(ValueError, match="obs_dtype"):
        gym_macm.make(env_id, n_agents=[2, 2], obs_dtype=dtype)
