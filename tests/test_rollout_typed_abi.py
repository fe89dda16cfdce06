"""CPU tests of the 16-bit rollout entry points (include/marlnav_b200_rollout_typed.h): each validates
obs_dtype and its pointers before it launches anything, the declarations compile and link from plain C,
and the binding's symbol list matches the header."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLLOUT_TYPED_H = os.path.join(ROOT, "include", "marlnav_b200_rollout_typed.h")
DECL = r"\b(marlnav_[a-z0-9_]+)\s*\("


def _lib():
    from marlnav_b200 import _lib, build
    build.build()
    return _lib, _lib.load()


def _params():
    from marlnav_b200 import _lib
    p = _lib.EnvParams(); p.num_envs, p.num_agents, p.num_obstacles = 64, 3, 3
    rs = _lib.ResetSpec(); rs.alias_first_step = 1
    return p, rs


def _calls(lib, code, obs):
    """(entry, error-text getter, call) for the three entries with observations `obs` and `obs_dtype` code;
    every other pointer is a non-NULL dummy, so only `obs` and the code can be refused."""
    from marlnav_b200 import _lib as L
    p, rs = _params()
    d = ctypes.c_void_p(16)
    sp = L.ActorSpec()
    sp.w1 = sp.b1 = sp.w_mu = sp.b_mu = sp.w_std = sp.b_std = 16
    sp.S, sp.H = 12, 50
    io = L.IoTransform()
    io.obs_mean = io.obs_scale = io.act_mean = io.act_scale = 16
    return [
        (lib.marlnav_rollout_last_error,
         lambda: lib.marlnav_actor_sample_typed(obs, code, 64, 12, 50, *([d] * 6), None, 0, 0, None, 0, d, d,
                                                None, None, None)),
        (lib.marlnav_rollout_last_error,
         lambda: lib.marlnav_critic_value_typed(obs, code, 64, 36, 50, d, d, d, d, d, None)),
        (lib.marlnav_last_error,
         lambda: lib.marlnav_act_step_typed(ctypes.byref(p), ctypes.byref(rs), *([d] * 5), ctypes.byref(sp), obs,
                                            d, d, ctypes.c_void_p(32), code, d, d, d, d, ctypes.byref(io), None)),
    ]


def test_rollout_typed_exports_match_the_header():
    _lib_mod, lib = _lib()
    declared = set(re.findall(DECL, open(ROLLOUT_TYPED_H).read()))
    assert declared == set(_lib_mod.ROLLOUT_TYPED_EXPORTS)
    assert not declared & set(_lib_mod.EXPORTS)
    assert not declared & set(_lib_mod.TYPED_EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    main = open(os.path.join(ROOT, "include", "marlnav_b200.h")).read()
    assert '#include "marlnav_b200_rollout_typed.h"' in main
    assert main.index('#include "marlnav_b200_typed.h"') < main.index('#include "marlnav_b200_rollout_typed.h"')


@pytest.mark.parametrize("code", [3, -1, 255])
def test_unknown_obs_dtype_is_rejected_before_launch(code):
    _lib_mod, lib = _lib()
    for err, call in _calls(lib, code, ctypes.c_void_p(16)):
        assert call() == -1
        assert b"obs_dtype" in err()


@pytest.mark.parametrize("code", [0, 1, 2])
def test_null_pointers_are_rejected(code):
    _lib_mod, lib = _lib()
    for err, call in _calls(lib, code, None):
        assert call() == -1
        assert b"NULL" in err()
    # shapes are checked as in the float32 entries
    d = ctypes.c_void_p(16)
    rc = lib.marlnav_actor_sample_typed(d, code, 64, 65, 50, *([d] * 6), None, 0, 0, None, 0, d, d, None, None, None)
    assert rc == -2 and b"obs_size" in lib.marlnav_rollout_last_error()
    rc = lib.marlnav_critic_value_typed(d, code, 64, 36, 65, d, d, d, d, d, None)
    assert rc == -2 and b"hidden" in lib.marlnav_rollout_last_error()


def test_rollout_typed_abi_from_plain_c(tmp_path):
    """The rollout typed declarations compile as C99 (-Wall -Werror) through marlnav_b200.h and link;
    argument errors come back as codes with a message."""
    from marlnav_b200 import build
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lib = build.build()
    exe = tmp_path / "rollout_typed_abi_check"
    src = os.path.join(ROOT, "tests", "c", "rollout_typed_abi_check.c")
    cmd = [gcc, "-std=c99", "-Wall", "-Werror", "-o", str(exe), src, "-L" + os.path.dirname(lib),
           "-lmarlnav_b200", "-Wl,-rpath," + os.path.dirname(lib)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    assert "rollout typed abi ok" in run.stdout
    declared = set(re.findall(DECL, open(ROLLOUT_TYPED_H).read()))
    assert all(name in open(src).read() for name in declared)
