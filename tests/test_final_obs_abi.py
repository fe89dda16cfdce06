"""CPU tests of the final-observation steps and the GAE scan (include/marlnav_b200_final.h): every
refusal happens before anything launches, the declarations compile and link from plain C, and the
binding's symbol list matches the header."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FINAL_H = os.path.join(ROOT, "include", "marlnav_b200_final.h")
DECL = r"\b(marlnav_[a-z0-9_]+)\s*\("


def _lib():
    from marlnav_b200 import _lib, build
    build.build()
    return _lib, _lib.load()


def _step_args(code, obs, final):
    """marlnav_step_final_typed arguments with observations `obs`, dtype `code` and `final_obs`; every
    other pointer is a non-NULL dummy, so only these can be refused."""
    from marlnav_b200 import _lib as L
    p = L.EnvParams(); p.num_envs, p.num_agents, p.num_obstacles = 64, 3, 3
    rs = L.ResetSpec(); rs.alias_first_step = 1
    d = ctypes.c_void_p(16)
    return (ctypes.byref(p), ctypes.byref(rs), d, d, d, d, d, d, obs, code, final, d, d, d, d, None, None), (p, rs)


def _call(lib, code, obs, final):
    from marlnav_b200 import _lib as L
    (args, keep) = _step_args(code, obs, final)
    call = L.StepCall()
    call.params, call.reset = ctypes.addressof(keep[0]), ctypes.addressof(keep[1])
    for name in ("states", "obstacles", "target", "step_num", "terminates", "actions", "rewards", "terminated",
                 "truncated", "stats"):
        setattr(call, name, 16)
    call.obs = obs.value if isinstance(obs, ctypes.c_void_p) else obs
    return [lib.marlnav_step_final_typed(*args), lib.marlnav_step_call_final_typed(ctypes.addressof(call), code, final)]


def test_final_exports_match_the_header():
    _lib_mod, lib = _lib()
    declared = set(re.findall(DECL, open(FINAL_H).read()))
    assert declared == set(_lib_mod.FINAL_EXPORTS)
    for other in (_lib_mod.EXPORTS, _lib_mod.TYPED_EXPORTS, _lib_mod.ROLLOUT_TYPED_EXPORTS):
        assert not declared & set(other)
    for name in declared:
        assert hasattr(lib, name), name
    main = open(os.path.join(ROOT, "include", "marlnav_b200.h")).read()
    assert main.index('#include "marlnav_b200_typed.h"') < main.index('#include "marlnav_b200_final.h"')


@pytest.mark.parametrize("code", [0, 1, 2])
def test_null_or_aliased_final_obs_is_refused(code):
    _lib_mod, lib = _lib()
    obs = ctypes.c_void_p(32)
    for rc in _call(lib, code, obs, None):
        assert rc == -1 and b"final_obs is NULL" in lib.marlnav_last_error()
    for rc in _call(lib, code, obs, obs):
        assert rc == -1 and b"different buffers" in lib.marlnav_last_error()


@pytest.mark.parametrize("code", [3, -1, 255])
def test_unknown_obs_dtype_is_refused(code):
    _lib_mod, lib = _lib()
    for rc in _call(lib, code, ctypes.c_void_p(32), ctypes.c_void_p(64)):
        assert rc == -1 and b"obs_dtype" in lib.marlnav_last_error()


def test_other_step_arguments_are_checked_as_in_the_typed_step():
    _lib_mod, lib = _lib()
    args, keep = _step_args(0, None, ctypes.c_void_p(64))
    assert lib.marlnav_step_final_typed(*args) == -1 and b"NULL tensor" in lib.marlnav_last_error()
    keep[0].num_agents = 1
    args2 = (ctypes.byref(keep[0]),) + args[1:8] + (ctypes.c_void_p(32),) + args[9:]
    assert lib.marlnav_step_final_typed(*args2) == -2 and b"num_agents" in lib.marlnav_last_error()
    assert lib.marlnav_step_call_final_typed(None, 0, ctypes.c_void_p(64)) == -1
    assert b"call is NULL" in lib.marlnav_last_error()


def test_gae_refusals():
    _lib_mod, lib = _lib()
    d, out1, out2 = ctypes.c_void_p(16), ctypes.c_void_p(32), ctypes.c_void_p(48)
    cases = [((None, d, d, d, None, None, 0.99, 0.95, 4, 8, out1, out2), b"NULL"),
             ((d, d, None, d, None, None, 0.99, 0.95, 4, 8, out1, out2), b"NULL"),
             ((d, d, d, d, None, None, 0.99, 0.95, 0, 8, out1, out2), b"empty"),
             ((d, d, d, d, None, None, 0.99, 0.95, 4, 0, out1, out2), b"empty"),
             ((d, d, d, d, None, None, 0.99, 0.95, 4, 8, out1, out1), b"different buffers")]
    for args, msg in cases:
        assert lib.marlnav_gae_f64(*args, None) == -1
        assert msg in lib.marlnav_rollout_last_error()


def test_final_abi_from_plain_c(tmp_path):
    """The declarations compile as C99 (-Wall -Werror) through marlnav_b200.h and link; refusals come
    back as codes with a message."""
    from marlnav_b200 import build
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lib = build.build()
    exe = tmp_path / "final_obs_abi_check"
    src = os.path.join(ROOT, "tests", "c", "final_obs_abi_check.c")
    cmd = [gcc, "-std=c99", "-Wall", "-Werror", "-o", str(exe), src, "-L" + os.path.dirname(lib),
           "-lmarlnav_b200", "-Wl,-rpath," + os.path.dirname(lib)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    assert "final abi ok" in run.stdout
    declared = set(re.findall(DECL, open(FINAL_H).read()))
    assert all(name in open(src).read() for name in declared)
