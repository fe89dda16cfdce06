"""CPU tests of the 16-bit observation entry points (include/marlnav_b200_typed.h): every one
validates obs_dtype and its pointers before it launches anything, the declarations compile and link
from plain C, and the binding's symbol list matches the header."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TYPED_H = os.path.join(ROOT, "include", "marlnav_b200_typed.h")


def _lib():
    from marlnav_b200 import _lib, build
    build.build()
    return _lib, _lib.load()


def _params():
    from marlnav_b200 import _lib
    p = _lib.EnvParams(); p.num_envs, p.num_agents, p.num_obstacles = 64, 3, 3
    rs = _lib.ResetSpec(); rs.alias_first_step = 1
    return p, rs


def test_typed_exports_match_the_header():
    _lib_mod, lib = _lib()
    declared = set(re.findall(r"\b(marlnav_[a-z0-9_]+)\s*\(", open(TYPED_H).read()))
    assert declared == set(_lib_mod.TYPED_EXPORTS)
    assert not declared & set(_lib_mod.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    main = open(os.path.join(ROOT, "include", "marlnav_b200.h")).read()
    assert '#include "marlnav_b200_typed.h"' in main


@pytest.mark.parametrize("code", [3, -1, 255])
def test_unknown_obs_dtype_is_rejected_before_launch(code):
    _lib_mod, lib = _lib()
    p, rs = _params()
    dummy = ctypes.c_void_p(16)
    checks = [
        lambda: lib.marlnav_observe_typed(ctypes.byref(p), dummy, dummy, dummy, dummy, code, None),
        lambda: lib.marlnav_step_typed(ctypes.byref(p), ctypes.byref(rs), *([dummy] * 7), code, *([dummy] * 4),
                                       None, None),
        lambda: lib.marlnav_step_call_typed(ctypes.byref(_lib_mod.StepCall()), code),
        lambda: lib.marlnav_step_host_typed(dummy, ctypes.byref(p), ctypes.byref(rs), *([dummy] * 16), None, None,
                                            code),
    ]
    for call in checks:
        assert call() == -1
        assert b"obs_dtype" in lib.marlnav_last_error()


@pytest.mark.parametrize("code", [0, 1, 2])
def test_null_pointers_are_rejected(code):
    _lib_mod, lib = _lib()
    p, rs = _params()
    rc = lib.marlnav_observe_typed(ctypes.byref(p), None, None, None, None, code, None)
    assert rc == -1 and b"NULL tensor pointer" in lib.marlnav_last_error()
    rc = lib.marlnav_step_typed(ctypes.byref(p), ctypes.byref(rs), *([None] * 7), code, *([None] * 4), None, None)
    assert rc == -1 and b"NULL tensor pointer" in lib.marlnav_last_error()
    rc = lib.marlnav_step_call_typed(None, code)
    assert rc == -1 and b"call is NULL" in lib.marlnav_last_error()
    call = _lib_mod.StepCall()
    call.params, call.reset = ctypes.addressof(p), ctypes.addressof(rs)
    rc = lib.marlnav_step_call_typed(ctypes.byref(call), code)
    assert rc == -1 and b"NULL tensor pointer" in lib.marlnav_last_error()
    rc = lib.marlnav_step_host_typed(ctypes.c_void_p(16), ctypes.byref(p), ctypes.byref(rs), *([None] * 16), None, None,
                                     code)
    assert rc == -1 and b"NULL host/staging pointer" in lib.marlnav_last_error()
    # shapes and struct sizes are checked as in the float32 entries
    p.num_agents = 1
    rc = lib.marlnav_observe_typed(ctypes.byref(p), None, None, None, None, code, None)
    assert rc == -2 and b"num_agents" in lib.marlnav_last_error()


def test_typed_abi_from_plain_c(tmp_path):
    """The typed declarations compile as C99 (-Wall -Werror) through marlnav_b200.h and link; argument
    errors come back as codes with a message."""
    from marlnav_b200 import build
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lib = build.build()
    exe = tmp_path / "typed_abi_check"
    src = os.path.join(ROOT, "tests", "c", "typed_abi_check.c")
    cmd = [gcc, "-std=c99", "-Wall", "-Werror", "-o", str(exe), src, "-L" + os.path.dirname(lib),
           "-lmarlnav_b200", "-Wl,-rpath," + os.path.dirname(lib)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0, (run.returncode, run.stdout, run.stderr)
    assert "typed abi ok" in run.stdout
    declared = set(re.findall(r"\b(marlnav_[a-z0-9_]+)\s*\(", open(TYPED_H).read()))
    assert all(name in open(src).read() for name in declared)
