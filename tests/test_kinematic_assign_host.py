"""CPU: the C-ABI surface of the kinematic model's assignment loss (reart_kin_assign) -- no GPU compute."""
import ctypes
import os
import re
import sys

import pytest

from conftest import ROOT


def header_params(name):
    """C parameter types of `REART_API <ret> <name>(...)` in include/reart_b200.h, in declaration order."""
    src = open(os.path.join(ROOT, "include", "reart_b200.h")).read()
    args = re.search(rf"REART_API \w+ {name}\((.*?)\);", src, flags=re.S).group(1)
    out = []
    for a in args.split(","):
        a = " ".join(a.split())
        out.append("ptr" if "*" in a else a[:a.rindex(" ")].replace("const ", ""))
    return out


def test_kin_assign_signature_matches_the_header():
    from reart_b200 import _lib
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_float: "float", ctypes.c_int: "int", ctypes.c_int64: "int64_t"}
    for name in ("reart_kin_assign", "reart_kin_assign_workspace_bytes"):
        res, args = _lib.SIGNATURES[name]
        assert [kinds[t] for t in args] == header_params(name), name
    assert _lib.SIGNATURES["reart_kin_assign"][0] is ctypes.c_int
    assert _lib.SIGNATURES["reart_kin_assign_workspace_bytes"][0] is ctypes.c_int64


def test_kin_assign_rejects_bad_arguments_without_touching_the_gpu():
    from reart_b200 import _lib
    L = _lib.lib()
    fake, null = ctypes.c_void_p(0x1000), None                  # never dereferenced: validation fails first
    ws_ok = L.reart_kin_assign_workspace_bytes(4, 3)
    assert ws_ok > 0

    def call(ptrs=None, T=4, N=64, n=16, P=3, ws=fake, ws_bytes=None):
        p = [fake] * 10 if ptrs is None else ptrs
        return L.reart_kin_assign(*p[:7], 0.3, T, N, n, P, *p[7:10], 1, ws, ws_ok if ws_bytes is None else ws_bytes, null)

    for k in range(10):                                           # every required pointer
        p = [fake] * 10
        p[k] = null
        assert call(p) == -1, k
    assert call(P=33) == -4
    assert call(P=0) == -1
    assert call(n=0) == -1
    assert call(T=-1) == -1
    assert call(ws_bytes=8) == -2                                 # workspace too small
    assert call(ws=null, ws_bytes=0) == -2
    assert call([null] * 10, T=0, ws=null, ws_bytes=0) == 0       # empty problem: nothing to do
    assert L.reart_kin_assign_workspace_bytes(4, 33) == -1
    assert L.reart_kin_assign_workspace_bytes(-1, 3) == -1


def test_kin_assign_kernel_carries_no_float_atomics():
    """The SASS of kin_assign_kernel has no float RED/ATOM: the (frame, part) sums and the loss have a fixed association."""
    import shutil
    from reart_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_summary
    build.build()
    _, kernels = sass_summary.census()
    found = [k for n, k in kernels.items() if "kin_assign_kernel" in n]
    assert found and all(k["float RED/ATOM"] == 0 for k in found)
