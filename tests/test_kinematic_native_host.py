"""CPU: the C-ABI surface of the native kinematic iteration (reart_kin_head / reart_kin_tail) -- no GPU compute."""
import ctypes
import os
import re
import sys

import pytest

from conftest import ROOT


def header_struct_fields(name):
    """(field, C type class) of `typedef struct <name> {...} <name>;` in include/reart_b200.h, in declaration order."""
    src = open(os.path.join(ROOT, "include", "reart_b200.h")).read()
    body = re.search(rf"typedef struct {name} \{{(.*?)\}} {name};", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for stmt in body.split(";"):
        stmt = stmt.strip()
        if not stmt:
            continue
        names = [n.strip() for n in stmt.split(",")]
        first = names[0]
        ctype = "ptr" if "*" in first else first[:first.rindex(" ")].strip()
        fields += [(re.search(r"(\w+)$", n).group(1), ctype) for n in names]
    return fields


def test_kin_tail_args_struct_matches_the_header_field_for_field():
    from reart_b200 import _lib
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_float: "float", ctypes.c_int32: "int32_t", ctypes.c_int64: "int64_t"}
    assert [(n, kinds[t]) for n, t in _lib.KinTailArgs._fields_] == header_struct_fields("reart_kin_tail_args")


def _tail_args(T=4, P=3, world=1, rank=0):
    from reart_b200 import _lib
    fake = ctypes.c_void_p(0x1000)                              # never dereferenced: validation fails first
    a = _lib.KinTailArgs()
    for n in ("fk", "gR", "gtr", "loss_local", "order", "parent", "edge", "axis", "moment", "theta", "grad", "m", "v", "step",
              "partials", "loss_out"):
        setattr(a, n, fake)
    a.lr, a.beta1, a.beta2, a.eps = 1e-2, 0.9, 0.999, 1e-8
    a.rank, a.world, a.T, a.P = rank, world, T, P
    return a


def test_kin_entry_points_reject_bad_arguments_without_touching_the_gpu():
    from reart_b200 import _lib
    L = _lib.lib()
    fake, null = ctypes.c_void_p(0x1000), None
    head = lambda *over, T=4, P=3: L.reart_kin_head(*over, T, P, fake, fake, fake, null)
    ok_ptrs = [fake, fake, fake, null, fake, fake, fake, null, null, null]
    assert head(*([null] + ok_ptrs[1:])) == -1                          # no axis
    assert head(*(ok_ptrs[:4] + [null] + ok_ptrs[5:])) == -1            # no tree order
    assert head(*(ok_ptrs[:8] + [fake, null])) == -1                    # root_6d without root_t
    assert head(*ok_ptrs, P=33) == -4                                   # P > 32
    assert head(*ok_ptrs, P=0) == -1
    assert head(*ok_ptrs, T=-1) == -1
    assert L.reart_kin_head(*([null] * 10), 0, 3, null, null, null, null) == 0     # empty problem: nothing to do
    assert L.reart_kin_tail(None, null) == -1
    assert L.reart_kin_tail(ctypes.byref(_tail_args(P=33)), null) == -4
    assert L.reart_kin_tail(ctypes.byref(_tail_args(world=2, rank=2)), null) == -1            # rank >= world
    assert L.reart_kin_tail(ctypes.byref(_tail_args(world=2, rank=1)), null) == -1            # one-shot without peer memory
    a = _tail_args(); a.grad = None
    assert L.reart_kin_tail(ctypes.byref(a), null) == -1
    a = _tail_args(); a.root_6d = fake
    assert L.reart_kin_tail(ctypes.byref(a), null) == -1
    a = _tail_args(); a.phase = 3
    assert L.reart_kin_tail(ctypes.byref(a), null) == -1
    assert L.reart_kin_tail_workspace_bytes(32, 8) >= 4 * (32 * 6 * 7 + 32 * 8 * 12)
    assert L.reart_kin_tail_workspace_bytes(-1, 8) == -1


def test_kin_kernels_carry_no_float_atomics():
    """The SASS of kin_head_kernel / kin_tail_kernel has no float RED/ATOM: the frame sums are fixed-order, so the native
    kinematic step is bit-reproducible (fk_bwd_kernel of the autograd path does use them)."""
    import shutil
    from reart_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_summary
    build.build()
    _, kernels = sass_summary.census()
    for frag in ("kin_head_kernel", "kin_tail_kernel"):
        found = [k for n, k in kernels.items() if frag in n]
        assert found and all(k["float RED/ATOM"] == 0 for k in found), frag
