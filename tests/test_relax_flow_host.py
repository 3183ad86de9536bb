"""CPU: the C-ABI surface of the flow loss's gradient w.r.t. the skinned cloud (reart_flow_grad), which the relaxation
model's native iteration runs with a flow loss -- no GPU compute."""
import ctypes
import os
import sys

import pytest

from conftest import ROOT
from test_kinematic_assign_host import header_params


def test_flow_grad_signature_matches_the_header():
    from reart_b200 import _lib
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_float: "float", ctypes.c_int: "int", ctypes.c_int64: "int64_t"}
    for name in ("reart_flow_grad", "reart_flow_grad_workspace_bytes"):
        res, args = _lib.SIGNATURES[name]
        assert [kinds[t] for t in args] == header_params(name), name
    assert _lib.SIGNATURES["reart_flow_grad"][0] is ctypes.c_int
    assert _lib.SIGNATURES["reart_flow_grad_workspace_bytes"][0] is ctypes.c_int64


def test_flow_grad_rejects_bad_arguments_without_touching_the_gpu():
    from reart_b200 import _lib
    L = _lib.lib()
    fake, null = ctypes.c_void_p(0x1000), None                  # never dereferenced: validation fails first
    ws_ok = L.reart_flow_grad_workspace_bytes(5, 64)
    assert ws_ok > 0

    def call(ptrs=None, K=5, N=64, T=3, q0=0, q1=4, ws=fake, ws_bytes=None):
        p = [fake] * 6 if ptrs is None else ptrs
        return L.reart_flow_grad(*p[:4], 1.0, 0, K, N, T, q0, q1, *p[4:6], 1, ws, ws_ok if ws_bytes is None else ws_bytes,
                                 null)

    for k in range(6):                                            # every required pointer
        p = [fake] * 6
        p[k] = null
        assert call(p) == -1, k
    assert call(K=1, q1=0) == -1
    assert call(N=0) == -1
    assert call(N=-1) == -1
    assert call(T=-1) == -1
    assert call(q0=-1) == -1                                      # pair ranges outside the window
    assert call(q0=3, q1=2) == -1
    assert call(q1=5) == -1
    assert call(ws_bytes=8) == -2                                 # workspace too small
    assert call(ws=null, ws_bytes=0) == -2
    assert call(N=4096) == -2                                     # more point chunks than the workspace holds
    assert call([null] * 6, T=0, ws=null, ws_bytes=0) == 0        # empty problem: nothing to do
    assert L.reart_flow_grad_workspace_bytes(1, 64) == -1
    assert L.reart_flow_grad_workspace_bytes(5, 0) == -1
    assert L.reart_flow_grad_workspace_bytes(64, 16384) >= 8 * 64 * 64 + 4          # a double per (slot, chunk) + the ticket


def test_flow_grad_kernel_carries_no_float_atomics():
    """The SASS of flow_grad_kernel has no float RED/ATOM: every gradient element has one writer and the loss has a fixed
    association."""
    import shutil
    from reart_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_summary
    build.build()
    _, kernels = sass_summary.census()
    found = [k for n, k in kernels.items() if "flow_grad_kernel" in n]
    assert found and all(k["float RED/ATOM"] == 0 for k in found)


def test_native_flow_fit_refuses_cull_and_a_flow_reference_of_the_wrong_length():
    """cull=True reorders the engine's clouds while the flow references stay in the caller's order; a flow reference needs
    one set per pair of the complete sequence.  Both are refused at set-up, before any device work."""
    import types
    import torch
    from reart_b200.engine import RelaxationEngine
    cano, frames = torch.zeros(64, 3), torch.zeros(4, 64, 3)
    with pytest.raises(ValueError, match="exact tile culling"):
        RelaxationEngine(cano, frames, 4, flow_ref=types.SimpleNamespace(T=4), native=True, cull=True)
    for T, c in ((3, 0), (5, 0), (4, 5), (4, -1)):
        with pytest.raises(ValueError, match="one set per pair"):
            RelaxationEngine(cano, frames, 4, flow_ref=types.SimpleNamespace(T=T), cano_idx=c, native=True)
