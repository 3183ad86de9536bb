"""CPU: the C-ABI surface of the kinematic model's flow loss (reart_kin_flow) and the window / exchange plan of the native
flow step under frame sharding (dist.flow_window_plan) -- no GPU compute."""
import ctypes
import os
import sys

import pytest

from conftest import ROOT
from test_kinematic_assign_host import header_params


def test_kin_flow_signature_matches_the_header():
    from reart_b200 import _lib
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_float: "float", ctypes.c_int: "int", ctypes.c_int64: "int64_t"}
    for name in ("reart_kin_flow", "reart_kin_flow_workspace_bytes"):
        res, args = _lib.SIGNATURES[name]
        assert [kinds[t] for t in args] == header_params(name), name
    assert _lib.SIGNATURES["reart_kin_flow"][0] is ctypes.c_int
    assert _lib.SIGNATURES["reart_kin_flow_workspace_bytes"][0] is ctypes.c_int64


def test_kin_flow_rejects_bad_arguments_without_touching_the_gpu():
    from reart_b200 import _lib
    L = _lib.lib()
    fake, null = ctypes.c_void_p(0x1000), None                  # never dereferenced: validation fails first
    ws_ok = L.reart_kin_flow_workspace_bytes(5, 3)
    assert ws_ok > 0

    def call(ptrs=None, K=5, N=64, P=3, T=3, q0=0, q1=4, ws=fake, ws_bytes=None):
        p = [fake] * 10 if ptrs is None else ptrs
        return L.reart_kin_flow(*p[:7], 1.0, 0, K, N, P, T, q0, q1, *p[7:10], 1, ws, ws_ok if ws_bytes is None else ws_bytes,
                                null)

    for k in range(10):                                           # every required pointer
        p = [fake] * 10
        p[k] = null
        assert call(p) == -1, k
    assert call(P=33) == -4                                       # P > 32: unsupported
    assert call(P=0) == -1
    assert call(K=1, q1=0) == -1
    assert call(N=0) == -1
    assert call(T=-1) == -1
    assert call(q0=-1) == -1                                      # pair ranges outside the window
    assert call(q0=3, q1=2) == -1
    assert call(q1=5) == -1
    assert call(ws_bytes=8) == -2                                 # workspace too small
    assert call(ws=null, ws_bytes=0) == -2
    assert call([null] * 10, T=0, ws=null, ws_bytes=0) == 0       # empty problem: nothing to do
    assert L.reart_kin_flow_workspace_bytes(5, 33) == -1
    assert L.reart_kin_flow_workspace_bytes(1, 3) == -1
    assert L.reart_kin_flow_workspace_bytes(64, 32) >= 8 * 64 * 32 + 4              # a double per (slot, part) + the ticket


def test_kin_flow_kernel_carries_no_float_atomics():
    """The SASS of kin_flow_kernel has no float RED/ATOM: the (frame, part) sums and the loss have a fixed association."""
    import shutil
    from reart_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_summary
    build.build()
    _, kernels = sass_summary.census()
    found = [k for n, k in kernels.items() if "kin_flow_kernel" in n]
    assert found and all(k["float RED/ATOM"] == 0 for k in found)


def _complete_index(g, c):
    return g if g < c else g + 1


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_flow_window_plan_counts_every_pair_once_and_matches_sends_to_receives(world):
    from reart_b200.dist import flow_pairs_for_rank, flow_window_plan, shard_bounds
    for T in range(1, 13):
        if T < world:
            continue
        for c in range(T + 1):
            bounds = [shard_bounds(T, world, r) for r in range(world)]
            plans = flow_window_plan(T, c, bounds)
            assert plans == flow_window_plan(T, c, bounds)           # plain arithmetic: every rank computes the same plan
            counted = []
            for r, ((lo, hi), pl) in enumerate(zip(bounds, plans)):
                j0, K, slots = pl["j0"], pl["K"], pl["slots"]
                assert K >= 2 and 0 <= j0 and j0 + K - 1 <= T
                # the slots are the complete sequence's frames [j0, j0 + K)
                for s, x in enumerate(slots):
                    k = j0 + s
                    g = None if k == c else (k if k < c else k - 1)
                    want = ("cano",) if g is None else ("local", g - lo) if lo <= g < hi else ("prev",) if g == lo - 1 \
                        else ("next",) if g == hi else None
                    assert x == want, (T, c, r, s)
                # every local frame has both its adjacent pairs (where they exist) inside the window
                for g in range(lo, hi):
                    k = _complete_index(g, c)
                    assert j0 <= max(k - 1, 0) and min(k + 1, T) <= j0 + K - 1, (T, c, r, g)
                # the counted pairs are flow_pairs_for_rank's, and each has a local slot
                p0, p1, _, _ = flow_pairs_for_rank(T, c, lo, hi)
                assert [j0 + q for q in range(pl["q0"], pl["q1"])] == list(range(p0, p1))
                for q in range(pl["q0"], pl["q1"]):
                    assert slots[q][0] == "local" or slots[q + 1][0] == "local"
                counted += list(range(j0 + pl["q0"], j0 + pl["q1"]))
                # receives: exactly the neighbour slots
                assert pl["recv_prev"] == next((s for s, x in enumerate(slots) if x == ("prev",)), None)
                assert pl["recv_next"] == next((s for s, x in enumerate(slots) if x == ("next",)), None)
                if r == 0:
                    assert pl["recv_prev"] is None and not pl["send_prev"]
                if r == world - 1:
                    assert pl["recv_next"] is None and not pl["send_next"]
            assert sorted(counted) == list(range(T)), (T, c, world)        # every pair's loss exactly once
            for r in range(world - 1):                                    # sends and receives match rank to rank
                a, b = plans[r], plans[r + 1]
                assert a["send_next"] == (b["recv_prev"] is not None)
                assert b["send_prev"] == (a["recv_next"] is not None)
                # nothing travels where the canonical frame separates the two shards
                boundary = _complete_index(bounds[r][1] - 1, c) + 1 == c
                assert a["send_next"] == b["send_prev"] == (not boundary), (T, c, r)
