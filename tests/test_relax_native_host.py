"""CPU: the C-ABI surface of the fused relaxation head / tail (reart_relax_head / reart_relax_tail) -- no GPU compute."""
import ctypes
import os
import sys

import pytest

from conftest import ROOT

# edges of the tail's point chunks (128 points) and first-level groups (8 chunks): one chunk, one ragged chunk, exactly
# one group, 16 groups, 17 groups, the cfg3_64k cloud
N_EDGES = (1, 127, 128, 129, 1024, 1025, 16384, 16385, 65536)


def _tail_args(N=1000, H=128, P=15, T=4, world=1, rank=0, phase=0):
    from reart_b200 import _lib
    fake = ctypes.c_void_p(0x1000)                              # never dereferenced: validation fails first
    a = _lib.RelaxTailArgs()
    for n in ("cano", "w0", "b0", "w2", "ysoft", "tau", "gW", "d6", "tr", "gR", "gtr", "m_seg", "v_seg", "m_d6", "v_d6",
              "m_tr", "v_tr", "step", "partials", "tickets", "loss_local", "bucket", "loss_out"):
        setattr(a, n, fake)
    a.lr_pose, a.lr_seg, a.beta1, a.beta2, a.eps = 1e-2, 1e-3, 0.9, 0.999, 1e-8
    a.rank, a.world, a.phase = rank, world, phase
    a.N, a.H, a.P, a.T = N, H, P, T
    return a


def test_relax_head_rejects_bad_arguments_without_touching_the_gpu():
    from reart_b200 import _lib
    L = _lib.lib()
    fake, null = ctypes.c_void_p(0x1000), None

    def head(N=100, H=128, P=15, T=4, hot=null):
        return L.reart_relax_head(fake, fake, fake, fake, fake, null, fake, fake, N, H, P, T, null, fake, fake, fake, hot, null)

    assert head(N=-1) == -1
    assert head(P=0) == -1
    assert head(P=33) == -4                                       # P > 32: no instantiation
    assert head(hot=ctypes.c_void_p(0x1004)) == -1                # the compact weights are written as int2: 16-byte aligned
    assert head(T=-1) == -1
    assert L.reart_relax_head(*([null] * 8), 0, 128, 15, 0, *([null] * 6)) == 0       # empty problem: nothing to do


def test_relax_tail_rejects_bad_arguments_without_touching_the_gpu():
    from reart_b200 import _lib
    L = _lib.lib()
    tail = lambda a: L.reart_relax_tail(None if a is None else ctypes.byref(a), None)
    assert tail(None) == -1
    assert tail(_tail_args(N=0)) == -1
    assert tail(_tail_args(T=0)) == -1
    assert tail(_tail_args(H=257)) == -4                          # Hpad <= 256: one thread per (unit, quarter), 1024 threads
    assert tail(_tail_args(P=33)) == -4
    assert tail(_tail_args(phase=3)) == -1
    assert tail(_tail_args(world=2, rank=2)) == -1                # rank >= world
    assert tail(_tail_args(world=2, rank=1)) == -1                # phase 0 over 2 ranks needs peer memory
    a = _tail_args(); a.gW = None
    assert tail(a) == -1


@pytest.mark.parametrize("N", N_EDGES)
def test_relax_tail_workspace_and_ticket_sizes_follow_their_formulas(N):
    """partials = one nseg row per 128-point chunk + one per group of 8 chunks, rounded up to 256 bytes plus 256 bytes of
    slack; tickets = the two launch-wide counters + one per group."""
    from reart_b200 import _lib
    L = _lib.lib()
    chunks = -(-N // 128)
    groups = -(-chunks // 8)
    assert L.reart_relax_tail_ticket_words(N) == 2 + groups
    for H, P in ((32, 1), (33, 15), (128, 15), (256, 32)):
        floats = (chunks + groups) * (4 * H + P * H)
        assert L.reart_relax_tail_workspace_bytes(N, H, P) == -(-floats * 4 // 256) * 256 + 256
    assert L.reart_relax_tail_ticket_words(-1) == -1
    assert L.reart_relax_tail_workspace_bytes(-1, 128, 15) == -1
    assert L.reart_relax_tail_workspace_bytes(N, 0, 15) == -1


def test_relax_head_carries_no_float_atomics():
    """The SASS of relax_head_kernel has no float RED/ATOM (relax_tail_kernel is covered with the search kernels): every
    point's logits and weights are computed by its own lanes in a fixed order."""
    import shutil
    from reart_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_summary
    build.build()
    _, kernels = sass_summary.census()
    found = [k for n, k in kernels.items() if "relax_head_kernel" in n]
    assert len(found) == 3 and all(k["float RED/ATOM"] == 0 for k in found)
