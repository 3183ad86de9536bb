"""CPU: the pieces of engine checkpoints that need no GPU -- the uneven-shard gather of per-frame state over gloo, and the
native tails' flat moment buffers <-> per-parameter tensors, pinned to the kernels' buffer order."""
import math
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

from reart_b200.engine import split_flat


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def join_flat(parts, layout):
    """Per-parameter tensors -> a flat buffer, written through split_flat's views (as load_checkpoint writes them)."""
    flat = torch.zeros(sum(math.prod(s) for _, s in layout))
    for k, view in split_flat(flat, layout).items():
        view.copy_(parts[k])
    return flat


def _full(T, dtype, tail):
    return (torch.arange(T * math.prod(tail), dtype=torch.float64).reshape((T,) + tail) * 1.5 - 7).to(dtype)


def _gather_worker(rank, world, port, cases, out_dir):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    from reart_b200.dist import DistContext, gather_frames
    ctx = DistContext.from_env(backend="gloo")
    for T, dtype, tail in cases:
        full = _full(T, dtype, tail)
        lo, hi = ctx.frames(T)
        got = gather_frames(ctx, full[lo:hi].clone(), T)
        assert got.dtype == full.dtype and torch.equal(got, full), (rank, T, dtype, tail)
        assert torch.equal(got[lo:hi], full[lo:hi])                # sliced again for this rank: its own shard
    open(os.path.join(out_dir, f"ok{rank}"), "w").close()
    ctx.barrier()
    ctx.destroy()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_gather_frames_over_uneven_shards_equals_the_unsharded_tensor(tmp_path, world):
    cases = [(T, dtype, tail) for T in (world, 5, 7, 8) for dtype, tail in
             ((torch.float32, (4, 6)), (torch.int32, (3,)), (torch.float64, (5,)), (torch.float32, ()))]
    mp.spawn(_gather_worker, args=(world, _free_port(), cases, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))


def test_gather_frames_on_one_rank_is_the_tensor():
    from reart_b200.dist import DistContext, gather_frames
    x = _full(5, torch.float32, (3,))
    assert gather_frames(DistContext(), x, 5) is x


@pytest.mark.parametrize("P", [8, 15, 32])
def test_seg_moment_layout_round_trip(P):
    from reart_b200.engine import relax_seg_layout
    H = 128
    lay = relax_seg_layout(H, P)
    flat = torch.randn(4 * H + P * H, generator=torch.Generator().manual_seed(P))
    parts = split_flat(flat, lay)
    w0, b0, w2 = parts["seg_head.model.0.weight"], parts["seg_head.model.0.bias"], parts["seg_head.model.2.weight"]
    assert w0.shape == (H, 3, 1) and b0.shape == (H,) and w2.shape == (P, H, 1)
    # relax_tail_kernel: out[3k + c] (w0), out[3H + k] (b0), out[4H + pH + k] (w2)
    for k in (0, 1, H - 1):
        for c in range(3):
            assert w0[k, c, 0] == flat[3 * k + c]
        assert b0[k] == flat[3 * H + k]
        for p in (0, P - 1):
            assert w2[p, k, 0] == flat[4 * H + p * H + k]
    assert torch.equal(join_flat(parts, lay), flat)
    fresh = {k: torch.randn(v.shape) for k, v in parts.items()}
    back = split_flat(join_flat(fresh, lay), lay)
    assert all(torch.equal(back[k], fresh[k]) for k in fresh)
    parts["seg_head.model.0.bias"].fill_(3.0)                         # views: writing a part writes the buffer
    assert torch.equal(flat[3 * H:4 * H], torch.full((H,), 3.0))


@pytest.mark.parametrize("distance,root", [(False, False), (True, False), (False, True), (True, True)])
def test_kinematic_moment_layout_round_trip(distance, root):
    from reart_b200.engine import kin_layout
    E, T = 5, 7
    lay = kin_layout(E, T, distance, root)
    n = 6 * E + 1 + T * E + (T * E if distance else 0) + (9 * T if root else 0)    # KinematicEngine's n_grad
    flat = torch.randn(n, generator=torch.Generator().manual_seed(n))
    parts = split_flat(flat, lay)
    names = ["axis_list", "moment_list", "theta_list"] + (["distance_list"] if distance else []) + (["root_6d", "root_t"] if root else [])
    assert list(parts) == names
    # kin_tail_kernel's offsets
    o_theta = 6 * E + 1
    o_dist = o_theta + T * E
    o_d6 = o_dist + (T * E if distance else 0)
    o_rt = o_d6 + 6 * T
    assert parts["axis_list"][E - 1, 2] == flat[3 * E - 1] and parts["moment_list"][0, 0] == flat[3 * E]
    assert parts["theta_list"][2, 3] == flat[o_theta + 2 * E + 3]
    if distance:
        assert parts["distance_list"][T - 1, E - 1] == flat[o_dist + T * E - 1]
    if root:
        assert parts["root_6d"][4, 5] == flat[o_d6 + 4 * 6 + 5] and parts["root_t"][6, 1] == flat[o_rt + 6 * 3 + 1]
    joined = join_flat(parts, lay)
    assert joined[6 * E] == 0                                          # the loss slot is not state
    want = flat.clone()
    want[6 * E] = 0
    assert torch.equal(joined, want)
    fresh = {k: torch.randn(v.shape) for k, v in parts.items()}
    back = split_flat(join_flat(fresh, lay), lay)
    assert all(torch.equal(back[k], fresh[k]) for k in fresh)
