"""The culled search on k-d ordered copies of the caller's clouds (reart_skinned_chamfer_fwd_bwd_ordered, the engine's
default from 8192 points on): every output must be BIT-IDENTICAL to the brute-force evaluation on the caller's order --
including which of several exactly equidistant points wins (the lowest caller index) -- and an optimisation run on it
must be the brute-force run, step for step."""
import numpy as np
import pytest
import torch

from conftest import synthetic_sequence
from test_cull_gpu import evaluate, same

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda")


def leaf_sorted(order, leaf):
    """Any permutation [B,n] made admissible: the points of every leaf in ascending caller index."""
    n = order.shape[1]
    leaf_of = torch.arange(n, device=order.device) // leaf
    return torch.sort(leaf_of[None] * n + order, dim=1).values % n


def inverse(order):
    inv = torch.empty_like(order)
    inv.scatter_(1, order, torch.arange(order.shape[1], device=order.device, dtype=order.dtype)[None].expand_as(order).contiguous())
    return inv


def evaluate_ordered(cano, W, R, tr, frames, row_order, tgt_order, nn):
    """One fused evaluation through the ordered C ABI; row_order [N], tgt_order [T,M] (int64, admissible)."""
    from reart_b200 import _lib, ops
    L = _lib.lib()
    T, P = R.shape[0], R.shape[1]
    N, M = cano.shape[0], frames.shape[1]
    out = dict(skinned=torch.empty(T, N, 3, device=dev()), loss=torch.empty(1, dtype=torch.float64, device=dev()),
               gW=torch.empty(N, P, device=dev()), gpose=torch.empty(T * P * 12, device=dev()),
               gs=torch.empty(T, N, 3, device=dev()), d_f=torch.empty(T, N, device=dev()),
               i_f=torch.empty(T, N, dtype=torch.int64, device=dev()), d_b=torch.empty(T, M, device=dev()),
               i_b=torch.empty(T, M, dtype=torch.int64, device=dev()))
    ro, ri = row_order.int().contiguous(), inverse(row_order[None])[0].int().contiguous()
    to, ti = tgt_order.int().contiguous(), inverse(tgt_order).int().contiguous()
    fs = torch.gather(frames, 1, tgt_order[:, :, None].expand(-1, -1, 3)).contiguous()
    fsp = ops.pack_cloud(fs)
    nbytes = L.reart_energy_workspace_bytes(T, N, M)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    p = _lib.ptr
    gR, gtr = out["gpose"][:T * P * 9], out["gpose"][T * P * 9:]
    _lib.check(L.reart_skinned_chamfer_fwd_bwd_ordered(
        p(cano), p(W), p(R), p(tr), p(frames), p(fs), p(fsp), T, N, M, P, p(ro), p(ri), p(to), p(ti), p(out["skinned"]),
        p(out["loss"]), p(out["gW"]), p(gR), p(gtr), p(out["gs"]), 1, p(out["d_f"]), p(out["i_f"]), p(out["d_b"]), p(out["i_b"]),
        p(nn[0]), p(nn[1]), p(nn[2]), p(ws), nbytes, _lib.stream_ptr()), "ordered")
    torch.cuda.synchronize()
    return out


def seeds(T, N, M):
    return (torch.full((T, N), -1, dtype=torch.int32, device=dev()), torch.full((T, M), -1, dtype=torch.int32, device=dev()),
            torch.zeros(3, dtype=torch.int64, device=dev()))


def random_scene(T, N, P, seed):
    """Synthetic sequence with both clouds in a random point order (the caller's order is arbitrary)."""
    seq = synthetic_sequence(T, N, P, seed=seed)
    g = torch.Generator().manual_seed(seed)
    pc = torch.randperm(N, generator=g)
    cano = torch.from_numpy(seq["cano"])[pc].contiguous().to(dev())
    part = torch.from_numpy(seq["part"].astype(np.int64))[pc].to(dev())
    pf = torch.stack([torch.randperm(N, generator=g) for _ in range(T)])
    frames = torch.gather(torch.from_numpy(seq["frames"]), 1, pf[:, :, None].expand(-1, -1, 3)).contiguous().to(dev())
    W = torch.eye(P, device=dev())[part].contiguous()
    R = torch.from_numpy(np.ascontiguousarray(seq["pose"][:, :, :3, :3])).to(dev())
    tr = torch.from_numpy(np.ascontiguousarray(seq["pose"][:, :, :3, 3])).to(dev())
    return cano, W, R, tr, frames


def orders(kind, cano, frames):
    from reart_b200 import ops
    T, N, M = frames.shape[0], cano.shape[0], frames.shape[1]
    if kind == "kd":
        return ops.search_order(cano[None], 256)[0], ops.search_order(frames, 32)
    if kind == "identity":
        return torch.arange(N, device=dev()), torch.arange(M, device=dev())[None].repeat(T, 1)
    assert kind == "reversed"
    return (leaf_sorted(torch.arange(N - 1, -1, -1, device=dev())[None], 256)[0],
            leaf_sorted(torch.arange(M - 1, -1, -1, device=dev())[None].repeat(T, 1), 32))


@pytest.mark.parametrize("T,N,P,kind", [(2, 300, 3, "kd"), (3, 5000, 4, "kd"), (1, 16384, 8, "kd"), (4, 8192, 5, "kd"),
                                        (3, 4096, 5, "identity"), (3, 4096, 5, "reversed")])
def test_ordered_evaluation_is_bit_identical_to_the_brute_force(T, N, P, kind):
    cano, W, R, tr, frames = random_scene(T, N, P, 11)
    M = frames.shape[1]
    ro, to = orders(kind, cano, frames)
    nn = seeds(T, N, M)
    brute = evaluate(cano, W, R, tr, frames)
    same(brute, evaluate_ordered(cano, W, R, tr, frames, ro, to, nn))
    # seeds from that evaluation, poses moved a little (the optimiser's situation)
    g = torch.Generator(device="cuda").manual_seed(3)
    tr2 = tr + 0.004 * torch.randn(tr.shape, device=dev(), generator=g)
    brute2 = evaluate(cano, W, R, tr2, frames)
    nn[2].zero_()
    same(brute2, evaluate_ordered(cano, W, R, tr2, frames, ro, to, nn))
    ev, off, _ = nn[2].tolist()
    if kind == "kd" and N >= 4096:
        assert ev < 0.6 * off, (ev, off)
    # garbage and out-of-range seeds: still exact
    nn[0].random_(0, M); nn[1].random_(0, N)
    same(brute2, evaluate_ordered(cano, W, R, tr2, frames, ro, to, nn))
    nn[0].fill_(M + 5); nn[1].fill_(-7)
    same(brute2, evaluate_ordered(cano, W, R, tr2, frames, ro, to, nn))


@pytest.mark.parametrize("N", [2048, 8192])
def test_ordered_evaluation_keeps_the_lowest_caller_index_on_lattices_and_duplicates(N):
    """Integer lattices and duplicated points: exact ties everywhere, across chunks of the search order too."""
    rng = np.random.default_rng(5)
    T, P = 2, 2
    cano_np = rng.integers(-6, 7, (N, 3)).astype(np.float32)
    cano_np[N // 2:] = cano_np[:N // 2][rng.permutation(N // 2)]                # every canonical point twice
    cano = torch.from_numpy(cano_np).to(dev())
    frames = torch.from_numpy(rng.integers(-6, 7, (T, N, 3)).astype(np.float32)).to(dev())
    W = torch.zeros(N, P, device=dev()); W[:, 0] = 1
    R = torch.eye(3, device=dev()).repeat(T, P, 1, 1).contiguous()
    tr = torch.zeros(T, P, 3, device=dev())
    ro, to = orders("kd", cano, frames)
    nn = seeds(T, N, N)
    brute = evaluate(cano, W, R, tr, frames)
    same(brute, evaluate_ordered(cano, W, R, tr, frames, ro, to, nn))
    assert nn[2][2] > 0
    same(brute, evaluate_ordered(cano, W, R, tr, frames, ro, to, nn))      # seeded by exact arg-mins: tight bounds


def far_cloud(n, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 3, generator=g) * 50.0 + 10.0                           # every point at distance > 10 from the origin
    return x


@pytest.mark.parametrize("M", [512, 16384])
def test_a_cross_chunk_tie_returns_the_lowest_caller_index(M):
    """A query with two exactly equidistant partners in DIFFERENT chunks of the search order, the higher caller index in
    the earlier chunk -- for a row (target chunks; at M = 16384 the two chunks lie in different target splits, whose
    partial keys meet through atomicMin) and for a column (256-row chunks)."""
    T, P, N = 1, 1, 512
    cano = far_cloud(N, 1)
    frames = far_cloud(M, 2)[None].clone()
    # row 3 at the origin; targets 7 and M-9 at distance 1 from it
    cano[3] = torch.tensor([0.0, 0.0, 0.0])
    frames[0, 7] = torch.tensor([1.0, 0.0, 0.0]); frames[0, M - 9] = torch.tensor([-1.0, 0.0, 0.0])
    # target 5 at (0, 30, 0); rows 20 and 400 at distance 2 from it
    frames[0, 5] = torch.tensor([0.0, 30.0, 0.0])
    cano[20] = torch.tensor([0.0, 32.0, 0.0]); cano[400] = torch.tensor([0.0, 28.0, 0.0])
    cano, frames = cano.to(dev()), frames.to(dev())
    # search orders: the HIGHER caller index first (first chunk / first 256-row block)
    def first_and_last(n, first, last):
        rest = torch.arange(n)
        return torch.cat((torch.tensor([first]), rest[(rest != first) & (rest != last)], torch.tensor([last])))
    to = first_and_last(M, M - 9, 7)
    ro = first_and_last(N, 400, 20)
    ro, to = leaf_sorted(ro[None].to(dev()), 256)[0], leaf_sorted(to[None].to(dev()), 32)
    assert int((ro == 400).nonzero()) // 256 < int((ro == 20).nonzero()) // 256
    assert int((to[0] == M - 9).nonzero()) // 32 < int((to[0] == 7).nonzero()) // 32
    W = torch.ones(N, P, device=dev())
    R = torch.eye(3, device=dev()).repeat(T, P, 1, 1).contiguous()
    tr = torch.zeros(T, P, 3, device=dev())
    nn = seeds(T, N, M)
    brute = evaluate(cano, W, R, tr, frames)
    assert int(brute["i_f"][0, 3]) == 7 and int(brute["i_b"][0, 5]) == 20
    same(brute, evaluate_ordered(cano, W, R, tr, frames, ro, to, nn))
    assert nn[2][2] >= 2
    same(brute, evaluate_ordered(cano, W, R, tr, frames, ro, to, nn))      # exact seeds


def run_engine(cano, frames, steps, use_graph, ingest=None, **kw):
    from reart_b200.engine import RelaxationEngine, tau_schedule
    eng = RelaxationEngine(cano, frames, num_parts=6, use_graph=use_graph, seed=2, **kw)
    torch.manual_seed(9)
    losses = []
    for i in range(steps):
        if ingest is None:
            losses.append(float(eng.step(tau_schedule(i, 100, 5.0, 1.0))))
        else:
            c, f = ingest[i & 1]
            losses.append(float(eng.step(tau_schedule(i, 100, 5.0, 1.0), ingest=(i & 1, c, f))))
    state = [q.detach().clone() for q in eng._opt_params()] + [eng.skinned.clone()]
    info = (eng.search_culled, eng.culling_stats(), eng.flagged_ties())
    eng.release()
    return losses, state, info


@pytest.mark.parametrize("assign", [None, dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=2, mode="add")])
def test_engine_default_search_is_the_brute_force_optimisation_bit_for_bit(assign):
    seq = synthetic_sequence(4, 8192, 6, seed=8)
    cano, frames = torch.from_numpy(seq["cano"]).to(dev()), torch.from_numpy(seq["frames"]).to(dev())
    ref, ref_state, ref_info = run_engine(cano, frames, 25, True, search="brute", assign=assign)
    got, state, info = run_engine(cano, frames, 25, True, assign=assign)
    assert not ref_info[0] and info[0]
    ev, off = info[1]
    assert 0 < ev < off
    assert got == ref                                                          # floats, not allclose
    for a, b in zip(state, ref_state):
        assert torch.equal(a, b)


def test_engine_default_search_with_ingest_is_the_brute_force_optimisation_bit_for_bit():
    seq = synthetic_sequence(4, 8192, 6, seed=8)
    seq2 = synthetic_sequence(4, 8192, 6, seed=9)
    stage = [(torch.from_numpy(s["cano"]).to(dev()).contiguous(), torch.from_numpy(s["frames"]).to(dev()).contiguous())
             for s in (seq, seq2)]
    ref, ref_state, _ = run_engine(stage[0][0].clone(), stage[0][1].clone(), 12, True, ingest=stage, search="brute")
    got, state, info = run_engine(stage[0][0].clone(), stage[0][1].clone(), 12, True, ingest=stage)
    assert info[0]
    assert got == ref
    for a, b in zip(state, ref_state):
        assert torch.equal(a, b)
