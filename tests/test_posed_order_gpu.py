"""The culled search with a row order computed per frame on the skinned cloud (reart_skinned_chamfer_fwd_bwd_posed, the
engine's default from 8192 up to reart_posed_order_max_points() points): every output must be BIT-IDENTICAL to the
brute-force evaluation on the caller's order, and the order it writes must be the sort-tile-recursive order on quantised
coordinates of csrc/order.cu, reproduced here in numpy."""
import numpy as np
import pytest
import torch

from test_cull_gpu import evaluate, same
from test_ordered_search_gpu import inverse, random_scene, seeds

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda")


def str_reference(p):
    """csrc/order.cu in numpy: axes by decreasing extent (lower axis first on equal extents); per level the rows ordered by
    (segment, quantised coordinate, caller index) and cut into runs of 2048 / 512 / 256 from the front; every leaf in
    ascending caller index."""
    p = p.astype(np.float32)
    lo = p.min(0)
    ext = p.max(0) - lo
    axes = sorted(range(3), key=lambda a: (-ext[a], a))
    n = len(p)
    idx = np.arange(n)
    seg = np.zeros(n, np.int64)
    order = idx
    for a, cells, size in zip(axes, (4096, 512, 128), (2048, 512, 256)):
        e = ext[a]
        scale = np.float32(cells) / e if 0 < e < np.inf else np.float32(0)
        v = (p[:, a] - lo[a]) * np.float32(scale)
        q = np.where(v > 0, np.minimum(np.float32(cells - 1), np.floor(v)), 0).astype(np.int64)
        order = np.lexsort((idx, seg * cells + q))
        seg[order] = np.arange(n) // size
    return np.concatenate([np.sort(order[s:s + 256]) for s in range(0, n, 256)])


def evaluate_posed(cano, W, R, tr, frames, tgt_order, nn):
    from reart_b200 import _lib, ops
    L = _lib.lib()
    T, P = R.shape[0], R.shape[1]
    N, M = cano.shape[0], frames.shape[1]
    out = dict(skinned=torch.empty(T, N, 3, device=dev()), loss=torch.empty(1, dtype=torch.float64, device=dev()),
               gW=torch.empty(N, P, device=dev()), gpose=torch.empty(T * P * 12, device=dev()),
               gs=torch.empty(T, N, 3, device=dev()), d_f=torch.empty(T, N, device=dev()),
               i_f=torch.empty(T, N, dtype=torch.int64, device=dev()), d_b=torch.empty(T, M, device=dev()),
               i_b=torch.empty(T, M, dtype=torch.int64, device=dev()),
               row_order=torch.full((T, N), -1, dtype=torch.int32, device=dev()),
               row_inv=torch.full((T, N), -1, dtype=torch.int32, device=dev()))
    to, ti = tgt_order.int().contiguous(), inverse(tgt_order).int().contiguous()
    fs = torch.gather(frames, 1, tgt_order[:, :, None].expand(-1, -1, 3)).contiguous()
    fsp = ops.pack_cloud(fs)
    nbytes = L.reart_energy_workspace_bytes(T, N, M)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev())
    p = _lib.ptr
    gR, gtr = out["gpose"][:T * P * 9], out["gpose"][T * P * 9:]
    rc = L.reart_skinned_chamfer_fwd_bwd_posed(
        p(cano), p(W), p(R), p(tr), p(frames), p(fs), p(fsp), T, N, M, P, p(to), p(ti), p(out["row_order"]),
        p(out["row_inv"]), p(out["skinned"]), p(out["loss"]), p(out["gW"]), p(gR), p(gtr), p(out["gs"]), 1, p(out["d_f"]),
        p(out["i_f"]), p(out["d_b"]), p(out["i_b"]), p(nn[0]), p(nn[1]), p(nn[2]), p(ws), nbytes, _lib.stream_ptr())
    torch.cuda.synchronize()
    out["rc"] = rc
    return out


def check_order(out):
    sk = out["skinned"].cpu().numpy()
    order, inv = out["row_order"].cpu().numpy(), out["row_inv"].cpu().numpy()
    T, N = order.shape
    for t in range(T):
        assert np.array_equal(np.sort(order[t]), np.arange(N)), t                 # a permutation
        assert np.array_equal(inv[t][order[t]], np.arange(N)), t
        for s in range(0, N, 256):
            assert np.all(np.diff(order[t, s:s + 256]) > 0), (t, s)               # leaves in caller order
        assert np.array_equal(order[t], str_reference(sk[t])), t


def articulated(T, N, P, seed):
    """random_scene's clouds with large random part transforms and a random hard part per point"""
    cano, _, _, _, frames = random_scene(T, N, P, seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    part = torch.randint(0, P, (N,), device=dev(), generator=g)
    W = torch.eye(P, device=dev())[part].contiguous()
    q, _ = torch.linalg.qr(torch.randn(T, P, 3, 3, device=dev(), generator=g))
    R = (q * torch.sign(torch.linalg.det(q))[..., None, None]).contiguous()
    tr = (0.3 * torch.randn(T, P, 3, device=dev(), generator=g)).contiguous()
    return cano, W, R, tr, frames


@pytest.mark.parametrize("T,N,P", [(1, 8192, 5), (8, 16384, 8), (2, 10000, 4), (64, 8192, 15)])
def test_posed_evaluation_is_bit_identical_to_the_brute_force(T, N, P):
    from reart_b200 import ops
    cano, W, R, tr, frames = articulated(T, N, P, 11)
    M = frames.shape[1]
    to = ops.search_order(frames, 32)
    nn = seeds(T, N, M)
    brute = evaluate(cano, W, R, tr, frames)
    got = evaluate_posed(cano, W, R, tr, frames, to, nn)
    assert got["rc"] == 0
    same(brute, got)
    check_order(got)
    # seeds from that evaluation (by caller index), poses moved a little
    g = torch.Generator(device="cuda").manual_seed(3)
    tr2 = tr + 0.004 * torch.randn(tr.shape, device=dev(), generator=g)
    brute2 = evaluate(cano, W, R, tr2, frames)
    nn[2].zero_()
    same(brute2, evaluate_posed(cano, W, R, tr2, frames, to, nn))
    ev, off, _ = nn[2].tolist()
    assert ev < off, (ev, off)
    # garbage and out-of-range seeds: still exact
    nn[0].random_(0, M); nn[1].random_(0, N)
    same(brute2, evaluate_posed(cano, W, R, tr2, frames, to, nn))
    nn[0].fill_(M + 5); nn[1].fill_(-7)
    same(brute2, evaluate_posed(cano, W, R, tr2, frames, to, nn))


def test_posed_seeds_carry_over_to_the_next_order():
    """Seeds by caller index carry over from one call's row order to the next: the seeded call culls at least as much."""
    from reart_b200 import ops
    T, N, P = 4, 16384, 8
    cano, W, R, tr, frames = articulated(T, N, P, 5)
    to = ops.search_order(frames, 32)
    nn = seeds(T, N, frames.shape[1])
    evaluate_posed(cano, W, R, tr, frames, to, nn)
    first = nn[2][0].item()
    nn[2].zero_()
    evaluate_posed(cano, W, R, tr, frames, to, nn)
    assert nn[2][0].item() <= first


@pytest.mark.parametrize("N", [2048, 8192])
def test_posed_evaluation_keeps_the_lowest_caller_index_on_lattices_and_duplicates(N):
    """Integer lattices and duplicated points: exact ties everywhere (many rows in one bucket of the order too), across
    leaves of the posed order."""
    from reart_b200 import ops
    rng = np.random.default_rng(5)
    T, P = 2, 2
    cano_np = rng.integers(-6, 7, (N, 3)).astype(np.float32)
    cano_np[N // 2:] = cano_np[:N // 2][rng.permutation(N // 2)]
    cano = torch.from_numpy(cano_np).to(dev())
    frames = torch.from_numpy(rng.integers(-6, 7, (T, N, 3)).astype(np.float32)).to(dev())
    W = torch.zeros(N, P, device=dev()); W[:, 0] = 1
    R = torch.eye(3, device=dev()).repeat(T, P, 1, 1).contiguous()
    tr = torch.zeros(T, P, 3, device=dev())
    to = ops.search_order(frames, 32)
    nn = seeds(T, N, N)
    brute = evaluate(cano, W, R, tr, frames)
    got = evaluate_posed(cano, W, R, tr, frames, to, nn)
    same(brute, got)
    check_order(got)
    assert nn[2][2] > 0
    same(brute, evaluate_posed(cano, W, R, tr, frames, to, nn))


@pytest.mark.parametrize("N", [20000, 65536])
def test_posed_evaluation_refuses_clouds_beyond_its_limit(N):
    from reart_b200 import _lib, ops
    assert _lib.lib().reart_posed_order_max_points() < N
    T, P = 1, 2
    g = torch.Generator(device="cuda").manual_seed(1)
    cano = torch.rand(N, 3, device=dev(), generator=g)
    frames = torch.rand(T, N, 3, device=dev(), generator=g)
    W = torch.zeros(N, P, device=dev()); W[:, 0] = 1
    R = torch.eye(3, device=dev()).repeat(T, P, 1, 1).contiguous()
    tr = torch.zeros(T, P, 3, device=dev())
    out = evaluate_posed(cano, W, R, tr, frames, torch.arange(N, device=dev())[None], seeds(T, N, N))
    assert out["rc"] == -4                                                        # REART_ERR_UNSUPPORTED
