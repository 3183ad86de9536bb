"""RelaxationEngine(native=True, flow_ref=...): the relaxation fit with the flow loss on the native iteration.
reart_flow_grad matches float64 autograd of loss.flow_loss w.r.t. the skinned cloud (plain and robust, both mask values,
errors below, at and above 1), a sub-window gives a frame the bits of the whole-sequence call, the native engine follows
the autograd engine (recon + flow, + assignment "add" / "replace"), and a native flow fit is bit-reproducible (run == run,
graph == eager across phase switches, culled == brute, fuse_producer == default, ingest == copying the clouds in)."""
import numpy as np
import pytest
import torch

from conftest import synthetic_sequence

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def dev():
    return torch.device("cuda")


# ---------------------------------------------------------------------------------------------- the kernel
def flow_problem(T, N, c, seed):
    """T skinned frames with the canonical cloud at c, as one window of the complete sequence.  Every fifth point sits
    still in every frame, so its predicted flow is exactly 0 and its targets (+-0.5, +-1, +-2) put its errors below,
    exactly at and above 1."""
    g = torch.Generator().manual_seed(seed)
    cano = 0.3 * torch.randn(N, 3, generator=g)
    sk = cano[None] + 0.2 * torch.randn(T, N, 3, generator=g)
    still = torch.arange(N) % 5 == 0
    sk[:, still] = cano[still]
    win = torch.cat((sk[:c], cano[None], sk[c:])).contiguous()
    tflow = 0.2 * torch.randn(T, N, 3, generator=g)
    levels = torch.tensor([-2.0, -1.0, -0.5, 0.5, 1.0, 2.0])
    tflow[:, still] = levels[torch.randint(0, 6, (T, int(still.sum()), 3), generator=g)]
    mask = (torch.rand(T, N, generator=g) < 0.7).to(torch.uint8)
    slot_frame = torch.tensor([-1 if k == c else (k if k < c else k - 1) for k in range(T + 1)], dtype=torch.int32)
    to = lambda x: x.to(dev()).contiguous()
    return dict(T=T, N=N, c=c, cano=to(cano), sk=to(sk), win=to(win), tflow=to(tflow), mask=to(mask), slot_frame=to(slot_frame))


def flow_grad(pb, lam, robust, g, loss, accumulate, win=None, tflow=None, mask=None, slot_frame=None, T=None, q=None):
    """reart_flow_grad on copies of g / loss; run twice (the kernel re-arms its ticket) and checked bit-reproducible."""
    from reart_b200 import _lib
    L, p = _lib.lib(), _lib.ptr
    win = pb["win"] if win is None else win
    tflow = pb["tflow"] if tflow is None else tflow
    mask = pb["mask"] if mask is None else mask
    slot_frame = pb["slot_frame"] if slot_frame is None else slot_frame
    K, N = win.shape[0], pb["N"]
    T = pb["T"] if T is None else T
    q0, q1 = (0, K - 1) if q is None else q
    nb = int(L.reart_flow_grad_workspace_bytes(K, N))
    ws = torch.zeros(nb, dtype=torch.uint8, device=dev())
    outs = []
    for _ in range(2):
        g1, l1 = g.clone(), loss.clone()
        _lib.check(L.reart_flow_grad(p(win), p(tflow), p(mask), p(slot_frame), lam, int(robust), K, N, T, q0, q1, p(g1), p(l1),
                                     accumulate, p(ws), nb, _lib.stream_ptr()), "reart_flow_grad")
        torch.cuda.synchronize()
        outs.append((g1, l1))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    return outs[0]


def reference(pb, lam, robust, drop=None):
    """float64 autograd of lam * loss.flow_loss over the complete sequence, w.r.t. the skinned frames (the kernel's float32
    inputs, exactly).  Returns (g [T,N,3], loss, element-wise majorant A of g, sum of |terms| of the loss).
    drop="pair": pair 0 left out;  drop="own": the term of the pair after every frame left out of that frame (controls)."""
    from reart_b200.loss import flow_loss
    c = pb["c"]
    sk = pb["sk"].double().requires_grad_(True)
    x = pb["cano"].double()
    complete = torch.cat((sk[:c], x[None], sk[c:]))
    pred = complete[1:] - complete[:-1]
    tf, keep = pb["tflow"].double(), pb["mask"].bool()
    if drop == "own":                                          # no frame sees the pair it opens
        pred = complete[1:] - complete[:-1].detach()
    loss = lam * flow_loss(tf, pred, flow_mask_list=keep, robust=robust)
    if drop == "pair":
        loss = loss - lam * flow_loss(tf[:1], pred[:1], flow_mask_list=keep[:1], robust=robust)
    gsk, = torch.autograd.grad(loss, sk)
    with torch.no_grad():
        err = pred - tf
        # |d| majorant per pair: the derivative of the rule times the magnitudes the float32 pred / err carry
        slope = 1.0 if robust else 2.0
        a = torch.where(keep[:, :, None], slope * (2 * pred.abs() + tf.abs() + err.abs()), 2e-2 * 2 * pred.abs()) * lam
        # a frame at complete index k sees pairs k-1 and k
        a_frame = torch.zeros(pb["T"] + 1, *a.shape[1:], dtype=torch.float64, device=dev())
        a_frame[1:] += a
        a_frame[:-1] += a
        A = torch.cat((a_frame[:c], a_frame[c + 1:]))
        per = torch.where(err.abs() < 1, 0.5 * err * err, err.abs() - 0.5) if robust else err * err
        # each term plus what the rounding of pred and err can move it by (|d term / d err| (|err| + |pred|))
        moved = slope * err.abs().clamp_max(1.0 if robust else float("inf")) * (err.abs() + pred.abs())
        terms = float((torch.where(keep[:, :, None], per.abs() + moved, 2e-2 * pred * pred)).sum() * lam)
    return gsk, float(loss.detach()), A, terms


# The gradient of one element is lam (d_prev - d_next): the rounding of pred, of err, of the rule's scale, of the
# difference and of lam's product -- five roundings, each within u of a term of A (C = 2 x headroom).
C_GRAD = 8
C_LOSS = 16            # the float sum of three components of each of two pairs, then double sums


def within(got, want, A):
    return bool(((got.double() - want).abs() <= C_GRAD * U * A + 1e-30).all())


def worst(got, want, A):
    return float(((got.double() - want).abs() / (C_GRAD * U * A + 1e-30)).max())


CASES = [(T, c) for T in (1, 7, 64) for c in sorted({0, T // 2, T})]


@pytest.mark.parametrize("T,c", CASES)
@pytest.mark.parametrize("robust", [False, True])
def test_flow_grad_matches_float64_autograd(T, c, robust):
    N = 3001 if T < 64 else 1025                                           # not a multiple of the 256-thread CTA
    pb = flow_problem(T, N, c, seed=T * 100 + c + 7 * robust)
    lam = 0.7
    want, wl, A, al = reference(pb, lam, robust)
    nan = torch.full((T, N, 3), float("nan"), device=dev())
    base_l = torch.full((1,), 1.25, dtype=torch.float64, device=dev())
    g, loss = flow_grad(pb, lam, robust, nan, base_l, 0)                  # overwrite: every element written
    assert not torch.isnan(g).any()
    assert within(g, want, A), worst(g, want, A)
    assert abs(float(loss) - wl) <= C_LOSS * U * al + 1e-30
    # accumulate: the overwrite result added onto what was there, bit for bit (one float add per element)
    base = torch.randn(T, N, 3, device=dev())
    ag, al_ = flow_grad(pb, lam, robust, base, base_l, 1)
    assert torch.equal(ag, base + g)
    assert float(al_) == 1.25 + float(loss)


def test_the_bound_catches_a_dropped_pair_or_a_frames_own_term():
    T, c, lam = 7, 3, 0.7
    pb = flow_problem(T, 3001, c, seed=11)
    z = torch.zeros(T, 3001, 3, device=dev())
    l0 = torch.zeros(1, dtype=torch.float64, device=dev())
    want, wl, A, al = reference(pb, lam, False)
    g, loss = flow_grad(pb, lam, False, z, l0, 0)
    assert within(g, want, A)
    for drop in ("pair", "own"):
        dwant, dl, _, _ = reference(pb, lam, False, drop=drop)
        assert not within(g, dwant, A), drop
        assert drop == "own" or abs(float(loss) - dl) > C_LOSS * U * al
    # the kernel's own pair range: leaving the last pair out of [q0, q1) must show in the loss
    _, dl = flow_grad(pb, lam, False, z, l0, 0, q=(0, T - 1))
    assert abs(float(dl) - wl) > C_LOSS * U * al


@pytest.mark.parametrize("c_at", ["start", "middle", "end"])
@pytest.mark.parametrize("world", [2, 3])
def test_sub_windows_give_the_whole_sequence_bits(c_at, world):
    """The windows of dist.flow_window_plan: each rank's frames get the whole-sequence call's bits; the ranks' losses add
    up to the whole sequence's (each pair counted once; only the association of the double sums differs)."""
    from reart_b200.dist import flow_window_plan, shard_bounds
    T, N, lam = 12, 2049, 0.7
    c = {"start": 0, "middle": 5, "end": T}[c_at]
    pb = flow_problem(T, N, c, seed=21 + c)
    l0 = lambda: torch.zeros(1, dtype=torch.float64, device=dev())
    for robust in (False, True):
        g, loss = flow_grad(pb, lam, robust, torch.zeros(T, N, 3, device=dev()), l0(), 0)
        bounds = [shard_bounds(T, world, r) for r in range(world)]
        total = 0.0
        for (lo, hi), pl in zip(bounds, flow_window_plan(T, c, bounds)):
            j0, K = pl["j0"], pl["K"]
            sf = torch.tensor([x[1] if x[0] == "local" else -1 for x in pl["slots"]], dtype=torch.int32, device=dev())
            sg, sl = flow_grad(pb, lam, robust, torch.zeros(hi - lo, N, 3, device=dev()), l0(), 0,
                               win=pb["win"][j0:j0 + K].contiguous(), tflow=pb["tflow"][j0:j0 + K - 1].contiguous(),
                               mask=pb["mask"][j0:j0 + K - 1].contiguous(), slot_frame=sf, T=hi - lo, q=(pl["q0"], pl["q1"]))
            assert torch.equal(sg, g[lo:hi]), (world, c, lo, hi)
            total += float(sl)
        assert abs(total - float(loss)) <= 1e-12 * float(loss)


# ---------------------------------------------------------------------------------------------- the engine
def flow_scene(T, N, P, c, seed=2):
    from reart_b200.flow_utils import FlowReference
    from reart_b200.synth import make_flow_reference
    seq = synthetic_sequence(T, N, P, seed=seed)
    refs, flows = make_flow_reference(seq, c, n_ref=N // 4)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    ref = FlowReference([cu(r) for r in refs], [cu(f) for f in flows])
    return cu(seq["cano"]), cu(seq["frames"]), ref


def relax(cano, frames, P, **kw):
    from reart_b200.engine import RelaxationEngine
    return RelaxationEngine(cano, frames, num_parts=P, seed=2, weight_decay=1e-3, **kw)


def params(eng):
    m = eng.model
    return [q.detach().clone() for q in (m.proposal_6d, m.proposal_t, m.seg_head.model[0].weight, m.seg_head.model[0].bias,
                                         m.seg_head.model[2].weight)]


def fit(eng, steps, ingest=None, by_hand=None):
    """``steps`` steps on the cosine tau schedule; returns (losses, parameters + skinned cloud)."""
    from reart_b200 import ops
    from reart_b200.engine import tau_schedule
    torch.manual_seed(3)
    losses = []
    for i in range(steps):
        if by_hand is not None:
            eng.cano.copy_(by_hand[0]); eng.frames.copy_(by_hand[1])
            ops.pack_cloud(eng.frames, out=eng.frames_packed)
        losses.append(float(eng.step(tau_schedule(i, 100, 5.0, 1.0), ingest=ingest)))
    state = params(eng) + [eng.skinned.clone()]
    eng.release()
    return losses, state


def assign_cfg(mode, **over):
    cfg = dict(downsample=4, assign_gap=3, lambda_assign=0.3, assign_iter=0, mode=mode)
    cfg.update(over)
    return cfg


@pytest.mark.parametrize("assign", [None, "add", "replace"])
@pytest.mark.parametrize("robust", [False, True])
def test_native_flow_fit_follows_the_autograd_fit(assign, robust):
    """Same seed, same gumbel draws: the first step to float rounding, the first four to 2e-5, a 12-step fit to 2e-3 (a
    flipped hard assignment moves the loss ~1/N), as for the recon-only native iteration."""
    c = 2
    cano, frames, ref = flow_scene(5, 3000, 7, c, seed=8)
    extra = dict(flow_ref=ref, cano_idx=c, lambda_flow=0.5, robust_flow=robust, use_graph=False)
    if assign is not None:
        extra["assign"] = assign_cfg(assign, assign_iter=2 if assign == "replace" else 0)
    out = {native: fit(relax(cano, frames, 7, native=native, **extra), 12) for native in (True, False)}
    la, lb = np.array(out[True][0]), np.array(out[False][0])
    assert abs(la[0] - lb[0]) <= 1e-6 * lb[0], (la[0], lb[0])
    np.testing.assert_allclose(la[:4], lb[:4], rtol=2e-5)
    np.testing.assert_allclose(la, lb, rtol=2e-3)
    for a, b in zip(out[True][1][:-1], out[False][1][:-1]):
        assert float((a - b).abs().max()) <= 2e-3 * float(b.abs().max())


def same_run(a, b):
    assert a[0] == b[0]
    for x, y in zip(a[1], b[1]):
        assert torch.equal(x, y)


@pytest.mark.parametrize("mode", [None, "add", "replace"])
def test_native_flow_fit_is_bit_reproducible_graph_and_eager(mode):
    cano, frames, ref = flow_scene(9, 2048, 6, 4, seed=6)
    extra = dict(flow_ref=ref, cano_idx=4, robust_flow=True, native=True, search="brute")
    if mode is not None:
        extra["assign"] = assign_cfg(mode, assign_iter=4)                  # phase switches at step 5, refreshes every 3
    first = fit(relax(cano, frames, 6, use_graph=False, **extra), 14)
    same_run(fit(relax(cano, frames, 6, use_graph=False, **extra), 14), first)
    same_run(fit(relax(cano, frames, 6, use_graph=True, **extra), 14), first)


def test_native_flow_culled_is_brute_and_fused_producer_is_default():
    cano, frames, ref = flow_scene(4, 8192, 8, 2, seed=8)
    extra = dict(flow_ref=ref, cano_idx=2, native=True, assign=assign_cfg("add", downsample=8))
    for graph in (True, False):
        brute = fit(relax(cano, frames, 8, use_graph=graph, search="brute", **extra), 8)
        culled = relax(cano, frames, 8, use_graph=graph, **extra)             # "auto" at 8192 points: culled
        assert culled.search_culled
        same_run(fit(culled, 8), brute)
        same_run(fit(relax(cano, frames, 8, use_graph=graph, fuse_producer=True, **extra), 8), brute)


def test_native_flow_ingest_is_copying_the_clouds_in_by_hand():
    cano, frames, ref = flow_scene(6, 2048, 6, 3, seed=9)
    g = torch.Generator(device="cuda").manual_seed(1)
    cano2 = (cano + 1e-3 * torch.randn(cano.shape, device=dev(), generator=g)).contiguous()
    frames2 = (frames + 1e-3 * torch.randn(frames.shape, device=dev(), generator=g)).contiguous()
    extra = dict(flow_ref=ref, cano_idx=3, native=True, search="brute", assign=assign_cfg("replace", assign_iter=3))
    # every engine gets its own copies: the engine adopts a float32 contiguous cloud without copying it, so the by-hand
    # copies would otherwise change the clouds the next engine samples its assignment points from
    hand = fit(relax(cano.clone(), frames.clone(), 6, use_graph=False, **extra), 8, by_hand=(cano2, frames2))
    for graph in (False, True):
        same_run(fit(relax(cano.clone(), frames.clone(), 6, use_graph=graph, **extra), 8, ingest=(0, cano2, frames2)), hand)


def test_native_flow_refusals():
    from reart_b200.engine import RelaxationEngine
    cano, frames, ref = flow_scene(4, 512, 4, 0)
    with pytest.raises(ValueError):
        RelaxationEngine(cano, frames, 4, native=True, flow_ref=ref, cull=True)
    with pytest.raises(ValueError):
        RelaxationEngine(cano, frames[:3], 4, native=True, flow_ref=ref)
    with pytest.raises(ValueError):
        RelaxationEngine(cano, frames, 4, native=True, flow_ref=ref, cano_idx=5)
    # native=None keeps the autograd composition with a flow loss
    assert not RelaxationEngine(cano, frames, 4, flow_ref=ref).native


# ---------------------------------------------------------------------------------------------- two GPUs
def _two_gpu_worker(rank, world, port, out_dir):
    import os
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    from reart_b200.dist import DistContext
    from reart_b200.engine import RelaxationEngine, tau_schedule
    ctx = DistContext.from_env()
    d = torch.device("cuda", rank)
    torch.cuda.set_device(d)
    out = {}
    for c in (0, 4, 8):                                                    # c = 4: the canonical frame between the shards
        cano, frames, ref = flow_scene(8, 4096, 6, c)
        extra = dict(flow_ref=ref, cano_idx=c, lambda_flow=0.5, native=True, seed=2)

        def steps(eng):
            torch.manual_seed(5); torch.cuda.manual_seed_all(5)
            ls = [float(eng.step(tau_schedule(i, 100, 5.0, 1.0))) for i in range(10)]
            w2 = eng.model.seg_head.model[2].weight.detach().cpu().numpy().copy()
            eng.release()
            return ls, w2
        for graph in (False, True):
            out[f"sharded_{c}_{int(graph)}"], out[f"w2_{c}_{int(graph)}"] = steps(
                RelaxationEngine(cano, frames, 6, ctx=ctx, use_graph=graph, **extra))
        if rank == 0:
            out[f"single_{c}"], _ = steps(RelaxationEngine(cano, frames, 6, ctx=DistContext(), use_graph=False, **extra))
    np.savez(os.path.join(out_dir, f"relaxflow{rank}.npz"), **out)
    dist.barrier()
    os._exit(0)


@pytest.mark.timeout(300)
def test_sharded_native_relaxation_flow_on_two_gpus(tmp_path):
    """Frame sharding: neighbour frames travel forward only; the sharded native flow fit reproduces the one-GPU fit's first
    step to 1e-6, graph == eager bit for bit, identical shared parameters on both ranks."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_two_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "relaxflow0.npz"), np.load(tmp_path / "relaxflow1.npz")
    for c in (0, 4, 8):
        assert list(r0[f"sharded_{c}_0"]) == list(r0[f"sharded_{c}_1"]) == list(r1[f"sharded_{c}_0"]) == list(r1[f"sharded_{c}_1"]), c
        assert np.array_equal(r0[f"w2_{c}_1"], r1[f"w2_{c}_1"]) and np.array_equal(r0[f"w2_{c}_0"], r0[f"w2_{c}_1"]), c
        assert abs(r0[f"sharded_{c}_0"][0] - r0[f"single_{c}"][0]) <= 1e-6 * r0[f"single_{c}"][0], c
        np.testing.assert_allclose(r0[f"sharded_{c}_0"], r0[f"single_{c}"], rtol=5e-3)
