"""KinematicEngine(flow_ref=...): the kinematic fit with the flow loss.  reart_kin_flow matches float64 autograd of
loss.flow_loss on one-hot skinning (plain and robust, both mask values, errors on both sides of 1 and at 1), a sub-window
gives a frame the bits of the whole-sequence call, the native engine matches the autograd engine (alone and with the
assignment loss), the autograd engine is the hand-written composition, and a native run is bit-reproducible (run == run,
graph == eager across phase switches, culled == brute, ingest == no ingest)."""
import math

import numpy as np
import pytest
import torch

from conftest import synthetic_sequence
from test_kinematic_native_gpu import clone, engine, params, scene

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda")


# ---------------------------------------------------------------------------------------------- the kernel
def flow_problem(T, N, P, c, seed):
    """The complete sequence of T one-hot skinned frames with the canonical cloud at c, as one window.  Part P-1 has no
    points; part 0 keeps the identity pose in every frame, so its predicted flow is exactly 0 and its targets (+-0.5,
    +-1, +-2) put its errors below, exactly at and above 1."""
    g = torch.Generator().manual_seed(seed)
    labels = torch.randint(0, max(P - 1, 1), (N,), generator=g)
    cano = 0.3 * torch.randn(N, 3, generator=g)
    R = torch.linalg.qr(torch.randn(T, P, 3, 3, generator=g))[0]
    tr = 0.3 * torch.randn(T, P, 3, generator=g)
    R[:, 0], tr[:, 0] = torch.eye(3), 0.0
    sk = torch.einsum("tnij,nj->tni", R[:, labels], cano) + tr[:, labels]
    win = torch.cat((sk[:c], cano[None], sk[c:])).contiguous()
    tflow = torch.randn(T, N, 3, generator=g)
    levels = torch.tensor([-2.0, -1.0, -0.5, 0.5, 1.0, 2.0])
    zero = labels == 0
    tflow[:, zero] = levels[torch.randint(0, 6, (T, int(zero.sum()), 3), generator=g)]
    mask = (torch.rand(T, N, generator=g) < 0.7).to(torch.uint8)
    slot_frame = torch.tensor([-1 if k == c else (k if k < c else k - 1) for k in range(T + 1)], dtype=torch.int32)
    to = lambda x: x.to(dev()).contiguous()
    return dict(T=T, N=N, P=P, c=c, labels=to(labels), cano=to(cano), R=to(R), tr=to(tr), sk=to(sk), win=to(win),
                tflow=to(tflow), mask=to(mask), slot_frame=to(slot_frame))


def grouping(labels, P):
    order = torch.argsort(labels, stable=True).int()
    offsets = torch.cat((labels.new_zeros(1), torch.bincount(labels, minlength=P).cumsum(0))).int()
    return order, offsets


def kin_flow(pb, lam, robust, gR, gtr, loss, accumulate, win=None, tflow=None, mask=None, slot_frame=None, T=None, q=None,
             order=None):
    from reart_b200 import _lib
    L, p = _lib.lib(), _lib.ptr
    win = pb["win"] if win is None else win
    tflow = pb["tflow"] if tflow is None else tflow
    mask = pb["mask"] if mask is None else mask
    slot_frame = pb["slot_frame"] if slot_frame is None else slot_frame
    K, N, P = win.shape[0], pb["N"], pb["P"]
    T = pb["T"] if T is None else T
    q0, q1 = (0, K - 1) if q is None else q
    o, offsets = grouping(pb["labels"], P)
    if order is not None:
        o, offsets = order
    nb = int(L.reart_kin_flow_workspace_bytes(K, P))
    ws = torch.zeros(nb, dtype=torch.uint8, device=dev())
    outs = []
    for _ in range(2):                                                    # twice: the kernel re-arms its ticket
        g1, t1, l1 = gR.clone(), gtr.clone(), loss.clone()
        _lib.check(L.reart_kin_flow(p(win), p(tflow), p(mask), p(slot_frame), p(pb["cano"]), p(o), p(offsets), lam,
                                    int(robust), K, N, P, T, q0, q1, p(g1), p(t1), p(l1), accumulate, p(ws), nb,
                                    _lib.stream_ptr()), "reart_kin_flow")
        torch.cuda.synchronize()
        outs.append((g1, t1, l1))
    assert all(torch.equal(a, b) for a, b in zip(*outs))                 # and bit-reproducible
    return outs[0]


def reference(pb, lam, robust):
    """float64 autograd of lam * loss.flow_loss over the complete sequence, on the float32 skinned values (the kernel's
    inputs) with the gradient of the one-hot skinning.  Returns (gR, gtr, loss, |terms| of gR, |terms| of gtr, |terms| of
    the loss, per-point gradient of the skinned cloud)."""
    from reart_b200.loss import flow_loss
    T, P, c = pb["T"], pb["P"], pb["c"]
    lab, x = pb["labels"], pb["cano"].double()
    R = pb["R"].double().requires_grad_(True)
    tr = pb["tr"].double().requires_grad_(True)
    sk64 = torch.einsum("tnij,nj->tni", R[:, lab], x) + tr[:, lab]
    sk = (pb["sk"].double() + (sk64 - sk64.detach())).detach().requires_grad_(True)
    complete = torch.cat((sk[:c], x[None], sk[c:]))
    pred = complete[1:] - complete[:-1]
    tf, keep = pb["tflow"].double(), pb["mask"].bool()
    loss = lam * flow_loss(tf, pred, flow_mask_list=keep, robust=robust)
    gsk, = torch.autograd.grad(loss, sk, retain_graph=True)
    (sk64 * gsk).sum().backward()
    with torch.no_grad():
        err = pred - tf
        per = torch.where(err.abs() < 1, 0.5 * err * err, err.abs() - 0.5) if robust else err * err
        terms = torch.where(keep[:, :, None], per, 1e-2 * pred * pred).abs().sum() * lam
        absR = torch.zeros(T, P, 3, 3, dtype=torch.float64, device=dev())
        absR.index_add_(1, lab, (gsk[:, :, :, None] * x[None, :, None, :]).abs())
        abst = torch.zeros(T, P, 3, dtype=torch.float64, device=dev())
        abst.index_add_(1, lab, gsk.abs())
    return R.grad, tr.grad, loss.item(), absR, abst, float(terms), gsk


def within(got, want, absterm, c):
    return bool(((got.double() - want).abs() <= c * 2.0 ** -24 * absterm + 1e-30).all())


def bound_c(pb):
    per_part = int(torch.bincount(pb["labels"], minlength=pb["P"]).max())
    return 4 * (math.ceil(per_part / 256) + 16)                           # per-point ops, the thread's chain, the trees


CASES = [(T, P, c) for T in (1, 7, 64) for P in (2, 8, 32) for c in sorted({0, T // 2, T})]


@pytest.mark.parametrize("T,P,c", CASES)
@pytest.mark.parametrize("robust", [False, True])
def test_kin_flow_matches_float64_autograd(T, P, c, robust):
    N = 4096 if T < 64 else 1024
    pb = flow_problem(T, N, P, c, seed=T * 100 + P + c)
    lam = 0.7
    wR, wt, wl, aR, at, al, _ = reference(pb, lam, robust)
    cc = bound_c(pb)
    base_R, base_t = torch.randn(T, P, 3, 3, device=dev()), torch.randn(T, P, 3, device=dev())
    base_l = torch.full((1,), 1.25, dtype=torch.float64, device=dev())
    gR, gtr, loss = kin_flow(pb, lam, robust, base_R, base_t, base_l, 0)
    used = slice(0, max(P - 1, 1))
    assert within(gR[:, used], wR[:, used], aR[:, used], cc) and within(gtr[:, used], wt[:, used], at[:, used], cc)
    assert abs(float(loss) - wl) <= cc * 2.0 ** -24 * al + 1e-30
    assert not gR[:, P - 1].any() and not gtr[:, P - 1].any()            # the part without points: zeros
    # accumulate: the same sums added onto what the energy wrote (bit for bit); the empty part is left untouched
    aR_, at_, al_ = kin_flow(pb, lam, robust, base_R, base_t, base_l, 1)
    assert torch.equal(aR_[:, used], base_R[:, used] + gR[:, used]) and torch.equal(at_[:, used], base_t[:, used] + gtr[:, used])
    assert torch.equal(aR_[:, P - 1], base_R[:, P - 1]) and torch.equal(at_[:, P - 1], base_t[:, P - 1])
    assert float(al_) == 1.25 + float(loss)


def test_the_bound_catches_a_dropped_point_or_pair():
    T, P, c, lam = 7, 8, 3, 0.7
    pb = flow_problem(T, 4096, P, c, seed=11)
    wR, wt, wl, aR, at, al, gsk = reference(pb, lam, False)
    cc = bound_c(pb)
    z = lambda *s: torch.zeros(*s, device=dev())
    l0 = torch.zeros(1, dtype=torch.float64, device=dev())
    gR, gtr, loss = kin_flow(pb, lam, False, z(T, P, 3, 3), z(T, P, 3), l0, 0)
    assert within(gR, wR, aR, cc) and within(gtr, wt, at, cc)
    # drop the point with the largest gradient from its part
    order, offsets = grouping(pb["labels"], P)
    i = int(gsk.abs().sum(dim=(0, 2)).argmax())
    part = int(pb["labels"][i])
    kept = order[order != i]
    offs = offsets.clone()
    offs[part + 1:] -= 1
    dR, dt, _ = kin_flow(pb, lam, False, z(T, P, 3, 3), z(T, P, 3), l0, 0, order=(kept.contiguous(), offs))
    assert not (within(dR, wR, aR, cc) and within(dt, wt, at, cc))
    # drop a pair from the loss
    _, _, dl = kin_flow(pb, lam, False, z(T, P, 3, 3), z(T, P, 3), l0, 0, q=(0, T - 1))
    assert abs(float(dl) - wl) > cc * 2.0 ** -24 * al


@pytest.mark.parametrize("c_at", ["start", "middle", "end"])
@pytest.mark.parametrize("world", [2, 3])
def test_sub_windows_give_the_whole_sequence_bits(c_at, world):
    from reart_b200.dist import flow_window_plan, shard_bounds
    T, P, lam = 12, 8, 0.7
    c = {"start": 0, "middle": 5, "end": T}[c_at]
    pb = flow_problem(T, 2048, P, c, seed=21 + c)
    z = lambda *s: torch.zeros(*s, device=dev())
    for robust in (False, True):
        gR, gtr, loss = kin_flow(pb, lam, robust, z(T, P, 3, 3), z(T, P, 3), torch.zeros(1, dtype=torch.float64, device=dev()), 0)
        bounds = [shard_bounds(T, world, r) for r in range(world)]
        total = 0.0
        for (lo, hi), pl in zip(bounds, flow_window_plan(T, c, bounds)):
            j0, K = pl["j0"], pl["K"]
            sf = torch.tensor([x[1] if x[0] == "local" else -1 for x in pl["slots"]], dtype=torch.int32, device=dev())
            sR, st, sl = kin_flow(pb, lam, robust, z(hi - lo, P, 3, 3), z(hi - lo, P, 3),
                                  torch.zeros(1, dtype=torch.float64, device=dev()), 0,
                                  win=pb["win"][j0:j0 + K].contiguous(), tflow=pb["tflow"][j0:j0 + K - 1].contiguous(),
                                  mask=pb["mask"][j0:j0 + K - 1].contiguous(), slot_frame=sf, T=hi - lo, q=(pl["q0"], pl["q1"]))
            assert torch.equal(sR, gR[lo:hi]) and torch.equal(st, gtr[lo:hi]), (world, c, lo, hi)
            total += float(sl)
        assert abs(total - float(loss)) <= 1e-12 * float(loss)


# ---------------------------------------------------------------------------------------------- the engine
def flow_scene(T, N, P, c, seed=2, n_ref=None, **kw):
    """scene() plus the synthetic flow reference of the same sequence."""
    from reart_b200.flow_utils import FlowReference
    from reart_b200.synth import make_flow_reference
    k, part, cano, frames = scene(T, N, P, seed=seed, **kw)
    refs, flows = make_flow_reference(synthetic_sequence(T, N, P, seed=seed), c, n_ref=n_ref or N // 4)
    ref = FlowReference([torch.from_numpy(r).to(dev()) for r in refs], [torch.from_numpy(f).to(dev()) for f in flows])
    return k, part, cano, frames, ref, (refs, flows)


def assign_cfg(mode, **over):
    cfg = dict(downsample=8, assign_gap=5, lambda_assign=0.3, assign_iter=0, mode=mode)
    cfg.update(over)
    return cfg


def grads_of_native_step(nat):
    m = nat.model
    g = nat._nat["grad"]
    E, T = m.axis_list.shape[0], m.theta_list.shape[0]
    sizes = [3 * E, 3 * E, 1, T * E] + ([T * E] if hasattr(m, "distance_list") else []) + ([6 * T, 3 * T] if hasattr(m, "root_6d") else [])
    parts = list(torch.split(g, sizes))
    del parts[2]                                                           # the loss slot
    return parts


@pytest.mark.parametrize("assign", [None, "add", "replace"])
@pytest.mark.parametrize("robust", [False, True])
@pytest.mark.parametrize("case,c", [("revolute", 0), ("mixed", 2), ("root", 5)])
def test_native_flow_gradients_and_a_short_fit_match_autograd(case, c, robust, assign):
    kw, part, cano, frames, ref_flow, _ = flow_scene(5, 2048, 6, c, prismatic=case != "revolute", root=case == "root", seed=4)
    extra = dict(flow_ref=ref_flow, cano_idx=c, robust_flow=robust, lambda_flow=0.5)
    if assign is not None:
        extra["assign"] = assign_cfg(assign)
    ref = engine(kw, part, cano, frames, use_graph=False, **extra)
    if hasattr(ref.model, "root_t"):                                       # fused Adam rejects the strided view (as in
        ref.model.root_t.data = ref.model.root_t.data.contiguous()         # test_kinematic_assign_gpu.py)
    ref.optimizer.zero_grad(set_to_none=True)
    ref.iteration = 1
    ref_loss = ref._iteration()
    ref_loss.backward()
    ref_grads = [q.grad.detach().clone() for q in ref._opt_params()]
    nat = engine(kw, part, cano, frames, use_graph=False, native=True, **extra)
    loss = float(nat.step())
    for got, want in zip(grads_of_native_step(nat), ref_grads):
        err = float((got - want.reshape(-1)).abs().max())
        assert err <= 1e-5 * float(want.abs().max()) + 1e-12, (case, robust, assign, err, float(want.abs().max()))
    assert abs(loss - ref_loss.item()) <= 1e-5 * ref_loss.item()
    for _ in range(11):
        nat.step()
    ref.iteration = 0
    for _ in range(12):
        ref.step()
    for a, b in zip(params(nat), params(ref)):
        assert float((a - b).abs().max()) <= 2e-3 * float(b.abs().max()), (case, robust, assign)


@pytest.mark.parametrize("c", [0, 3, 6])
def test_autograd_flow_path_is_the_hand_written_composition(c):
    from reart_b200 import ops
    from reart_b200.flow_utils import blend_anchor_motion
    from reart_b200.knn_module import KNN
    from reart_b200.loss import flow_loss
    kw, part, cano, frames, ref_flow, (refs, flows) = flow_scene(6, 2048, 5, c, prismatic=True, seed=9)
    eng = engine(kw, part, cano, frames, use_graph=False, flow_ref=ref_flow, cano_idx=c, lambda_flow=0.5)
    eng.iteration = 1
    loss = eng._iteration()
    loss.backward()
    got = [q.grad.detach().clone() for q in eng._opt_params()]
    hand = engine(kw, part, cano, frames, use_graph=False)
    trans = hand.model.transforms()
    R, tr = trans[:, :, :3, :3].contiguous(), trans[:, :, :3, 3].contiguous()
    chamfer, skinned = ops.skinned_chamfer_loss(hand.cano, hand.weight, R, tr, hand.frames, hand.frames_packed, unit_grad=True)
    complete = torch.cat((skinned[:c], hand.cano[None], skinned[c:]))
    knn = KNN(k=3, transpose_mode=True)
    tgt, masks = [], []
    with torch.no_grad():
        for k in range(complete.shape[0] - 1):
            t_, m_ = blend_anchor_motion(complete[k].detach(), torch.from_numpy(refs[k]).to(dev()),
                                         torch.from_numpy(flows[k]).to(dev()), knn, return_mask=True)
            tgt.append(t_); masks.append(m_)
    want_loss = chamfer + 0.5 * flow_loss(torch.stack(tgt), complete[1:] - complete[:-1], flow_mask_list=torch.stack(masks))
    want_loss.backward()
    assert abs(loss.item() - want_loss.item()) <= 1e-6 * want_loss.item()
    for a, q in zip(got, hand._opt_params()):
        assert float((a - q.grad).abs().max()) <= 1e-5 * float(q.grad.abs().max()) + 1e-12


def run(kw, part, cano, frames, steps, ingest=None, **extra):
    eng = engine(kw, part, cano, frames, native=True, **extra)
    losses = [float(eng.step(ingest=ingest)) for _ in range(steps)]
    state = params(eng) + [eng.skinned.clone()]
    eng.release()
    return losses, state


def same_run(a, b):
    assert a[0] == b[0]
    for x, y in zip(a[1], b[1]):
        assert torch.equal(x, y)


@pytest.mark.parametrize("mode", [None, "add", "replace"])
def test_native_flow_fit_is_bit_reproducible_graph_and_eager(mode):
    kw, part, cano, frames, ref_flow, _ = flow_scene(9, 2048, 6, 4, prismatic=True, root=True, seed=6)
    extra = dict(flow_ref=ref_flow, cano_idx=4, robust_flow=True, search="brute")
    if mode is not None:
        extra["assign"] = assign_cfg(mode, downsample=4, assign_iter=4, assign_gap=3)       # phase switches at step 5
    first = run(kw, part, cano, frames, 14, use_graph=False, **extra)
    same_run(run(kw, part, cano, frames, 14, use_graph=False, **extra), first)
    same_run(run(kw, part, cano, frames, 14, use_graph=True, **extra), first)


def test_native_flow_culled_is_brute_and_ingest_is_no_ingest_bit_for_bit():
    kw, part, cano, frames, ref_flow, _ = flow_scene(4, 8192, 8, 2, seed=8)
    extra = dict(flow_ref=ref_flow, cano_idx=2)
    for graph in (True, False):
        brute = run(kw, part, cano, frames, 8, use_graph=graph, search="brute", **extra)
        culled = run(kw, part, cano, frames, 8, use_graph=graph, **extra)                  # "auto" at 8192 points: culled
        same_run(culled, brute)
        ingest = run(kw, part, cano, frames, 8, use_graph=graph, search="brute", ingest=(0, cano.clone(), frames.clone()),
                     **extra)
        same_run(ingest, brute)


def test_flow_reference_must_cover_the_complete_sequence():
    kw, part, cano, frames, ref_flow, _ = flow_scene(4, 512, 4, 0)
    with pytest.raises(ValueError):
        engine(kw, part, cano, frames[:3], flow_ref=ref_flow)
    with pytest.raises(ValueError):
        engine(kw, part, cano, frames, flow_ref=ref_flow, cano_idx=5)


# ---------------------------------------------------------------------------------------------- two GPUs
def _two_gpu_worker(rank, world, port, out_dir):
    import os
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    from reart_b200.dist import DistContext
    from reart_b200.engine import KinematicEngine
    ctx = DistContext.from_env()
    d = torch.device("cuda", rank)
    torch.cuda.set_device(d)
    out = {}
    for c in (0, 4, 8):                                                    # c = 4: the canonical frame between the shards
        kw, part, cano, frames, ref_flow, _ = flow_scene(8, 4096, 6, c, prismatic=True)
        extra = dict(flow_ref=ref_flow, cano_idx=c, lambda_flow=0.5)
        for name, over in (("nat0", dict(native=True, use_graph=False)), ("nat1", dict(native=True, use_graph=True)),
                           ("auto", dict(use_graph=False))):
            eng = KinematicEngine(clone(kw), part, cano, frames, ctx=ctx, **over, **extra)
            if hasattr(eng.model, "root_t"):
                eng.model.root_t.data = eng.model.root_t.data.contiguous()
            out[f"{name}_{c}"] = [float(eng.step()) for _ in range(12)]
            out[f"{name}_{c}_axis"] = eng.model.axis_list.detach().cpu().numpy().copy()
            out[f"{name}_{c}_moment"] = eng.model.moment_list.detach().cpu().numpy().copy()
            eng.release()
        if rank == 0:
            single = KinematicEngine(clone(kw), part, cano, frames, ctx=DistContext(), use_graph=False, native=True, **extra)
            out[f"single_{c}"] = [float(single.step()) for _ in range(12)]
            out[f"single_{c}_axis"] = single.model.axis_list.detach().cpu().numpy().copy()
            single.release()
    np.savez(os.path.join(out_dir, f"kinflow{rank}.npz"), **out)
    dist.barrier()
    os._exit(0)


@pytest.mark.timeout(300)
def test_sharded_native_kinematic_flow_on_two_gpus(tmp_path):
    """Frame sharding: neighbour frames travel forward only; the sharded native fit follows the 1-GPU native fit and the
    sharded autograd fit, graph == eager on every rank, identical shared parameters on both ranks."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_two_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "kinflow0.npz"), np.load(tmp_path / "kinflow1.npz")
    for c in (0, 4, 8):
        assert list(r0[f"nat0_{c}"]) == list(r0[f"nat1_{c}"]) == list(r1[f"nat0_{c}"]) == list(r1[f"nat1_{c}"]), c
        for k in ("axis", "moment"):
            assert np.array_equal(r0[f"nat0_{c}_{k}"], r1[f"nat0_{c}_{k}"]) and np.array_equal(r0[f"nat0_{c}_{k}"], r0[f"nat1_{c}_{k}"])
        for other in ("single", "auto"):
            a, b = np.array(r0[f"nat0_{c}"]), np.array(r0[f"{other}_{c}"])
            assert np.all(np.abs(a - b) <= 1e-3 * np.abs(b)), (c, other, a, b)
            assert np.abs(r0[f"nat0_{c}_axis"] - r0[f"{other}_{c}_axis"]).max() <= 2e-3, (c, other)
