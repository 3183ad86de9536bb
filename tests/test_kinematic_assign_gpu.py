"""KinematicEngine(assign=...): the kinematic fit with the assignment loss.  reart_kin_assign equals the composition
reart_assign_loss_grad + reart_skin_bwd (and float64 autograd) on one-hot weights; the native engine matches the autograd
engine in both flavours ("add": Chamfer + assignment, "replace": assignment only), its assignments are the host solver's,
a run is bit-reproducible (graph == eager, run == run), the culled search is the brute force bit for bit, and a
"replace" fit recovers the joint angles."""
import numpy as np
import pytest
import torch

from test_kinematic_native_gpu import clone, engine, params, scene

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda")


# ---------------------------------------------------------------------------------------------- the kernel
def assign_problem(T, n, P, seed):
    """Random one-hot scene: labels with part P-1 never sampled, n distinct samples, random matchings."""
    g = torch.Generator().manual_seed(seed)
    N = max(2 * n, 256)
    labels = torch.randint(0, P, (N,), generator=g)
    src_idx = torch.randperm(N, generator=g)[:n]
    labels[src_idx] = torch.randint(0, P - 1, (n,), generator=g)           # part P-1: no samples
    cano = torch.randn(N, 3, generator=g)
    R = torch.linalg.qr(torch.randn(T, P, 3, 3, generator=g))[0]
    tr = 0.1 * torch.randn(T, P, 3, generator=g)
    tgt = torch.randn(T, n, 3, generator=g)
    col4row = torch.stack([torch.randperm(n, generator=g) for _ in range(T)]).int()
    to = lambda x: x.to(dev()).contiguous()
    return dict(T=T, N=N, n=n, P=P, labels=to(labels), src_idx=to(src_idx), cano=to(cano), R=to(R), tr=to(tr), tgt=to(tgt),
                col4row=to(col4row))


def kin_assign(pb, skinned, lam, gR, gtr, loss, accumulate):
    from reart_b200 import _lib
    L, p = _lib.lib(), _lib.ptr
    sample_part = pb["labels"][pb["src_idx"]]
    order = torch.argsort(sample_part, stable=True).int()
    offsets = torch.cat((sample_part.new_zeros(1), torch.bincount(sample_part, minlength=pb["P"]).cumsum(0))).int()
    nb = int(L.reart_kin_assign_workspace_bytes(pb["T"], pb["P"]))
    ws = torch.zeros(nb, dtype=torch.uint8, device=dev())
    outs = []
    for _ in range(2):                                                    # twice: the kernel re-arms its ticket
        g1, t1, l1 = gR.clone(), gtr.clone(), loss.clone()
        _lib.check(L.reart_kin_assign(p(skinned), p(pb["cano"]), p(pb["src_idx"]), p(pb["tgt"]), p(pb["col4row"]), p(order),
                                      p(offsets), lam, pb["T"], pb["N"], pb["n"], pb["P"], p(g1), p(t1), p(l1), accumulate,
                                      p(ws), nb, _lib.stream_ptr()), "reart_kin_assign")
        torch.cuda.synchronize()
        outs.append((g1, t1, l1))
    assert all(torch.equal(a, b) for a, b in zip(*outs))                 # and bit-reproducible
    return outs[0]


def composition(pb, skinned, lam):
    """reart_assign_loss_grad into a [T,N,3] gradient, then the full skin backward with the one-hot W."""
    from reart_b200 import _lib
    L, p = _lib.lib(), _lib.ptr
    T, N, n, P = pb["T"], pb["N"], pb["n"], pb["P"]
    W = torch.nn.functional.one_hot(pb["labels"], P).float().contiguous()
    gs = torch.zeros(T, N, 3, device=dev())
    loss = torch.zeros(1, dtype=torch.float64, device=dev())
    _lib.check(L.reart_assign_loss_grad(p(skinned), p(pb["src_idx"]), p(pb["tgt"]), p(pb["col4row"]), T, N, n, lam, p(gs), 0,
                                        p(loss), _lib.stream_ptr()), "reart_assign_loss_grad")
    gW, gR, gtr = torch.empty(N, P, device=dev()), torch.empty(T, P, 3, 3, device=dev()), torch.empty(T, P, 3, device=dev())
    nb = int(L.reart_skin_bwd_workspace_bytes(T, N, P))
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev())
    _lib.check(L.reart_skin_bwd(p(pb["cano"]), p(W), p(pb["R"]), p(pb["tr"]), p(gs), T, N, P, p(gW), p(gR), p(gtr), p(ws), nb,
                                _lib.stream_ptr()), "reart_skin_bwd")
    torch.cuda.synchronize()
    return gR, gtr, float(loss)


def skinned_of(pb):
    from reart_b200 import ops
    W = torch.nn.functional.one_hot(pb["labels"], pb["P"]).float()
    return ops.skin(pb["cano"], W, pb["R"], pb["tr"]).contiguous()


def close(got, want, rel):
    return float((got - want).abs().max()) <= rel * float(want.abs().max()) + 1e-30


@pytest.mark.parametrize("T", [1, 7, 64])
@pytest.mark.parametrize("n", [37, 1024, 4096])
@pytest.mark.parametrize("P", [2, 8, 32])
def test_kin_assign_is_the_composition_of_assign_grad_and_skin_backward(T, n, P):
    pb = assign_problem(T, n, P, seed=T * 1000 + n + P)
    skinned, lam = skinned_of(pb), 0.3
    wR, wt, wl = composition(pb, skinned, lam)
    base_R, base_t = torch.randn(T, P, 3, 3, device=dev()), torch.randn(T, P, 3, device=dev())
    base_l = torch.full((1,), 1.25, dtype=torch.float64, device=dev())
    for accumulate in (0, 1):
        gR, gtr, loss = kin_assign(pb, skinned, lam, base_R, base_t, base_l, accumulate)
        want_R, want_t = (base_R + wR, base_t + wt) if accumulate else (wR, wt)
        want_l = 1.25 * accumulate + wl
        assert close(gR[:, :P - 1], want_R[:, :P - 1], 1e-5) and close(gtr[:, :P - 1], want_t[:, :P - 1], 1e-5), accumulate
        assert abs(float(loss) - want_l) <= 1e-6 * want_l, (float(loss), want_l)
        # the part without samples: untouched when accumulating, zeros otherwise
        if accumulate:
            assert torch.equal(gR[:, P - 1], base_R[:, P - 1]) and torch.equal(gtr[:, P - 1], base_t[:, P - 1])
        else:
            assert not gR[:, P - 1].any() and not gtr[:, P - 1].any()


@pytest.mark.parametrize("T,n,P", [(1, 37, 2), (7, 1024, 8), (64, 4096, 32)])
def test_kin_assign_matches_float64_autograd(T, n, P):
    pb = assign_problem(T, n, P, seed=7 + T + n + P)
    skinned, lam = skinned_of(pb), 0.3
    gR, gtr, loss = kin_assign(pb, skinned, lam, torch.zeros(T, P, 3, 3, device=dev()), torch.zeros(T, P, 3, device=dev()),
                               torch.zeros(1, dtype=torch.float64, device=dev()), 0)
    R = pb["R"].double().requires_grad_(True)
    tr = pb["tr"].double().requires_grad_(True)
    lab, x = pb["labels"], pb["cano"].double()
    sk = torch.einsum("tnij,nj->tni", R[:, lab], x) + tr[:, lab]
    a = sk[:, pb["src_idx"]]
    b = torch.gather(pb["tgt"].double(), 1, pb["col4row"].long()[:, :, None].expand(-1, -1, 3))
    ref = lam * ((a - b) ** 2).sum()
    ref.backward()
    assert close(gR.double(), R.grad, 1e-5) and close(gtr.double(), tr.grad, 1e-5)
    assert abs(float(loss) - ref.item()) <= 1e-6 * ref.item()


# ---------------------------------------------------------------------------------------------- the engine
def assign_cfg(mode, **over):
    cfg = dict(downsample=8, assign_gap=5, lambda_assign=0.3, assign_iter=0, mode=mode)
    cfg.update(over)
    return cfg


@pytest.mark.parametrize("mode", ["add", "replace"])
@pytest.mark.parametrize("case", ["revolute", "mixed", "root"])
def test_native_assign_gradients_and_a_short_fit_match_autograd(mode, case):
    kw, part, cano, frames = scene(5, 2048, 6, prismatic=case != "revolute", root=case == "root", seed=4)
    cfg = assign_cfg(mode)
    ref = engine(kw, part, cano, frames, use_graph=False, assign=cfg)
    # KinematicModel keeps root_t as a strided view of root_trans, whose gradient torch's fused Adam rejects; the reference
    # optimisation runs on a contiguous copy of the same values
    if hasattr(ref.model, "root_t"):
        ref.model.root_t.data = ref.model.root_t.data.contiguous()
    ref.optimizer.zero_grad(set_to_none=True)
    ref.iteration = 1                                                      # the phase of the first step: assignment, refresh
    ref_loss = ref._iteration()
    ref_loss.backward()
    ref_grads = [q.grad.detach().clone() for q in ref._opt_params()]
    nat = engine(kw, part, cano, frames, use_graph=False, native=True, assign=cfg)
    loss = float(nat.step())
    m = ref.model
    g = nat._nat["grad"]
    E, T = m.axis_list.shape[0], m.theta_list.shape[0]
    sizes = [3 * E, 3 * E, 1, T * E] + ([T * E] if hasattr(m, "distance_list") else []) + ([6 * T, 3 * T] if hasattr(m, "root_6d") else [])
    parts = list(torch.split(g, sizes))
    del parts[2]                                                           # the loss slot
    for got, want in zip(parts, ref_grads):
        err = float((got - want.reshape(-1)).abs().max())
        assert err <= 1e-5 * float(want.abs().max()) + 1e-12, (mode, case, err, float(want.abs().max()))
    assert abs(loss - ref_loss.item()) <= 1e-5 * ref_loss.item()
    for _ in range(11):
        nat.step()
    ref.iteration = 0                                                      # the same phases and refreshes as the native run
    for _ in range(12):                                                    # the manual evaluation above took no Adam step
        ref.step()
    for a, b in zip(params(nat), params(ref)):
        assert float((a - b).abs().max()) <= 2e-3 * float(b.abs().max()), (mode, case)


def test_native_refresh_matches_the_host_solver():
    from reart_b200.assign import AssignLoss
    kw, part, cano, frames = scene(4, 2048, 6, seed=5)
    nat = engine(kw, part, cano, frames, use_graph=False, native=True, assign=assign_cfg("add", downsample=4))
    for _ in range(6):                                                     # steps 0 and 5 refresh
        nat.step()
    host = AssignLoss(nat.cano, nat.frames, downsample=4, solver="scipy")
    host.refresh(nat.skinned)                                              # the cloud the step-5 solve saw
    assert torch.equal(nat.assign.col4row, host.col4row)


def run(kw, part, cano, frames, steps, **extra):
    eng = engine(kw, part, cano, frames, native=True, **extra)
    losses = [float(eng.step()) for _ in range(steps)]
    state = params(eng) + [eng.skinned.clone()]
    info = (eng.search_culled, eng.culling_stats())
    eng.release()
    return losses, state, info


def same_run(a, b):
    assert a[0] == b[0]
    for x, y in zip(a[1], b[1]):
        assert torch.equal(x, y)


@pytest.mark.parametrize("mode", ["add", "replace"])
def test_native_assign_fit_is_bit_reproducible_graph_and_eager(mode):
    kw, part, cano, frames = scene(16, 2048, 6, prismatic=True, root=True, seed=6)
    cfg = assign_cfg(mode, downsample=4, assign_iter=4, assign_gap=3)
    first = run(kw, part, cano, frames, 22, use_graph=False, search="brute", assign=cfg)
    same_run(run(kw, part, cano, frames, 22, use_graph=False, search="brute", assign=cfg), first)
    same_run(run(kw, part, cano, frames, 22, use_graph=True, search="brute", assign=cfg), first)


def test_culled_search_with_assignment_is_the_brute_force_bit_for_bit():
    kw, part, cano, frames = scene(4, 8192, 8, seed=8)
    cfg = assign_cfg("add", downsample=16, assign_iter=4, assign_gap=3)
    for graph in (True, False):
        brute = run(kw, part, cano, frames, 25, use_graph=graph, search="brute", assign=cfg)
        culled = run(kw, part, cano, frames, 25, use_graph=graph, assign=cfg)       # "auto" at 8192 points: culled
        assert not brute[2][0] and culled[2][0]
        same_run(culled, brute)


def test_native_replace_fit_recovers_joint_angles_on_a_synthetic_tree():
    """The scenario of test_kinematic_native_gpu.py::test_native_engine_recovers_joint_angles_on_a_synthetic_tree, fitted
    with the assignment loss alone (run_robot.py's "replace" flavour)."""
    import oracle
    from reart_b200.engine import KinematicEngine
    rng = np.random.default_rng(3)
    T, N, P = 5, 3000, 4
    E = P - 1
    axis = rng.standard_normal((E, 3)); axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    anchor = np.cumsum(np.full((E, 3), 0.08), axis=0) * np.array([1.0, 0.2, 0.1])
    moment = np.cross(anchor, axis)
    theta_gt = rng.uniform(-0.8, 0.8, (T, E)).astype(np.float32)
    order = np.arange(P, dtype=np.int32); parent = np.arange(-1, P - 1, dtype=np.int32); edge = np.arange(-1, P - 1, dtype=np.int32)
    part = rng.integers(0, P, N)
    cano = (rng.uniform(-0.04, 0.04, (N, 3)) + np.concatenate([[np.zeros(3)], anchor])[part] * 1.0).astype(np.float32)
    poses = oracle.fk(axis, moment, theta_gt, None, order, parent, edge)
    W = np.eye(P, dtype=np.float32)[part]
    frames = oracle.skin_fwd(cano, W, poses[:, :, :3, :3], poses[:, :, :3, 3])
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    kw = dict(edge_index={f"{c}_{c-1}": c - 1 for c in range(1, P)}, paths_to_base={c: list(range(c, -1, -1)) for c in range(P)},
              reverse_topo=list(range(P)), axis_list=cu(axis.astype(np.float32)), moment_list=cu(moment.astype(np.float32)),
              theta_list=cu(theta_gt + rng.normal(0, 0.15, theta_gt.shape).astype(np.float32)))
    # every point sampled: at the true angles the optimal matching is the exact correspondence (loss 0)
    cfg = dict(downsample=1, assign_gap=5, lambda_assign=1.0, assign_iter=0, mode="replace")
    for graph in (False, True):
        eng = KinematicEngine(clone(kw), torch.from_numpy(part), cu(cano), cu(frames), lr=1e-2, use_graph=graph, native=True,
                              assign=cfg)
        first = float(eng.step())
        for _ in range(150):
            last = float(eng.step())
        assert last < 0.2 * first, (graph, first, last)
        assert np.abs(eng.model.theta_list.detach().cpu().numpy() - theta_gt).mean() < 0.06
        eng.release()


def test_assignment_rejects_ingest_and_a_bad_mode():
    kw, part, cano, frames = scene(2, 512, 4)
    eng = engine(kw, part, cano, frames, native=True, use_graph=False, assign=assign_cfg("add"))
    with pytest.raises(ValueError):
        eng.step(ingest=(0, cano.clone(), frames.clone()))
    with pytest.raises(ValueError):
        engine(kw, part, cano, frames, native=True, assign=assign_cfg("both"))
    with pytest.raises(ValueError):
        engine(kw, part, cano, frames, assign=assign_cfg("add", downsample=1024))      # no samples left


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
    kw, part, cano, frames = scene(8, 4096, 6, prismatic=True)
    kw = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in kw.items()}
    cano, frames = cano.to(d), frames.to(d)
    cfg = assign_cfg("add", downsample=8, assign_iter=2, assign_gap=3)
    out = {}
    for graph in (False, True):
        eng = KinematicEngine(clone(kw), part, cano, frames, ctx=ctx, use_graph=graph, native=True, assign=cfg)
        out[f"kin_{int(graph)}"] = [float(eng.step()) for _ in range(10)]
        out[f"axis_{int(graph)}"] = eng.model.axis_list.detach().cpu().numpy().copy()
        out[f"moment_{int(graph)}"] = eng.model.moment_list.detach().cpu().numpy().copy()
        eng.release()
    first_cfg = assign_cfg("add", downsample=8, assign_iter=0)            # the first step already has the assignment
    if rank == 0:
        single = KinematicEngine(clone(kw), part, cano, frames, ctx=DistContext(), use_graph=False, native=True, assign=first_cfg)
        out["kin_single"] = [float(single.step())]
        single.release()
    first = KinematicEngine(clone(kw), part, cano, frames, ctx=ctx, use_graph=False, native=True, assign=first_cfg)
    out["kin_first"] = [float(first.step())]
    first.release()
    np.savez(os.path.join(out_dir, f"kinassign{rank}.npz"), **out)
    dist.barrier()
    os._exit(0)


@pytest.mark.timeout(300)
def test_sharded_native_kinematic_assignment_on_two_gpus(tmp_path):
    """Frame sharding: each rank samples and solves its own frames; the first step's loss is the single-GPU loss to 1e-6
    (only the association of the sums differs), graph == eager bit for bit, identical axis/moment on both ranks."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_two_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "kinassign0.npz"), np.load(tmp_path / "kinassign1.npz")
    assert list(r0["kin_0"]) == list(r0["kin_1"]) == list(r1["kin_0"]) == list(r1["kin_1"])
    for k in ("axis_0", "axis_1", "moment_0", "moment_1"):
        assert np.array_equal(r0[k], r1[k]), k
    assert np.array_equal(r0["axis_0"], r0["axis_1"]) and np.array_equal(r0["moment_0"], r0["moment_1"])
    assert abs(r0["kin_first"][0] - r0["kin_single"][0]) <= 1e-6 * r0["kin_single"][0]
