"""KinematicEngine(native=True): the kinematic fit on kin_head -> fused energy -> kin_tail.  The head's poses are the tree
FK's bit for bit, the tail's gradients are autograd's, a run is bit-reproducible (graph == eager, run == run), the culled
search is the brute force bit for bit, and the fit still recovers the joint angles."""
import numpy as np
import pytest
import torch

from conftest import synthetic_sequence

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda")


def _rot(axis, angle):
    axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * (K @ K)


def scene(T, N, P, seed=2, prismatic=False, root=False, theta_noise=0.1):
    """(model kwargs, part labels, cano, frames) of a synthetic articulated sequence; prismatic: every other joint slides
    (with a learned distance per frame); root: a learned root pose per frame."""
    from reart_b200.synth import kinematic_init
    seq = synthetic_sequence(T, N, P, seed=seed)
    kw = {k: (torch.from_numpy(v).to(dev()) if isinstance(v, np.ndarray) else v)
          for k, v in kinematic_init(seq, theta_noise=theta_noise).items()}
    rng = np.random.default_rng(seed + 5)
    E = P - 1
    if prismatic:
        kw["joint_type_list"] = ["prismatic" if e % 2 else "revolute" for e in range(E)]
        kw["distance_list"] = torch.from_numpy(rng.uniform(-0.05, 0.05, (T, E)).astype(np.float32)).to(dev())
    if root:
        rt = np.tile(np.eye(4, dtype=np.float32), (T, 1, 1))
        for t in range(T):
            rt[t, :3, :3] = _rot(rng.standard_normal(3), rng.uniform(-0.05, 0.05))
            rt[t, :3, 3] = rng.uniform(-0.02, 0.02, 3)
        kw["root_trans"] = torch.from_numpy(rt).to(dev())
    return kw, torch.from_numpy(seq["part"]), torch.from_numpy(seq["cano"]).to(dev()), torch.from_numpy(seq["frames"]).to(dev())


def clone(kw):
    return {k: (v.clone() if torch.is_tensor(v) else v) for k, v in kw.items()}


def engine(kw, part, cano, frames, **extra):
    from reart_b200.engine import KinematicEngine
    return KinematicEngine(clone(kw), part, cano, frames, lr=1e-2, **extra)


def params(eng):
    m = eng.model
    return [getattr(m, n).detach().clone() for n in ("axis_list", "moment_list", "theta_list", "distance_list", "root_6d",
                                                     "root_t") if hasattr(m, n)]


def run_head(model):
    from reart_b200 import _lib
    L, p = _lib.lib(), _lib.ptr
    T, P = model.theta_list.shape[0], model.num_parts
    tree = model.tree(dev())
    R, tr, fk = torch.empty(T, P, 3, 3, device=dev()), torch.empty(T, P, 3, device=dev()), torch.empty(T, P, 12, device=dev())
    root = hasattr(model, "root_6d")
    _lib.check(L.reart_kin_head(p(model.axis_list), p(model.moment_list), p(model.theta_list),
                                p(getattr(model, "distance_list", None)), p(tree.order), p(tree.parent), p(tree.edge),
                                p(tree.joint_type), p(model.root_6d.contiguous()) if root else None,
                                p(model.root_t.contiguous()) if root else None, T, P, p(R), p(tr), p(fk), _lib.stream_ptr()),
               "reart_kin_head")
    torch.cuda.synchronize()
    return R, tr


@pytest.mark.parametrize("prismatic", [False, True])
def test_head_is_the_tree_fk_bit_for_bit(prismatic):
    from reart_b200.engine import KinematicEngine
    kw, part, cano, frames = scene(6, 1024, 6, prismatic=prismatic)
    eng = KinematicEngine(clone(kw), part, cano, frames, use_graph=False)
    with torch.no_grad():
        want = eng.model.transforms()
    R, tr = run_head(eng.model)
    assert torch.equal(R, want[:, :, :3, :3]) and torch.equal(tr, want[:, :, :3, 3])


def test_head_with_a_root_pose_matches_the_model_transforms():
    from reart_b200.engine import KinematicEngine
    kw, part, cano, frames = scene(6, 1024, 6, prismatic=True, root=True)
    eng = KinematicEngine(clone(kw), part, cano, frames, use_graph=False)
    with torch.no_grad():
        want = eng.model.transforms()
    R, tr = run_head(eng.model)
    assert (R - want[:, :, :3, :3]).abs().max() <= 1e-6 and (tr - want[:, :, :3, 3]).abs().max() <= 1e-6


@pytest.mark.parametrize("case", ["revolute", "mixed", "root"])
def test_tail_gradients_and_a_short_fit_match_autograd(case):
    kw, part, cano, frames = scene(5, 2048, 6, prismatic=case != "revolute", root=case == "root", seed=4)
    ref = engine(kw, part, cano, frames, use_graph=False)
    # KinematicModel keeps root_t as a strided view of root_trans, whose gradient torch's fused Adam rejects; the reference
    # optimisation runs on a contiguous copy of the same values
    if hasattr(ref.model, "root_t"):
        ref.model.root_t.data = ref.model.root_t.data.contiguous()
    ref.optimizer.zero_grad(set_to_none=True)
    ref_loss = ref._iteration()
    ref_loss.backward()
    m = ref.model
    ref_grads = [q.grad.detach().clone() for q in ref._opt_params()]
    nat = engine(kw, part, cano, frames, use_graph=False, native=True)
    loss = float(nat.step())
    g = nat._nat["grad"]
    E = m.axis_list.shape[0]
    T = m.theta_list.shape[0]
    sizes = [3 * E, 3 * E, 1, T * E] + ([T * E] if hasattr(m, "distance_list") else []) + ([6 * T, 3 * T] if hasattr(m, "root_6d") else [])
    parts = list(torch.split(g, sizes))
    del parts[2]                                                           # the loss slot
    names = [n for n in ("axis_list", "moment_list", "theta_list", "distance_list", "root_6d", "root_t") if hasattr(m, n)]
    assert len(parts) == len(ref_grads) == len(names)
    for name, got, want in zip(names, parts, ref_grads):
        err = float((got - want.reshape(-1)).abs().max())
        assert err <= 1e-5 * float(want.abs().max()) + 1e-12, (case, name, err, float(want.abs().max()))
    if case != "root":
        assert loss == ref_loss.item()                                     # same R/tr, same energy kernel: equal as floats
    for _ in range(11):
        nat.step()
    for _ in range(12):                                                    # the manual evaluation above took no Adam step
        ref.step()
    for a, b in zip(params(nat), params(ref)):
        assert float((a - b).abs().max()) <= 2e-3 * float(b.abs().max()), case
    # the model's own parameters were updated in place: a forward pass sees the fitted values
    with torch.no_grad():
        _, _, trans = nat.model(nat.cano)
    R, tr = run_head(nat.model)
    assert torch.allclose(trans[:, :, :3, :3], R, atol=1e-6)


def run(kw, part, cano, frames, steps, ingest=None, **extra):
    eng = engine(kw, part, cano, frames, native=True, **extra)
    losses = []
    for i in range(steps):
        if ingest is None:
            losses.append(float(eng.step()))
        else:
            c, f = ingest[i & 1]
            losses.append(float(eng.step(ingest=(i & 1, c, f))))
    state = params(eng) + [eng.skinned.clone()]
    info = (eng.search_culled, eng.culling_stats(), eng.flagged_ties())
    eng.release()
    return losses, state, info


def same_run(a, b):
    assert a[0] == b[0]
    for x, y in zip(a[1], b[1]):
        assert torch.equal(x, y)


def test_native_fit_is_bit_reproducible_graph_and_eager():
    kw, part, cano, frames = scene(64, 2048, 6, prismatic=True, root=True, seed=6)
    first = run(kw, part, cano, frames, 20, use_graph=False, search="brute")
    same_run(run(kw, part, cano, frames, 20, use_graph=False, search="brute"), first)
    same_run(run(kw, part, cano, frames, 20, use_graph=True, search="brute"), first)


def test_culled_search_is_the_brute_force_bit_for_bit():
    kw, part, cano, frames = scene(4, 8192, 8, seed=8)
    for graph in (True, False):
        brute = run(kw, part, cano, frames, 25, use_graph=graph, search="brute")
        culled = run(kw, part, cano, frames, 25, use_graph=graph)                 # "auto" at 8192 points: culled
        assert not brute[2][0] and culled[2][0]
        ev, off = culled[2][1]
        assert 0 < ev < off
        same_run(culled, brute)
    seq2 = synthetic_sequence(4, 8192, 8, seed=9)
    stage = [(cano.clone(), frames.clone()),
             (torch.from_numpy(seq2["cano"]).to(dev()), torch.from_numpy(seq2["frames"]).to(dev()))]
    brute = run(kw, part, cano.clone(), frames.clone(), 12, ingest=stage, use_graph=True, search="brute")
    culled = run(kw, part, cano.clone(), frames.clone(), 12, ingest=stage, use_graph=True, search="culled")
    same_run(culled, brute)


def test_culled_search_needs_the_native_iteration():
    kw, part, cano, frames = scene(2, 512, 4)
    with pytest.raises(ValueError):
        engine(kw, part, cano, frames, search="culled")


def test_native_engine_recovers_joint_angles_on_a_synthetic_tree():
    """The scenario of test_gpu_parity.py::test_kinematic_engine_recovers_joint_angles_on_a_synthetic_tree, native."""
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
    for graph in (False, True):
        eng = KinematicEngine(clone(kw), torch.from_numpy(part), cu(cano), cu(frames), lr=1e-2, use_graph=graph, native=True)
        first = float(eng.step())
        for _ in range(150):
            last = float(eng.step())
        assert last < 0.2 * first, (graph, first, last)
        assert np.abs(eng.model.theta_list.detach().cpu().numpy() - theta_gt).mean() < 0.06
        eng.release()


def _two_gpu_worker(rank, world, port, out_dir):
    import os
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    from reart_b200.dist import DistContext
    from reart_b200.engine import KinematicEngine, RelaxationEngine, tau_schedule
    ctx = DistContext.from_env()
    d = torch.device("cuda", rank)
    torch.cuda.set_device(d)
    kw, part, cano, frames = scene(8, 4096, 6, prismatic=True)
    kw = {k: (v.to(d) if torch.is_tensor(v) else v) for k, v in kw.items()}
    cano, frames = cano.to(d), frames.to(d)
    out = {}
    for graph in (False, True):
        eng = KinematicEngine(clone(kw), part, cano, frames, ctx=ctx, use_graph=graph, native=True)
        out[f"kin_{int(graph)}"] = [float(eng.step()) for _ in range(10)]
        out[f"axis_{int(graph)}"] = eng.model.axis_list.detach().cpu().numpy().copy()
        out[f"moment_{int(graph)}"] = eng.model.moment_list.detach().cpu().numpy().copy()
        eng.release()
    if rank == 0:
        single = KinematicEngine(clone(kw), part, cano, frames, ctx=DistContext(), use_graph=False, native=True)
        out["kin_single"] = [float(single.step()) for _ in range(10)]
        single.release()
    seq = synthetic_sequence(8, 4096, 6, seed=2)
    rc, rf = torch.from_numpy(seq["cano"]).to(d), torch.from_numpy(seq["frames"]).to(d)
    for search in ("brute", "culled"):
        eng = RelaxationEngine(rc, rf, 6, ctx=ctx, use_graph=True, seed=2, search=search)
        torch.manual_seed(5); torch.cuda.manual_seed_all(5)
        out[f"relax_{search}"] = [float(eng.step(tau_schedule(i, 100, 5.0, 1.0))) for i in range(10)]
        out[f"relax_w2_{search}"] = eng.model.seg_head.model[2].weight.detach().cpu().numpy().copy()
        out[f"relax_t_{search}"] = eng.model.proposal_t.detach().cpu().numpy().copy()
        eng.release()
    np.savez(os.path.join(out_dir, f"kin{rank}.npz"), **out)
    dist.barrier()
    os._exit(0)


@pytest.mark.timeout(300)
def test_sharded_native_kinematic_and_culled_relaxation_on_two_gpus(tmp_path):
    """Frame sharding: the native kinematic step reproduces the single-GPU step (first step to 1e-6: only the association
    of the frame sums differs), graph == eager bit for bit with identical axis/moment on both ranks; the sharded
    RelaxationEngine's culled search is its brute force bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_two_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "kin0.npz"), np.load(tmp_path / "kin1.npz")
    assert list(r0["kin_0"]) == list(r0["kin_1"]) == list(r1["kin_0"]) == list(r1["kin_1"])
    for k in ("axis_0", "axis_1", "moment_0", "moment_1"):
        assert np.array_equal(r0[k], r1[k]), k
    assert np.array_equal(r0["axis_0"], r0["axis_1"]) and np.array_equal(r0["moment_0"], r0["moment_1"])
    assert abs(r0["kin_0"][0] - r0["kin_single"][0]) <= 1e-6 * r0["kin_single"][0]
    for r in (r0, r1):
        assert list(r["relax_brute"]) == list(r["relax_culled"])
        assert np.array_equal(r["relax_w2_brute"], r["relax_w2_culled"]) and np.array_equal(r["relax_t_brute"], r["relax_t_culled"])
