"""Engine checkpoints: ``checkpoint()`` / ``load_checkpoint()`` / ``fit_relaxation(resume=...)``.

The native iterations give the same bits from run to run, so a resume is checked exactly: k steps, a checkpoint through
``torch.save`` / ``torch.load(weights_only=True)``, a fresh engine built with ANOTHER seed (so the RNG must come from the
file), k more steps == 2k uninterrupted steps, every loss, every parameter and the skinned cloud ``torch.equal``."""
import io
import os

import numpy as np
import pytest
import torch

from conftest import synthetic_sequence
from test_kinematic_native_gpu import clone, scene
from test_relax_flow_gpu import flow_scene

pytestmark = pytest.mark.gpu

RTOL = 1e-5                                                  # test_gpu_parity's


def dev():
    return torch.device("cuda")


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def through_file(ck):
    buf = io.BytesIO()
    torch.save(ck, buf)
    buf.seek(0)
    return torch.load(buf, weights_only=True)


def assert_same(a, b, where="ck"):
    """Nested dicts / lists of tensors and plain values, tensor for tensor."""
    if isinstance(a, dict):
        assert isinstance(b, dict) and set(a) == set(b), (where, sorted(a), sorted(b))
        for k in a:
            assert_same(a[k], b[k], f"{where}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), where
        for i, (x, y) in enumerate(zip(a, b)):
            assert_same(x, y, f"{where}[{i}]")
    elif torch.is_tensor(a):
        assert torch.is_tensor(b) and a.dtype == b.dtype and torch.equal(a, b), where
    else:
        assert a == b, (where, a, b)


# ---------------------------------------------------------------------------------------------- engines of the flavours
def relax_scene(T=6, N=2048, P=8, seed=2):
    seq = synthetic_sequence(T, N, P, seed=seed)
    return cu(seq["cano"]), cu(seq["frames"])


def relax_maker(cano, frames, P, **kw):
    from reart_b200.engine import RelaxationEngine
    return lambda seed: RelaxationEngine(cano, frames, num_parts=P, seed=seed, weight_decay=1e-3, **kw)


def kin_maker(kw, part, cano, frames, **extra):
    from reart_b200.engine import KinematicEngine
    return lambda seed: KinematicEngine(clone(kw), part, cano, frames, lr=1e-2, **extra)


def state(eng):
    m = eng.model
    return [q.detach().clone() for _, q in sorted(m.named_parameters())] + [eng.skinned.clone()]


def stepper(n_total):
    from reart_b200.engine import RelaxationEngine, tau_schedule

    def step(eng, i):
        if isinstance(eng, RelaxationEngine):
            return float(eng.step(tau_schedule(i, n_total, 5.0, 1.0)))
        return float(eng.step())
    return step


def run(make, seed, steps, start=0, n_total=None, ck=None):
    step = stepper(n_total or steps)
    eng = make(seed)
    if ck is not None:
        eng.load_checkpoint(ck)
        assert eng.iteration == start
    losses = [step(eng, i) for i in range(start, steps)]
    return eng, losses


def check_resume(make, k):
    """2k uninterrupted steps == k steps, checkpoint, file, fresh engine with another seed, k steps."""
    full, la = run(make, 2, 2 * k)
    want = state(full)
    full.release()
    first, lb = run(make, 2, k, n_total=2 * k)
    ck = through_file(first.checkpoint())
    first.release()
    assert ck["engine"]["iteration"] == k
    second, lc = run(make, 11, 2 * k, start=k, ck=ck)
    got = state(second)
    second.release()
    assert lb + lc == la
    assert len(got) == len(want)
    for x, y in zip(got, want):
        assert torch.equal(x, y)
    return ck


# ---------------------------------------------------------------------------------------------- 1. exact resume, native
@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("flavour", ["brute", "culled_posed", "cull", "fuse_producer"])
def test_native_relaxation_resume_is_exact(flavour, graph):
    if flavour == "culled_posed":
        cano, frames = relax_scene(T=4, N=8192, P=8)
        extra = dict(search="culled")
    else:
        cano, frames = relax_scene()
        extra = dict(brute=dict(search="brute"), cull=dict(cull=True), fuse_producer=dict(fuse_producer=True))[flavour]
    make = relax_maker(cano, frames, 8, use_graph=graph, native=True, **extra)
    if flavour == "culled_posed":
        eng = make(2)
        assert eng.search_culled and eng.search_posed
        eng.release()
    check_resume(make, 5)


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("mode", ["add", "replace"])
def test_native_relaxation_assignment_resume_is_exact(mode, graph):
    """Refreshes at i = 2 (assign_iter) and every i % 3 == 0 after: k = 1 resumes before the assignment starts, k = 4
    between two refreshes (the matches and warm-start duals come from the file)."""
    cano, frames = relax_scene()
    cfg = dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=2, mode=mode)
    make = relax_maker(cano, frames, 8, use_graph=graph, native=True, search="brute", assign=cfg)
    for k in (1, 4):
        ck = check_resume(make, k)
        assert ck["engine"]["assign"]["have_assignment"] == (k > 2)


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("assign", [None, "add"])
def test_native_relaxation_flow_resume_is_exact(assign, graph):
    cano, frames, ref = flow_scene(6, 2048, 6, c=2)
    cfg = None if assign is None else dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=0, mode=assign)
    make = relax_maker(cano, frames, 6, use_graph=graph, native=True, flow_ref=ref, cano_idx=2, assign=cfg)
    check_resume(make, 4)


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("flavour", ["brute", "culled", "assign", "flow", "prismatic_root"])
def test_native_kinematic_resume_is_exact(flavour, graph):
    extra = dict(use_graph=graph, native=True)
    if flavour == "culled":
        kw, part, cano, frames = scene(4, 8192, 8, seed=8)
        extra["search"] = "culled"
    elif flavour == "flow":
        from test_kinematic_flow_gpu import flow_scene as kin_flow_scene
        kw, part, cano, frames, ref, _ = kin_flow_scene(6, 2048, 6, 2)
        extra.update(flow_ref=ref, cano_idx=2)
    else:
        kw, part, cano, frames = scene(6, 2048, 6, seed=4, prismatic=flavour == "prismatic_root", root=flavour == "prismatic_root")
        extra["search"] = "brute"
        if flavour == "assign":
            extra["assign"] = dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=2, mode="add")
    ck = check_resume(kin_maker(kw, part, cano, frames, **extra), 4)
    if flavour == "prismatic_root":
        assert {"distance_list", "root_6d", "root_t"} <= set(ck["state_dict"]) and ck["joint_type_list"][1] == "prismatic"


# ---------------------------------------------------------------------------------------------- 2. load after capture
def test_a_captured_engine_loads_another_engines_checkpoint_mid_run():
    """b captures its graphs on a fit of its own, then loads a's checkpoint of step 7: b's next steps are a's.  The RNG is
    the process's: a's continuation runs first, b's after the load (which restores the generator of step 7)."""
    from reart_b200.engine import tau_schedule
    cano, frames = relax_scene()
    cfg = dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=0, mode="add")
    make = relax_maker(cano, frames, 8, use_graph=True, native=True, search="brute", assign=cfg)
    kw, part, kc, kf = scene(6, 2048, 6, seed=4)
    kmake = kin_maker(kw, part, kc, kf, use_graph=True, native=True)
    for mk, seeds, tau in ((make, (2, 5), lambda i: tau_schedule(i, 20, 5.0, 1.0)), (kmake, (0, 0), lambda i: None)):
        a, b = mk(seeds[0]), mk(seeds[1])
        for i in range(4):                                    # b's graphs exist, its state is another fit's
            b.step(tau(i))
        graphs = dict(b._graphs)
        for i in range(7):
            a.step(tau(i))
        ck = a.checkpoint()
        want = [float(a.step(tau(i))) for i in range(7, 13)]
        b.load_checkpoint(ck)
        got = [float(b.step(tau(i))) for i in range(7, 13)]
        assert got == want
        assert all(b._graphs[key] is g for key, g in graphs.items())   # the graphs captured before the load ran
        for x, y in zip(state(a), state(b)):
            assert torch.equal(x, y)
        a.release(); b.release()


# ---------------------------------------------------------------------------------------------- 3. autograd paths
def close_runs(la, lb, sa, sb):
    """The tolerance of the native-vs-autograd tests (test_gpu_parity / test_relax_flow_gpu)."""
    np.testing.assert_allclose(la, lb, rtol=2e-3)
    for x, y in zip(sa, sb):
        assert float((x - y).abs().max()) <= 2e-3 * float(y.abs().max())


@pytest.mark.parametrize("graph", [True, False])
@pytest.mark.parametrize("model", ["relaxation_flow", "kinematic"])
def test_autograd_resume_follows_the_uninterrupted_run(model, graph):
    if model == "relaxation_flow":
        cano, frames, ref = flow_scene(6, 2048, 6, c=2)
        make = relax_maker(cano, frames, 6, use_graph=graph, flow_ref=ref, cano_idx=2)
    else:
        kw, part, cano, frames = scene(6, 2048, 6, seed=4, prismatic=True)
        make = kin_maker(kw, part, cano, frames, use_graph=graph)
    k = 5
    full, la = run(make, 2, 2 * k)
    assert not full.native
    want = state(full)
    full.release()
    first, lb = run(make, 2, k, n_total=2 * k)
    ck = through_file(first.checkpoint())
    first.release()
    assert ck["engine"]["adam"]["step"] == k
    eng = make(11)
    eng.load_checkpoint(ck)                                   # before the first step: torch's Adam state does not exist yet
    assert_same(eng.checkpoint()["engine"]["adam"], ck["engine"]["adam"])
    step = stepper(2 * k)
    lc = [step(eng, k)]
    # the first step (with graph: warm-up + capture + replay) continued the loaded state: a capture that took it for
    # torch's lazily created state would have zeroed it, and the step count would restart at 1
    assert eng.checkpoint()["engine"]["adam"]["step"] == k + 1
    lc += [step(eng, i) for i in range(k + 1, 2 * k)]
    close_runs(lb + lc, la, state(eng), want)
    eng.release()


# ---------------------------------------------------------------------------------------------- 4. cross-path
@pytest.mark.parametrize("model", ["relaxation", "kinematic"])
def test_a_native_checkpoint_loads_into_the_autograd_engine_unchanged(model):
    if model == "relaxation":
        cano, frames = relax_scene()
        nat = relax_maker(cano, frames, 8, use_graph=False, native=True)(2)
        auto = relax_maker(cano, frames, 8, use_graph=True, native=False)(7)
        step = stepper(10)
    else:
        kw, part, cano, frames = scene(6, 2048, 6, seed=4, prismatic=True)
        nat = kin_maker(kw, part, cano, frames, use_graph=False, native=True)(0)
        auto = kin_maker(kw, part, cano, frames, use_graph=True)(0)
        step = stepper(10)
    for i in range(4):
        step(nat, i)
    ck = through_file(nat.checkpoint())
    auto.load_checkpoint(ck)
    assert_same(through_file(auto.checkpoint()), ck)
    step(auto, 4)                                             # and it steps from there
    nat.release(); auto.release()


# ---------------------------------------------------------------------------------------------- 5. reference layout
def test_state_dict_loads_strictly_into_the_reference_models():
    from reart_b200.knn_module import KNN
    from reart_b200.model import BaseModel, KinematicModel
    cano, frames = relax_scene(T=7)
    eng = relax_maker(cano, frames, 8, use_graph=False, native=True)(2)
    for i in range(3):
        stepper(10)(eng, i)
    ck = through_file(eng.checkpoint())
    BaseModel(num_parts=8, pose_len=7).load_state_dict(ck["state_dict"], strict=True)
    assert ck["state_dict"]["proposal_6d"].shape == (7, 8, 6) and ck["cano_idx"] == 0 and ck["tau"] == float(eng.tau)
    eng.release()
    kw, part, kc, kf = scene(7, 2048, 6, seed=4, prismatic=True, root=True)
    eng = kin_maker(kw, part, kc, kf, use_graph=False, native=True)(0)
    eng.step()
    ck = through_file(eng.checkpoint())
    km = KinematicModel(pose_len=7, seg_part=ck["seg_part"], cano_pc=ck["cano_pc"], knn=KNN(k=1, transpose_mode=True),
                        edge_index=ck["edge_index"], paths_to_base=ck["paths_to_base"], reverse_topo=ck["reverse_topo"],
                        joint_type_list=ck["joint_type_list"], load_distance=True, load_root_trans=True)
    km.load_state_dict(ck["state_dict"], strict=True)
    eng.release()


def test_a_model_built_from_the_file_skins_like_the_resumed_engine():
    """oracle/make_golden.py's construction of KinematicModel from a checkpoint, on the canonical cloud, against the first
    step of an engine resumed from the same file."""
    from reart_b200.knn_module import KNN
    from reart_b200.model import KinematicModel
    kw, part, cano, frames = scene(6, 2048, 6, seed=4)
    make = kin_maker(kw, part, cano, frames, use_graph=False, native=True)
    eng = make(0)
    for _ in range(5):
        eng.step()
    ck = through_file(eng.checkpoint())
    eng.release()
    km = KinematicModel(pose_len=6, seg_part=ck["seg_part"], cano_pc=ck["cano_pc"], knn=KNN(k=1, transpose_mode=True),
                        edge_index=ck["edge_index"], paths_to_base=ck["paths_to_base"], reverse_topo=ck["reverse_topo"])
    km.load_state_dict(ck["state_dict"], strict=True)
    km.to(dev())
    with torch.no_grad():
        pc_trans, _, _ = km(km.cano_pc)
    eng = make(0)
    eng.load_checkpoint(ck)
    eng.step()
    assert torch.allclose(pc_trans, eng.skinned, rtol=RTOL, atol=2e-6)
    eng.release()


@pytest.mark.parametrize("native", [False, True])
def test_shipped_layout_nao_weights_give_the_reference_loss(nao, native):
    """A reference-layout dict (no "engine" section) of nao.npz's katC_* weights: the first loss is katC_loss, the optimiser
    starts afresh at iteration 0."""
    from reart_b200.engine import KinematicEngine
    g, cano, pc_list = nao
    order, parent, edge = g["katC_order"], g["katC_parent"], g["katC_edge"]
    edge_index = {f"{c}_{parent[c]}": int(edge[c]) for c in range(len(order)) if parent[c] >= 0}
    paths = {}
    for c in range(len(order)):
        path, x = [c], c
        while parent[x] >= 0:
            x = int(parent[x]); path.append(x)
        paths[c] = path
    seg_part = torch.from_numpy(g["katC_seg_part"].astype(np.int64))
    ck = dict(state_dict={"axis_list": torch.from_numpy(g["katC_axis"]), "moment_list": torch.from_numpy(g["katC_moment"]),
                          "theta_list": torch.from_numpy(g["katC_theta"])},
              seg_part=seg_part, cano_pc=torch.from_numpy(cano), edge_index=edge_index, paths_to_base=paths,
              reverse_topo=[int(o) for o in order])
    ck = through_file(ck)
    kw = dict(edge_index=edge_index, paths_to_base=paths, reverse_topo=[int(o) for o in order])
    eng = KinematicEngine(kw, seg_part, cu(cano), cu(pc_list), use_graph=False, native=native)
    eng.load_checkpoint(ck)
    assert eng.iteration == 0
    loss = float(eng.step())
    assert abs(loss - float(g["katC_loss"])) <= RTOL * float(g["katC_loss"])      # 4.810586452
    adam = eng.checkpoint()["engine"]["adam"]
    assert adam["step"] == 1
    eng.release()


# ---------------------------------------------------------------------------------------------- 6. fit_relaxation
def test_fit_relaxation_resumes_from_iteration_20_of_40():
    from reart_b200.engine import RelaxationEngine, fit_relaxation
    cano, frames = relax_scene()
    full, lf = fit_relaxation(cano, frames, 8, 40, seed=2)
    want = state(full)
    full.release()
    first, _ = run(lambda seed: RelaxationEngine(cano, frames, 8, seed=seed), 2, 20, n_total=40)
    ck = through_file(first.checkpoint())
    first.release()
    eng, lr = fit_relaxation(cano, frames, 8, 40, seed=9, resume=ck)
    assert eng.iteration == 40 and lr[-1] == lf[-1]
    for x, y in zip(state(eng), want):
        assert torch.equal(x, y)
    eng.release()


# ---------------------------------------------------------------------------------------------- 7. refusals
def test_mismatched_checkpoints_are_refused():
    import copy
    cano, frames = relax_scene()
    make = relax_maker(cano, frames, 8, use_graph=False, native=True, search="brute")
    eng = make(2)
    eng.step(1.0)
    ck = eng.checkpoint()
    for field, value in (("kind", "kinematic"), ("N", 1), ("M", 1), ("P", 3), ("H", 64), ("T_total", 5)):
        bad = copy.deepcopy(ck)
        bad["engine"][field] = value
        with pytest.raises(ValueError, match=field):
            eng.load_checkpoint(bad)
    # a real engine of another size, another part count, another frame count
    for other in (relax_maker(cano[:1024], frames, 8, use_graph=False, native=True),
                  relax_maker(cano, frames[:, :1024], 8, use_graph=False, native=True),
                  relax_maker(cano, frames, 6, use_graph=False, native=True),
                  relax_maker(cano, frames[:5], 8, use_graph=False, native=True)):
        with pytest.raises(ValueError):
            other(2).load_checkpoint(ck)
    # assignment state present without an assignment loss, and the other way round; another sample count
    cfg = dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=0, mode="add")
    with_assign = relax_maker(cano, frames, 8, use_graph=False, native=True, assign=cfg)(2)
    with pytest.raises(ValueError, match="assign"):
        with_assign.load_checkpoint(ck)
    with_assign.step(1.0)
    ck_a = with_assign.checkpoint()
    with pytest.raises(ValueError, match="assign"):
        eng.load_checkpoint(ck_a)
    with pytest.raises(ValueError, match="num_fps"):
        relax_maker(cano, frames, 8, use_graph=False, native=True, assign=dict(cfg, downsample=4))(2).load_checkpoint(ck_a)
    # the kinematic parameter set: distance / root pose present or not
    kw, part, kc, kf = scene(6, 2048, 6, seed=4)
    kwp, _, _, _ = scene(6, 2048, 6, seed=4, prismatic=True, root=True)
    plain = kin_maker(kw, part, kc, kf, use_graph=False, native=True)(0)
    full = kin_maker(kwp, part, kc, kf, use_graph=False, native=True)(0)
    with pytest.raises(ValueError, match="parameter set"):
        plain.load_checkpoint(full.checkpoint())
    with pytest.raises(ValueError, match="parameter set"):
        full.load_checkpoint(plain.checkpoint())
    with pytest.raises(ValueError, match="kind"):
        plain.load_checkpoint(ck)
    # nothing was changed by a refused load: the engine still resumes its own checkpoint exactly
    eng.load_checkpoint(ck)
    assert eng.iteration == 1


# ---------------------------------------------------------------------------------------------- 8. two GPUs
def _two_gpu_worker(rank, world, port, out_dir):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    from reart_b200.dist import DistContext
    ctx = DistContext.from_env()
    d = torch.device("cuda", rank)
    torch.cuda.set_device(d)
    seq = synthetic_sequence(7, 2048, 8, seed=2)                          # 7 frames: shards of 4 and 3
    cano, frames = torch.from_numpy(seq["cano"]).to(d), torch.from_numpy(seq["frames"]).to(d)
    cfg = dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=0, mode="add")
    make = relax_maker(cano, frames, 8, ctx=ctx, use_graph=True, native=True, assign=cfg)
    k = 4
    full, la = run(make, 2, 2 * k)
    want = state(full)
    full.release()
    first, lb = run(make, 2, k, n_total=2 * k)
    ck = through_file(first.checkpoint())
    first.release()
    second, lc = run(make, 11, 2 * k, start=k, ck=ck)
    ok = lb + lc == la and all(torch.equal(x, y) for x, y in zip(state(second), want))
    second.release()
    if rank == 0:
        torch.save(ck, os.path.join(out_dir, "ck2.pt"))
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), ok=ok, la=np.array(la))
    dist.barrier()
    os._exit(0)


@pytest.mark.timeout(600)
def test_sharded_checkpoint_resumes_exactly_and_loads_on_one_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    from reart_b200.dist import DistContext
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_two_gpu_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        assert bool(np.load(tmp_path / f"r{r}.npz")["ok"]), f"rank {r}: the sharded resume differs"
    ck2 = torch.load(tmp_path / "ck2.pt", weights_only=True)
    seq = synthetic_sequence(7, 2048, 8, seed=2)
    cfg = dict(downsample=8, assign_gap=3, lambda_assign=0.3, assign_iter=0, mode="add")
    one = relax_maker(cu(seq["cano"]), cu(seq["frames"]), 8, ctx=DistContext(), use_graph=True, native=True, assign=cfg)(5)
    one.load_checkpoint(ck2)
    assert_same(through_file(one.checkpoint()), ck2)
    stepper(8)(one, 4)
    one.release()
