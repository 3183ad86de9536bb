"""Generate tests/golden/*.npz by running the UNMODIFIED reference Python in this container.

    python -m oracle.make_golden

TEST INFRASTRUCTURE ONLY.  Needs /root/reference (read-only, container only).  The vectors
are committed so that the GPU box (which has no reference tree) can check the CUDA path and
the C oracle against what the reference itself computes.  Third-party stand-ins used for
``chamferdist._C`` / ``knn_cuda`` are described in oracle/ref_harness.py.
"""
from __future__ import annotations

import math
import os
import pickle

import numpy as np
import torch

from . import ref_harness as rh

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
REF = rh.REFERENCE_ROOT


def flatten_tree(edge_index, paths_to_base, reverse_topo):
    """dict-based tree of utils/kinematic_utils.py:151-198 -> (order, parent, edge) int32 arrays."""
    P = len(reverse_topo)
    order = np.array([int(p) for p in reverse_topo], np.int32)
    parent = -np.ones(P, np.int32)
    edge = -np.ones(P, np.int32)
    for part, path in paths_to_base.items():
        part = int(part)
        if len(path) > 1:
            par = int(path[1])
            parent[part] = par
            edge[part] = int(edge_index[f"{part}_{par}"])
    return order, parent, edge


def gen_nao(ref):
    torch.manual_seed(0)
    pcs64, parts = rh.load_nao()
    res = pickle.load(open(f"{REF}/demo_data/pretrained/nao/base-2/result_14999.pkl", "rb"))
    complete = torch.from_numpy(res["complete_pc_list"]).float()          # [10,4096,3]
    assert np.array_equal(complete.numpy(), pcs64.astype(np.float32))
    cano_idx = int(res["cano_idx"])
    cano = torch.from_numpy(res["cano_pc"]).float()
    pc_list = torch.from_numpy(res["pc_list"]).float()
    assert torch.equal(cano, complete[cano_idx])
    assert torch.equal(pc_list, torch.cat([complete[:cano_idx], complete[cano_idx + 1:]]))
    cd = ref.chamfer.ChamferDistance()
    out = {"complete_pc_list": complete.numpy(), "cano_idx": np.int64(cano_idx),
           "gt_part": parts.astype(np.int16)}

    # KAT-A: hard-label skin of the base-2 relaxation result + Chamfer both ways
    pose = torch.from_numpy(res["pred_pose_list"]).float()
    part = torch.from_numpy(res["pred_cano_part"]).long()
    skinned = ref.model_utils.compute_pc_transform(cano, pose, part)
    d_f, i_f = cd(skinned, pc_list, return_index=True)
    d_b, i_b = cd(skinned, pc_list, reverse=True, return_index=True)
    out.update(katA_pose=pose.numpy(), katA_part=part.numpy().astype(np.int16), katA_skinned_s16=skinned.numpy()[:, ::16],
               katA_sum_fwd=np.float64(d_f.double().sum().item()), katA_sum_bwd=np.float64(d_b.double().sum().item()),
               katA_idx_fwd=i_f.numpy().astype(np.int16), katA_idx_bwd=i_b.numpy().astype(np.int16),
               katA_d_fwd=d_f.numpy())      # d_b is not stored: no test reads it, and it would take nao.npz past 1 MB

    # KAT-B: raw frames 0 <-> 1, bidirectional
    tot, i01, i10 = cd(complete[0:1], complete[1:2], bidirectional=True, return_index=True)
    out.update(katB_sum=np.float64(tot.double().sum().item()), katB_idx_fwd=i01.numpy().astype(np.int16),
               katB_idx_bwd=i10.numpy().astype(np.int16), katB_total=tot.numpy())

    # KAT-C: kinematic-2 checkpoint -> KinematicModel.forward -> recon_loss (+ grads)
    ck = torch.load(f"{REF}/demo_data/pretrained/nao/kinematic-2/model.pth.tar", map_location="cpu",
                    weights_only=False)
    km = ref.model.KinematicModel(pose_len=pc_list.shape[0], seg_part=ck["seg_part"], cano_pc=ck["cano_pc"],
                                  knn=ref.KNN(k=1, transpose_mode=True), edge_index=ck["edge_index"],
                                  paths_to_base=ck["paths_to_base"], reverse_topo=ck["reverse_topo"])
    km.load_state_dict(ck["state_dict"], strict=True)
    assert torch.equal(ck["cano_pc"].float().cpu(), cano)
    pc_trans, seg_part, trans_list = km(cano)
    loss = ref.loss.recon_loss(pc_trans, pc_list, cd)
    loss.backward()
    order, parent, edge = flatten_tree(ck["edge_index"], ck["paths_to_base"], ck["reverse_topo"])
    out.update(katC_axis=km.axis_list.detach().numpy(), katC_moment=km.moment_list.detach().numpy(),
               katC_theta=km.theta_list.detach().numpy(), katC_seg_part=ck["seg_part"].cpu().numpy().astype(np.int16),
               katC_order=order, katC_parent=parent, katC_edge=edge,
               katC_trans_list=trans_list.detach().numpy(), katC_pc_trans_s16=pc_trans.detach().numpy()[:, ::16],
               katC_loss=np.float64(loss.item()), katC_g_axis=km.axis_list.grad.numpy(),
               katC_g_moment=km.moment_list.grad.numpy(), katC_g_theta=km.theta_list.grad.numpy(),
               katC_seg_out=seg_part.numpy().astype(np.int16))

    # KAT-D: base-2 checkpoint -> BaseModel.forward (gumbel weights captured) -> recon_loss (+ grads)
    cb = torch.load(f"{REF}/demo_data/pretrained/nao/base-2/model.pth.tar", map_location="cpu", weights_only=False)
    bm = ref.model.BaseModel(num_parts=20, pose_len=pc_list.shape[0])
    bm.load_state_dict(cb["state_dict"], strict=False)
    captured = {}
    import torch.nn.functional as F
    orig = F.gumbel_softmax

    def capture(logits, tau=1.0, hard=False, **kw):
        w = orig(logits, tau=tau, hard=hard, **kw)
        captured["w"] = w
        captured["logits"] = logits
        return w

    F.gumbel_softmax = capture
    try:
        torch.manual_seed(2)
        pc_trans, seg_arg, trans_list = bm(cano, tau=1.0)
    finally:
        F.gumbel_softmax = orig
    W = captured["w"]
    W.retain_grad()
    loss = ref.loss.recon_loss(pc_trans, pc_list, cd)
    loss.backward()
    Wd = W.detach()
    hot = Wd.argmax(dim=1)
    assert int((Wd != 0).sum()) == Wd.shape[0]
    out.update(katD_6d=bm.proposal_6d.detach().numpy(), katD_t=bm.proposal_t.detach().numpy(),
               katD_w0=bm.seg_head.model[0].weight.detach().numpy(), katD_b0=bm.seg_head.model[0].bias.detach().numpy(),
               katD_w2=bm.seg_head.model[2].weight.detach().numpy(),
               katD_hot=hot.numpy().astype(np.int8), katD_hotval=Wd.gather(1, hot[:, None])[:, 0].numpy(),
               katD_logits_s16=captured["logits"].detach().numpy()[::16], katD_seg_argmax=seg_arg.numpy().astype(np.int8),
               katD_pc_trans_s16=pc_trans.detach().numpy()[:, ::16], katD_trans_list=trans_list.detach().numpy(),
               katD_loss=np.float64(loss.item()), katD_g_6d=bm.proposal_6d.grad.numpy(),
               katD_g_t=bm.proposal_t.grad.numpy(), katD_g_W_s8=W.grad.numpy()[::8])
    np.savez_compressed(os.path.join(OUT, "nao.npz"), **out)
    print("nao.npz  katA", out["katA_sum_fwd"], out["katA_sum_bwd"], "katB", out["katB_sum"],
          "katC", out["katC_loss"], "katD", out["katD_loss"])


def gen_se3(ref):
    g = torch.Generator().manual_seed(7)
    B = 64
    l = torch.randn(B, 3, generator=g)
    l = l / l.norm(dim=1, keepdim=True) * (0.5 + torch.rand(B, 1, generator=g))    # un-normalised axes (Q17)
    m = torch.randn(B, 3, generator=g) * 0.3
    theta = (torch.rand(B, generator=g) * 2 - 1) * 2.5
    d = (torch.rand(B, generator=g) * 2 - 1) * 0.2
    # edge cases (SURVEY Q8-Q10)
    theta[0] = 1e-6; d[0] = 0.13            # exactly eps: with-rot branch, prismatic-like
    theta[1] = 5e-7; d[1] = 0.2             # no-rot branch ignores d
    theta[2] = math.pi                      # |theta-pi|<eps -> no-rot
    theta[3] = 0.005                        # clamp theta^2*|l|^2 at 1e-4
    theta[4] = -0.004
    theta[5] = 0.0
    theta[6] = 1e-6; d[6] = 1e-6
    l.requires_grad_(True); m.requires_grad_(True); theta.requires_grad_(True); d.requires_grad_(True)
    expc = ref.screw_se3.screw_param_to_exponential_coordinates(l, m, theta, d)
    M = ref.screw_se3.transform_from_exponential_coordinates(expc)
    coef = torch.randn(B, 4, 4, generator=g)
    (M * coef).sum().backward()
    d6 = torch.randn(50, 6, generator=g)
    d6[0] = torch.tensor([1., 0, 0, 0, 1, 0])
    d6.requires_grad_(True)
    R = ref.screw_se3.rotation_6d_to_matrix(d6)
    coefR = torch.randn(50, 3, 3, generator=g)
    (R * coefR).sum().backward()
    np.savez_compressed(os.path.join(OUT, "se3.npz"), l=l.detach().numpy(), m=m.detach().numpy(),
                        theta=theta.detach().numpy(), d=d.detach().numpy(), expc=expc.detach().numpy(),
                        M=M.detach().numpy(), coef=coef.numpy(), g_l=l.grad.numpy(), g_m=m.grad.numpy(),
                        g_theta=theta.grad.numpy(), g_d=d.grad.numpy(), d6=d6.detach().numpy(),
                        R=R.detach().numpy(), coefR=coefR.numpy(), g_d6=d6.grad.numpy())
    print("se3.npz", M.shape, R.shape)


def gen_fk(ref):
    """fk on a synthetic mixed revolute/prismatic tree (sapien-shaped, cfg4) with root pose."""
    g = torch.Generator().manual_seed(11)
    T, P = 6, 8
    E = P - 1
    # random tree: parent of part c (c>=1 in a shuffled labelling) is an earlier part
    perm = torch.randperm(P, generator=g).tolist()
    root = perm[0]
    par = {perm[0]: None}
    edge_index, k = {}, 0
    import networkx as nx
    G = nx.DiGraph()
    G.add_node(root)
    for i in range(1, P):
        c = perm[i]
        p = perm[int(torch.randint(0, i, (1,), generator=g))]
        par[c] = p
        edge_index[f"{c}_{p}"] = k
        k += 1
        G.add_edge(c, p)
    paths_to_base = nx.shortest_path(G, target=root)
    reverse_topo = list(reversed(list(nx.topological_sort(G))))
    axis = torch.randn(E, 3, generator=g); axis = axis / axis.norm(dim=1, keepdim=True) * (0.6 + 0.6 * torch.rand(E, 1, generator=g))
    moment = torch.randn(E, 3, generator=g) * 0.2
    theta = (torch.rand(T, E, generator=g) * 2 - 1)
    dist = (torch.rand(T, E, generator=g) * 2 - 1) * 0.1
    jt = ["prismatic" if i % 3 == 1 else "revolute" for i in range(E)]
    outs = {}
    for tag, (dl, jtl) in {"plain": (None, None), "dist": (dist, None), "typed": (dist, jt)}.items():
        a, mo, th = axis.clone().requires_grad_(True), moment.clone().requires_grad_(True), theta.clone().requires_grad_(True)
        di = dl.clone().requires_grad_(True) if dl is not None else None
        out = ref.kinematic_utils.fk(paths_to_base, reverse_topo, edge_index, a, mo, th, distance_list=di,
                                     joint_type_list=jtl)
        coef = torch.randn(T, P, 4, 4, generator=g)
        (out * coef).sum().backward()
        outs.update({f"{tag}_out": out.detach().numpy(), f"{tag}_coef": coef.numpy(), f"{tag}_g_axis": a.grad.numpy(),
                     f"{tag}_g_moment": mo.grad.numpy(), f"{tag}_g_theta": th.grad.numpy()})
        if di is not None and di.grad is not None:
            outs[f"{tag}_g_dist"] = di.grad.numpy()
    order, parent, edge = flatten_tree(edge_index, paths_to_base, reverse_topo)
    np.savez_compressed(os.path.join(OUT, "fk.npz"), axis=axis.numpy(), moment=moment.numpy(), theta=theta.numpy(),
                        dist=dist.numpy(), joint_type=np.array([2 if j == "prismatic" else 1 for j in jt], np.int32),
                        order=order, parent=parent, edge=edge, **outs)
    print("fk.npz", order, parent, edge)


def gen_chamfer_small(ref):
    g = torch.Generator().manual_seed(3)
    cd = ref.chamfer.ChamferDistance()
    out = {}
    for tag, (B, N, M) in {"a": (3, 257, 300), "b": (5, 20, 20), "c": (1, 1, 7), "d": (2, 1000, 33)}.items():
        src = torch.randn(B, N, 3, generator=g).requires_grad_(True)
        tgt = torch.randn(B, M, 3, generator=g).requires_grad_(True)
        d_f, i_f = cd(src, tgt, return_index=True)
        d_b, i_b = cd(src, tgt, reverse=True, return_index=True)
        wf = torch.rand(B, N, generator=g); wb = torch.rand(B, M, generator=g)
        ((d_f * wf).sum() + (d_b * wb).sum()).backward()
        out.update({f"{tag}_src": src.detach().numpy(), f"{tag}_tgt": tgt.detach().numpy(), f"{tag}_d_fwd": d_f.detach().numpy(),
                    f"{tag}_i_fwd": i_f.numpy(), f"{tag}_d_bwd": d_b.detach().numpy(), f"{tag}_i_bwd": i_b.numpy(),
                    f"{tag}_wf": wf.numpy(), f"{tag}_wb": wb.numpy(), f"{tag}_g_src": src.grad.numpy(),
                    f"{tag}_g_tgt": tgt.grad.numpy()})
    # exact ties: integer lattice points => many equal distances, lowest index must win
    src = torch.randint(-2, 3, (2, 64, 3), generator=g).float()
    tgt = torch.randint(-2, 3, (2, 96, 3), generator=g).float()
    d_f, i_f = cd(src, tgt, return_index=True)
    out.update(tie_src=src.numpy(), tie_tgt=tgt.numpy(), tie_d_fwd=d_f.numpy(), tie_i_fwd=i_f.numpy())
    np.savez_compressed(os.path.join(OUT, "chamfer_small.npz"), **out)
    print("chamfer_small.npz")


def gen_flow(ref):
    g = torch.Generator().manual_seed(5)
    m, n, T = 500, 180, 3
    knn = ref.KNN(k=3, transpose_mode=True)
    out = {}
    blended, masks, queries, refs, flows = [], [], [], [], []
    for t in range(T):
        q = torch.rand(m, 3, generator=g) * 0.6 - 0.3
        r = q[torch.randperm(m, generator=g)[:n]] + 0.01 * torch.randn(n, 3, generator=g)
        if t == 0:
            r[:5] = q[:5]                      # zero distances -> 1e-10 clamp (flow_utils.py:160)
        f = 0.05 * torch.randn(n, 3, generator=g)
        if t == 1:
            f = f * 0.001                      # tiny flows: mask decided by the 0.05 threshold
        b, mk = ref.flow_utils.blend_anchor_motion(q, r, f, knn, return_mask=True)
        blended.append(b); masks.append(mk); queries.append(q); refs.append(r); flows.append(f)
    gt = torch.stack(blended); mask = torch.stack(masks)
    pred = (gt + 0.02 * torch.randn(gt.shape, generator=g)).requires_grad_(True)
    l_mse = ref.loss.flow_loss(gt, pred, flow_mask_list=mask, robust=False)
    g_mse, = torch.autograd.grad(l_mse, pred)
    l_hub = ref.loss.flow_loss(gt, pred, flow_mask_list=mask, robust=True)
    g_hub, = torch.autograd.grad(l_hub, pred)
    l_nomask = ref.loss.flow_loss(gt, pred)
    np.savez_compressed(os.path.join(OUT, "flow.npz"), query=torch.stack(queries).numpy(), ref=torch.stack(refs).numpy(),
                        flow=torch.stack(flows).numpy(), blended=gt.numpy(), mask=mask.numpy(),
                        pred=pred.detach().numpy(), l_mse=np.float64(l_mse.item()), g_mse=g_mse.numpy(),
                        l_hub=np.float64(l_hub.item()), g_hub=g_hub.numpy(), l_nomask=np.float64(l_nomask.item()))
    print("flow.npz", mask.float().mean().item())


def _fps_from_zero(xyz, npoint):
    """CUDA semantics of furthest point sampling (sampling_gpu.cu:113-115 starts at index 0; the reference's CPU
    fallback starts at a random index, SURVEY Q13).  Used as the FPS stand-in for the structure goldens."""
    B, N, _ = xyz.shape
    out = torch.zeros(B, npoint, dtype=torch.long)
    for b in range(B):
        dist = torch.full((N,), 1e10)
        far = 0
        for i in range(npoint):
            out[b, i] = far
            d = ((xyz[b] - xyz[b, far]) ** 2).sum(-1)
            dist = torch.minimum(dist, d)
            far = int(torch.argmax(dist))
    return out


def _random_screw_sequence(T, P, gen, prismatic=(), static=()):
    """[T,P,4,4] rigid transforms: part p moves about its own fixed screw axis (revolute unless listed)."""
    import importlib
    se3 = importlib.import_module("screw_se3")
    out = torch.eye(4).repeat(T, P, 1, 1)
    for p in range(P):
        if p in static:
            continue
        l = torch.nn.functional.normalize(torch.randn(1, 3, generator=gen), dim=-1)
        pt = 0.3 * torch.randn(1, 3, generator=gen)
        m = torch.cross(pt, l, dim=-1)
        for t in range(T):
            if p in prismatic:
                th, d = torch.tensor([1e-6]), 0.05 + 0.3 * torch.rand(1, generator=gen)
            else:
                th, d = 0.2 + 1.2 * torch.rand(1, generator=gen), torch.tensor([1e-6])
            out[t, p] = se3.transform_from_exponential_coordinates(
                se3.screw_param_to_exponential_coordinates(l, m, th, d))[0]
    return out


def gen_structure(ref):
    """Structure-extraction stage (SURVEY 8f rank 4): utils/graph_utils.py:62-421, utils/kinematic_utils.py:20-148,
    screw_se3/dq_utils.py:134-182, utils/model_utils.py:92-118 run on (1) the shipped nao relaxation result and
    (2) a synthetic mixed revolute / prismatic / static sequence."""
    import importlib
    import warnings
    import networkx as nx
    g = importlib.import_module("utils.graph_utils")
    k = importlib.import_module("utils.kinematic_utils")
    mu = ref.model_utils
    se3 = ref.screw_se3
    g.farthest_point_sample = _fps_from_zero
    cd = ref.chamfer.ChamferDistance()
    warnings.simplefilter("ignore")
    out = {}

    # ---- (1) nao base-2 result
    res = pickle.load(open(f"{REF}/demo_data/pretrained/nao/base-2/result_14999.pkl", "rb"))
    cano = torch.from_numpy(res["cano_pc"]).float()
    pc_list = torch.from_numpy(res["pc_list"]).float()
    pose = torch.from_numpy(res["pred_pose_list"]).float()
    part = torch.from_numpy(res["pred_cano_part"]).long()
    out["nao_pose"], out["nao_part"], out["nao_cano"] = pose.numpy(), part.numpy().astype(np.int16), cano.numpy()
    uni = torch.unique(part, sorted=True)
    out["nao_uni"] = uni.numpy()

    dq = se3.transform_to_dq(pose.reshape(-1, 4, 4))
    l, m, th, d = se3.dq_to_screw(dq)
    out["nao_dq"], out["nao_l"], out["nao_m"], out["nao_th"], out["nao_d"] = (x.numpy() for x in (dq, l, m, th, d))

    ax, mo, th, di, rel = g.compute_relative_trans(pose, return_trans=True)
    sel = lambda x: x[:, uni, :][:, :, uni]
    geo = g.compute_geo_cost(sel(rel), sel(ax), sel(mo), sel(th), sel(di))
    out["nao_rel_theta"], out["nao_rel_dist"] = sel(th).numpy(), sel(di).numpy()
    out["nao_rel_axis"], out["nao_rel_moment"] = sel(ax).numpy(), sel(mo).numpy()
    out["nao_geo_cost"] = geo.numpy()
    out["nao_root_cost"] = g.compute_root_cost(pose).numpy()

    pred = mu.compute_pc_transform(cano, pose, part)
    fps_pts, fps_idx = g.fps_sample_cano(cano, part, uni, num_fps=20)
    part_fps = g.fps_index_list(pred, fps_idx)
    cano_dist, pair = g.compute_spatial_cost(fps_pts, cd, return_index=True)
    P = len(uni)
    px, py = torch.meshgrid(torch.arange(P), torch.arange(P), indexing="ij")
    conn_all = torch.stack([px, py], dim=2).reshape(-1, 2)
    joint = g.compute_joint_cost(part_fps, conn_all, pair.reshape(-1, 2)).reshape(-1, P, P).sum(dim=0)
    out["nao_fps_idx"], out["nao_cano_dist"], out["nao_pair"], out["nao_joint_cost"] = \
        fps_idx.numpy(), cano_dist.numpy(), pair.numpy(), joint.numpy()

    merged = g.merging_wrapper(part.clone(), pose, cano, cd, 3e-2, n_it=2)
    out["nao_merged_part"] = merged.numpy().astype(np.int16)
    conn = g.mst_wrapper(merged, pose, cano, cd, verbose=False, num_fps=20, cano_dist_thr=1e-2, joint_cost_weight=100)
    out["nao_connection"] = conn.numpy()
    new_seg, new_trans, new_conn = k.extract_kinematic(merged, pose, conn.clone())
    out["nao_new_seg"], out["nao_new_conn"] = new_seg.numpy().astype(np.int16), new_conn.numpy()
    G, root, axis_list, moment_list, theta_list, edge_index = k.build_graph(new_conn, new_trans, verbose=False)
    names = list(edge_index.keys())
    out["nao_root"] = np.int64(root)
    out["nao_edges"] = np.array([[int(a) for a in n.split("_")] for n in names], np.int64)
    out["nao_edge_ids"] = np.array([edge_index[n] for n in names], np.int64)
    out["nao_axis_list"], out["nao_moment_list"], out["nao_theta_list"] = \
        axis_list.numpy(), moment_list.numpy(), theta_list.numpy()
    out["nao_reverse_topo"] = np.array(list(reversed(list(nx.topological_sort(G)))), np.int64)
    out["nao_screw_cost"] = np.float64(g.compute_screw_cost(new_trans, new_conn).item())
    pred2 = mu.compute_pc_transform(cano, new_trans, new_seg)
    cidx = int(res["cano_idx"])
    complete = torch.cat((pred2[:cidx], cano[None], pred2[cidx:]), dim=0)
    out["nao_group_err"] = np.float64(float(mu.compute_group_temporal_err(complete, new_seg)))
    sub = torch.arange(0, cano.shape[0], 8)                      # 512-point subsample keeps the Hungarian solves short
    out["nao_ass_sub"] = sub.numpy()
    out["nao_ass_err"] = np.float64(mu.compute_ass_err(pred2[:, sub], pc_list[:, sub], use_nproc=False).item())

    # ---- (2) synthetic mixed joints: part 0 static, 2 and 4 prismatic, others revolute; chain 0-1-2, 1-3, 0-4
    gen = torch.Generator().manual_seed(7)
    T, P = 6, 5
    local = _random_screw_sequence(T, P, gen, prismatic=(2, 4), static=(0,))
    parent = [-1, 0, 1, 1, 0]
    world = torch.eye(4).repeat(T, P, 1, 1)
    for p in range(1, P):
        world[:, p] = torch.bmm(world[:, parent[p]], local[:, p])
    out["syn_trans"] = world.numpy()
    T_recon, cost = g.compute_screw_trans(local.clone(), return_cost=True)
    out["syn_local"], out["syn_recon"], out["syn_recon_cost"] = local.numpy(), T_recon.numpy(), np.float64(cost.item())
    conn = torch.tensor([[1, 0], [2, 1], [3, 1], [4, 0]])
    out["syn_conn"] = conn.numpy()
    out["syn_screw_cost"] = np.float64(g.compute_screw_cost(world, conn).item())
    ax, mo, th, di, rel = g.compute_relative_trans(world, return_trans=True)
    out["syn_geo_cost"] = g.compute_geo_cost(rel, ax, mo, th, di).numpy()
    out["syn_root_cost"] = g.compute_root_cost(world).numpy()
    G, root, a_l, m_l, t_l, d_l, e_i, jt = k.build_graph(conn.clone(), world, verbose=False, revolute_only=False,
                                                         return_joint_type=True)
    names = list(e_i.keys())
    out["syn_root"] = np.int64(root)
    out["syn_edges"] = np.array([[int(a) for a in n.split("_")] for n in names], np.int64)
    out["syn_axis_list"], out["syn_moment_list"] = a_l.numpy(), m_l.numpy()
    out["syn_theta_list"], out["syn_distance_list"] = t_l.numpy(), d_l.numpy()
    out["syn_joint_prismatic"] = np.array([j == "prismatic" for j in jt])

    # ---- (3) greedy spanning tree on seeded cost matrices, with and without relabelling / early stop
    cost = torch.rand(7, 7, generator=gen)
    cost = cost + cost.T + 1e4 * torch.eye(7)
    out["mst_cost"] = cost.numpy()
    out["mst_plain"] = g.mst(cost).numpy()
    lab = torch.tensor([2, 3, 5, 8, 11, 12, 19])
    out["mst_labels"] = lab.numpy()
    out["mst_relabelled"] = g.mst(cost, uni_label=lab).numpy()
    out["mst_capped"] = g.mst(cost, uni_label=lab, max_cost=0.55).numpy()
    out["mst_cap"] = np.float64(0.55)

    # ---- (4) merge pass with real contractions: parts {1,2,5} move together, {3,6} move together, 0 and 4 alone
    T, P = 5, 7
    motion = _random_screw_sequence(T, 3, gen)
    trans = torch.eye(4).repeat(T, P, 1, 1)
    for p, grp in {1: 0, 2: 0, 5: 0, 3: 1, 6: 1, 4: 2}.items():
        trans[:, p] = motion[:, grp]
    seg = torch.randint(0, P, (300,), generator=gen)
    conn = torch.tensor([[0, 1], [2, 1], [2, 5], [5, 3], [3, 6], [4, 0]])
    m_seg, m_conn = g.merge_graph(seg.clone(), conn, trans, 3e-2, verbose=False)
    out["mrg_trans"], out["mrg_seg"], out["mrg_conn"] = trans.numpy(), seg.numpy(), conn.numpy()
    out["mrg_new_seg"], out["mrg_new_conn"] = m_seg.numpy(), m_conn.numpy()

    np.savez_compressed(os.path.join(OUT, "structure.npz"), **out)
    print("structure.npz", out["nao_connection"].tolist(), out["nao_root"], out["nao_screw_cost"],
          out["syn_joint_prismatic"], out["mst_capped"].shape)


def gen_nao_eval(ref):
    """KAT-E (SURVEY section 6 / 8c): the rows of result.txt that the UNMODIFIED run_robot.py --evaluate writes for the
    shipped nao checkpoints (run_robot.py:224-338), produced by scripts/run_reference_dropin.py --backend stubs in this
    container, together with the dataset-side inputs of that evaluation (ground-truth flow / clouds / parts, the three
    sparse novel states of ik(), the kinematic-2 tree), so that a GPU test can reproduce the rows without the reference
    tree."""
    import importlib
    import json
    import subprocess
    import sys
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rows = {}
    # base_fps0: the reference's CUDA FPS kernel starts at index 0, its CPU fallback at torch.randint (SURVEY Q13), and the
    # structure stage of the relaxation evaluation depends on the samples -- "base" is the CPU row of BASELINE.md, "base_fps0"
    # what the same reference code gives with the CUDA start index (= what it prints on a GPU box over the drop-in)
    for tag, model, ck, extra in (("kin", "kinematic", "kinematic-2", []), ("base", "base", "base-2", []),
                                  ("base_fps0", "base", "base-2", ["--fps-from-zero"])):
        tmp = tempfile.mkdtemp()
        summ = os.path.join(tmp, "s.json")
        subprocess.check_call([sys.executable, os.path.join(root, "scripts", "run_reference_dropin.py"), "--backend", "stubs",
                               *extra, "--ref-root", REF, "--summary", summ, "--", f"--seq_path={REF}/demo_data/data/nao",
                               f"--save_root={tmp}", "--cano_idx=2", "--evaluate", f"--model={model}",
                               f"--resume={REF}/demo_data/pretrained/nao/{ck}/model.pth.tar"],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        rows[tag] = json.load(open(summ))["result_txt"]
    ds = importlib.import_module("dataset.dataset_robot")
    du = importlib.import_module("utils.dataset_utils")
    dataset = ds.Sequence(f"{REF}/demo_data/data/nao", num_points=4096, cano_idx=2)
    sample = dataset[0]
    cano_pose = dataset.pose_list[dataset.cano_idx]
    states = [du.sparse_sample_novel_state(sample["cano_pc"], sample["gt_cano_part"], cano_pose, nov, sparse_sample_per_part=1)
              for nov in dataset.novel_pose_list]
    ck = torch.load(f"{REF}/demo_data/pretrained/nao/kinematic-2/model.pth.tar", map_location="cpu", weights_only=False)
    tree = {"edge_index": {k: int(v) for k, v in ck["edge_index"].items()},
            "paths_to_base": {str(int(k)): [int(x) for x in v] for k, v in ck["paths_to_base"].items()},
            "reverse_topo": [int(x) for x in ck["reverse_topo"]]}
    out = dict(gt_flow_list=sample["gt_flow_list"].astype(np.float32),
               complete_gt_pc_list=sample["complete_gt_pc_list"].astype(np.float32),
               gt_cano_part=np.asarray(sample["gt_cano_part"]).astype(np.int16),
               sparse_cano_pc=np.asarray(states[0]["sparse_cano_pc"], np.float32),
               sparse_novel_pc=np.stack([np.asarray(s["sparse_novel_pc"], np.float32) for s in states]),
               novel_pc=np.stack([np.asarray(s["novel_pc"], np.float32) for s in states]),
               kin_tree_json=np.array(json.dumps(tree)),
               kin_rows_json=np.array(json.dumps(rows["kin"])), base_rows_json=np.array(json.dumps(rows["base"])),
               base_rows_fps0_json=np.array(json.dumps(rows["base_fps0"])))
    for s in states[1:]:
        assert np.array_equal(s["sparse_cano_pc"], states[0]["sparse_cano_pc"])
    np.savez_compressed(os.path.join(OUT, "nao_eval.npz"), **out)
    print("nao_eval.npz", rows)


def gen_assign(ref):
    """The assignment-loss refresh block of run_robot.py:164-187 run with the reference's own helpers on the nao demo
    (skinned cloud = the base-2 relaxation result, KAT-A), FPS with the CUDA start index 0 (SURVEY Q13):
    sample indices, per-frame optimal assignment cost, the matching, and the loss."""
    import importlib
    from scipy.optimize import linear_sum_assignment
    pn2 = importlib.import_module("networks.pointnet2_utils")
    mu = ref.model_utils
    res = pickle.load(open(f"{REF}/demo_data/pretrained/nao/base-2/result_14999.pkl", "rb"))
    cano = torch.from_numpy(res["cano_pc"]).float()
    pc_list = torch.from_numpy(res["pc_list"]).float()
    pose = torch.from_numpy(res["pred_pose_list"]).float()
    part = torch.from_numpy(res["pred_cano_part"]).long()
    pc_trans_list = mu.compute_pc_transform(cano, pose, part)
    downsample, lambda_assign = 4, 3e-1
    num_fps = pc_trans_list.shape[1] // downsample
    src_idx = _fps_from_zero(cano.unsqueeze(dim=0), num_fps).expand(pc_trans_list.shape[0], num_fps)
    pc_src = pn2.index_points(pc_trans_list, src_idx)
    tgt_idx = _fps_from_zero(pc_list, num_fps)
    pc_tgt = pn2.index_points(pc_list, tgt_idx)
    cost = torch.cdist(pc_src, pc_tgt).cpu().numpy()
    indices = [linear_sum_assignment(c) for c in cost]
    assign_indices = [(torch.as_tensor(i, dtype=torch.int64), torch.as_tensor(j, dtype=torch.int64)) for i, j in indices]
    ass_src_idx = mu.get_src_permutation_idx(assign_indices)
    ass_tgt_idx = mu.get_tgt_permutation_idx(assign_indices)
    ass_loss = lambda_assign * ((pc_src[ass_src_idx] - pc_tgt[ass_tgt_idx]) ** 2).sum(dim=-1).sum()
    totals = np.array([c[i, j].astype(np.float64).sum() for c, (i, j) in zip(cost, indices)])
    np.savez_compressed(os.path.join(OUT, "assign.npz"), src_idx=src_idx[0].numpy().astype(np.int16),
                        tgt_idx=tgt_idx.numpy().astype(np.int16), col_ind=np.stack([j for _, j in indices]).astype(np.int16),
                        totals=totals, ass_loss=np.float64(ass_loss.item()), lambda_assign=np.float64(lambda_assign),
                        downsample=np.int64(downsample))
    print("assign.npz", totals.sum(), ass_loss.item())


def gen_total_err(ref):
    """The model-selection energy of run_robot.py:224-240,306-314 for the shipped base-2 relaxation checkpoint on the nao
    demo, computed by the reference's own functions (structure tail with the CUDA FPS start index, then
    total_err = 100 * ass_err + screw_err + group_err)."""
    import importlib
    g = importlib.import_module("utils.graph_utils")
    k = importlib.import_module("utils.kinematic_utils")
    mu = ref.model_utils
    g.farthest_point_sample = _fps_from_zero
    cd = ref.chamfer.ChamferDistance()
    res = pickle.load(open(f"{REF}/demo_data/pretrained/nao/base-2/result_14999.pkl", "rb"))
    cano = torch.from_numpy(res["cano_pc"]).float()
    pc_list = torch.from_numpy(res["pc_list"]).float()
    cidx = int(res["cano_idx"])
    cb = torch.load(f"{REF}/demo_data/pretrained/nao/base-2/model.pth.tar", map_location="cpu", weights_only=False)
    bm = ref.model.BaseModel(num_parts=20, pose_len=pc_list.shape[0])
    bm.load_state_dict(cb["state_dict"], strict=False)
    with torch.no_grad():
        _, seg_part, trans_list = bm(cano)
    seg_part = g.denoise_seg_label(seg_part, cano, ref.KNN(k=1, transpose_mode=True), min_num=20)
    seg_part = g.merging_wrapper(seg_part, trans_list, cano, cd, 3e-2, n_it=2)
    conn = g.mst_wrapper(seg_part, trans_list, cano, cd, verbose=False, num_fps=20, cano_dist_thr=1e-2, joint_cost_weight=100)
    seg_part, trans_list, conn = k.extract_kinematic(seg_part, trans_list, conn)
    pred = mu.compute_pc_transform(cano, trans_list, seg_part)
    ass_err = 100 * mu.compute_ass_err(pred, pc_list, use_nproc=True)
    screw_err = g.compute_screw_cost(trans_list, conn)
    complete = torch.cat((pred[:cidx], cano[None], pred[cidx:]), dim=0)
    group_err = mu.compute_group_temporal_err(complete, seg_part)
    total = ass_err + screw_err + group_err
    np.savez_compressed(os.path.join(OUT, "total_err.npz"), ass_err=np.float64(float(ass_err)), screw_err=np.float64(float(screw_err)),
                        group_err=np.float64(float(group_err)), total_err=np.float64(float(total)))
    print("total_err.npz", float(ass_err), float(screw_err), float(group_err), float(total))


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    ref = rh.import_reference()
    gen_chamfer_small(ref)
    gen_se3(ref)
    gen_fk(ref)
    gen_flow(ref)
    gen_nao(ref)
    gen_structure(ref)
    gen_nao_eval(ref)
    gen_assign(ref)
    gen_total_err(ref)


if __name__ == "__main__":
    main()
