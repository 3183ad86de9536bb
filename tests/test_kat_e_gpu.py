"""KAT-E on the GPU: the rows of ``result.txt`` that the reference's ``run_robot.py --evaluate --cano_idx=2`` writes for
the shipped nao checkpoints (run_robot.py:224-338; README.md:60-76), reproduced WITHOUT the reference tree from
``tests/golden/nao.npz`` + ``tests/golden/nao_eval.npz`` through ``reart_b200.{model,structure,model_utils,eval_utils,
retarget}`` -- i.e. the evaluation block of the run script re-played on the package's own modules.

Golden rows (reference Python on CPU, oracle/make_golden.py::gen_nao_eval, 3 decimals as the script prints them):
  kinematic-2: recon_err 0.896  retarget_err 2.234  flow_epe 0.447  acc5 0.609  acc10 0.911  angle 0.282  seg_ri 0.890
  base-2:      recon_err 1.194  (retarget 9999 by design)  flow_epe 0.636  acc5 0.412  acc10 0.853  seg_ri 0.882   [CPU]
  base-2 with the CUDA FPS start index 0 (what the reference prints on a GPU box, profiles/r02_run_robot_dropin.md):
               recon_err 0.903  flow_epe 0.478  acc5 0.604  acc10 0.913  angle 0.372  seg_ri 0.890
The relaxation rows are device dependent IN THE REFERENCE: its CPU FPS fallback starts at torch.randint, its CUDA kernel
at index 0 (SURVEY Q13), and the merging / spanning-tree stage that precedes the rows consumes those samples.  On a GPU
the reference -- and this package -- follow the CUDA semantics, so the base test is pinned on the fps0 rows.
"""
import json

import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

ROW_TOL = 1e-3            # the script prints 3 decimals
RETARGET_TOL = 5e-2       # 200 Adam(amsgrad) steps from theta = 1e-6: fp32 trajectory noise, stated in VERDICT item 1


def dev():
    return torch.device("cuda")


def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    return t if dtype is None else t.to(dtype)


def _rows(pred_pc_list, cano, cano_idx, seg_part, ev):
    """run_robot.py:247-268 on device tensors -> dict of the printed rows."""
    from reart_b200.eval_utils import eval_flow, eval_seg
    complete = torch.cat((pred_pc_list[:cano_idx], cano[None], pred_pc_list[cano_idx:]), dim=0)
    pred_flow = complete[1:] - complete[:-1]
    epe, acc1, acc2, angle = eval_flow(pred_flow, cu(ev["gt_flow_list"]), acc1_thre=0.005, acc2_thre=0.01)
    ri = eval_seg(cu(ev["gt_cano_part"].astype(np.int64)), seg_part)
    gt = cu(ev["complete_gt_pc_list"])
    recon = 100.0 * float((complete - gt).square().sum(-1).sqrt().mean(dim=1).mean())
    return {"recon_err": recon, "flow_epe": 100.0 * epe, "flow_acc5": acc1, "flow_acc10": acc2, "flow_angle": angle,
            "seg_ri": float(ri)}


def _check(rows, golden, keys):
    for k in keys:
        assert abs(rows[k] - golden[k]) <= ROW_TOL, (k, rows[k], golden[k])


def test_kat_e_kinematic_rows(nao):
    from reart_b200.knn_module import KNN
    from reart_b200.model import KinematicModel
    from reart_b200.model_utils import compute_pc_transform
    from reart_b200.retarget import retarget, retarget_error
    from reart_b200.structure import denoise_seg_label, edge_index2edges, extract_kinematic
    g, cano_np, _ = nao
    ev = load_golden("nao_eval.npz")
    golden = json.loads(str(ev["kin_rows_json"]))
    tree = json.loads(str(ev["kin_tree_json"]))
    paths = {int(k): v for k, v in tree["paths_to_base"].items()}
    cano = cu(cano_np)
    model = KinematicModel(pose_len=9, seg_part=torch.from_numpy(g["katC_seg_part"].astype(np.int64)),
                           cano_pc=torch.from_numpy(cano_np), knn=KNN(k=1, transpose_mode=True),
                           edge_index=tree["edge_index"], paths_to_base=paths, reverse_topo=tree["reverse_topo"])
    model.load_state_dict({"axis_list": torch.from_numpy(g["katC_axis"]), "moment_list": torch.from_numpy(g["katC_moment"]),
                           "theta_list": torch.from_numpy(g["katC_theta"])}, strict=True)
    model.to(dev()).eval()
    cano_idx = int(g["cano_idx"])
    with torch.no_grad():
        _, seg_part, trans_list = model(cano)                                             # run_robot.py:159
    knn = KNN(k=1, transpose_mode=True)
    seg_part = denoise_seg_label(seg_part, cano, knn, min_num=20)                          # :229
    joint_connection = torch.tensor(edge_index2edges(model.edge_index), dtype=torch.long, device=dev())   # :233-235
    seg_part, trans_list, joint_connection = extract_kinematic(seg_part, trans_list, joint_connection)    # :240
    pred = compute_pc_transform(cano, trans_list, seg_part)                                # :244
    rows = _rows(pred, cano, cano_idx, seg_part, ev)
    _check(rows, golden, ("recon_err", "flow_epe", "flow_acc5", "flow_acc10", "flow_angle", "seg_ri"))
    # ik() retargeting (run_robot.py:292-295, kinematic_utils.py:201-266): three novel states, 200 Adam steps each
    fitted = retarget(model, cu(ev["sparse_cano_pc"]), cu(ev["sparse_novel_pc"]), n_iter=200)
    err, _, _ = retarget_error(model, cano, cu(ev["novel_pc"]), fitted)
    assert abs(float(err.mean()) - golden["retarget_err"]) <= RETARGET_TOL, (err.tolist(), golden["retarget_err"])


def test_kat_e_base_rows(nao):
    """base-2 checkpoint: the relaxation model's evaluation rows.  The structure stage that precedes them in the script
    (denoise -> merging_wrapper -> mst_wrapper -> extract_kinematic, run_robot.py:229-240) relabels and merges parts;
    recon / flow rows depend on the merged labels, so the whole chain runs here on the package's structure module."""
    from reart_b200.chamfer import ChamferDistance
    from reart_b200.knn_module import KNN
    from reart_b200.model import BaseModel
    from reart_b200.model_utils import compute_pc_transform
    from reart_b200.structure import denoise_seg_label, extract_kinematic, merging_wrapper, mst_wrapper
    g, cano_np, _ = nao
    ev = load_golden("nao_eval.npz")
    golden = json.loads(str(ev["base_rows_fps0_json"]))
    cano = cu(cano_np)
    model = BaseModel(num_parts=20, pose_len=9)
    sd = {"proposal_6d": torch.from_numpy(g["katD_6d"]), "proposal_t": torch.from_numpy(g["katD_t"]),
          "seg_head.model.0.weight": torch.from_numpy(g["katD_w0"]), "seg_head.model.0.bias": torch.from_numpy(g["katD_b0"]),
          "seg_head.model.2.weight": torch.from_numpy(g["katD_w2"])}
    model.load_state_dict(sd, strict=False)
    model.to(dev()).eval()
    cano_idx = int(g["cano_idx"])
    with torch.no_grad():
        _, seg_part, trans_list = model(cano, tau=1.0)
    cd, knn = ChamferDistance(), KNN(k=1, transpose_mode=True)
    seg_part = denoise_seg_label(seg_part, cano, knn, min_num=20)
    seg_part = merging_wrapper(seg_part, trans_list, cano, cd, 3e-2, n_it=2)
    conn = mst_wrapper(seg_part, trans_list, cano, cd, verbose=False, num_fps=20, cano_dist_thr=1e-2, joint_cost_weight=100)
    seg_part, trans_list, conn = extract_kinematic(seg_part, trans_list, conn)
    pred = compute_pc_transform(cano, trans_list, seg_part)
    rows = _rows(pred, cano, cano_idx, seg_part, ev)
    _check(rows, golden, ("recon_err", "flow_epe", "flow_acc5", "flow_acc10", "flow_angle", "seg_ri"))
