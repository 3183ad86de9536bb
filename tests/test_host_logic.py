"""CPU: host-side logic and the C-ABI surface (no GPU compute)."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden


def header_symbols():
    src = open(os.path.join(ROOT, "include", "reart_b200.h")).read()
    return sorted(set(re.findall(r"REART_API\s+[\w\s\*]+?\b(reart_\w+)\s*\(", src)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    import ctypes
    from reart_b200 import _lib, build
    so = build.build()
    assert os.path.exists(so)
    handle = ctypes.CDLL(so)
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(handle, s), f"{s} declared in include/reart_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == syms, "ctypes SIGNATURES out of sync with the header"
    L = _lib.lib()
    assert b"sm_100a" in L.reart_version()
    assert L.reart_error_string(-2).decode().startswith("workspace")
    assert L.reart_knn1_workspace_bytes(2, 100, 100) > 0 and L.reart_chamfer_workspace_bytes(1, 1, 1) > 0
    assert L.reart_packed_bytes(1, 33) >= 64 * 12


def test_ctypes_signatures_match_the_header_prototypes():
    """Argument count and the int64 / int / float / pointer class of every parameter, parsed from the header."""
    import ctypes
    from reart_b200 import _lib
    src = open(os.path.join(ROOT, "include", "reart_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    protos = re.findall(r"REART_API\s+([\w\s\*]+?)\b(reart_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S)
    assert len(protos) == len(_lib.SIGNATURES)

    def kind(decl):
        decl = decl.strip()
        if "*" in decl:
            return "ptr"
        for key in ("int64_t", "float", "double", "int"):
            if re.search(rf"\b{key}\b", decl):
                return key
        raise AssertionError(decl)

    ctype_kind = {ctypes.c_int64: "int64_t", ctypes.c_int: "int", ctypes.c_float: "float", ctypes.c_void_p: "ptr",
                  ctypes.c_char_p: "ptr"}
    for ret, name, params in protos:
        restype, argtypes = _lib.SIGNATURES[name]
        decls = [] if params.strip() in ("", "void") else [p for p in params.split(",")]
        assert len(decls) == len(argtypes), name
        for d, a in zip(decls, argtypes):
            assert kind(d) == ctype_kind.get(a, "ptr"), (name, d.strip(), a)
        assert kind(ret + " ") == ctype_kind.get(restype, "ptr"), (name, ret)


def test_relax_tail_args_struct_matches_the_header_field_for_field():
    """ctypes mirror of reart_relax_tail_args: same field names in the same order, same C type class, so the layouts agree."""
    import ctypes
    from reart_b200 import _lib
    src = open(os.path.join(ROOT, "include", "reart_b200.h")).read()
    body = re.search(r"typedef struct reart_relax_tail_args \{(.*?)\} reart_relax_tail_args;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for stmt in body.split(";"):
        stmt = stmt.strip()
        if not stmt:
            continue
        names = [n.strip() for n in stmt.split(",")]
        first = names[0]
        ctype = first[:first.rindex(" ")].strip() if "*" not in first else first[:first.rindex("*") + 1].strip()
        for n in names:
            ident = re.search(r"(\w+)$", n).group(1)
            if "*" in first:
                fields.append((ident, "ptr"))
            else:
                fields.append((ident, ctype))
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_float: "float", ctypes.c_int32: "int32_t", ctypes.c_int64: "int64_t"}
    mirror = [(n, kinds[t]) for n, t in _lib.RelaxTailArgs._fields_]
    assert mirror == fields


def test_header_cites_reference_for_every_entry_point():
    src = open(os.path.join(ROOT, "include", "reart_b200.h")).read()
    for name in ("utils/chamfer.py:174", "utils/chamfer.py:206", "networks/model.py:63-69", "networks/loss.py:24-29",
                 "screw_se3/geo_utils.py:632-651", "screw_se3/screw_utils.py:6-30", "utils/kinematic_utils.py:151-198",
                 "utils/flow_utils.py:147-170", "pointnet2_utils.py:29,263"):
        assert name in src


def test_built_library_is_sm100a_sass_with_bulk_tma_and_packed_fp32():
    """Checks the BINARY (cuobjdump -sass of the in-tree .so), not the source: sm_100a only; the search kernels stage
    their tiles with 1-D bulk TMA (UBLKCP) and run packed FP32 (FFMA2/FADD2/FMUL2) with FMNMX3 / REDUX minima; no
    tensor-core opcode anywhere (contraction depth 3); the deterministic kernels carry no float RED/ATOM at all."""
    import shutil
    import sys
    from reart_b200 import build
    assert "arch=compute_100a,code=sm_100a" in " ".join(build.NVCC_FLAGS) and "-lineinfo" in build.NVCC_FLAGS
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_summary
    build.build()
    arch, kernels = sass_summary.census()
    assert arch == ["sm_100a"]
    by = lambda frag: [k for n, k in kernels.items() if frag in n]
    sym = by("chamfer_sym_kernelILi8ELi1E")                   # brute-force, culled and fused-producer instantiations
    assert len(sym) == 3
    for k in sym:
        assert k["UBLKCP"] >= 2 and k["FFMA2"] > 100 and k["FADD2"] > 100 and k["FMNMX3"] > 50 and k["REDUX"] > 10
    assert all(k["UBLKCP"] >= 1 and k["FFMA2"] > 0 for k in by("knn1_main_kernel"))
    assert sum(k["UTCMMA|HGMMA|HMMA"] for k in kernels.values()) == 0
    for frag in ("skin_bwd_fused_kernel", "skin_bwd_reduce_kernel", "energy_rows_kernel", "skin_fwd_sorted_kernel",
                 "relax_head_kernel"):
        assert by(frag) and all(k["float RED/ATOM"] == 0 for k in by(frag)), frag
    for frag in ("energy_cols_kernel", "relax_tail_kernel", "lap_jv_kernel", "assign_loss_grad_kernel"):
        assert by(frag) and all(k["float RED/ATOM"] == 0 for k in by(frag)), frag      # integer tickets / fixed point only


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "reart_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            path = os.path.join(dirpath, f)
            if f.endswith(".py"):
                text = open(path).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", text, re.M), path
                assert "libreart_oracle" not in text and "oracle/_build" not in text, path
            elif f.endswith((".cu", ".cuh", ".h")):
                for line in open(path):
                    if line.lstrip().startswith("#include"):
                        assert "oracle" not in line, path


def test_chamfer_argument_validation_matches_reference():
    from reart_b200 import ReartError
    from reart_b200.chamfer import ChamferDistance, knn_gather, knn_points
    cd = ChamferDistance()
    a, b = torch.randn(2, 5, 3), torch.randn(2, 6, 3)
    with pytest.raises(TypeError):
        cd(a.numpy(), b)
    with pytest.raises(ValueError, match="same batchsize"):
        cd(a, torch.randn(3, 6, 3))
    with pytest.raises(ValueError, match="same dimensionality"):
        cd(a, torch.randn(2, 6, 2))
    with pytest.raises(ValueError, match="Reduction"):
        cd(a, b, reduction="max")
    with pytest.raises(ValueError, match="same batch dimension"):
        knn_points(a, torch.randn(3, 6, 3))
    with pytest.raises(ValueError, match="same point dimension"):
        knn_points(a, torch.randn(2, 6, 4))
    with pytest.raises(ReartError):                     # CPU tensors: no fallback
        cd(a, b)
    x = torch.arange(24.0).reshape(2, 4, 3)
    idx = torch.tensor([[[0], [3]], [[1], [1]]])
    out = knn_gather(x, idx)
    assert out.shape == (2, 2, 1, 3) and torch.equal(out[0, 1, 0], x[0, 3]) and torch.equal(out[1, 0, 0], x[1, 1])


def test_flow_loss_matches_reference_golden():
    from reart_b200.loss import flow_loss
    g = load_golden("flow.npz")
    gt, mask = torch.from_numpy(g["blended"]), torch.from_numpy(g["mask"])
    for robust, lk, gk in ((False, "l_mse", "g_mse"), (True, "l_hub", "g_hub")):
        pred = torch.from_numpy(g["pred"]).requires_grad_(True)
        l = flow_loss(gt, pred, flow_mask_list=mask, robust=robust)
        assert abs(l.item() - float(g[lk])) <= 1e-5 * float(g[lk])
        l.backward()
        np.testing.assert_allclose(pred.grad.numpy(), g[gk], rtol=1e-5, atol=1e-8)
    l = flow_loss(gt, torch.from_numpy(g["pred"]))
    assert abs(l.item() - float(g["l_nomask"])) <= 1e-5 * float(g["l_nomask"])


def test_torch_restatements_of_screw_helpers_match_reference_golden():
    from reart_b200 import screw_se3
    g = load_golden("se3.npz")
    l, m, th, d = (torch.from_numpy(g[k]) for k in ("l", "m", "theta", "d"))
    expc = screw_se3.screw_param_to_exponential_coordinates(l, m, th, d)
    np.testing.assert_allclose(expc.numpy(), g["expc"], rtol=1e-5, atol=1e-7)
    M = screw_se3.transform_from_exponential_coordinates(expc)
    np.testing.assert_allclose(M.numpy(), g["M"], rtol=1e-5, atol=2e-6)
    inv = screw_se3.inverse_transformation(M)
    np.testing.assert_allclose(torch.bmm(inv, M).numpy(), np.tile(np.eye(4, dtype=np.float32), (M.shape[0], 1, 1)), atol=2e-5)
    R = torch.from_numpy(g["R"])
    assert screw_se3.matrix_to_rotation_6d(R).shape == (R.shape[0], 6)


def test_tree_flattening_and_model_state_dict_keys():
    from reart_b200.kinematic import flatten_tree
    from reart_b200.model import BaseModel, KinematicModel
    g = load_golden("nao.npz")
    order, parent, edge = g["katC_order"], g["katC_parent"], g["katC_edge"]
    edge_index = {f"{c}_{parent[c]}": int(edge[c]) for c in range(len(order)) if parent[c] >= 0}
    paths = {}
    for c in range(len(order)):
        path, x = [c], c
        while parent[x] >= 0:
            x = int(parent[x]); path.append(x)
        paths[c] = path
    o2, p2, e2 = flatten_tree(paths, [int(o) for o in order], edge_index)
    assert np.array_equal(o2, order) and np.array_equal(p2, parent) and np.array_equal(e2, edge)
    bm = BaseModel(num_parts=20, pose_len=9)
    assert set(bm.state_dict()) == {"proposal_6d", "proposal_t", "joint_connection", "seg_head.model.0.weight",
                                    "seg_head.model.0.bias", "seg_head.model.2.weight"}
    assert bm.state_dict()["seg_head.model.0.weight"].shape == (128, 3, 1)
    km = KinematicModel(pose_len=9, seg_part=torch.from_numpy(g["katC_seg_part"].astype(np.int64)),
                        cano_pc=torch.zeros(4096, 3), knn=None, edge_index=edge_index, paths_to_base=paths,
                        reverse_topo=[int(o) for o in order])
    assert set(km.state_dict()) == {"axis_list", "moment_list", "theta_list"}
    km2 = KinematicModel(pose_len=9, seg_part=torch.from_numpy(g["katC_seg_part"].astype(np.int64)),
                         cano_pc=torch.zeros(4096, 3), knn=None, edge_index=edge_index, paths_to_base=paths,
                         reverse_topo=[int(o) for o in order], load_distance=True, load_root_trans=True)
    assert set(km2.state_dict()) == {"axis_list", "moment_list", "theta_list", "distance_list", "root_6d", "root_t"}


def test_model_utils_small_helpers():
    from reart_b200.model_utils import create_transformation, tau_cosine, th_with_zeros
    x = torch.randn(5, 3, 4)
    y = th_with_zeros(x)
    assert y.shape == (5, 4, 4) and torch.equal(y[:, 3], torch.tensor([0.0, 0, 0, 1]).expand(5, 4))
    T = create_transformation(torch.eye(3)[None].repeat(2, 1, 1), torch.ones(2, 3, 1))
    assert T.shape == (2, 4, 4) and float(T[0, 3, 3]) == 1 and float(T[0, 0, 3]) == 1
    assert tau_cosine(0, 100, 1.0, 5.0) == 5.0 and abs(tau_cosine(100, 100, 1.0, 5.0) - 1.0) < 1e-12


def test_dropin_registers_the_three_native_module_names():
    import sys
    from reart_b200 import dropin
    dropin.install(force=True)
    assert hasattr(sys.modules["chamferdist"]._C, "knn_points_idx")
    assert hasattr(sys.modules["chamferdist"]._C, "knn_points_backward")
    assert sys.modules["knn_cuda"].KNN(k=3, transpose_mode=True).k == 3
    assert hasattr(sys.modules["pointnet2_cuda"], "furthest_point_sampling_wrapper")
    assert hasattr(sys.modules["pointnet2_cuda"], "ball_query_wrapper")
    for k in ("chamferdist", "chamferdist._C", "knn_cuda", "pointnet2_cuda"):
        sys.modules.pop(k, None)


def test_synthetic_generator_is_deterministic_and_in_range():
    from reart_b200.synth import make_sequence
    a = make_sequence(4, 512, 5, seed=2); b = make_sequence(4, 512, 5, seed=2)
    assert np.array_equal(a["cano"], b["cano"]) and np.array_equal(a["frames"], b["frames"])
    assert a["cano"].shape == (512, 3) and a["frames"].shape == (4, 512, 3) and a["pose"].shape == (4, 5, 4, 4)
    assert np.abs(a["cano"]).max() < 0.4


def test_c_abi_rejects_bad_arguments_without_touching_the_gpu():
    """Error behaviour at the boundary (include/reart_b200.h): negative codes, never exit(); the argument and
    workspace checks run on the host before any CUDA call, so they are testable here."""
    import ctypes
    from reart_b200 import _lib
    L = _lib.lib()
    fake = ctypes.c_void_p(0x1000)                      # never dereferenced: every call below fails validation first
    null = None
    assert L.reart_knn1_fwd(null, null, 1, 4, 4, null, null, null, 0, null) == -1
    assert L.reart_knn1_fwd(fake, fake, -1, 4, 4, fake, fake, fake, 0, null) == -1
    assert L.reart_knn1_fwd(fake, fake, 1, 4, 4, fake, fake, null, 0, null) == -2          # no workspace
    need = L.reart_knn1_workspace_bytes(1, 4, 4)
    assert L.reart_knn1_fwd(fake, fake, 1, 4, 4, fake, fake, fake, 64, null) == -2         # too small
    assert L.reart_chamfer_bidir_fwd(fake, fake, 2, 8, 8, fake, fake, fake, fake, fake, 16, null) == -2
    assert L.reart_chamfer_bidir_fwd(null, fake, 2, 8, 8, fake, fake, fake, fake, fake, 1 << 20, null) == -1
    assert L.reart_knn(fake, fake, 1, 10, 10, 9, fake, fake, null) == -1                   # k > 8
    assert L.reart_knn(fake, fake, 1, 2, 10, 3, fake, fake, null) == -1                    # fewer refs than k
    assert L.reart_fk_fwd(fake, fake, fake, null, null, null, null, null, 3, 4, fake, null) == -1
    assert L.reart_skinned_chamfer_fwd_bwd(fake, fake, fake, fake, fake, fake, 2, 16, 16, 3, fake, fake, fake, fake,
                                           fake, null, 1, fake, 8, null) == -2
    assert L.reart_allreduce_oneshot(fake, 3, 2, 10, 12, fake, fake, null) == -1           # rank >= world
    assert L.reart_knn1_workspace_bytes(-1, 1, 1) == -1
    # empty problems are successes and touch nothing
    assert L.reart_knn1_fwd(null, null, 0, 4, 4, null, null, null, 0, null) == 0
    assert L.reart_skin_fwd(null, null, null, null, 0, 0, 3, null, null) == 0
    for code in (0, -1, -2, -3, -4, -99):
        assert len(L.reart_error_string(code)) > 0


def test_bench_reference_arm_contract_on_cpu():
    """`bench.py --impl reference` is the CPU arm (oracle port on the host cores): it must run without a GPU and
    print one JSON line with the contract's keys."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "skinned_chamfer_fwd_bwd_directed_point_pairs_per_s"
    assert d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["dtype"] == "f32" and d["data"] == "synthetic"


def test_kd_order_is_a_permutation_and_refining_it_keeps_the_coarse_blocks():
    """ops.kd_order (pure torch, runs on the CPU too): a permutation; the engine orders the canonical cloud with leaf 8 but the
    search works on blocks of 256 rows -- refining the order must leave every 256-block the same SET of points as the leaf-256
    order (only their order inside the block changes), and make runs of 8 much tighter."""
    from reart_b200 import ops
    torch.manual_seed(0)
    for N in (16384, 5000, 3001):
        pts = torch.rand(2, N, 3)
        coarse, fine = ops.kd_order(pts, 256), ops.kd_order(pts, 8)
        for perm in (coarse, fine):
            assert all(sorted(perm[i].tolist()) == list(range(N)) for i in range(2))
        for i in range(2):
            for blk in range(0, N - 255, 256):
                assert set(coarse[i, blk:blk + 256].tolist()) == set(fine[i, blk:blk + 256].tolist())

        def spread(perm, chunk):
            q = torch.gather(pts, 1, perm[:, :, None].expand(-1, -1, 3))
            n = (N // chunk) * chunk
            c = q[:, :n].reshape(2, -1, chunk, 3)
            return float((c.amax(2) - c.amin(2)).norm(dim=-1).mean())
        assert spread(fine, 8) < 0.5 * spread(coarse, 8)
        assert spread(coarse, 256) < 0.6 * spread(torch.arange(N)[None].expand(2, N), 256)
