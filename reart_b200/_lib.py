"""ctypes binding of libreart_b200.so (include/reart_b200.h).

The product path has no CPU fallback: if the shared library is missing or a call fails the
caller gets an exception.  Tensors are passed as raw device pointers on the current CUDA stream.
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "csrc", "libreart_b200.so")

_c_i64 = ctypes.c_int64
_c_int = ctypes.c_int
_vp = ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/reart_b200.h one to one
SIGNATURES = {
    "reart_version": (ctypes.c_char_p, []),
    "reart_error_string": (ctypes.c_char_p, [_c_int]),
    "reart_last_cuda_error": (ctypes.c_char_p, []),
    "reart_knn1_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "reart_knn1_fwd": (_c_int, [_vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _c_i64, _vp]),
    "reart_chamfer_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "reart_chamfer_bidir_fwd": (_c_int, [_vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _c_i64, _vp]),
    "reart_chamfer_sym_search": (_c_int, [_vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp, ctypes.POINTER(ctypes.c_int32), _c_int,
                                          _vp]),
    "reart_knn1_bwd": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp]),
    "reart_chamfer_bidir_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp]),
    "reart_packed_bytes": (_c_i64, [_c_i64, _c_i64]),
    "reart_pack_cloud": (_c_int, [_vp, _c_i64, _c_i64, _vp, _vp]),
    "reart_skin_fwd": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp]),
    "reart_skin_bwd_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "reart_skin_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _c_i64, _vp]),
    "reart_energy_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "reart_skinned_chamfer_fwd_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _c_i64, _vp, _vp,
                                               _vp, _vp, _vp, _vp, _c_int, _vp, _c_i64, _vp]),
    "reart_skinned_chamfer_fwd_bwd_ex": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _c_i64, _vp, _vp,
                                                  _vp, _vp, _vp, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _c_i64, _vp]),
    "reart_skinned_chamfer_fwd_bwd_culled": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _c_i64, _vp, _vp,
                                                      _vp, _vp, _vp, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64,
                                                      _vp]),
    "reart_skinned_chamfer_fwd_bwd_ordered": (_c_int, [_vp] * 7 + [_c_i64] * 4 + [_vp] * 10 + [_c_int] + [_vp] * 8 +
                                              [_c_i64, _vp]),
    "reart_skinned_chamfer_fwd_bwd_posed": (_c_int, [_vp] * 7 + [_c_i64] * 4 + [_vp] * 10 + [_c_int] + [_vp] * 8 +
                                            [_c_i64, _vp]),
    "reart_posed_order_max_points": (_c_i64, []),
    "reart_segmlp_fwd": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp]),
    "reart_segmlp_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp]),
    "reart_gumbel_st_fwd": (_c_int, [_vp, _vp, _vp, _c_i64, _c_i64, _vp, _vp, _vp]),
    "reart_gumbel_st_bwd": (_c_int, [_vp, _vp, _vp, _c_i64, _c_i64, _vp, _vp]),
    "reart_rot6d_fwd": (_c_int, [_vp, _c_i64, _vp, _vp]),
    "reart_rot6d_bwd": (_c_int, [_vp, _vp, _c_i64, _vp, _vp]),
    "reart_screw_to_transform_fwd": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _vp, _vp]),
    "reart_screw_to_transform_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _vp, _vp, _vp, _vp, _vp]),
    "reart_fk_fwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _vp, _vp]),
    "reart_fk_bwd": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _vp,
                              _vp, _vp]),
    "reart_knn": (_c_int, [_vp, _vp, _c_i64, _c_i64, _c_i64, _c_int, _vp, _vp, _vp]),
    "reart_knn_sq": (_c_int, [_vp, _vp, _c_i64, _c_i64, _c_i64, _c_int, _vp, _vp, _vp]),
    "reart_knn3_blend": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_i64, _vp, _vp, _vp]),
    "reart_flow_refs_sorted_bytes": (_c_i64, [_c_i64, _c_i64]),
    "reart_flow_refs_sort": (_c_int, [_vp, _vp, _c_i64, _c_i64, _vp, _c_i64, _c_i64, _vp, _vp]),
    "reart_knn3_blend_sorted": (_c_int, [_vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _vp, _vp, _vp, _vp]),
    "reart_fps": (_c_int, [_vp, _c_i64, _c_i64, _c_i64, _vp, _vp]),
    "reart_fps_temp": (_c_int, [_vp, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp]),
    "reart_ball_query": (_c_int, [_vp, _vp, _c_i64, _c_i64, _c_i64, ctypes.c_float, _c_int, _vp, _vp]),
    "reart_allreduce_oneshot": (_c_int, [_vp, _c_int, _c_int, _c_i64, _c_i64, _vp, _vp, _vp]),
    "reart_fp32_probe": (_c_int, [_c_int, _c_int, _c_int, _vp, _vp, ctypes.POINTER(ctypes.c_double),
                                  ctypes.POINTER(ctypes.c_double), _vp]),
}



class RelaxTailArgs(ctypes.Structure):
    """reart_relax_tail_args of include/reart_b200.h (field for field)."""
    _fields_ = [(n, _vp) for n in ("cano", "w0", "b0", "w2", "ysoft", "tau", "gW", "d6", "tr", "gR", "gtr", "m_seg", "v_seg",
                                   "m_d6", "v_d6", "m_tr", "v_tr", "step")] + \
               [(n, ctypes.c_float) for n in ("lr_pose", "lr_seg", "beta1", "beta2", "eps", "weight_decay")] + \
               [(n, _vp) for n in ("partials", "tickets", "loss_local", "bucket", "loss_out", "peer_base", "epoch")] + \
               [(n, ctypes.c_int32) for n in ("rank", "world", "n_pad", "phase")] + \
               [(n, _c_i64) for n in ("N", "H", "P", "T")]


class KinTailArgs(ctypes.Structure):
    """reart_kin_tail_args of include/reart_b200.h (field for field)."""
    _fields_ = [(n, _vp) for n in ("fk", "gR", "gtr", "loss_local", "order", "parent", "edge", "joint_type", "axis", "moment",
                                   "theta", "distance", "root_6d", "root_t", "grad", "m", "v", "step")] + \
               [(n, ctypes.c_float) for n in ("lr", "beta1", "beta2", "eps", "weight_decay")] + \
               [(n, _vp) for n in ("partials", "loss_out", "peer_base", "epoch")] + \
               [(n, ctypes.c_int32) for n in ("rank", "world", "n_pad", "phase")] + \
               [(n, _c_i64) for n in ("T", "P")]


SIGNATURES.update({
    "reart_kin_head": (_c_int, [_vp] * 10 + [_c_i64, _c_i64] + [_vp] * 4),
    "reart_kin_tail_workspace_bytes": (_c_i64, [_c_i64, _c_i64]),
    "reart_kin_tail": (_c_int, [ctypes.POINTER(KinTailArgs), _vp]),
    "reart_kin_assign_workspace_bytes": (_c_i64, [_c_i64, _c_i64]),
    "reart_kin_assign": (_c_int, [_vp] * 7 + [ctypes.c_float] + [_c_i64] * 4 + [_vp] * 3 + [_c_int, _vp, _c_i64, _vp]),
    "reart_kin_flow_workspace_bytes": (_c_i64, [_c_i64, _c_i64]),
    "reart_kin_flow": (_c_int, [_vp] * 7 + [ctypes.c_float, _c_int] + [_c_i64] * 6 + [_vp] * 3 + [_c_int, _vp, _c_i64, _vp]),
    "reart_flow_grad_workspace_bytes": (_c_i64, [_c_i64, _c_i64]),
    "reart_flow_grad": (_c_int, [_vp] * 4 + [ctypes.c_float, _c_int] + [_c_i64] * 5 + [_vp] * 2 + [_c_int, _vp, _c_i64, _vp]),
    "reart_relax_head": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "reart_skinned_chamfer_fwd_bwd_fused": (_c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, _c_i64, _vp, _vp, _vp,
                                                     _vp, _vp, _vp, _c_int, _vp, _c_i64, _vp]),
    "reart_relax_tail_workspace_bytes": (_c_i64, [_c_i64, _c_i64, _c_i64]),
    "reart_relax_tail_ticket_words": (_c_i64, [_c_i64]),
    "reart_relax_tail": (_c_int, [ctypes.POINTER(RelaxTailArgs), _vp]),
    "reart_lap": (_c_int, [_vp, _vp, _c_i64, _vp, _c_i64, _c_i64, _vp, _vp, _vp, _c_int, _vp]),
    "reart_assign_loss_grad": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_i64, _c_i64, ctypes.c_float, _vp, _c_int, _vp, _vp]),
})

_lib = None


class ReartError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Load the C-ABI library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ReartError(
                f"{SO_PATH} not found: build it with `python -m reart_b200.build` "
                "(reart_b200 has no CPU or PyTorch fallback)")
        handle = ctypes.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(code: int, what: str) -> None:
    if code != 0:
        extra = f"; CUDA: {lib().reart_last_cuda_error().decode()}" if code == -3 else ""
        raise ReartError(f"{what} failed: {lib().reart_error_string(code).decode()} ({code}){extra}")


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise ReartError("reart_b200 kernels need CUDA tensors (there is no CPU fallback); got a tensor on "
                             f"{t.device}")


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
