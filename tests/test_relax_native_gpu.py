"""The fused relaxation head / tail (csrc/relax.cu: relax_head_kernel, relax_tail_kernel) at every part-count
instantiation (<8>, <16>, <32>), called through the C ABI, against float64 references built from the very float32 inputs
the kernels received.

Reading the tail's gradients exactly: with m = 0, beta1 = 0 and weight_decay = 0, Adam's first moment becomes
m = 0 + 1 * (g - 0) = g, so after one call m_seg / m_d6 / m_tr hold the float32 gradients bit for bit (and bucket[:nseg]
holds the seg gradients too).  Adam itself is then checked on the kernel's own gradient, read the same way from a twin.

Tolerances scale with the sum of absolute terms: for an output y = sum of d products, |y32 - y64| <= c (d + k) u S with
S the same sum over absolute values, k the roundings inside one term and u = 2^-24.  Negative controls show that the
bounds are tight enough to see one point, one part or one hidden unit go missing."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, synthetic_sequence

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
# Every output is a float32 sum of d terms, each a product of factors that carry at most P + ~10 roundings of their own
# (the gumbel backward's dot product over P parts, 1/tau, the three roundings of h, the seg-MLP backward's sum over P
# parts).  First-order error analysis gives |err| <= (d + P + 10) u S; with d >= 10 that is <= 2 (d + P) u S.
C = 2.0
# depth of the tail's seg sums: 32 points in registers per (unit, quarter), + 3 quarters, + 7 chunks per group, + groups
TAIL_POINTS, TAIL_GROUP = 128, 8


def dev():
    return torch.device("cuda")


def lib():
    from reart_b200 import _lib
    return _lib, _lib.lib()


def worst(got, ref, bound):
    """max |got - ref| / bound over the elements (0/0 counts as 0, x/0 as inf)."""
    err = (got.double().cpu().reshape(-1) - ref.reshape(-1)).abs()
    b = bound.reshape(-1)
    r = torch.where(b > 0, err / torch.where(b > 0, b, torch.ones_like(b)), torch.where(err > 0, float("inf"), 0.0))
    return float(r.max()) if r.numel() else 0.0


def report(tag, **ratios):
    line = f"[{tag}] " + "  ".join(f"{k} {v:.3g}" for k, v in ratios.items())
    print(line)
    return line


# ------------------------------------------------------------------------------------------------------ launches
def run_head(x, w0, b0, w2, expo, tau, d6, noise_index=None, logits=True, hot=True):
    """reart_relax_head; N = len(x) (0: pose only), T = len(d6) (None: points only)."""
    _lib, L = lib()
    N, H, P = x.shape[0], w0.shape[0], w2.shape[0]
    T = 0 if d6 is None else d6.shape[0]
    e = lambda *s: torch.empty(*s, device=dev())
    out = dict(W=e(N, P), ysoft=e(N, P), R=e(T, P, 3, 3) if T else None, logits=e(N, P) if logits else None,
               hot=e(N, 2) if hot else None)
    _lib.check(L.reart_relax_head(_lib.ptr(x), _lib.ptr(w0), _lib.ptr(b0), _lib.ptr(w2), _lib.ptr(expo), _lib.ptr(noise_index),
                                  _lib.ptr(tau), _lib.ptr(d6), N, H, P, T, _lib.ptr(out["logits"]), _lib.ptr(out["W"]),
                                  _lib.ptr(out["ysoft"]), _lib.ptr(out["R"]), _lib.ptr(out["hot"]), _lib.stream_ptr()), "relax_head")
    return out


def tail_inputs(N, H, P, T, seed):
    """Random tail inputs; ysoft from the head on random noise (the tail does not care where its inputs come from).
    d6 stays near the identity frame so that the Gram-Schmidt of the 6D map is well conditioned."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *s: torch.randn(*s, device=dev(), generator=g)
    x = torch.rand(N, 3, device=dev(), generator=g) - 0.5
    w0, b0, w2 = r(H, 3), r(H) * 0.3, r(P, H) * 0.2
    expo = torch.empty(N, P, device=dev()).exponential_(generator=g)
    tau = torch.full((1,), 1.7, device=dev())
    ysoft = run_head(x, w0, b0, w2, expo, tau, None, logits=False, hot=False)["ysoft"]
    d6 = torch.tensor([1.0, 0.0, 0.0, 0.0, 1.0, 0.0], device=dev()) + 0.3 * r(T, P, 6)
    return dict(N=N, H=H, P=P, T=T, cano=x, w0=w0, b0=b0, w2=w2, d6=d6, tr=r(T, P, 3) * 0.1, ysoft=ysoft, tau=tau,
                gW=r(N, P), gR=r(T, P, 3, 3), gtr=r(T, P, 3))


class Tail:
    """One reart_relax_tail problem: its parameters, Adam state, step counter, tickets and workspace (world = 1)."""
    PARAMS = ("w0", "b0", "w2", "d6", "tr")

    def __init__(self, inp, params=None):
        _lib, L = lib()
        self.inp = inp
        N, H, P, T = inp["N"], inp["H"], inp["P"], inp["T"]
        self.nseg = 4 * H + P * H
        src = inp if params is None else params
        for k in self.PARAMS:
            setattr(self, k, src[k].clone())
        z = lambda *s: torch.zeros(*s, device=dev())
        self.m_seg, self.v_seg = z(self.nseg), z(self.nseg)
        self.m_d6, self.v_d6, self.m_tr, self.v_tr = z(T, P, 6), z(T, P, 6), z(T, P, 3), z(T, P, 3)
        self.step = z(1)
        self.partials = _lib.workspace(int(L.reart_relax_tail_workspace_bytes(N, H, P)), dev())
        self.tickets = torch.zeros(int(L.reart_relax_tail_ticket_words(N)), dtype=torch.int32, device=dev())
        self.loss_local = torch.full((1,), 0.8125, dtype=torch.float64, device=dev())
        self.bucket, self.loss_out = z(self.nseg + 1), z(1)

    def params(self):
        return {k: getattr(self, k) for k in self.PARAMS}

    def twin(self):
        """Same parameters and inputs, fresh Adam state, step counter, tickets and workspace."""
        return Tail(self.inp, self.params())

    def run(self, phase=0, beta1=0.0, beta2=0.999, wd=0.0, lr_pose=1e-2, lr_seg=1e-3, eps=1e-8):
        _lib, L = lib()
        p = _lib.ptr
        i = self.inp
        a = _lib.RelaxTailArgs()
        a.cano, a.w0, a.b0, a.w2, a.ysoft, a.tau, a.gW = p(i["cano"]), p(self.w0), p(self.b0), p(self.w2), p(i["ysoft"]), p(i["tau"]), p(i["gW"])
        a.d6, a.tr, a.gR, a.gtr = p(self.d6), p(self.tr), p(i["gR"]), p(i["gtr"])
        a.m_seg, a.v_seg, a.m_d6, a.v_d6, a.m_tr, a.v_tr = (p(t) for t in (self.m_seg, self.v_seg, self.m_d6, self.v_d6, self.m_tr, self.v_tr))
        a.step = p(self.step)
        a.lr_pose, a.lr_seg, a.beta1, a.beta2, a.eps, a.weight_decay = lr_pose, lr_seg, beta1, beta2, eps, wd
        a.partials, a.tickets, a.loss_local, a.bucket, a.loss_out = (p(t) for t in (self.partials, self.tickets, self.loss_local,
                                                                                     self.bucket, self.loss_out))
        a.rank, a.world, a.n_pad, a.phase = 0, 1, 0, phase
        a.N, a.H, a.P, a.T = i["N"], i["H"], i["P"], i["T"]
        _lib.check(L.reart_relax_tail(ctypes.byref(a), _lib.stream_ptr()), "reart_relax_tail")

    def seg_params(self):
        return torch.cat([self.w0.reshape(-1), self.b0.reshape(-1), self.w2.reshape(-1)])

    def state(self):
        return dict(self.params(), m_seg=self.m_seg, v_seg=self.v_seg, m_d6=self.m_d6, v_d6=self.v_d6, m_tr=self.m_tr,
                    v_tr=self.v_tr, step=self.step, bucket=self.bucket, loss_out=self.loss_out)


# ---------------------------------------------------------------------------------------------- float64 references
def f64(t):
    return t.detach().double().cpu()


def seg_reference(x, w0, b0, w2, ysoft, gW, tau, drop_part=False):
    """Float64 gradients of the seg MLP's parameters through the straight-through gumbel backward, in the tail's layout
    [w0 (H,3) | b0 (H) | w2 (P,H)], with the abs-sum S of every output and the ReLU-tie allowance.
    drop_part: part P-1 left out (a negative control)."""
    x, w0, b0, w2, y, g = (f64(t).reshape(s) for t, s in ((x, (-1, 3)), (w0, (-1, 3)), (b0, (-1,)), (w2, (w2.shape[0], -1)),
                                                          (ysoft, ysoft.shape), (gW, gW.shape)))
    tau = float(f64(tau).reshape(-1)[0])
    keep = torch.ones(y.shape[1], dtype=torch.float64)
    if drop_part:
        keep[-1] = 0.0
    dot = (g * y * keep).sum(1, keepdim=True)
    glog = y * (g - dot) / tau * keep
    sglog = y.abs() * (g.abs() + (g.abs() * y.abs()).sum(1, keepdim=True)) / tau
    pre = x @ w0.T + b0
    habs = x.abs() @ w0.abs().T + b0.abs()
    act = (pre > 0).double()
    tie = (pre.abs() <= 8 * U * habs).double()              # the float32 mask may differ from float64's here
    h = pre.clamp_min(0.0)
    gh, sgh = glog @ w2, sglog @ w2.abs()
    gpre, sgpre = gh * act, sgh * act
    grad = torch.cat([(gpre.T @ x).reshape(-1), gpre.sum(0), (glog.T @ h).reshape(-1)])
    S = torch.cat([(sgpre.T @ x.abs()).reshape(-1), sgpre.sum(0), (sglog.T @ (habs * act)).reshape(-1)])
    ties = torch.cat([((sgh * tie).T @ x.abs()).reshape(-1), (sgh * tie).sum(0), (sglog.T @ (16 * U * habs * tie)).reshape(-1)])
    # the last point's own contribution (the control "last point of the last, ragged chunk dropped")
    last = torch.cat([(gpre[-1][:, None] * x[-1][None]).reshape(-1), gpre[-1], (glog[-1][:, None] * h[-1][None]).reshape(-1)])
    return dict(grad=grad, S=S, ties=ties, last=last)


def tail_bound(ref, N, P):
    groups = -(-(-(-N // TAIL_POINTS)) // TAIL_GROUP)
    d = TAIL_POINTS // 4 + 3 + (TAIL_GROUP - 1) + groups
    return C * (d + P) * U * ref["S"] + ref["ties"]


def rot6d64(d6):
    """The Gram-Schmidt of screw_se3.rotation_6d_to_matrix (rows b1, b2, b1 x b2), restated in float64 torch: the library
    function itself runs on the float32 kernel."""
    a1, a2 = d6[..., :3], d6[..., 3:]
    b1 = a1 / a1.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    u = a2 - (b1 * a2).sum(-1, keepdim=True) * b1
    b2 = u / u.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    return torch.stack([b1, b2, torch.cross(b1, b2, dim=-1)], dim=-2)


def pose_reference(d6, gR):
    """g_d6 = J^T gR by float64 autograd, and its bound.  The kernel's derivatives come out of ~20 dual-number roundings
    (two normalisations, the projection, the cross product), then a sum of 9: bound = C (9 + 32) u sum_o |gR_o| max|J|."""
    d = f64(d6).reshape(-1, 6).requires_grad_(True)
    R = rot6d64(d).reshape(-1, 9)
    J = torch.stack([torch.autograd.grad(R[:, o].sum(), d, retain_graph=True)[0] for o in range(9)], dim=1)   # [TP,9,6]
    gr = f64(gR).reshape(-1, 9, 1)
    grad = (gr * J).sum(1)
    S = (gr.abs().sum(1) * J.abs().amax(dim=(1, 2))[:, None]).expand_as(grad)
    return grad, C * (9 + 32) * U * S


# ---------------------------------------------------------------------------------------------- 1. tail vs float64
# (P, H, N, T, negative controls): every instantiation x a spread of the reduction edges
TAIL_CASES = [
    (1, 32, 1, 2, False),          # <8>: one point, P=1 (exactly zero logit gradients), one pose block
    (7, 100, 1025, 3, True),       # <8>: ragged last chunk (1 point), idle units (Hpad 128), 2 groups
    (8, 128, 128, 64, False),      # <8>: exactly one chunk; T*P = 512 = one pose block of 4*Hpad threads
    (8, 256, 16385, 300, False),   # <8>: 17 groups (second pass of the 16-load loop), 3 pose blocks
    (9, 32, 127, 5, False),        # <16>: one ragged chunk
    (15, 33, 129, 40, True),       # <16>: scalar path (nseg = 627), 600 poses over 3 blocks of 256
    (15, 128, 16384, 64, True),    # <16>: the headline cfg3_16k shape, 16 groups
    (15, 128, 65536, 64, False),   # <16>: the cfg3_64k shape, 64 groups
    (16, 256, 1024, 8, False),     # <16>: exactly one group, Hpad = 256
    (17, 100, 16385, 4, False),    # <32>: 17 groups
    (31, 33, 16385, 3, False),     # <32>: scalar path (nseg = 1155) with 17 groups
    (31, 128, 1025, 50, True),     # <32>: ragged chunk, 1550 poses over 4 blocks
    (32, 256, 65536, 2, False),    # <32>: Hpad = 256 at 64 groups
]


@pytest.mark.parametrize("P,H,N,T,controls", TAIL_CASES, ids=[f"P{c[0]}-H{c[1]}-N{c[2]}-T{c[3]}" for c in TAIL_CASES])
def test_tail_gradients_match_float64(P, H, N, T, controls):
    inp = tail_inputs(N, H, P, T, seed=1000 + 7 * P + H + N % 997)
    before = {k: f64(inp[k]) for k in Tail.PARAMS}
    tail = Tail(inp)
    tail.run(beta1=0.0, wd=0.0)
    torch.cuda.synchronize()
    # the gradients are read bit for bit: bucket == m_seg, m_tr == gtr; the loss is passed through
    assert torch.equal(tail.bucket[:tail.nseg], tail.m_seg)
    assert torch.equal(tail.m_tr, inp["gtr"])
    assert float(tail.loss_out) == float(np.float32(0.8125)) and float(tail.step) == 1.0
    ref = seg_reference(inp["cano"], before["w0"], before["b0"], before["w2"], inp["ysoft"], inp["gW"], inp["tau"])
    bound = tail_bound(ref, N, P)
    seg = worst(tail.m_seg, ref["grad"], bound)
    gd6, bd6 = pose_reference(before["d6"], inp["gR"])
    pose = worst(tail.m_d6, gd6, bd6)
    ratios = dict(seg=seg, pose=pose)
    if P == 1:
        assert torch.count_nonzero(tail.m_seg) == 0, "P=1: the straight-through weights have no logit gradient"
    if controls:
        # the bound must see one point, one part and one unit go missing
        ratios["ctl_last_point"] = worst(tail.m_seg, ref["grad"] - ref["last"], bound)
        ratios["ctl_part"] = worst(tail.m_seg, seg_reference(inp["cano"], before["w0"], before["b0"], before["w2"], inp["ysoft"],
                                                             inp["gW"], inp["tau"], drop_part=True)["grad"], bound)
        g = ref["grad"].clone()
        g[3 * (H - 1):3 * H] = 0.0; g[3 * H + H - 1] = 0.0; g[4 * H + H - 1::H] = 0.0
        ratios["ctl_unit"] = worst(tail.m_seg, g, bound)
    line = report(f"tail P={P} H={H} N={N} T={T}", **ratios)
    assert seg < 1 and pose < 1, line
    if controls:
        assert min(ratios["ctl_last_point"], ratios["ctl_part"], ratios["ctl_unit"]) > 1, line


# ---------------------------------------------------------------------------------------------- 2. Adam
@pytest.mark.parametrize("P,H,N,T", [(15, 128, 3001, 10), (31, 33, 1025, 12)])
def test_adam_from_the_kernels_own_gradient(P, H, N, T):
    """Four steps with betas (0.9, 0.999) and weight decay: each step's exact gradient is read from a twin (same
    parameters, beta1 = 0, no weight decay), then m, v and p are checked against torch.optim.Adam's formula in float64.
    Covers the bias corrections, the step counter and the ticket re-arm (without it w0/b0/w2 would stop moving)."""
    inp = tail_inputs(N, H, P, T, seed=77 + P)
    f32 = lambda v: float(np.float32(v))                      # the hyper-parameters the kernel receives
    b1, b2, wd, eps = f32(0.9), f32(0.999), f32(1e-3), f32(1e-8)
    lrs = dict(seg=f32(1e-3), d6=f32(1e-2), tr=f32(1e-2))
    tail = Tail(inp)
    for step in range(1, 5):
        twin = tail.twin()
        twin.run(beta1=0.0, wd=0.0)
        torch.cuda.synchronize()
        g = dict(seg=f64(twin.m_seg), d6=f64(twin.m_d6), tr=f64(twin.m_tr))
        prev = dict(seg=(f64(tail.seg_params()), f64(tail.m_seg), f64(tail.v_seg)), d6=(f64(tail.d6), f64(tail.m_d6), f64(tail.v_d6)),
                    tr=(f64(tail.tr), f64(tail.m_tr), f64(tail.v_tr)))
        tail.run(beta1=0.9, beta2=0.999, wd=1e-3)
        torch.cuda.synchronize()
        assert float(tail.step) == step
        new = dict(seg=(f64(tail.seg_params()), f64(tail.m_seg), f64(tail.v_seg)), d6=(f64(tail.d6), f64(tail.m_d6), f64(tail.v_d6)),
                   tr=(f64(tail.tr), f64(tail.m_tr), f64(tail.v_tr)))
        bc1, bc2 = 1.0 - b1 ** step, 1.0 - b2 ** step
        for k in ("seg", "d6", "tr"):
            p0, m0, v0 = (t.reshape(-1) for t in prev[k])
            p1, m1, v1 = (t.reshape(-1) for t in new[k])
            gk = g[k].reshape(-1)
            gw = gk + wd * p0                                 # weight decay is added to g in float32
            tol_g = 2 * U * (gk.abs() + (wd * p0).abs())
            m_ref = b1 * m0 + (1 - b1) * gw
            tol_m = 4 * U * (m0.abs() + gw.abs()) + (1 - b1) * tol_g
            v_ref = b2 * v0 + (1 - b2) * gw * gw
            tol_v = 4 * U * v_ref + (1 - b2) * 2 * gw.abs() * tol_g
            upd = lrs[k] / bc1 * m1 / (v1.sqrt() / np.sqrt(bc2) + eps)         # from the kernel's own m, v
            p_ref = p0 - upd
            tol_p = 4 * U * p0.abs() + 16 * U * upd.abs()
            r = dict(m=worst(m1, m_ref, tol_m), v=worst(v1, v_ref, tol_v), p=worst(p1, p_ref, tol_p))
            line = report(f"adam P={P} H={H} step {step} {k}", **r)
            assert max(r.values()) < 1, line
            assert k != "seg" or bool((p1 != p0).any()), f"step {step}: the seg parameters did not move"


# ---------------------------------------------------------------------------------------------- 3. phases, 4. graph
def assert_same_state(a, b, what):
    for k, t in a.state().items():
        assert torch.equal(t, b.state()[k]), f"{what}: {k} differs"


@pytest.mark.parametrize("P,H,N,T", [(15, 128, 3001, 10), (32, 100, 16385, 5)])
def test_phase1_then_phase2_equals_phase0(P, H, N, T):
    """The NCCL fallback (gradients -> bucket, [all-reduce], Adam from the bucket) with nothing in between (one rank)
    is the one-launch step bit for bit, over several steps."""
    inp = tail_inputs(N, H, P, T, seed=5)
    a, b = Tail(inp), Tail(inp)
    for s in range(3):
        for t in (a, b):
            t.loss_local.fill_(1.0 / 3.0 + s)
        a.run(phase=0, beta1=0.9, wd=1e-3)
        b.run(phase=1, beta1=0.9, wd=1e-3)
        b.run(phase=2, beta1=0.9, wd=1e-3)
        torch.cuda.synchronize()
        assert_same_state(a, b, f"step {s}")
        assert float(b.loss_out) == float(np.float32(1.0 / 3.0 + s))
        assert float(b.step) == s + 1


@pytest.mark.parametrize("P,H,N,T", [(32, 256, 16385, 4), (15, 33, 1025, 40)])
def test_tail_graph_replay_equals_eager(P, H, N, T):
    inp = tail_inputs(N, H, P, T, seed=6)
    a, b = Tail(inp), Tail(inp)
    for _ in range(5):
        a.run(beta1=0.9, wd=1e-3)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.run(beta1=0.9, wd=1e-3)
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize()
    assert_same_state(a, b, "graph replay")


# ---------------------------------------------------------------------------------------------- 5./6. head
# (P, H, N, T, noise_index, logits/hot outputs)
HEAD_CASES = [
    (1, 32, 1, 3, False, True),
    (2, 100, 31, 2, True, True),
    (8, 256, 32, 5, False, False),
    (9, 32, 33, 7, True, True),
    (15, 128, 3001, 7, True, True),
    (16, 100, 3001, 4, True, False),
    (17, 256, 3001, 9, False, True),
    (31, 100, 33, 1, True, True),
    (32, 256, 3001, 7, True, True),
    (32, 32, 31, 0, False, True),      # points only
    (15, 128, 0, 40, False, True),     # poses only
]


def head_inputs(P, H, N, T, noise, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(N, 3, device=dev(), generator=g) - 0.5
    w0, b0 = torch.randn(H, 3, device=dev(), generator=g), torch.randn(H, device=dev(), generator=g) * 0.3
    w2 = torch.randn(P, H, device=dev(), generator=g) * 0.2
    expo = torch.empty(N, P, device=dev()).exponential_(generator=g)
    idx = torch.randperm(N, device=dev(), generator=g) if noise else None
    d6 = torch.randn(T, P, 6, device=dev(), generator=g) if T else None
    return x, w0, b0, w2, expo, idx, torch.full((1,), 1.3, device=dev()), d6


@pytest.mark.parametrize("P,H,N,T,noise,outs", HEAD_CASES, ids=[f"P{c[0]}-H{c[1]}-N{c[2]}-T{c[3]}" + ("-perm" if c[4] else "")
                                                                 for c in HEAD_CASES])
def test_head_equals_the_separate_kernels(P, H, N, T, noise, outs):
    """reart_relax_head == reart_segmlp_fwd + reart_gumbel_st_fwd (on expo[noise_index]) + reart_rot6d_fwd, bit for bit;
    hot holds each row's one non-zero of W."""
    _lib, L = lib()
    x, w0, b0, w2, expo, idx, tau, d6 = head_inputs(P, H, N, T, noise, seed=P * 31 + H + N)
    out = run_head(x, w0, b0, w2, expo, tau, d6, noise_index=idx, logits=outs, hot=outs)
    if N:
        lg = torch.empty(N, P, device=dev())
        _lib.check(L.reart_segmlp_fwd(_lib.ptr(x), _lib.ptr(w0), _lib.ptr(b0), _lib.ptr(w2), N, H, P, _lib.ptr(lg), _lib.stream_ptr()), "segmlp")
        e = expo[idx].contiguous() if noise else expo
        W2, ys2 = torch.empty(N, P, device=dev()), torch.empty(N, P, device=dev())
        _lib.check(L.reart_gumbel_st_fwd(_lib.ptr(lg), _lib.ptr(e), _lib.ptr(tau), N, P, _lib.ptr(W2), _lib.ptr(ys2), _lib.stream_ptr()), "gumbel")
        assert torch.equal(out["W"], W2) and torch.equal(out["ysoft"], ys2)
        if outs:
            assert torch.equal(out["logits"], lg)
            assert torch.equal(torch.count_nonzero(out["W"], dim=1), torch.ones(N, dtype=torch.int64, device=dev()))
            part = out["hot"].view(torch.int32)[:, 0].long()
            assert torch.equal(part, (out["W"] != 0).float().argmax(dim=1))
            assert torch.equal(out["hot"][:, 1], out["W"].gather(1, part[:, None])[:, 0])
    if T:
        R2 = torch.empty(T, P, 3, 3, device=dev())
        _lib.check(L.reart_rot6d_fwd(_lib.ptr(d6), T * P, _lib.ptr(R2), _lib.stream_ptr()), "rot6d")
        assert torch.equal(out["R"], R2)


@pytest.mark.parametrize("P,H,N,T,noise,outs", [c for c in HEAD_CASES if c[2] > 0],
                         ids=[f"P{c[0]}-H{c[1]}-N{c[2]}" + ("-perm" if c[4] else "") for c in HEAD_CASES if c[2] > 0])
def test_head_matches_float64(P, H, N, T, noise, outs):
    """logits and ysoft within the abs-sum bound of a float64 forward (ReLU ties allowed for); W one-hot with value
    (1 - y) + y in float32; the hot part is float64's argmax except where the top-two gap is within the bound."""
    x, w0, b0, w2, expo, idx, tau, d6 = head_inputs(P, H, N, T, noise, seed=P * 31 + H + N)
    out = run_head(x, w0, b0, w2, expo, tau, d6, noise_index=idx, logits=True, hot=True)
    torch.cuda.synchronize()
    X, W0, B0, W2 = f64(x), f64(w0), f64(b0), f64(w2)
    E = f64(expo[idx] if noise else expo)
    t = float(f64(tau)[0])
    pre = X @ W0.T + B0
    habs = X.abs() @ W0.abs().T + B0.abs()
    act = (pre > 0).double()
    tie = (pre.abs() <= 8 * U * habs).double()
    lg = pre.clamp_min(0.0) @ W2.T
    d = -(-H // 8) + 3                                        # 8 lanes per point: H/8 units each, then a 3-level xor tree
    bl = C * (d + P) * U * ((habs * act) @ W2.abs().T) + (16 * U * habs * tie) @ W2.abs().T
    r_logit = worst(out["logits"], lg, bl)
    le = E.log()
    z = (lg - le) / t
    y = torch.softmax(z, dim=1)
    zb = (bl + 4 * U * (lg.abs() + le.abs())) / t + 4 * U * z.abs() + 2 * U * z.abs().amax(1, keepdim=True)
    yb = y * (zb + zb.amax(1, keepdim=True)) + C * (P + 8) * U * y
    r_y = worst(out["ysoft"], y, yb)
    ys = out["ysoft"].cpu().numpy()
    Wk = out["W"].cpu().numpy()
    hot = (Wk != 0).argmax(1)
    assert ((Wk != 0).sum(1) == 1).all()
    yh = ys[np.arange(N), hot]
    assert np.array_equal(Wk[np.arange(N), hot], (np.float32(1.0) - yh) + yh)
    top2 = torch.topk(y, min(2, P), dim=1)
    want = top2.indices[:, 0].numpy()
    if P > 1:
        gap = (top2.values[:, 0] - top2.values[:, 1]).numpy()
        near = gap <= (yb.gather(1, top2.indices).sum(1)).numpy()
    else:
        near = np.zeros(N, dtype=bool)
    bad = (hot != want) & ~near
    line = report(f"head P={P} H={H} N={N}", logits=r_logit, ysoft=r_y, argmax_ties=float(near.sum()))
    assert r_logit < 1 and r_y < 1 and not bad.any(), line


# ---------------------------------------------------------------------------------------------- 7. engine wiring
@pytest.mark.parametrize("P,N", [(8, 3000), (8, 16384), (15, 3000), (15, 16384), (32, 3000), (32, 16384)])
def test_engine_hands_the_tail_its_own_buffers(P, N):
    """One native step with beta1 = 0 and no weight decay: the engine's m_* are the gradients of its own gW/gR/gtr/ysoft
    buffers, its tau and its parameters from before the step -- a wrong buffer, tau or parameter fails the bound."""
    from reart_b200.engine import RelaxationEngine, tau_schedule
    T = 64 if (P, N) == (15, 16384) else 6
    seq = synthetic_sequence(T, N, P, seed=5)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    eng = RelaxationEngine(cu(seq["cano"]), cu(seq["frames"]), num_parts=P, use_graph=False, seed=2, native=True,
                           betas=(0.0, 0.999), weight_decay=0.0)
    m = eng.model
    conv0, conv2 = m.seg_head.model[0], m.seg_head.model[2]
    H = conv0.weight.shape[0]
    w0, b0, w2, d6 = (f64(q) for q in (conv0.weight.reshape(H, 3), conv0.bias, conv2.weight.reshape(P, H), m.proposal_6d))
    eng.step(tau_schedule(0, 100, 5.0, 1.0))
    torch.cuda.synchronize()
    b = eng._nat
    ref = seg_reference(eng.cano, w0, b0, w2, b["ysoft"], b["gW"], eng.tau.reshape(1))
    seg = worst(b["m_seg"], ref["grad"], tail_bound(ref, N, P))
    gd6, bd6 = pose_reference(d6, b["gR"])
    pose = worst(b["m_d6"], gd6, bd6)
    line = report(f"engine P={P} N={N} T={T}", seg=seg, pose=pose)
    assert torch.equal(b["m_tr"].reshape(-1), b["gtr"].reshape(-1)), line
    assert seg < 1 and pose < 1, line


# ---------------------------------------------------------------------------------------------- 8. smem opt-in
# Each size below is launched in a fresh child process so that the per-process, per-device opt-in state starts clean.
# The sequences run different kernel instantiations (tail <32>, tail <16>, LAP with 256 / 512 / 1024 threads), so they
# share a child without touching each other's state; every sequence starts with its smaller size.
OPT_IN_ORDERS = [("tail", 20, 96), ("tail", 20, 128), ("tail", 20, 256), ("tail", 12, 160), ("tail", 12, 256),
                 ("lap", 700), ("lap", 1024), ("lap", 1100), ("lap", 2048), ("lap", 2100), ("lap", 4096)]
OPT_IN_ALONE = [[("tail", 20, 128), ("tail", 12, 256), ("lap", 1024), ("lap", 2048), ("lap", 4096)], [("tail", 20, 256)]]


def _child_run(items, out_path):
    """In the child: run `items` in order, save every result to out_path (npz)."""
    from reart_b200.assign import lap_assign
    out = {}
    for it in items:
        if it[0] == "tail":
            _, P, H = it
            tail = Tail(tail_inputs(1500, H, P, 5, seed=H * 100 + P))
            tail.run(beta1=0.9, wd=1e-3)
            for k, v in tail.state().items():
                out[f"tail{P}_{H}_{k}"] = v.cpu().numpy()
        else:
            n = it[1]
            src, tgt = lap_inputs(n)
            cols, total = lap_assign(torch.from_numpy(src).to(dev()), torch.from_numpy(tgt).to(dev()), want_total=True)
            out[f"lap{n}_cols"], out[f"lap{n}_total"] = cols.cpu().numpy(), total.cpu().numpy()
    torch.cuda.synchronize()
    np.savez(out_path, **out)


def lap_inputs(n):
    rng = np.random.default_rng(500 + n)
    src = (rng.random((1, n, 3)) * 0.7 - 0.35).astype(np.float32)
    tgt = (src[:, rng.permutation(n)] + rng.normal(0, 0.02, (1, n, 3))).astype(np.float32)
    return src, tgt


def _spawn(items, path):
    code = ("import sys; sys.path[:0] = [sys.argv[1], sys.argv[2]]; import json, test_relax_native_gpu as t; "
            "t._child_run([tuple(i) for i in json.loads(sys.argv[3])], sys.argv[4])")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code, ROOT, os.path.join(ROOT, "tests"),
                                                                          json.dumps(items), str(path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, f"child {items} failed:\n{r.stderr[-4000:]}"
    return dict(np.load(path))


def test_shared_memory_opt_in_covers_every_size_of_an_instantiation(tmp_path):
    """A later call with a larger shared-memory footprint than the first one of its instantiation must launch (the opt-in
    above 48 KB covers the instantiation's largest size) and give the bits of a fresh process, and the LAP's cost must be
    scipy's optimum."""
    from scipy.optimize import linear_sum_assignment
    seq = _spawn(OPT_IN_ORDERS, tmp_path / "orders.npz")
    alone = {}
    for i, items in enumerate(OPT_IN_ALONE):
        alone.update(_spawn(items, tmp_path / f"alone{i}.npz"))
    for k, v in alone.items():
        assert np.array_equal(seq[k], v), k
    for n in (1024, 2048, 4096):
        src, tgt = lap_inputs(n)
        cols = seq[f"lap{n}_cols"][0]
        assert sorted(cols.tolist()) == list(range(n))
        d = src[0][:, None, :] - tgt[0][None, :, :]
        c = np.sqrt((d * d).sum(-1, dtype=np.float32)).astype(np.float64)
        r, col = linear_sum_assignment(c)
        np.testing.assert_allclose(seq[f"lap{n}_total"][0], c[r, col].sum(), rtol=1e-6, atol=1e-9)
