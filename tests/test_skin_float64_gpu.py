"""The skinning kernels of csrc/skin.cu -- skin_fwd_kernel, skin_fwd_sorted_kernel (1, 2 or 4 frames per CTA),
skin_fwd_sorted8_kernel, and skin_bwd_fused_kernel<8|16|32> with its frame groups and skin_bwd_reduce_kernel -- called
through the C ABI at every launch variant (selection mirrored in test_skin_float64_host.py), against float64 references
built from the very float32 inputs the kernels received.  Also every producer of the x-sorted copy of a cloud (the two
sorted skinning kernels, the fused producer of chamfer_sym.cu, pack_cloud_sorted_kernel of knn1.cu, posed_order_kernel
of order.cu) against one numpy reference of the copy.

Forward: out[t,n] = sum_p W[n,p] (R[t,p] c_n + tr[t,p]).  Every skinning kernel computes one axis as common.cuh skin_axis
(a product, two fmas, an add) and accumulates the non-zero weights with one fma each, so element-wise
    |got - ref| <= C u (nnz + 3) sum_p |W[n,p]| (|c_x m0| + |c_y m1| + |c_z m2| + |t|),   u = 2^-24, C = 2
(skin_axis rounds the c_y m1 term 4 times, the fma chain adds at most nnz more).  The skinned cloud must be BIT-IDENTICAL
across every producer, and each x-sorted copy bit-equal to sorted_blocks() of the rows that producer was given.

Backward: gW[n,p] = sum_t g[t,n] . (R[t,p] c_n + tr[t,p]); gR[t,p] = sum_n W[n,p] g[t,n] c_n^T; gtr[t,p] = sum_n W[n,p] g[t,n],
from float64 autograd of sum g . skin.  The bounds follow the kernel's association (skin.cu, "backward"):
    gW:   C u (7 + 4 tiles_per_group + 1 + groups) sum_t sum_a |g_a| (|c_x m_a0| + |c_y m_a1| + |c_z m_a2| + |t_a|)
          (7: the 3x4 product and the dot with g; a thread adds 4 frames per tile of its group; two frame halves; the
          groups in order);
    pose: C u (2 + 64 + 1 + ceil(chunks / 8) + 8) sum_n |W g c|   (|W g| for gtr)
          (g c and its fma; 64 points per half; two halves; the chunks of one reduce slice; the 8 slices).
The per-group gW slices in the workspace are checked the same way, and groups that own no tile must hold exact zeros.
Negative controls (the largest term dropped from one gR sum, the largest frame dropped from one gW sum, the largest
non-empty group counted twice) must fail the bound.  Every test prints its worst ratio |got - ref| / bound."""
import math

import numpy as np
import pytest
import torch

from test_skin_float64_host import (BWD_SHAPES, FWD_SHAPES, PRODUCER_M, PRODUCER_SHAPES, RAW_N, bits,
                                    chamfer_sorted_copy_layout, energy_sorted_copy_layout, group_frames, pmax,
                                    skin_bwd_groups, skin_fwd_fpb, skin_fwd_sorted_fpb, sorted_blocks, tiles_per_group)

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
C = 2.0
F64 = torch.float64


def dev():
    return torch.device("cuda")


def lib():
    from reart_b200 import _lib
    return _lib, _lib.lib()


def worst(got, ref, bound):
    """max |got - ref| / bound over the elements (0/0 counts as 0, x/0 as inf)."""
    err = (got.double().reshape(-1) - ref.double().reshape(-1)).abs()
    b = bound.double().reshape(-1)
    r = torch.where(b > 0, err / torch.where(b > 0, b, torch.ones_like(b)), torch.where(err > 0, float("inf"), 0.0))
    return float(r.max()) if r.numel() else 0.0


def report(tag, **ratios):
    line = f"[{tag}] " + "  ".join(f"{k} {v:.3g}" if isinstance(v, float) else f"{k} {v}" for k, v in ratios.items())
    print(line)
    return line


def nan_like(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), dtype=dtype, device=dev())


# ------------------------------------------------------------------------------------------------ inputs
def make_inputs(T, N, P, weights, scale=1.0, seed=0):
    """float32 cano [N,3], W [N,P], R [T,P,3,3], tr [T,P,3] on the GPU, and the hard part of every row (one-hot classes)."""
    g = torch.Generator().manual_seed(1000 * seed + 17 * T + N + P)
    part = torch.randint(0, P, (N,), generator=g)
    if weights == "lattice":
        cano = torch.randint(-6, 7, (N, 3), generator=g).float()
        perm = torch.stack([torch.randperm(3, generator=g) for _ in range(T * P)])
        sign = torch.randint(0, 2, (T * P, 3), generator=g).float() * 2 - 1
        R = torch.zeros(T * P, 3, 3)
        R.scatter_(2, perm[:, :, None], sign[:, :, None])
        R = R.view(T, P, 3, 3)
        tr = torch.randint(-3, 4, (T, P, 3), generator=g).float()
        W = torch.zeros(N, P)
        W[torch.arange(N), part] = 1.0
    else:
        cano = (torch.randn(N, 3, generator=g, dtype=F64) * scale).float()
        q, _ = torch.linalg.qr(torch.randn(T, P, 3, 3, generator=g, dtype=F64))
        R = q.float()
        tr = (0.3 * scale * torch.randn(T, P, 3, generator=g, dtype=F64)).float()
        W = torch.zeros(N, P, dtype=F64)
        if weights == "onehot" or (weights == "two" and P == 1):
            k = torch.randint(-3, 4, (N,), generator=g).double()
            W[torch.arange(N), part] = 1.0 + torch.where(k > 0, k * 2.0 ** -23, k * 2.0 ** -24)   # 1 +- a few ulps, exact
        elif weights == "two":
            other = (part + torch.randint(1, P, (N,), generator=g)) % P
            W[torch.arange(N), part] = 0.1 + 0.9 * torch.rand(N, generator=g, dtype=F64)
            W[torch.arange(N), other] = 0.1 + 0.9 * torch.rand(N, generator=g, dtype=F64)
        elif weights == "dense":
            W = torch.softmax(2.0 * torch.randn(N, P, generator=g, dtype=F64), dim=1)
        else:
            assert weights == "sparse"
            W = -0.3 + 1.3 * torch.rand(N, P, generator=g, dtype=F64)
            W[torch.rand(N, P, generator=g) < 0.5] = 0.0
            W[::7] = 0.0                                                       # rows without any weight
        W = W.float()
    to = lambda a: a.contiguous().to(dev())
    return to(cano), to(W), to(R), to(tr), part.to(dev())


def targets(T, M, weights, seed=0):
    g = torch.Generator().manual_seed(7 + seed)
    if weights == "lattice":
        return torch.randint(-7, 8, (T, M, 3), generator=g).float().contiguous().to(dev())
    return (1.5 * torch.randn(T, M, 3, generator=g)).contiguous().to(dev())


def hot_rows(W, part):
    """reart_relax_head's compact one-hot form: (part as int32 bits, weight value) [N,2]"""
    val = W[torch.arange(W.shape[0], device=W.device), part].contiguous()
    return torch.stack([part.int(), val.view(torch.int32)], 1).contiguous().view(torch.float32)


def is_one_hot(W):
    return bool(((W != 0).sum(1) == 1).all())


# ------------------------------------------------------------------------------------------------ float64 references
def transformed64(cano, R, tr):
    """v [T,P,N,3] = R[t,p] c_n + tr[t,p] and its majorant |R||c| + |tr|, float64"""
    c, R, tr = cano.double(), R.double(), tr.double()
    v = torch.einsum("tpab,nb->tpna", R, c) + tr[:, :, None, :]
    av = torch.einsum("tpab,nb->tpna", R.abs(), c.abs()) + tr.abs()[:, :, None, :]
    return v, av


def forward_check(got, cano, W, R, tr):
    """worst ratio of a skinned cloud against the float64 forward and its bound"""
    v, av = transformed64(cano, R, tr)
    W64 = W.double()
    ref = torch.einsum("np,tpna->tna", W64, v)
    nnz = (W != 0).sum(1).double()
    bound = C * U * (nnz[None, :, None] + 3) * torch.einsum("np,tpna->tna", W64.abs(), av)
    return worst(got, ref, bound), ref, bound


def skin_fwd(cano, W, R, tr):
    _lib, L = lib()
    T, P, N = R.shape[0], R.shape[1], cano.shape[0]
    out = nan_like(T, N, 3)
    p = _lib.ptr
    _lib.check(L.reart_skin_fwd(p(cano), p(W), p(R), p(tr), T, N, P, p(out), _lib.stream_ptr()), "reart_skin_fwd")
    torch.cuda.synchronize()
    return out


def skin_bwd(cano, W, R, tr, g, ws_fill=None):
    """reart_skin_bwd -> (gW, gR [T,P,3,3], gtr, workspace); outputs and workspace pre-filled with NaN"""
    _lib, L = lib()
    T, P, N = R.shape[0], R.shape[1], cano.shape[0]
    gW, gR, gtr = nan_like(N, P), nan_like(T, P, 3, 3), nan_like(T, P, 3)
    nbytes = L.reart_skin_bwd_workspace_bytes(T, N, P)
    ws = torch.full((nbytes,), 255, dtype=torch.uint8, device=dev())
    p = _lib.ptr
    _lib.check(L.reart_skin_bwd(p(cano), p(W), p(R), p(tr), p(g), T, N, P, p(gW), p(gR), p(gtr), p(ws), nbytes,
                                _lib.stream_ptr()), "reart_skin_bwd")
    torch.cuda.synchronize()
    return gW, gR, gtr, ws


# ------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("T,N,P,weights,scale", FWD_SHAPES)
def test_skin_fwd_against_float64(T, N, P, weights, scale):
    cano, W, R, tr, _ = make_inputs(T, N, P, weights, scale)
    got = skin_fwd(cano, W, R, tr)
    assert not torch.isnan(got).any()
    r, ref, bound = forward_check(got, cano, W, R, tr)
    report(f"skin_fwd T={T} N={N} P={P} {weights} x{scale:g} fpb={skin_fwd_fpb(T, N)}", worst=r)
    assert r <= 1.0
    # negative control: the largest weighted term of one row left out must fail the bound
    v, _ = transformed64(cano, R, tr)
    terms = W.double().t()[None, :, :, None] * v                                  # [T,P,N,3]
    k = int(terms.abs().reshape(-1).argmax())
    t, p, n, a = np.unravel_index(k, tuple(terms.shape))
    bad = got.double().clone()
    bad[t, n, a] -= terms[t, p, n, a]
    assert worst(bad, ref, bound) > 1.0


# ------------------------------------------------------------------------------------------------ the producers
def workspace(nbytes):
    return torch.full((nbytes,), 255, dtype=torch.uint8, device=dev())


def read_sorted_copy(ws, lay, T):
    """(packed, perm, xq) of the x-sorted copy out of a workspace, at the offsets of `lay`"""
    n_pad = lay["n_pad"]
    nblk = n_pad // 256
    host = ws[:lay["end"]].cpu().numpy()
    packed = host[lay["psrc"]:lay["psrc"] + T * n_pad * 12].view(np.float32).reshape(T, n_pad * 3)
    perm = host[lay["perm"]:lay["perm"] + T * n_pad].reshape(T, n_pad)
    xq = host[lay["xq"]:lay["xq"] + T * nblk * 64].view(np.float32).reshape(T, nblk, 16)
    return packed, perm, xq


def assert_sorted_copy(ws, lay, rows, what):
    T = rows.shape[0]
    got = read_sorted_copy(ws, lay, T)
    want = sorted_blocks(rows, lay["n_pad"])
    for name, a, b in zip(("packed", "perm", "xq"), got, want):
        if a.dtype == np.float32:
            assert np.array_equal(bits(a), bits(b)), (what, name)
        else:
            assert np.array_equal(a, b), (what, name)


def energy_outputs(T, N, M, P):
    return dict(skinned=nan_like(T, N, 3), loss=nan_like(1, dtype=F64), gW=nan_like(N, P), gR=nan_like(T, P, 3, 3),
                gtr=nan_like(T, P, 3), gs=nan_like(T, N, 3), d_f=nan_like(T, N), i_f=torch.full((T, N), -1, dtype=torch.int64, device=dev()),
                d_b=nan_like(T, M), i_b=torch.full((T, M), -1, dtype=torch.int64, device=dev()))


def run_energy(kind, cano, W, R, tr, tgt, part=None):
    """One energy evaluation through the C ABI: kind = brute | ordered | posed | fused -> (outputs, workspace, row order
    [T,N] of the rows the search copy was built from)"""
    from reart_b200 import ops
    _lib, L = lib()
    p = _lib.ptr
    T, P, N, M = R.shape[0], R.shape[1], cano.shape[0], tgt.shape[1]
    o = energy_outputs(T, N, M, P)
    nbytes = L.reart_energy_workspace_bytes(T, N, M)
    ws = workspace(nbytes)
    st = _lib.stream_ptr()
    head = (p(o["skinned"]), p(o["loss"]), p(o["gW"]), p(o["gR"]), p(o["gtr"]), p(o["gs"]), 1)
    rows = torch.arange(N, device=dev())[None].repeat(T, 1)
    if kind in ("brute", "fused"):
        packed = ops.pack_cloud(tgt)
        if kind == "brute":
            rc = L.reart_skinned_chamfer_fwd_bwd(p(cano), p(W), p(R), p(tr), p(tgt), p(packed), T, N, M, P, *head,
                                                 p(ws), nbytes, st)
        else:
            hot = hot_rows(W, part)
            rc = L.reart_skinned_chamfer_fwd_bwd_fused(p(cano), p(hot), p(W), p(R), p(tr), p(tgt), p(packed), T, N, M, P,
                                                       *head, p(ws), nbytes, st)
    else:
        to = ops.search_order(tgt, 32).int().contiguous()
        ti = torch.empty_like(to)
        ti.scatter_(1, to.long(), torch.arange(M, dtype=torch.int32, device=dev())[None].expand(T, M).contiguous())
        fs = torch.gather(tgt, 1, to.long()[:, :, None].expand(-1, -1, 3)).contiguous()
        fsp = ops.pack_cloud(fs)
        nn = (torch.full((T, N), -1, dtype=torch.int32, device=dev()), torch.full((T, M), -1, dtype=torch.int32, device=dev()),
              torch.zeros(3, dtype=torch.int64, device=dev()))
        tail = (p(o["d_f"]), p(o["i_f"]), p(o["d_b"]), p(o["i_b"]), p(nn[0]), p(nn[1]), p(nn[2]), p(ws), nbytes, st)
        if kind == "ordered":
            ro = ops.search_order(cano[None], 256)[0].int().contiguous()           # the engine's row order
            ri = torch.empty_like(ro)
            ri[ro.long()] = torch.arange(N, dtype=torch.int32, device=dev())
            rc = L.reart_skinned_chamfer_fwd_bwd_ordered(p(cano), p(W), p(R), p(tr), p(tgt), p(fs), p(fsp), T, N, M, P,
                                                         p(ro), p(ri), p(to), p(ti), *head, *tail)
            rows = ro.long()[None].repeat(T, 1)
        else:
            assert kind == "posed"
            ro = torch.full((T, N), -1, dtype=torch.int32, device=dev())
            ri = torch.full((T, N), -1, dtype=torch.int32, device=dev())
            rc = L.reart_skinned_chamfer_fwd_bwd_posed(p(cano), p(W), p(R), p(tr), p(tgt), p(fs), p(fsp), T, N, M, P,
                                                       p(to), p(ti), p(ro), p(ri), *head, *tail)
            rows = ro.long()
    torch.cuda.synchronize()
    _lib.check(rc, f"energy ({kind})")
    return o, ws, rows


@pytest.mark.parametrize("T,N,P,weights", PRODUCER_SHAPES)
def test_every_producer_gives_the_same_cloud_and_the_reference_sorted_copy(T, N, P, weights):
    """reart_skin_fwd is checked against float64; the energy entries (brute, ordered, posed, fused) must return that very
    cloud, an x-sorted copy bit-equal to sorted_blocks() of the rows they were given, and the gradients reart_skin_bwd
    computes from the g_skinned the same call returned."""
    _, L = lib()
    cano, W, R, tr, part = make_inputs(T, N, P, weights)
    tgt = targets(T, PRODUCER_M, weights)
    ref = skin_fwd(cano, W, R, tr)
    r, _, _ = forward_check(ref, cano, W, R, tr)
    assert r <= 1.0
    ref_np = ref.cpu().numpy()
    if weights == "lattice" and N > 1:                                         # the ties the copy has to order by offset
        x = np.concatenate([ref_np[:, :, 0], np.full((T, -N % 256), np.inf, np.float32)], 1).reshape(T, -1, 256)
        assert any(len(np.unique(b[np.isfinite(b)])) < np.isfinite(b).sum() for b in x.reshape(-1, 256))
    kinds = ["brute", "ordered"]
    if N <= L.reart_posed_order_max_points():
        kinds.append("posed")
    if is_one_hot(W):
        kinds.append("fused")
    lay = energy_sorted_copy_layout(T, N, PRODUCER_M)
    for kind in kinds:
        o, ws, rows = run_energy(kind, cano, W, R, tr, tgt, part)
        assert torch.equal(o["skinned"], ref), kind
        rows_np = rows.cpu().numpy()
        assert all(np.array_equal(np.sort(rows_np[t]), np.arange(N)) for t in range(T)), kind
        assert_sorted_copy(ws, lay, np.take_along_axis(ref_np, rows_np[:, :, None], 1), kind)
        gW, gR, gtr, _ = skin_bwd(cano, W, R, tr, o["gs"])
        assert not torch.isnan(o["gs"]).any(), kind
        assert torch.equal(o["gW"], gW) and torch.equal(o["gR"], gR) and torch.equal(o["gtr"], gtr), kind
    report(f"producers T={T} N={N} P={P} {weights} sorted fpb={skin_fwd_sorted_fpb(T, N)}", worst=r,
           bit_identical="+".join(kinds))


@pytest.mark.parametrize("N", RAW_N)
def test_pack_cloud_sorted_gives_the_reference_sorted_copy(N):
    """pack_cloud_sorted_kernel (reart_chamfer_bidir_fwd's copy of src): raw rows with -0.0 and +0.0 x values and exact
    ties in every block, -0.0 before +0.0."""
    _lib, L = lib()
    B, M = 2, 300
    rng = np.random.default_rng(N)
    src = rng.integers(-2, 3, (B, N, 3)).astype(np.float32)
    x = src[:, :, 0]                                                             # a view: writes land in src
    x[(x == 0) & (rng.random((B, N)) < 0.5)] = np.float32(-0.0)
    for s in range(0, N, 256):                                                   # +0.0 at a LOWER offset than two -0.0
        x[:, s] = np.float32(0.0) if s + 1 < N else np.float32(-0.0)
        x[:, s + 1:s + 3] = np.float32(-0.0)
    sb = bits(x)
    for b in range(B):
        for s in range(0, N, 256):
            blk = sb[b, s:s + 256]
            assert (blk == 0x80000000).any()                                     # -0.0 in every block
            if len(blk) >= 3:
                assert (blk == 0).any() and len(np.unique(blk)) < len(blk)     # +0.0 and exact ties
    tgt = rng.standard_normal((B, M, 3)).astype(np.float32)
    s_t, t_t = torch.from_numpy(src).to(dev()), torch.from_numpy(tgt).to(dev())
    nbytes = L.reart_chamfer_workspace_bytes(B, N, M)
    ws = workspace(nbytes)
    out = [nan_like(B, N), torch.empty(B, N, dtype=torch.int64, device=dev()), nan_like(B, M),
           torch.empty(B, M, dtype=torch.int64, device=dev())]
    p = _lib.ptr
    _lib.check(L.reart_chamfer_bidir_fwd(p(s_t), p(t_t), B, N, M, *[p(t) for t in out], p(ws), nbytes, _lib.stream_ptr()),
               "reart_chamfer_bidir_fwd")
    torch.cuda.synchronize()
    assert_sorted_copy(ws, chamfer_sorted_copy_layout(B, N, M), src, "pack_cloud_sorted")
    report(f"pack_cloud_sorted N={N}", bit_identical="yes")


# ------------------------------------------------------------------------------------------------ backward
def backward_reference(cano, W, R, tr, g):
    """float64 autograd of sum g . skin, and the majorants the bounds scale"""
    c = cano.double()
    W64 = W.double().requires_grad_(True)
    R64 = R.double().requires_grad_(True)
    t64 = tr.double().requires_grad_(True)
    g64 = g.double()
    v = torch.einsum("tpab,nb->tpna", R64, c) + t64[:, :, None, :]
    (torch.einsum("np,tpna->tna", W64, v) * g64).sum().backward()
    _, av = transformed64(cano, R, tr)
    absW, absg = W.double().abs(), g64.abs()
    return dict(gW=W64.grad, gR=R64.grad, gtr=t64.grad, v=v.detach(),
                SW_t=torch.einsum("tna,tpna->tnp", absg, av),                     # per-frame gW majorant [T,N,P]
                SR=torch.einsum("np,tna,nb->tpab", absW, absg, c.abs()),
                St=torch.einsum("np,tna->tpa", absW, absg))


def depths(T, N):
    groups, tpg = skin_bwd_groups(T, N), tiles_per_group(T, N)
    chunks = math.ceil(N / 128)
    return 7 + 4 * tpg + 1 + groups, 2 + 64 + 1 + math.ceil(chunks / 8) + 8, 7 + 4 * tpg + 1


@pytest.mark.parametrize("T,N,P,weights,scale", BWD_SHAPES)
def test_skin_bwd_against_float64(T, N, P, weights, scale):
    cano, W, R, tr, _ = make_inputs(T, N, P, weights, scale, seed=1)
    g = torch.randn(T, N, 3, generator=torch.Generator().manual_seed(T + N)).contiguous().to(dev())
    gW, gR, gtr, ws = skin_bwd(cano, W, R, tr, g)
    for t in (gW, gR, gtr):
        assert not torch.isnan(t).any()
    ref = backward_reference(cano, W, R, tr, g)
    dW, dP, dG = depths(T, N)
    bW = C * U * dW * ref["SW_t"].sum(0)
    bR, bt = C * U * dP * ref["SR"], C * U * dP * ref["St"]
    rW, rR, rt = worst(gW, ref["gW"], bW), worst(gR, ref["gR"], bR), worst(gtr, ref["gtr"], bt)

    # the per-group gW slices [groups][N][P] behind the pose partials in the workspace (skin.cu launch_skin_bwd_p)
    groups = skin_bwd_groups(T, N)
    chunks = math.ceil(N / 128)
    rG, terms_W = 0.0, None
    terms_W = torch.einsum("tna,tpna->tnp", g.double(), ref["v"])                    # [T,N,P] signed frame terms
    part_ref = []
    if groups > 1:
        parts = ws[:groups * N * P * 4 + chunks * T * 12 * P * 4].view(torch.float32)[chunks * T * 12 * P:]
        parts = parts.view(groups, N, P)
        for q in range(groups):
            lo, hi = group_frames(T, N, q)
            if lo == hi:
                assert torch.equal(parts[q], torch.zeros_like(parts[q])), q          # a group without tiles adds exact zeros
                part_ref.append(torch.zeros(N, P, dtype=F64, device=dev()))
                continue
            pr = terms_W[lo:hi].sum(0)
            part_ref.append(pr)
            rG = max(rG, worst(parts[q], pr, C * U * dG * ref["SW_t"][lo:hi].sum(0)))
    report(f"skin_bwd T={T} N={N} P={P} {weights} x{scale:g} PMAX={pmax(P)} groups={groups} tpg={tiles_per_group(T, N)}",
           gW=rW, gR=rR, gtr=rt, group_slices=rG)
    assert max(rW, rR, rt, rG) <= 1.0

    # bit-identical on a second call
    gW2, gR2, gtr2, _ = skin_bwd(cano, W, R, tr, g)
    assert torch.equal(gW, gW2) and torch.equal(gR, gR2) and torch.equal(gtr, gtr2)

    # negative controls
    # (1) the largest term W[n,p] g[t,n,a] c[n,b] dropped from its gR sum
    c64, g64, W64 = cano.double(), g.double(), W.double()
    gc = g64[:, :, :, None] * c64[None, :, None, :]                                # [T,N,3,3]
    best, arg = -1.0, None
    for p in range(P):
        m = (W64[:, p][None, :, None, None] * gc).abs()
        k = int(m.reshape(-1).argmax())
        if float(m.reshape(-1)[k]) > best:
            best, arg = float(m.reshape(-1)[k]), (p,) + tuple(int(i) for i in np.unravel_index(k, tuple(m.shape)))
    p, t, n, a, b = arg
    bad = gR.double().clone()
    bad[t, p, a, b] -= W64[n, p] * gc[t, n, a, b]
    assert worst(bad, ref["gR"], bR) > 1.0
    # (2) the largest frame term dropped from its gW sum
    t, n, p = np.unravel_index(int(terms_W.abs().reshape(-1).argmax()), tuple(terms_W.shape))
    bad = gW.double().clone()
    bad[n, p] -= terms_W[t, n, p]
    assert worst(bad, ref["gW"], bW) > 1.0
    # (3) the largest non-empty frame group counted twice
    if groups > 1:
        pr = torch.stack(part_ref)
        q, n, p = np.unravel_index(int(pr.abs().reshape(-1).argmax()), tuple(pr.shape))
        assert group_frames(T, N, q) != (0, 0)
        bad = gW.double().clone()
        bad[n, p] += pr[q, n, p]
        assert worst(bad, ref["gW"], bW) > 1.0


def test_skin_bwd_empty_sides_and_unsupported_parts():
    _lib, L = lib()
    p = _lib.ptr
    st = _lib.stream_ptr()
    T, N, P = 3, 10, 5
    ws = workspace(L.reart_skin_bwd_workspace_bytes(T, N, P))
    # no points: the pose gradients are zero
    gR, gtr = nan_like(T, P, 3, 3), nan_like(T, P, 3)
    assert L.reart_skin_bwd(None, None, None, None, None, T, 0, P, None, p(gR), p(gtr), p(ws), ws.numel(), st) == 0
    # no frames: the weight gradient is zero
    gW = nan_like(N, P)
    assert L.reart_skin_bwd(None, None, None, None, None, 0, N, P, p(gW), None, None, p(ws), ws.numel(), st) == 0
    torch.cuda.synchronize()
    for t in (gR, gtr, gW):
        assert torch.equal(t, torch.zeros_like(t))
    # 33 parts: no instantiation
    cano, W, R, tr, _ = make_inputs(2, N, 33, "dense")
    g = torch.randn(2, N, 3, device=dev())
    nb = L.reart_skin_bwd_workspace_bytes(2, N, 33)
    ws = workspace(nb)
    outs = nan_like(N, 33), nan_like(2, 33, 9), nan_like(2, 33, 3)
    assert L.reart_skin_bwd(p(cano), p(W), p(R), p(tr), p(g), 2, N, 33, *[p(t) for t in outs], p(ws), nb, st) == -4
    report("skin_bwd empty sides", zero_filled="yes", P33="REART_ERR_UNSUPPORTED")
