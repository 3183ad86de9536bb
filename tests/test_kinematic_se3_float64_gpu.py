"""The SE(3) kernels of the kinematic fit -- reart_rot6d_*, reart_screw_to_transform_*, reart_fk_fwd / _bwd and the fused
kinematic head / tail (csrc/se3.cu, csrc/kin.cu over csrc/se3_device.cuh) -- called through the C ABI, against float64
references built from the very float32 inputs the kernels received.

The float64 reference restates the reference's screw map with its quirks (se3.cu header): the no-rot branch
(|theta| < 1e-6 or |theta - pi| < 1e-6: w = 0, v = l theta, d ignored), h = d / theta, |l theta|^2 clamped at 1e-4 before
the square root with a zero gradient below the clamp, axes never normalised; the 6D map with F.normalize's eps 1e-12; the
tree walk in `order`; and the joint inputs of fk_joint_inputs (revolute: d := 1e-6f, prismatic: theta := 1e-6f, type 0
or no joint types: both as given, d = 1e-6f without distances).  Gradients are float64 autograd of
sum gR.R + sum gtr.tr -- not the kernels' forward-mode dual numbers.  The branch decisions are made in float32 as the
kernels make them: 1e-6f < 1e-6 holds in float64 but not in float32, so a float64 predicate would send every prismatic
joint down the no-rot branch.  The clamp is decided on the float64 |l theta|^2, and every generated input keeps it at
least 1e-3 relative away from 1e-4 (asserted), so that float32 decides the same way.

Bounds are element-wise: |got - ref| <= C u S with u = 2^-24 and S a running-error majorant from a second float64 pass
(class Run) that replays the kernels' own operation sequence (the dual-number screw and 6D maps, the 3x4 products, the
leaves-first fold, the frame sums in frame order) and gives every rounded result z the term
sum_i |dz/dx_i| S(x_i) + |z| (4 |z| for sinf / cosf, which are within 2 ulp).  Each rounding thus adds one absolute
term, so the (k + depth) of a sum-of-products bound lives inside S, and the ill-conditioned spots -- the theta
derivative of h = d / theta near small theta, 1 - cos and ang - sin near the clamp, a nearly parallel second 6D column,
chains of 31 joints -- get exactly the slack their cancellations need.  fk_bwd adds over frames with float atomics in
any order: its axis / moment bound adds (T - 1) sum_t |term_t|.
C = 2 covers the first-order analysis and the 2-ulp sinf / cosf; every test prints its worst ratio |got - ref| / bound.
The same Run pass also yields a second float64 value, asserted to agree with autograd far inside the bound, so a slip in
the mirrored sequence cannot inflate S unnoticed.  Negative controls (a frame left out of the axis / moment frame sum, one
leaf's fold into its parent skipped in one frame, the root-pose chain rule dropped for one part) must fail the bound."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
C = 2.0
F64 = torch.float64
EPS_F = float(np.float32(1e-6))                  # the kernels' 1e-6f: the no-rot window and the fixed joint input
PI_F = float(np.float32(np.pi))
CLAMP_F = float(np.float32(1e-4))


def dev():
    return torch.device("cuda")


def lib():
    from reart_b200 import _lib
    return _lib, _lib.lib()


def worst(got, ref, bound):
    """max |got - ref| / bound over the elements (0/0 counts as 0, x/0 as inf)."""
    err = (got.double().cpu().reshape(-1) - ref.double().cpu().reshape(-1)).abs()
    b = bound.double().cpu().reshape(-1)
    r = torch.where(b > 0, err / torch.where(b > 0, b, torch.ones_like(b)), torch.where(err > 0, float("inf"), 0.0))
    return float(r.max()) if r.numel() else 0.0


def report(tag, **ratios):
    line = f"[{tag}] " + "  ".join(f"{k} {v:.3g}" for k, v in ratios.items())
    print(line)
    return line


# ------------------------------------------------------------------------------------------------ branch decisions
def no_rot32(theta32):
    """The kernels' strict no-rot predicate, evaluated on the float32 angles with pi rounded to float32."""
    th = theta32.detach().float().cpu()
    eps, pi = torch.tensor(EPS_F, dtype=torch.float32), torch.tensor(PI_F, dtype=torch.float32)
    return (th.abs() < eps) | ((th - pi).abs() < eps)


def clamp_margin(l, theta, norot):
    """min |(|l theta|^2) / 1e-4f - 1| over the rotating elements (l [B,3], theta [B], float64)."""
    nrm = (l * theta[:, None]).pow(2).sum(-1)
    rel = (nrm / CLAMP_F - 1.0).abs()
    rel = rel[~norot]
    return float(rel.min()) if rel.numel() else float("inf")


# ------------------------------------------------------------------------------------------------ float64 reference
def skew(w):
    z = torch.zeros_like(w[..., 0])
    return torch.stack([torch.stack([z, -w[..., 2], w[..., 1]], -1), torch.stack([w[..., 2], z, -w[..., 0]], -1),
                        torch.stack([-w[..., 1], w[..., 0], z], -1)], -2)


def screw64(l, m, th, d, norot):
    """l, m [B,3], th, d [B] (float64), norot [B] (decided in float32) -> [B,3,4]"""
    ths = torch.where(norot, torch.ones_like(th), th)              # keeps the unused branch finite at theta = 0
    q = torch.cross(l, m, dim=-1)
    c = torch.cross(q, l, dim=-1)
    h = d / ths
    w = torch.where(norot[:, None], torch.zeros_like(l), l * th[:, None])
    v = torch.where(norot[:, None], l * th[:, None], (c + h[:, None] * l) * th[:, None])
    nrm = (w * w).sum(-1)
    ang = torch.where(nrm >= CLAMP_F, nrm, torch.full_like(nrm, CLAMP_F)).sqrt()
    sn, cs = ang.sin(), ang.cos()
    K = skew(w)
    K2 = K @ K
    eye = torch.eye(3, dtype=F64).expand_as(K)
    f = lambda x: x[:, None, None]
    Rm = f(sn / ang) * K + f((1 - cs) / ang ** 2) * K2 + eye
    V = eye + K * f((1 - cs) / ang ** 2) + K2 * f((ang - sn) / ang ** 3)
    return torch.cat([Rm, (V @ v[..., None])], -1)


def rot6d64(d6):
    """rows b1, b2, b1 x b2 of the Gram-Schmidt of rotation_6d_to_matrix (F.normalize: x / max(|x|, 1e-12))."""
    a1, a2 = d6[..., :3], d6[..., 3:]
    b1 = a1 / a1.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    u = a2 - (b1 * a2).sum(-1, keepdim=True) * b1
    b2 = u / u.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    return torch.stack([b1, b2, torch.cross(b1, b2, dim=-1)], dim=-2)


def mat34(A, B):
    return torch.cat([A[..., :3] @ B[..., :3], A[..., :3] @ B[..., 3:] + A[..., 3:]], -1)


def f64(t):
    return t.detach().double().cpu()


# ------------------------------------------------------------------------------------------------ running-error pass
class Run:
    """A float64 value v with S (s): u * s majorises the rounding error of the same sequence of float32 operations.
    Forward-mode dual parts d [B,K] carry their own S (ds), mirroring the kernels' Dual<K>."""
    __slots__ = ("v", "s", "d", "ds")

    def __init__(self, v, s, d, ds):
        self.v, self.s, self.d, self.ds = v, s, d, ds

    @staticmethod
    def exact(v, K=0, k=None):
        d = torch.zeros(*v.shape, K, dtype=F64)
        if k is not None:
            d[..., k] = 1.0
        return Run(v, torch.zeros_like(v), d, torch.zeros_like(d))

    def const(self, c):
        return Run(torch.full_like(self.v, c), torch.zeros_like(self.v), torch.zeros_like(self.d), torch.zeros_like(self.d))

    def plain(self):
        """the value as a dual-free Run"""
        e = torch.zeros(*self.v.shape, 0, dtype=F64)
        return Run(self.v, self.s, e, e)

    def part(self, k):
        """dual component k as a dual-free Run"""
        e = torch.zeros(*self.v.shape, 0, dtype=F64)
        return Run(self.d[..., k], self.ds[..., k], e, e)

    def __add__(a, b):
        v, d = a.v + b.v, a.d + b.d
        return Run(v, a.s + b.s + v.abs(), d, a.ds + b.ds + d.abs())

    def __sub__(a, b):
        v, d = a.v - b.v, a.d - b.d
        return Run(v, a.s + b.s + v.abs(), d, a.ds + b.ds + d.abs())

    def __neg__(a):
        return Run(-a.v, a.s, -a.d, a.ds)

    def __mul__(a, b):
        v = a.v * b.v
        av, bv, as_, bs = a.v[..., None], b.v[..., None], a.s[..., None], b.s[..., None]
        p1, p2 = a.d * bv, av * b.d
        ds = bv.abs() * a.ds + a.d.abs() * bs + av.abs() * b.ds + b.d.abs() * as_ + p1.abs() + p2.abs() + (p1 + p2).abs()
        return Run(v, b.v.abs() * a.s + a.v.abs() * b.s + v.abs(), p1 + p2, ds)

    def __truediv__(a, b):
        # r.v = a.v / b.v; inv = 1 / b.v; r.d = (a.d - r.v * b.d) * inv
        r = a.v / b.v
        sr = a.s / b.v.abs() + a.v.abs() * b.s / b.v ** 2 + r.abs()
        inv = 1.0 / b.v
        sinv = b.s / b.v ** 2 + inv.abs()
        rv, srv, iv, siv = r[..., None], sr[..., None], inv[..., None], sinv[..., None]
        t = rv * b.d
        st = b.d.abs() * srv + rv.abs() * b.ds + t.abs()
        w = a.d - t
        sw = a.ds + st + w.abs()
        d = w * iv
        return Run(r, sr, d, iv.abs() * sw + w.abs() * siv + d.abs())

    def sin(a):
        v, c = a.v.sin(), a.v.cos()
        sc = v.abs() * a.s + 4 * c.abs()
        d = c[..., None] * a.d
        return Run(v, c.abs() * a.s + 4 * v.abs(), d, c.abs()[..., None] * a.ds + a.d.abs() * sc[..., None] + d.abs())

    def cos(a):
        v, sn = a.v.cos(), -a.v.sin()
        ss = v.abs() * a.s + 4 * sn.abs()
        d = sn[..., None] * a.d
        return Run(v, sn.abs() * a.s + 4 * v.abs(), d, sn.abs()[..., None] * a.ds + a.d.abs() * ss[..., None] + d.abs())

    def sqrt(a):
        v = a.v.sqrt()
        s = a.s / (2 * v) + v.abs()
        k = 0.5 / v
        sk = k.abs() * (s / v.abs() + 1.0)
        d = k[..., None] * a.d
        return Run(v, s, d, k.abs()[..., None] * a.ds + a.d.abs() * sk[..., None] + d.abs())

    def clamp_min(a, lo, keep):
        """torch.clamp(min=lo) with the decision `keep` (a >= lo) given: the gradient is zero below."""
        c = a.const(lo)
        return select(keep, a, c)


def select(mask, a, b):
    m = mask[..., None]
    return Run(torch.where(mask, a.v, b.v), torch.where(mask, a.s, b.s), torch.where(m, a.d, b.d), torch.where(m, a.ds, b.ds))


def screw_run(l, m, th, d, norot):
    """screw_eval of se3_device.cuh, operation for operation, on Run (l, m: 3 Runs, th, d: Runs) -> 12 Runs"""
    one, zero = th.const(1.0), th.const(0.0)
    q = [l[1] * m[2] - l[2] * m[1], l[2] * m[0] - l[0] * m[2], l[0] * m[1] - l[1] * m[0]]
    ths = select(norot, one, th)
    h = d / ths
    c = [q[1] * l[2] - q[2] * l[1], q[2] * l[0] - q[0] * l[2], q[0] * l[1] - q[1] * l[0]]
    w = [select(norot, zero * th, l[k] * th) for k in range(3)]
    v = [select(norot, l[k] * th, (c[k] + h * l[k]) * th) for k in range(3)]
    nrm = w[0] * w[0] + w[1] * w[1] + w[2] * w[2]
    ang = nrm.clamp_min(CLAMP_F, nrm.v >= CLAMP_F).sqrt()
    inv = one / ang
    sn, cs = ang.sin(), ang.cos()
    fac1 = inv * sn
    fac2 = inv * inv * (one - cs)
    facV1 = (one - cs) / (ang * ang)
    facV2 = (ang - sn) / (ang * ang * ang)
    K = [zero, -w[2], w[1], w[2], zero, -w[0], -w[1], w[0], zero]
    K2 = [K[3 * i] * K[j] + K[3 * i + 1] * K[3 + j] + K[3 * i + 2] * K[6 + j] for i in range(3) for j in range(3)]
    M = [None] * 12
    for i in range(3):
        Vr = []
        for j in range(3):
            I = one if i == j else zero
            M[4 * i + j] = fac1 * K[3 * i + j] + fac2 * K2[3 * i + j] + I
            Vr.append(I + K[3 * i + j] * facV1 + K2[3 * i + j] * facV2)
        M[4 * i + 3] = Vr[0] * v[0] + Vr[1] * v[1] + Vr[2] * v[2]
    return M


def normalize_run(v):
    n = (v[0] * v[0] + v[1] * v[1] + v[2] * v[2]).sqrt()
    den = n.clamp_min(1e-12, n.v >= 1e-12)
    return [v[0] / den, v[1] / den, v[2] / den]


def rot6d_run(d6):
    """rot6d_eval of se3_device.cuh on Run (6 Runs) -> 9 Runs"""
    b1 = normalize_run(d6[:3])
    dot = b1[0] * d6[3] + b1[1] * d6[4] + b1[2] * d6[5]
    b2 = normalize_run([d6[3 + k] - dot * b1[k] for k in range(3)])
    return b1 + b2 + [b1[1] * b2[2] - b1[2] * b2[1], b1[2] * b2[0] - b1[0] * b2[2], b1[0] * b2[1] - b1[1] * b2[0]]


def mat34_run(A, B):
    out = []
    for i in range(3):
        for j in range(4):
            s = A[4 * i] * B[j] + A[4 * i + 1] * B[4 + j] + A[4 * i + 2] * B[8 + j]
            out.append(s + A[4 * i + 3] if j == 3 else s)
    return out


def contract(g, outs, k):
    """sum_o g[o] * outs[o].d[k] in o order (the kernels' backward contractions); g exact float32 inputs [B, n]"""
    acc = None
    for o, x in enumerate(outs):
        t = Run.exact(g[:, o]) * x.part(k)
        acc = t if acc is None else acc + t
    return acc


def seq_sum(v, s):
    """sum over dim 0 in index order: (value, S)"""
    acc_v, acc_s = torch.zeros_like(v[0]), torch.zeros_like(s[0])
    for t in range(v.shape[0]):
        acc_v = acc_v + v[t]
        acc_s = acc_s + s[t] + acc_v.abs()
    return acc_v, acc_s


# ------------------------------------------------------------------------------------------------ trees
def _tree_dicts(parent_of, order, edge_of):
    paths = {}
    for c in order:
        p, path = c, [c]
        while parent_of[p] >= 0:
            p = parent_of[p]
            path.append(p)
        paths[c] = path
    return paths, list(order), {f"{c}_{parent_of[c]}": edge_of[c] for c in order if parent_of[c] >= 0}


def tree_spec(name):
    """(paths_to_base, reverse_topo, edge_index) written out by hand for each tree shape."""
    if name == "p1":
        return {0: [0]}, [0], {}
    if name == "p2":
        return {0: [0], 1: [1, 0]}, [0, 1], {"1_0": 0}
    if name == "chain32":                           # depth 31
        return {c: list(range(c, -1, -1)) for c in range(32)}, list(range(32)), {f"{c}_{c - 1}": c - 1 for c in range(1, 32)}
    if name == "star32":
        return {0: [0], **{c: [c, 0] for c in range(1, 32)}}, list(range(32)), {f"{c}_0": c - 1 for c in range(1, 32)}
    if name == "perm17":                            # random tree, part ids permuted, edges numbered independently
        rng = np.random.default_rng(17)
        P = 17
        topo_parent = [-1] + [int(rng.integers(0, k)) for k in range(1, P)]
        ids = rng.permutation(P)
        while ids[0] == 0:
            ids = rng.permutation(P)
        eids = rng.permutation(P - 1)
        parent_of, edge_of = {}, {}
        for k in range(P):
            parent_of[int(ids[k])] = -1 if k == 0 else int(ids[topo_parent[k]])
            if k:
                edge_of[int(ids[k])] = int(eids[k - 1])
        return _tree_dicts(parent_of, [int(i) for i in ids], edge_of)
    raise KeyError(name)


def flat_tree(name, jt_codes):
    from reart_b200.kinematic import FlatTree
    paths, topo, edges = tree_spec(name)
    tree = FlatTree(paths, topo, edges, device=dev())
    if jt_codes is not None:                         # codes set directly: type 0 ("as given") has no joint name
        tree.joint_type = torch.tensor(jt_codes, dtype=torch.int32, device=dev())
    return tree


# ------------------------------------------------------------------------------------------------ inputs
# angles planted at chosen (frame, joint) cells; every one lands in a known branch of the screw map
PLANTED = {
    "zero": 0.0,                                                         # no-rot
    "eps": EPS_F,                                                        # 1e-6f: NOT no-rot (1e-6f < 1e-6f is false)
    "below_eps": float(np.nextafter(np.float32(1e-6), np.float32(0))),    # no-rot
    "pi": PI_F,                                                          # no-rot, d ignored
    "pi+4ulp": float(np.float32(PI_F) + 4 * np.spacing(np.float32(PI_F))),   # 9.5e-7 away: no-rot
    "pi+5ulp": float(np.float32(PI_F) + 5 * np.spacing(np.float32(PI_F))),   # 1.19e-6 away: rotates
    "pi-5ulp": float(np.float32(PI_F) - 5 * np.spacing(np.float32(PI_F))),
    "-pi": -PI_F,                                                        # rotates (a reference quirk)
    "2.5pi": float(np.float32(2.5 * np.pi)),
    "clamp": 0.003,                                                      # |l theta| < 0.01: clamp active
}
PLANTED_NOROT = {"zero": True, "eps": False, "below_eps": True, "pi": True, "pi+4ulp": True, "pi+5ulp": False,
                 "pi-5ulp": False, "-pi": False, "2.5pi": False, "clamp": False}
AXIS_NORMS = (0.3, 1.0, 3.0)


def random_axes(rng, n):
    a = rng.standard_normal((n, 3))
    a /= np.linalg.norm(a, axis=1, keepdims=True)
    return (a * np.array(AXIS_NORMS)[np.arange(n) % 3][:, None]).astype(np.float32)


def keep_off_the_clamp(l, theta, fixed):
    """Nudge the random angles whose |l theta|^2 falls within 1e-3 relative of 1e-4 (fixed: cells left alone)."""
    for _ in range(4):
        nrm = (l.astype(np.float64) ** 2).sum(-1) * theta.astype(np.float64) ** 2
        close = (np.abs(nrm / CLAMP_F - 1.0) < 2e-3) & ~fixed
        if not close.any():
            break
        theta[close] = (theta[close] * 1.01).astype(np.float32)
    return theta


JOINTS = ("none", "none_dist", "revolute_dist", "prismatic", "mixed")


class Kin:
    """One kinematic problem on the device: tree, parameters (float32, as the kernels receive them), pose gradients."""

    def __init__(self, tree_name, joints, root, T, seed):
        rng = np.random.default_rng(seed)
        paths, topo, _ = tree_spec(tree_name)
        P = len(topo)
        E = P - 1
        self.name = f"{tree_name}-{joints}-{'root' if root else 'noroot'}-T{T}"
        self.T, self.P, self.E = T, P, E
        codes = None
        if joints == "revolute_dist":
            codes = [1] * E
        elif joints == "prismatic":
            codes = [2] * E
        elif joints == "mixed":
            codes = [(1, 2, 0)[e % 3] for e in range(E)]
        self.codes = codes
        self.tree = flat_tree(tree_name, codes)
        self.has_dist = joints != "none"
        axis = random_axes(rng, E)
        moment = (rng.standard_normal((E, 3)) * 0.1).astype(np.float32)
        theta = rng.uniform(-np.pi, np.pi, (T, E)).astype(np.float32)
        fixed = np.zeros((T, E), bool)
        for k, val in enumerate(PLANTED.values()):
            if E:
                t, e = (3 * k) % T, (5 * k) % E
                theta[t, e] = np.float32(val)
                fixed[t, e] = True
        dist = rng.uniform(-0.1, 0.1, (T, E)).astype(np.float32) if self.has_dist else None
        jt = np.zeros(E, np.int32) if codes is None else np.array(codes, np.int32)
        if E:
            th_eff = np.where(jt[None] == 2, np.float32(EPS_F), theta)
            theta = np.where(jt[None] == 2, theta, keep_off_the_clamp(np.broadcast_to(axis, (T, E, 3)), th_eff, fixed))
        cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
        self.axis, self.moment, self.theta = cu(axis), cu(moment), cu(theta.astype(np.float32))
        self.distance = cu(dist) if dist is not None else None
        self.root_6d = self.root_t = None
        if root:
            self.root_6d = cu((np.array([1, 0, 0, 0, 1, 0]) + 0.4 * rng.standard_normal((T, 6))).astype(np.float32))
            self.root_t = cu((0.2 * rng.standard_normal((T, 3))).astype(np.float32))
        self.gR = cu(rng.standard_normal((T, P, 3, 3)).astype(np.float32))
        self.gtr = cu(rng.standard_normal((T, P, 3)).astype(np.float32))

    # ---------------------------------------------------------------------------------------- effective joint inputs
    def joint_inputs(self):
        """(theta, d) as fk_joint_inputs hands them to the screw map (float32 CPU [T,E]) and the masks of the variables."""
        T, E = self.T, self.E
        jt = torch.zeros(E, dtype=torch.int32) if self.codes is None else torch.tensor(self.codes, dtype=torch.int32)
        th = self.theta.detach().cpu().clone()
        d = self.distance.detach().cpu().clone() if self.has_dist else torch.full((T, E), EPS_F)
        th_var = (jt != 2).expand(T, E)
        d_var = (jt != 1).expand(T, E) & self.has_dist
        d = torch.where((jt == 1).expand(T, E), torch.full_like(d, EPS_F), d)
        th = torch.where((jt == 2).expand(T, E), torch.full_like(th, EPS_F), th)
        return th, d, th_var, d_var

    def params(self):
        return [q for q in (self.axis, self.moment, self.theta, self.distance, self.root_6d, self.root_t) if q is not None]

    def layout(self):
        """(name, size) of the tail's grad buffer slices (kin.cu)."""
        T, E = self.T, self.E
        out = [("axis", 3 * E), ("moment", 3 * E), ("loss", 1), ("theta", T * E)]
        if self.has_dist:
            out.append(("distance", T * E))
        if self.root_6d is not None:
            out += [("root_6d", 6 * T), ("root_t", 3 * T)]
        return out

    def split(self, g):
        names, sizes = zip(*self.layout())
        return dict(zip(names, torch.split(g.reshape(-1), list(sizes))))

    # ---------------------------------------------------------------------------------------- float64 autograd
    def reference(self, gR=None, gtr=None, drop_root_part=None):
        T, P, E = self.T, self.P, self.E
        gR = f64(self.gR if gR is None else gR)
        gtr = f64(self.gtr if gtr is None else gtr)
        th32, d32, th_var, d_var = self.joint_inputs()
        norot = no_rot32(th32)
        axis = f64(self.axis).requires_grad_(True)
        moment = f64(self.moment).requires_grad_(True)
        theta = f64(self.theta).requires_grad_(True)
        dist = f64(self.distance).requires_grad_(True) if self.has_dist else None
        th = torch.where(th_var, theta, th32.double())
        d = torch.where(d_var, dist, d32.double()) if dist is not None else d32.double()
        order, parent, edge = (self.tree.order.tolist(), self.tree.parent.tolist(), self.tree.edge.tolist())
        poses = [None] * P
        for c in order:
            if parent[c] < 0:
                poses[c] = torch.eye(3, 4, dtype=F64).expand(T, 3, 4)
            else:
                e = edge[c]
                rel = screw64(axis[e].expand(T, 3), moment[e].expand(T, 3), th[:, e], d[:, e], norot[:, e])
                poses[c] = mat34(poses[parent[c]], rel)
        F = torch.stack(poses, 1)
        leaves = [axis, moment, theta] + ([dist] if dist is not None else [])
        out = F
        if self.root_6d is not None:
            r6 = f64(self.root_6d).requires_grad_(True)
            rt = f64(self.root_t).requires_grad_(True)
            leaves += [r6, rt]
            root = torch.cat([rot6d64(r6), rt[:, :, None]], -1)[:, None].expand(T, P, 3, 4)
            out = mat34(root, F)
            if drop_root_part is not None:
                keep = torch.ones(P, dtype=torch.bool)
                keep[drop_root_part] = False
                out = torch.where(keep[None, :, None, None], out, F)
        R, tr = out[..., :3], out[..., 3]
        obj = (gR * R).sum() + (gtr * tr).sum()
        grads = torch.autograd.grad(obj, leaves, allow_unused=True, materialize_grads=True) if E or len(leaves) > 3 else []
        names = ["axis", "moment", "theta"] + (["distance"] if dist is not None else []) + \
                (["root_6d", "root_t"] if self.root_6d is not None else [])
        g = {n: q.reshape(-1) for n, q in zip(names, grads)} if grads else {n: torch.zeros(0, dtype=F64) for n in names}
        return dict(R=R.detach(), tr=tr.detach(), fk=F.detach().reshape(T, P, 12), grad=g, norot=norot, th32=th32)

    # ---------------------------------------------------------------------------------------- running-error bounds
    def bounds(self):
        """The Run pass of head + tail (+ fk_bwd's order-free frame sums): Run values and S of every output."""
        T, P, E = self.T, self.P, self.E
        th32, d32, th_var, d_var = self.joint_inputs()
        norot = no_rot32(th32)
        order, parent, edge = (self.tree.order.tolist(), self.tree.parent.tolist(), self.tree.edge.tolist())
        axis, moment = f64(self.axis), f64(self.moment)
        ones, zeros = torch.ones(T, dtype=F64), torch.zeros(T, dtype=F64)
        ident = [Run.exact(ones if k % 5 == 0 else zeros) for k in range(12)]
        F, rel = [None] * P, [None] * P
        for c in order:
            if parent[c] < 0:
                F[c] = ident
                continue
            e = edge[c]
            L = [Run.exact(axis[e, k].expand(T).clone(), 8, k) for k in range(3)]
            Mo = [Run.exact(moment[e, k].expand(T).clone(), 8, 3 + k) for k in range(3)]
            rel[c] = screw_run(L, Mo, Run.exact(th32[:, e].double(), 8, 6), Run.exact(d32[:, e].double(), 8, 7), norot[:, e])
            F[c] = mat34_run(F[parent[c]], [x.plain() for x in rel[c]])
        out = {"fk_v": torch.stack([torch.stack([x.v for x in F[c]], -1) for c in range(P)], 1),
               "fk_s": torch.stack([torch.stack([x.s for x in F[c]], -1) for c in range(P)], 1)}
        G = f64(self.gR).reshape(T, P, 9)
        Gt = f64(self.gtr)
        Gc = [[Run.exact(G[:, c, 3 * i + j]) if j < 3 else Run.exact(Gt[:, c, i]) for i in range(3) for j in range(4)]
              for c in range(P)]
        head = F
        if self.root_6d is not None:
            r6 = f64(self.root_6d)
            Rr = rot6d_run([Run.exact(r6[:, k], 6, k) for k in range(6)])
            root = []
            for i in range(3):
                root += [Rr[3 * i].plain(), Rr[3 * i + 1].plain(), Rr[3 * i + 2].plain(), Run.exact(f64(self.root_t)[:, i])]
            head = [mat34_run(root, F[c]) for c in range(P)]
            gRr, gtr_acc = [None] * 9, [None] * 3
            gw = [None] * P
            for c in range(P):                       # kin_tail: part-id order
                for i in range(3):
                    for k in range(3):
                        t = (Gc[c][4 * i] * F[c][4 * k] + Gc[c][4 * i + 1] * F[c][4 * k + 1] + Gc[c][4 * i + 2] * F[c][4 * k + 2]
                             + Gc[c][4 * i + 3] * F[c][4 * k + 3])
                        gRr[3 * i + k] = t if gRr[3 * i + k] is None else gRr[3 * i + k] + t
                    gtr_acc[i] = Gc[c][4 * i + 3] if gtr_acc[i] is None else gtr_acc[i] + Gc[c][4 * i + 3]
                gw[c] = [Rr[k].plain() * Gc[c][j] + Rr[3 + k].plain() * Gc[c][4 + j] + Rr[6 + k].plain() * Gc[c][8 + j]
                         for k in range(3) for j in range(4)]
            g6 = []
            for k in range(6):
                acc = None
                for o in range(9):
                    t = gRr[o] * Rr[o].part(k)
                    acc = t if acc is None else acc + t
                g6.append(acc)
            out["root_6d"] = (torch.stack([x.v for x in g6], -1).reshape(-1), torch.stack([x.s for x in g6], -1).reshape(-1))
            out["root_t"] = (torch.stack([x.v for x in gtr_acc], -1).reshape(-1), torch.stack([x.s for x in gtr_acc], -1).reshape(-1))
        else:
            gw = [list(g) for g in Gc]
        out["R_v"] = torch.stack([torch.stack([head[c][4 * i + j].v for i in range(3) for j in range(3)], -1) for c in range(P)], 1)
        out["R_s"] = torch.stack([torch.stack([head[c][4 * i + j].s for i in range(3) for j in range(3)], -1) for c in range(P)], 1)
        out["tr_v"] = torch.stack([torch.stack([head[c][4 * i + 3].v for i in range(3)], -1) for c in range(P)], 1)
        out["tr_s"] = torch.stack([torch.stack([head[c][4 * i + 3].s for i in range(3)], -1) for c in range(P)], 1)
        fv, fs = torch.zeros(T, 6 * E, dtype=F64), torch.zeros(T, 6 * E, dtype=F64)
        th_v, th_s = torch.zeros(T, E, dtype=F64), torch.zeros(T, E, dtype=F64)
        d_v, d_s = torch.zeros(T, E, dtype=F64), torch.zeros(T, E, dtype=F64)
        for oi in range(P - 1, -1, -1):              # leaves first
            c = order[oi]
            par = parent[c]
            if par < 0:
                continue
            e = edge[c]
            A, Gm, r = F[par], gw[c], rel[c]
            g8 = [None] * 8
            for i in range(3):
                for j in range(4):
                    dT = A[i] * Gm[j] + A[4 + i] * Gm[4 + j] + A[8 + i] * Gm[8 + j]
                    for k in range(8):
                        t = dT * r[4 * i + j].part(k)
                        g8[k] = t if g8[k] is None else g8[k] + t
            for i in range(3):
                for j in range(4):
                    if j < 3:
                        s = (Gm[4 * i] * r[4 * j].plain() + Gm[4 * i + 1] * r[4 * j + 1].plain() + Gm[4 * i + 2] * r[4 * j + 2].plain()
                             + Gm[4 * i + 3] * r[4 * j + 3].plain())
                    else:
                        s = Gm[4 * i + 3]
                    gw[par][4 * i + j] = gw[par][4 * i + j] + s
            for k in range(3):
                fv[:, 3 * e + k], fs[:, 3 * e + k] = g8[k].v, g8[k].s
                fv[:, 3 * E + 3 * e + k], fs[:, 3 * E + 3 * e + k] = g8[3 + k].v, g8[3 + k].s
            th_v[:, e], th_s[:, e] = g8[6].v, g8[6].s
            d_v[:, e], d_s[:, e] = g8[7].v, g8[7].s
        sv, ss = seq_sum(fv, fs)                     # kin_tail: frame order
        ss_any = fs.sum(0) + max(T - 1, 0) * fv.abs().sum(0)   # fk_bwd: atomics, any order
        out["axis"], out["moment"] = (sv[:3 * E], ss[:3 * E]), (sv[3 * E:], ss[3 * E:])
        out["axis_any"], out["moment_any"] = ss_any[:3 * E], ss_any[3 * E:]
        out["theta"] = (th_v.reshape(-1), th_s.reshape(-1))
        out["distance"] = (d_v.reshape(-1), d_s.reshape(-1))
        out["th_var"], out["d_var"] = th_var.reshape(-1), d_var.reshape(-1)
        return out

    # ---------------------------------------------------------------------------------------- launches
    def head(self, params=None):
        _lib, L = lib()
        p = _lib.ptr
        q = self if params is None else params
        T, P = self.T, self.P
        R, tr, fk = (torch.empty(T, P, 3, 3, device=dev()), torch.empty(T, P, 3, device=dev()),
                     torch.empty(T, P, 12, device=dev()))
        th = q.theta if self.E else None                 # a one-part model has no joints: null pointers
        _lib.check(L.reart_kin_head(p(q.axis if self.E else None), p(q.moment if self.E else None), p(th), p(q.distance),
                                    p(self.tree.order), p(self.tree.parent), p(self.tree.edge), p(self.tree.joint_type),
                                    p(q.root_6d), p(q.root_t), T, P, p(R), p(tr), p(fk), _lib.stream_ptr()), "reart_kin_head")
        return R, tr, fk

    def fk_fwd(self):
        _lib, L = lib()
        p = _lib.ptr
        out = torch.empty(self.T, self.P, 4, 4, device=dev())
        _lib.check(L.reart_fk_fwd(p(self.axis), p(self.moment), p(self.theta), p(self.distance), p(self.tree.order),
                                  p(self.tree.parent), p(self.tree.edge), p(self.tree.joint_type), self.T, self.P, p(out),
                                  _lib.stream_ptr()), "reart_fk_fwd")
        return out

    def fk_bwd(self, fk_out):
        _lib, L = lib()
        p = _lib.ptr
        T, P, E = self.T, self.P, self.E
        g_out = torch.zeros(T, P, 4, 4, device=dev())
        g_out[:, :, :3, :3] = self.gR
        g_out[:, :, :3, 3] = self.gtr
        e = lambda *s: torch.full(s, float("nan"), device=dev())
        g = dict(axis=e(E, 3), moment=e(E, 3), theta=e(T, E), distance=e(T, E) if self.has_dist else None)
        ws = torch.empty(T * P * 16, device=dev())
        _lib.check(L.reart_fk_bwd(p(self.axis), p(self.moment), p(self.theta), p(self.distance), p(self.tree.order),
                                  p(self.tree.parent), p(self.tree.edge), p(self.tree.joint_type), T, P, p(fk_out), p(g_out),
                                  p(g["axis"]), p(g["moment"]), p(g["theta"]), p(g["distance"]), p(ws), _lib.stream_ptr()),
                   "reart_fk_bwd")
        return {k: v for k, v in g.items() if v is not None}


class Tail:
    """reart_kin_tail state for one Kin problem (world = 1): its own copy of the parameters, Adam moments, workspace."""

    def __init__(self, kin, params=None):
        _lib, L = lib()
        self.kin = kin
        src = kin if params is None else params
        cl = lambda t: None if t is None else t.clone()
        self.axis, self.moment, self.theta = cl(src.axis), cl(src.moment), cl(src.theta)
        self.distance, self.root_6d, self.root_t = cl(src.distance), cl(src.root_6d), cl(src.root_t)
        n = sum(s for _, s in kin.layout())
        z = lambda *s: torch.zeros(*s, device=dev())
        self.grad, self.m, self.v, self.step, self.loss_out = z(n), z(n), z(n), z(1), z(1)
        self.partials = _lib.workspace(int(L.reart_kin_tail_workspace_bytes(kin.T, kin.P)), dev())
        self.loss_local = torch.full((1,), 0.8125, dtype=torch.float64, device=dev())

    def twin(self):
        return Tail(self.kin, self)

    def params(self):
        return {k: getattr(self, k) for k in ("axis", "moment", "theta", "distance", "root_6d", "root_t")
                if getattr(self, k) is not None}

    def flat_params(self):
        """the parameters in the grad buffer's layout (no loss slot)"""
        P = self.params()
        return torch.cat([P[n].reshape(-1) for n, _ in self.kin.layout() if n != "loss"])

    def state(self):
        return dict(self.params(), grad=self.grad, m=self.m, v=self.v, step=self.step, loss_out=self.loss_out)

    def iterate(self, phase=0, beta1=0.9, beta2=0.999, wd=1e-3, lr=1e-2, eps=1e-8, gR=None, gtr=None):
        """kin_head on this state's parameters, then kin_tail"""
        _lib, L = lib()
        p = _lib.ptr
        k = self.kin
        _, _, fk = self.fk = k.head(self)
        E = k.E
        a = _lib.KinTailArgs()
        a.fk, a.gR, a.gtr, a.loss_local = p(fk), p(k.gR if gR is None else gR), p(k.gtr if gtr is None else gtr), p(self.loss_local)
        a.order, a.parent, a.edge, a.joint_type = p(k.tree.order), p(k.tree.parent), p(k.tree.edge), p(k.tree.joint_type)
        a.axis, a.moment = p(self.axis if E else None), p(self.moment if E else None)
        a.theta, a.distance = p(self.theta if E else None), p(self.distance)
        a.root_6d, a.root_t = p(self.root_6d), p(self.root_t)
        a.grad, a.m, a.v, a.step = p(self.grad), p(self.m), p(self.v), p(self.step)
        a.lr, a.beta1, a.beta2, a.eps, a.weight_decay = lr, beta1, beta2, eps, wd
        a.partials, a.loss_out = p(self.partials), p(self.loss_out)
        a.rank, a.world, a.n_pad, a.phase = 0, 1, 0, phase
        a.T, a.P = k.T, k.P
        self.args = a                                  # kept alive for graph replay
        _lib.check(L.reart_kin_tail(ctypes.byref(a), _lib.stream_ptr()), "reart_kin_tail")


# ------------------------------------------------------------------------------------------------ cases
TREES = ("p1", "p2", "chain32", "star32", "perm17")
TS = (1, 31, 33, 257, 600)


def _cases():
    out, i = [], 0
    for tree in TREES:
        for joints in (("none",) if tree == "p1" else JOINTS):
            for root in (False, True):
                out.append((tree, joints, root, TS[i % len(TS)]))
                i += 1
    return out


CASES = _cases()
CASE_IDS = [f"{t}-{j}-{'root' if r else 'noroot'}-T{T}" for t, j, r, T in CASES]
_REF = {}


def problem(case):
    """(Kin, float64 reference, Run bounds), cached per case: head, fk and tail tests share them."""
    if case not in _REF:
        tree, joints, root, T = case
        kin = Kin(tree, joints, root, T, seed=100 + CASES.index(case))
        assert_margins(kin)
        ref, bnd = kin.reference(), kin.bounds()
        _check_run_agrees(kin, ref, bnd)
        _REF[case] = (kin, ref, bnd)
    return _REF[case]


def _check_run_agrees(kin, ref, bnd):
    """The Run pass recomputes every output in float64 by the kernels' sequence: it must agree with the autograd
    reference far inside the float32 bound (else S would not describe the computation it claims to)."""
    pairs = [(bnd["R_v"], ref["R"].reshape(kin.T, kin.P, 9), bnd["R_s"]), (bnd["tr_v"], ref["tr"], bnd["tr_s"]),
             (bnd["fk_v"], ref["fk"], bnd["fk_s"])]
    for n in ("axis", "moment", "root_6d", "root_t"):
        if n in bnd and n in ref["grad"]:
            pairs.append((bnd[n][0], ref["grad"][n], bnd[n][1]))
    for n, var in (("theta", "th_var"), ("distance", "d_var")):
        if n in ref["grad"]:
            keep = bnd[var]
            pairs.append((bnd[n][0][keep], ref["grad"][n][keep], bnd[n][1][keep]))
    for v, r, s in pairs:
        assert worst(v, r, 1e-6 * C * U * s) <= 1.0, kin.name


def assert_margins(kin):
    """every rotating joint input keeps |l theta|^2 at least 1e-3 relative away from the clamp"""
    if kin.E == 0:
        return
    th32, _, _, _ = kin.joint_inputs()
    norot = no_rot32(th32)
    l = f64(kin.axis)
    for e in range(kin.E):
        assert clamp_margin(l[e].expand(kin.T, 3), th32[:, e].double(), norot[:, e]) >= 1e-3, (kin.name, e)


# ------------------------------------------------------------------------------------------------ 1. screw and 6D kernels
def screw_sweep(B=333, seed=3):
    """B screw inputs (not a multiple of the 64 / 128 thread blocks): every planted angle at every axis norm with
    random and zero distances first, then random angles in (-pi, pi)."""
    rng = np.random.default_rng(seed)
    l = random_axes(rng, B)
    m = (rng.standard_normal((B, 3)) * 0.2).astype(np.float32)
    th = rng.uniform(-np.pi, np.pi, B).astype(np.float32)
    d = rng.uniform(-0.2, 0.2, B).astype(np.float32)
    fixed = np.zeros(B, bool)
    i = 0
    for val in PLANTED.values():
        for norm_k in range(3):
            for dz in (False, True):
                l[i] = l[i] / np.linalg.norm(l[i]) * AXIS_NORMS[norm_k]
                th[i], fixed[i] = np.float32(val), True
                if dz:
                    d[i] = 0.0
                i += 1
    th = keep_off_the_clamp(l, th, fixed)
    return l.astype(np.float32), m, th.astype(np.float32), d


def test_screw_kernels_match_float64():
    _lib, L = lib()
    p = _lib.ptr
    l, m, th, d = screw_sweep()
    B = len(th)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    lt, mt, tt, dt = cu(l), cu(m), cu(th), cu(d)
    norot = no_rot32(tt)
    assert norot.sum() == 3 * 2 * sum(PLANTED_NOROT.values())               # exactly the planted no-rot cells
    assert clamp_margin(torch.from_numpy(l).double(), torch.from_numpy(th).double(), norot) >= 1e-3
    M = torch.empty(B, 16, device=dev())
    _lib.check(L.reart_screw_to_transform_fwd(p(lt), p(mt), p(tt), p(dt), B, p(M), _lib.stream_ptr()), "screw_fwd")
    gM = torch.randn(B, 16, device=dev())
    gl, gm, gth, gd = (torch.full((B, 3), float("nan"), device=dev()), torch.full((B, 3), float("nan"), device=dev()),
                       torch.full((B,), float("nan"), device=dev()), torch.full((B,), float("nan"), device=dev()))
    _lib.check(L.reart_screw_to_transform_bwd(p(lt), p(mt), p(tt), p(dt), p(gM), B, p(gl), p(gm), p(gth), p(gd),
                                              _lib.stream_ptr()), "screw_bwd")
    torch.cuda.synchronize()
    assert torch.equal(M[:, 12:].cpu(), torch.tensor([0.0, 0.0, 0.0, 1.0]).expand(B, 4))
    # float64 autograd
    L64, M64, T64, D64 = (f64(x).requires_grad_(True) for x in (lt, mt, tt, dt))
    ref = screw64(L64, M64, T64, D64, norot).reshape(B, 12)
    g12 = f64(gM)[:, :12]
    grads = torch.autograd.grad((g12 * ref).sum(), [L64, M64, T64, D64])
    # bounds
    run = screw_run([Run.exact(f64(lt)[:, k], 8, k) for k in range(3)], [Run.exact(f64(mt)[:, k], 8, 3 + k) for k in range(3)],
                    Run.exact(f64(tt), 8, 6), Run.exact(f64(dt), 8, 7), norot)
    s_fwd = torch.stack([x.s for x in run], -1)
    gb = [contract(g12, run, k) for k in range(8)]
    bl = torch.stack([gb[k].s for k in range(3)], -1)
    bm = torch.stack([gb[3 + k].s for k in range(3)], -1)
    r = dict(M=worst(M[:, :12], ref.detach(), C * U * s_fwd), l=worst(gl, grads[0], C * U * bl), m=worst(gm, grads[1], C * U * bm),
             theta=worst(gth, grads[2], C * U * gb[6].s), d=worst(gd, grads[3], C * U * gb[7].s))
    flat = [grads[0][:, 0], grads[0][:, 1], grads[0][:, 2], grads[1][:, 0], grads[1][:, 1], grads[1][:, 2], grads[2], grads[3]]
    for x, want in zip(gb, flat):                    # the mirrored sequence computes the same derivatives
        assert worst(x.v, want, 1e-6 * C * U * x.s) <= 1.0
    line = report(f"screw B={B}", **r)
    assert max(r.values()) < 1, line
    # the no-rot branch ignores d: its d-gradient is exactly zero
    assert torch.count_nonzero(gd.cpu()[norot]) == 0, line


def rot6d_sweep(B=333, seed=4):
    """random 6D inputs, then second columns down to nearly parallel to the first (sin of the angle 1e-1 .. 1e-3)"""
    rng = np.random.default_rng(seed)
    d6 = rng.standard_normal((B, 6))
    for i, eps in enumerate(np.repeat([1e-1, 1e-2, 3e-3, 1e-3], 20)):
        a1 = d6[i, :3]
        perp = np.cross(a1, rng.standard_normal(3))
        perp /= np.linalg.norm(perp)
        d6[i, 3:] = a1 * rng.uniform(0.5, 2.0) + eps * np.linalg.norm(a1) * perp
    return d6.astype(np.float32)


def test_rot6d_kernels_match_float64():
    _lib, L = lib()
    p = _lib.ptr
    d6 = torch.from_numpy(rot6d_sweep()).to(dev())
    B = d6.shape[0]
    R = torch.empty(B, 9, device=dev())
    _lib.check(L.reart_rot6d_fwd(p(d6), B, p(R), _lib.stream_ptr()), "rot6d_fwd")
    gR = torch.randn(B, 9, device=dev())
    g = torch.full((B, 6), float("nan"), device=dev())
    _lib.check(L.reart_rot6d_bwd(p(d6), p(gR), B, p(g), _lib.stream_ptr()), "rot6d_bwd")
    torch.cuda.synchronize()
    x = f64(d6).requires_grad_(True)
    ref = rot6d64(x).reshape(B, 9)
    gref = torch.autograd.grad((f64(gR) * ref).sum(), x)[0]
    run = rot6d_run([Run.exact(f64(d6)[:, k], 6, k) for k in range(6)])
    gb = [contract(f64(gR), run, k) for k in range(6)]
    bg = torch.stack([y.s for y in gb], -1)
    assert worst(torch.stack([y.v for y in gb], -1), gref, 1e-6 * C * U * bg) <= 1.0
    r = dict(R=worst(R, ref.detach(), C * U * torch.stack([y.s for y in run], -1)), g=worst(g, gref, C * U * bg))
    line = report(f"rot6d B={B}", **r)
    assert max(r.values()) < 1, line


# ------------------------------------------------------------------------------------------------ 2. fk_fwd / fk_bwd
# fk_fwd / fk_bwd have no root pose: gR / gtr are the gradients of the tree poses themselves, which is the reference's
# gradient only without a root pose
FK_CASES = [(c, i) for c, i in zip(CASES, CASE_IDS) if c[0] != "p1" and not c[2]]


@pytest.mark.parametrize("case", [c for c, _ in FK_CASES], ids=[i for _, i in FK_CASES])
def test_fk_kernels_match_float64(case):
    kin, ref, bnd = problem(case)
    out = kin.fk_fwd()
    g = kin.fk_bwd(out)
    torch.cuda.synchronize()
    T, P = kin.T, kin.P
    assert torch.equal(out[:, :, 3].cpu(), torch.tensor([0.0, 0.0, 0.0, 1.0]).expand(T, P, 4))
    r = dict(fk=worst(out[:, :, :3].reshape(T, P, 12), ref["fk"], C * U * bnd["fk_s"]),
             axis=worst(g["axis"], ref["grad"]["axis"], C * U * bnd["axis_any"]),
             moment=worst(g["moment"], ref["grad"]["moment"], C * U * bnd["moment_any"]),
             theta=worst(g["theta"], ref["grad"]["theta"], C * U * bnd["theta"][1] * bnd["th_var"]))
    if kin.has_dist:
        r["distance"] = worst(g["distance"], ref["grad"]["distance"], C * U * bnd["distance"][1] * bnd["d_var"])
    line = report(f"fk {kin.name}", **r)
    assert max(r.values()) < 1, line


# ------------------------------------------------------------------------------------------------ 3. head
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_head_matches_float64(case):
    kin, ref, bnd = problem(case)
    R, tr, fk = kin.head()
    torch.cuda.synchronize()
    T, P = kin.T, kin.P
    r = dict(R=worst(R.reshape(T, P, 9), ref["R"].reshape(T, P, 9), C * U * bnd["R_s"]),
             tr=worst(tr, ref["tr"], C * U * bnd["tr_s"]), fk=worst(fk, ref["fk"], C * U * bnd["fk_s"]))
    line = report(f"head {kin.name}", **r)
    assert max(r.values()) < 1, line
    if kin.root_6d is None:
        if P > 1:                                    # the same device arithmetic as fk_fwd_kernel: bit for bit
            want = kin.fk_fwd()
            assert torch.equal(R, want[:, :, :3, :3]) and torch.equal(tr, want[:, :, :3, 3]), line
        assert torch.equal(fk.reshape(T, P, 3, 4)[..., :3], R) and torch.equal(fk.reshape(T, P, 3, 4)[..., 3], tr), line


# ------------------------------------------------------------------------------------------------ 4. tail gradients
# one case per tree runs the negative controls
CONTROL_CASES = {("p2", "none_dist", True), ("chain32", "mixed", True), ("star32", "prismatic", True),
                 ("perm17", "none_dist", True), ("perm17", "revolute_dist", True)}


def tail_ratios(kin, grad, ref, bnd):
    got = kin.split(grad)
    out = {}
    for n, _ in kin.layout():
        if n == "loss":
            continue
        if n in ("theta", "distance"):
            bound = C * U * bnd[n][1] * bnd["th_var" if n == "theta" else "d_var"]
        else:
            bound = C * U * bnd[n][1]
        out[n] = worst(got[n], ref["grad"][n], bound)
    return out


def leaf_of(kin):
    parents = set(kin.tree.parent.tolist())
    return max(c for c in range(kin.P) if kin.tree.parent[c] >= 0 and c not in parents)


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_tail_gradients_match_float64(case):
    kin, ref, bnd = problem(case)
    tail = Tail(kin)
    tail.iterate(wd=0.0)
    again = Tail(kin)
    again.iterate(wd=0.0)
    torch.cuda.synchronize()
    got = kin.split(tail.grad)
    r = tail_ratios(kin, tail.grad, ref, bnd)
    line = report(f"tail {kin.name}", **r)
    assert max(r.values(), default=0.0) < 1, line
    assert torch.equal(tail.grad, again.grad), "the tail's gradient is not bit-reproducible"
    assert float(got["loss"]) == float(np.float32(0.8125)) and float(tail.loss_out) == float(np.float32(0.8125))
    # where the joint type fixes theta or d, the gradient is exactly zero
    _, _, th_var, d_var = kin.joint_inputs()
    assert torch.count_nonzero(got["theta"].cpu()[~th_var.reshape(-1)]) == 0, line
    if kin.has_dist:
        assert torch.count_nonzero(got["distance"].cpu()[~d_var.reshape(-1)]) == 0, line
    if kin.P == 1:                                   # no joints: only the root pose has parameters
        assert [n for n, s in kin.layout() if s] == (["loss", "root_6d", "root_t"] if kin.root_6d is not None else ["loss"])
    if case[:3] in CONTROL_CASES:
        T, t0 = kin.T, kin.T // 2
        ctl = {}
        gR, gtr = kin.gR.clone(), kin.gtr.clone()
        gR[t0], gtr[t0] = 0.0, 0.0
        off = kin.reference(gR=gR, gtr=gtr)["grad"]          # frame t0 left out of the axis / moment frame sum
        ctl["ctl_frame"] = max(worst(got[n], off[n], C * U * bnd[n][1]) for n in ("axis", "moment"))
        leaf = leaf_of(kin)
        gR, gtr = kin.gR.clone(), kin.gtr.clone()
        gR[t0, leaf], gtr[t0, leaf] = 0.0, 0.0
        ctl["ctl_fold"] = max(tail_ratios(kin, tail.grad, kin.reference(gR=gR, gtr=gtr), bnd).values())
        ctl["ctl_root"] = max(tail_ratios(kin, tail.grad, kin.reference(drop_root_part=leaf), bnd).values())
        line = report(f"controls {kin.name}", **ctl)
        assert min(ctl.values()) > 1, line


# ------------------------------------------------------------------------------------------------ 5. Adam
@pytest.mark.parametrize("case", [("perm17", "mixed", True, 33), ("p1", "none", True, 31), ("chain32", "none_dist", False, 257)],
                         ids=["perm17-mixed-root-T33", "p1-root-T31", "chain32-none_dist-T257"])
def test_tail_adam_matches_the_formula(case):
    """Three steps with betas (0.9, 0.999) and weight decay, each from the tail's own gradient (the grad buffer, written
    before the update), against torch.optim.Adam's formula in float64; step counts, loss_out passes the loss through."""
    tree, joints, root, T = case
    kin = Kin(tree, joints, root, T, seed=91)
    f32 = lambda v: float(np.float32(v))
    b1, b2, wd, eps, lr = f32(0.9), f32(0.999), f32(1e-3), f32(1e-8), f32(1e-2)
    tail = Tail(kin)
    for step in range(1, 4):
        p0, m0, v0 = f64(tail.flat_params()), f64(tail.m), f64(tail.v)
        tail.loss_local.fill_(0.25 * step + 1.0 / 3.0)
        tail.iterate(beta1=0.9, beta2=0.999, wd=1e-3, lr=1e-2)
        torch.cuda.synchronize()
        assert float(tail.step) == step
        assert float(tail.loss_out) == float(np.float32(0.25 * step + 1.0 / 3.0))
        keep = torch.ones(tail.grad.numel(), dtype=torch.bool)
        keep[6 * kin.E] = False                       # the loss slot
        g, m0, v0 = f64(tail.grad)[keep], m0[keep], v0[keep]
        p1, m1, v1 = f64(tail.flat_params()), f64(tail.m)[keep], f64(tail.v)[keep]
        bc1, bc2 = 1.0 - b1 ** step, 1.0 - b2 ** step
        gw = g + wd * p0
        tol_g = 2 * U * (g.abs() + (wd * p0).abs())
        m_ref = b1 * m0 + (1 - b1) * gw
        tol_m = 4 * U * (m0.abs() + gw.abs()) + (1 - b1) * tol_g
        v_ref = b2 * v0 + (1 - b2) * gw * gw
        tol_v = 4 * U * v_ref + (1 - b2) * 2 * gw.abs() * tol_g
        upd = lr / bc1 * m1 / (v1.sqrt() / np.sqrt(bc2) + eps)
        p_ref = p0 - upd
        tol_p = 4 * U * p0.abs() + 16 * U * upd.abs()
        r = dict(m=worst(m1, m_ref, tol_m), v=worst(v1, v_ref, tol_v), p=worst(p1, p_ref, tol_p))
        line = report(f"adam {kin.name} step {step}", **r)
        assert max(r.values()) < 1, line
        assert bool((p1 != p0).all()), f"step {step}: a parameter did not move"


# ------------------------------------------------------------------------------------------------ 6. phases, 7. graph
def assert_same_state(a, b, what):
    for k, t in a.state().items():
        assert torch.equal(t, b.state()[k]), f"{what}: {k} differs"


@pytest.mark.parametrize("case", [("perm17", "mixed", True, 257), ("star32", "none_dist", False, 33), ("p1", "none", True, 5)],
                         ids=["perm17-mixed-root-T257", "star32-none_dist-T33", "p1-root-T5"])
def test_phase1_then_phase2_equals_phase0(case):
    kin = Kin(*case, seed=7)
    a, b = Tail(kin), Tail(kin)
    for s in range(3):
        for t in (a, b):
            t.loss_local.fill_(1.0 / 3.0 + s)
        a.iterate(phase=0)
        b.iterate(phase=1)
        b.iterate(phase=2)
        torch.cuda.synchronize()
        assert_same_state(a, b, f"step {s}")
        assert float(b.step) == s + 1 and float(b.loss_out) == float(np.float32(1.0 / 3.0 + s))


@pytest.mark.parametrize("case", [("chain32", "mixed", True, 600), ("p1", "none", True, 33)], ids=["chain32-mixed-root-T600", "p1-root-T33"])
def test_head_and_tail_graph_replay_equals_eager(case):
    kin = Kin(*case, seed=8)
    a, b = Tail(kin), Tail(kin)
    for _ in range(5):
        a.iterate()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.iterate()
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize()
    assert_same_state(a, b, "graph replay")


# ------------------------------------------------------------------------------------------------ 8. one part
def test_one_part_model_trains_only_its_root_pose():
    """P = 1 has no joints: head and tail take null axis / moment / theta, and a step moves the root pose alone."""
    kin = Kin("p1", "none", True, 9, seed=5)
    tail = Tail(kin)
    before = {k: v.clone() for k, v in tail.params().items() if v.numel()}
    assert set(before) == {"root_6d", "root_t"}                            # axis, moment, theta are empty
    tail.iterate()
    torch.cuda.synchronize()
    assert tail.grad.numel() == 1 + 9 * kin.T
    for k in before:
        assert bool((getattr(tail, k) != before[k]).any()), k
    R, tr, _ = kin.head(tail)
    torch.cuda.synchronize()
    want = rot6d64(f64(tail.root_6d))
    assert (f64(R)[:, 0] - want).abs().max() < 1e-6 and torch.equal(tr[:, 0], tail.root_t)
