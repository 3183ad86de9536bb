"""The kinematic fit with the assignment loss (KinematicEngine(assign=...)) on three iterations, alternated in one process:
the autograd composition, and native=True with search="brute" / "culled", in both flavours ("add": Chamfer + assignment,
"replace": assignment only).  Per (workload, mode, arm): ms/step under the CUDA graph (events, 256 MiB L2 flush between
steps) separately for refresh steps (reart_lap runs) and the others, and our kernels per step of each kind
(bench.kernels_of_one_step).  Then the kernel alone: reart_kin_assign against the composition it replaces,
reart_assign_loss_grad + reart_skin_bwd on a [T,N,3] gradient, timed with CUDA events at the same shapes.
One JSON line per row.

    python scripts/gpu_kinematic_assign.py [--steps 20] [--rounds 2] --out OUT.jsonl
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ARMS = ("autograd", "native_brute", "native_culled")
# (name, T, N, P, downsample): cfg4 of bench.WORKLOADS at two sample counts, and the nao-shaped sequence
WORKLOADS = (("cfg4_ds16", 32, 16384, 8, 16), ("cfg4_ds4", 32, 16384, 8, 4), ("nao", 9, 4096, 10, 2))
GAP = 5


def make(arm, T, N, P, downsample, mode):
    import numpy as np
    import torch
    from reart_b200.engine import KinematicEngine
    from reart_b200.synth import kinematic_init, make_sequence
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    dev = torch.device("cuda")
    kw = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else v) for k, v in kinematic_init(seq).items()}
    extra = {} if arm == "autograd" else dict(native=True, search=arm.split("_")[1])
    assign = dict(downsample=downsample, assign_gap=GAP, lambda_assign=0.3, assign_iter=0, mode=mode)
    return KinematicEngine(kw, torch.from_numpy(seq["part"]), torch.from_numpy(seq["cano"]).to(dev),
                           torch.from_numpy(seq["frames"]).to(dev), assign=assign, **extra)


def timed(eng, steps, flush):
    """[(refresh step?, ms)] of ``steps`` steps."""
    import torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    kinds = []
    for i in range(steps):
        flush.fill_(i & 0xff)
        ev[i][0].record()
        eng.step()
        ev[i][1].record()
        kinds.append(bool(eng._cur_variant[2]))                            # the flavour the step just ran
    torch.cuda.synchronize()
    return [(k, a.elapsed_time(b)) for k, (a, b) in zip(kinds, ev)]


def census(eng):
    """Our kernels / all kernels of one eager non-refresh and one eager refresh iteration."""
    from bench import kernels_of_one_step
    out = {}
    for refresh in (False, True):
        eng._cur_variant = (eng.assign_mode == "add", True, refresh)
        ours, names = kernels_of_one_step(eng)
        out["refresh" if refresh else "plain"] = (ours, sum(names.values()) if names else None)
    return out


def kernel_timing(T, N, P, n, reps=200):
    """ms per call of reart_kin_assign vs reart_assign_loss_grad + reart_skin_bwd on a random one-hot problem."""
    import torch
    from reart_b200 import _lib, ops
    L, p, sp = _lib.lib(), _lib.ptr, _lib.stream_ptr
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1)
    labels = torch.randint(0, P, (N,), device=dev, generator=g)
    src_idx = torch.randperm(N, device=dev, generator=g)[:n].contiguous()
    cano = torch.randn(N, 3, device=dev, generator=g)
    W = torch.nn.functional.one_hot(labels, P).float().contiguous()
    R = torch.linalg.qr(torch.randn(T, P, 3, 3, device=dev, generator=g))[0].contiguous()
    tr = torch.randn(T, P, 3, device=dev, generator=g)
    skinned = ops.skin(cano, W, R, tr).contiguous()
    tgt = torch.randn(T, n, 3, device=dev, generator=g)
    col4row = torch.stack([torch.randperm(n, device=dev, generator=g) for _ in range(T)]).int()
    sample_part = labels[src_idx]
    order = torch.argsort(sample_part, stable=True).int()
    offsets = torch.cat((sample_part.new_zeros(1), torch.bincount(sample_part, minlength=P).cumsum(0))).int()
    gR, gtr = torch.zeros(T, P, 3, 3, device=dev), torch.zeros(T, P, 3, device=dev)
    loss = torch.zeros(1, dtype=torch.float64, device=dev)
    ka_bytes = int(L.reart_kin_assign_workspace_bytes(T, P))
    ka_ws = torch.zeros(ka_bytes, dtype=torch.uint8, device=dev)
    gs, gW = torch.zeros(T, N, 3, device=dev), torch.empty(N, P, device=dev)
    sb_bytes = int(L.reart_skin_bwd_workspace_bytes(T, N, P))
    sb_ws = torch.empty(sb_bytes, dtype=torch.uint8, device=dev)

    def fused():
        _lib.check(L.reart_kin_assign(p(skinned), p(cano), p(src_idx), p(tgt), p(col4row), p(order), p(offsets), 0.3, T, N, n,
                                      P, p(gR), p(gtr), p(loss), 1, p(ka_ws), ka_bytes, sp()), "reart_kin_assign")

    def composed():
        _lib.check(L.reart_assign_loss_grad(p(skinned), p(src_idx), p(tgt), p(col4row), T, N, n, 0.3, p(gs), 1, p(loss), sp()),
                   "reart_assign_loss_grad")
        _lib.check(L.reart_skin_bwd(p(cano), p(W), p(R), p(tr), p(gs), T, N, P, p(gW), p(gR), p(gtr), p(sb_ws), sb_bytes, sp()),
                   "reart_skin_bwd")

    res = {}
    for rnd in range(3):                                                    # alternated; the first round is warm-up
        for name, fn in (("kin_assign", fused), ("assign_loss_grad+skin_bwd", composed)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            if rnd:
                res.setdefault(name, []).append(a.elapsed_time(b) / reps)
    return {k: min(v) for k, v in res.items()}


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the three arms")
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--out", required=True, help="JSON lines are appended here")
    args = ap.parse_args()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    props = torch.cuda.get_device_properties(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > L2: every step starts cold, as in bench.py
    with open(args.out, "a") as f:
        def emit(row):
            row["gpu"] = props.name
            print(json.dumps(row), flush=True)
            f.write(json.dumps(row) + "\n")

        for name, T, N, P, ds in WORKLOADS:
            n = N // ds
            for mode in ("add", "replace"):
                engines = {arm: make(arm, T, N, P, ds, mode) for arm in ARMS}
                for eng in engines.values():                                # capture every flavour, same steps for all
                    for _ in range(args.warmup):
                        eng.step()
                ms = {a: [] for a in ARMS}
                for _ in range(args.rounds):
                    for arm in ARMS:
                        ms[arm] += timed(engines[arm], args.steps, flush)
                for arm in ARMS:
                    eng = engines[arm]
                    k = census(eng)
                    row = {"workload": name, "T": T, "N": N, "P": P, "n": n, "mode": mode, "arm": arm, "gap": GAP,
                           "rounds": args.rounds}
                    for kind, sel in (("plain", False), ("refresh", True)):
                        v = [t for r, t in ms[arm] if r == sel]
                        row[f"ms_{kind}"] = sum(v) / len(v) if v else None
                        row[f"steps_{kind}"] = len(v)
                        row[f"our_kernels_{kind}"], row[f"all_kernels_{kind}"] = k[kind]
                    row["ms_mean_over_gap"] = sum(t for _, t in ms[arm]) / len(ms[arm])
                    emit(row)
                for eng in engines.values():
                    eng.release()
                del engines
                torch.cuda.empty_cache()
            emit(dict({"kernel": "pose gradient of the assignment loss", "workload": name, "T": T, "N": N, "P": P, "n": n},
                      **{f"ms_{k}": v for k, v in kernel_timing(T, N, P, n).items()}))


if __name__ == "__main__":
    main()
