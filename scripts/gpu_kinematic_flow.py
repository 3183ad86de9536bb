"""The kinematic fit with the flow loss (KinematicEngine(flow_ref=...)) on three iterations, alternated in one process: the
autograd composition, and native=True with search="brute" / "culled".  cfg4 of bench.WORKLOADS (T=32 x 16 384, P=8) with
synth.make_flow_reference(seq, cano_idx, n_ref=N//4), cano_idx in {0, 16}, without and with the assignment loss ("add").
Per (cano_idx, assign, arm): ms/step under the CUDA graph (events, 256 MiB L2 flush before each step).  Then the kernel
alone: reart_kin_flow against the composition it replaces, loss.flow_loss forward + backward on the window and
reart_skin_bwd of the local frames' [T,N,3] gradient, timed with CUDA events over many launches.  One JSON line per row.

    python scripts/gpu_kinematic_flow.py [--steps 20] [--rounds 2] --out OUT.jsonl
    python scripts/gpu_kinematic_flow.py --census --out OUT.jsonl     # kernels per step (torch profiler), a separate run
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ARMS = ("autograd", "native_brute", "native_culled")
T, N, P = 32, 16384, 8                                                      # cfg4
CANO = (0, 16)
ASSIGN = (None, dict(downsample=16, assign_gap=5, lambda_assign=0.3, assign_iter=0, mode="add"))


def make(arm, cano_idx, assign):
    import numpy as np
    import torch
    from reart_b200.engine import KinematicEngine
    from reart_b200.flow_utils import FlowReference
    from reart_b200.synth import kinematic_init, make_flow_reference, make_sequence
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    dev = torch.device("cuda")
    kw = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else v) for k, v in kinematic_init(seq).items()}
    refs, flows = make_flow_reference(seq, cano_idx, n_ref=N // 4)
    ref = FlowReference([torch.from_numpy(r).to(dev) for r in refs], [torch.from_numpy(f).to(dev) for f in flows])
    extra = {} if arm == "autograd" else dict(native=True, search=arm.split("_")[1])
    if assign is not None:
        extra["assign"] = dict(assign)
    return KinematicEngine(kw, torch.from_numpy(seq["part"]), torch.from_numpy(seq["cano"]).to(dev),
                           torch.from_numpy(seq["frames"]).to(dev), flow_ref=ref, cano_idx=cano_idx, **extra)


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
        kinds.append(bool(eng._cur_variant[2]))
    torch.cuda.synchronize()
    return [(k, a.elapsed_time(b)) for k, (a, b) in zip(kinds, ev)]


def kernel_timing(cano_idx, reps=200):
    """ms per call of reart_kin_flow vs flow_loss forward + backward + reart_skin_bwd on a random one-hot window of cfg4."""
    import torch
    from reart_b200 import _lib
    from reart_b200.loss import flow_loss
    L, p, sp = _lib.lib(), _lib.ptr, _lib.stream_ptr
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1)
    K = T + 1
    labels = torch.randint(0, P, (N,), device=dev, generator=g)
    cano = torch.randn(N, 3, device=dev, generator=g)
    W = torch.nn.functional.one_hot(labels, P).float().contiguous()
    R = torch.linalg.qr(torch.randn(T, P, 3, 3, device=dev, generator=g))[0].contiguous()
    tr = torch.randn(T, P, 3, device=dev, generator=g)
    sk = (torch.einsum("tnij,nj->tni", R[:, labels], cano) + tr[:, labels]).contiguous()
    win = torch.cat((sk[:cano_idx], cano[None], sk[cano_idx:])).contiguous()
    tflow = torch.randn(K - 1, N, 3, device=dev, generator=g)
    mask = (torch.rand(K - 1, N, device=dev, generator=g) < 0.7).to(torch.uint8)
    slot_frame = torch.tensor([-1 if k == cano_idx else (k if k < cano_idx else k - 1) for k in range(K)], dtype=torch.int32,
                              device=dev)
    order = torch.argsort(labels, stable=True).int()
    offsets = torch.cat((labels.new_zeros(1), torch.bincount(labels, minlength=P).cumsum(0))).int()
    gR, gtr = torch.zeros(T, P, 3, 3, device=dev), torch.zeros(T, P, 3, device=dev)
    loss = torch.zeros(1, dtype=torch.float64, device=dev)
    kf_bytes = int(L.reart_kin_flow_workspace_bytes(K, P))
    kf_ws = torch.zeros(kf_bytes, dtype=torch.uint8, device=dev)
    gW = torch.empty(N, P, device=dev)
    sb_bytes = int(L.reart_skin_bwd_workspace_bytes(T, N, P))
    sb_ws = torch.empty(sb_bytes, dtype=torch.uint8, device=dev)
    keep = slot_frame >= 0
    mask_b = mask.bool()

    def fused():
        _lib.check(L.reart_kin_flow(p(win), p(tflow), p(mask), p(slot_frame), p(cano), p(order), p(offsets), 1.0, 0, K, N, P, T,
                                    0, K - 1, p(gR), p(gtr), p(loss), 1, p(kf_ws), kf_bytes, sp()), "reart_kin_flow")

    def composed():
        w = win.detach().requires_grad_(True)
        fl = flow_loss(tflow, w[1:] - w[:-1], flow_mask_list=mask_b)
        gs = torch.autograd.grad(fl, w)[0][keep].contiguous()
        _lib.check(L.reart_skin_bwd(p(cano), p(W), p(R), p(tr), p(gs), T, N, P, p(gW), p(gR), p(gtr), p(sb_ws), sb_bytes, sp()),
                   "reart_skin_bwd")

    res = {}
    for rnd in range(3):                                                    # alternated; the first round is warm-up
        for name, fn in (("kin_flow", fused), ("flow_loss_fwd_bwd+skin_bwd", composed)):
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
    ap.add_argument("--census", action="store_true", help="only count the kernels of one eager step per arm (torch profiler)")
    ap.add_argument("--out", required=True, help="JSON lines are appended here")
    args = ap.parse_args()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    props = torch.cuda.get_device_properties(0)
    with open(args.out, "a") as f:
        def emit(row):
            row["gpu"] = props.name
            print(json.dumps(row), flush=True)
            f.write(json.dumps(row) + "\n")

        if args.census:
            from bench import kernels_of_one_step
            for c in CANO:
                for assign in ASSIGN:
                    for arm in ARMS:
                        eng = make(arm, c, assign)
                        eng.iteration = 1
                        eng._cur_variant = eng._variant()
                        ours, names = kernels_of_one_step(eng)
                        emit({"census": True, "T": T, "N": N, "P": P, "cano_idx": c, "assign": assign is not None, "arm": arm,
                              "our_kernels": ours, "all_kernels": sum(names.values()) if names else None,
                              "names": names})
                        eng.release()
            return
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > L2: every step starts cold, as in bench.py
        for c in CANO:
            for assign in ASSIGN:
                engines = {arm: make(arm, c, assign) for arm in ARMS}
                for eng in engines.values():
                    for _ in range(args.warmup):
                        eng.step()
                ms = {a: [] for a in ARMS}
                for _ in range(args.rounds):
                    for arm in ARMS:
                        ms[arm] += timed(engines[arm], args.steps, flush)
                for arm in ARMS:
                    row = {"workload": "cfg4", "T": T, "N": N, "P": P, "cano_idx": c, "assign": assign is not None, "arm": arm,
                           "rounds": args.rounds}
                    for kind, sel in (("plain", False), ("refresh", True)):
                        v = [t for r, t in ms[arm] if r == sel]
                        row[f"ms_{kind}"] = sum(v) / len(v) if v else None
                        row[f"steps_{kind}"] = len(v)
                    row["ms_mean"] = sum(t for _, t in ms[arm]) / len(ms[arm])
                    emit(row)
                for eng in engines.values():
                    eng.release()
                del engines
                torch.cuda.empty_cache()
            emit(dict({"kernel": "pose gradient of the flow loss", "workload": "cfg4", "T": T, "N": N, "P": P, "cano_idx": c},
                      **{f"ms_{k}": v for k, v in kernel_timing(c).items()}))


if __name__ == "__main__":
    main()
