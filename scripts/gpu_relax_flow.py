"""The relaxation fit with the flow loss (RelaxationEngine(flow_ref=...)) on its iterations, alternated in one process: the
autograd composition (the default with a flow loss), and native=True with search="brute" / "culled".  Workloads built as
bench.py builds cfg2 (synth.make_sequence, synth.make_flow_reference(seq, cano_idx, n_ref=N//4)):
  cfg2      T=16 x 4 096, P=15, recon + flow + assignment "add", cano_idx 0 (brute only: 4 096 points are below the culled
            search's threshold);
  cfg3_16k  T=64 x 16 384, P=15, recon + flow, cano_idx 0 and 32.
Per (workload, cano_idx, arm): ms/step under the CUDA graph (events, 256 MiB L2 flush before each step).  Then the kernel
alone: reart_flow_grad against the composition it replaces, loss.flow_loss forward + backward on the window, timed with
CUDA events over many launches.  One JSON line per row.

    python scripts/gpu_relax_flow.py [--steps 20] [--rounds 2] --out OUT.jsonl
    python scripts/gpu_relax_flow.py --census --out OUT.jsonl     # kernels per step (torch profiler), a separate run
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ASSIGN = dict(downsample=4, assign_gap=5, lambda_assign=0.3)               # bench.py's cfg2
# (workload, T, N, P, cano_idx, assignment, arms)
CASES = [("cfg2", 16, 4096, 15, 0, True, ("autograd", "native_brute")),
         ("cfg3_16k", 64, 16384, 15, 0, False, ("autograd", "native_brute", "native_culled")),
         ("cfg3_16k", 64, 16384, 15, 32, False, ("autograd", "native_brute", "native_culled"))]


def make(arm, T, N, P, cano_idx, assign):
    import torch
    from reart_b200.engine import RelaxationEngine
    from reart_b200.flow_utils import FlowReference
    from reart_b200.synth import make_flow_reference, make_sequence
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    dev = torch.device("cuda")
    refs, flows = make_flow_reference(seq, cano_idx=cano_idx, n_ref=N // 4)
    ref = FlowReference([torch.from_numpy(r).to(dev) for r in refs], [torch.from_numpy(f).to(dev) for f in flows])
    extra = {} if arm == "autograd" else dict(native=True, search=arm.split("_")[1])
    if assign:
        extra["assign"] = dict(ASSIGN)
    return RelaxationEngine(torch.from_numpy(seq["cano"]).to(dev), torch.from_numpy(seq["frames"]).to(dev), num_parts=P,
                            flow_ref=ref, cano_idx=cano_idx, **extra)


def timed(eng, steps, flush):
    """[(refresh step?, ms)] of ``steps`` steps."""
    import torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    kinds = []
    for i in range(steps):
        flush.fill_(i & 0xff)
        ev[i][0].record()
        eng.step(2.0)
        ev[i][1].record()
        kinds.append(bool(eng._cur_variant[2]))
    torch.cuda.synchronize()
    return [(k, a.elapsed_time(b)) for k, (a, b) in zip(kinds, ev)]


def kernel_timing(T, N, cano_idx, reps=200):
    """ms per call of reart_flow_grad vs loss.flow_loss forward + backward w.r.t. the window, on a random window."""
    import torch
    from reart_b200 import _lib
    from reart_b200.loss import flow_loss
    L, p, sp = _lib.lib(), _lib.ptr, _lib.stream_ptr
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1)
    K = T + 1
    win = torch.randn(K, N, 3, device=dev, generator=g)
    tflow = torch.randn(K - 1, N, 3, device=dev, generator=g)
    mask = (torch.rand(K - 1, N, device=dev, generator=g) < 0.7).to(torch.uint8)
    slot_frame = torch.tensor([-1 if k == cano_idx else (k if k < cano_idx else k - 1) for k in range(K)], dtype=torch.int32,
                              device=dev)
    gs = torch.zeros(T, N, 3, device=dev)
    loss = torch.zeros(1, dtype=torch.float64, device=dev)
    nb = int(L.reart_flow_grad_workspace_bytes(K, N))
    ws = torch.zeros(nb, dtype=torch.uint8, device=dev)
    keep = slot_frame >= 0
    mask_b = mask.bool()

    def fused():
        _lib.check(L.reart_flow_grad(p(win), p(tflow), p(mask), p(slot_frame), 1.0, 0, K, N, T, 0, K - 1, p(gs), p(loss), 1,
                                     p(ws), nb, sp()), "reart_flow_grad")

    def composed():
        w = win.detach().requires_grad_(True)
        fl = flow_loss(tflow, w[1:] - w[:-1], flow_mask_list=mask_b)
        gs.add_(torch.autograd.grad(fl, w)[0][keep])

    res = {}
    for rnd in range(3):                                                    # alternated; the first round is warm-up
        for name, fn in (("flow_grad", fused), ("flow_loss_fwd_bwd", composed)):
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
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the arms")
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
            for wl, T, N, P, c, assign, arms in CASES:
                for arm in arms:
                    eng = make(arm, T, N, P, c, assign)
                    eng.iteration = 1
                    eng._cur_variant = eng._phase()
                    ours, names = kernels_of_one_step(eng)
                    emit({"census": True, "workload": wl, "T": T, "N": N, "P": P, "cano_idx": c, "assign": assign, "arm": arm,
                          "our_kernels": ours, "all_kernels": sum(names.values()) if names else None, "names": names})
                    eng.release()
            return
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > L2: every step starts cold, as in bench.py
        for wl, T, N, P, c, assign, arms in CASES:
            engines = {arm: make(arm, T, N, P, c, assign) for arm in arms}
            for eng in engines.values():
                for _ in range(args.warmup):
                    eng.step(2.0)
            ms = {a: [] for a in arms}
            for _ in range(args.rounds):
                for arm in arms:
                    ms[arm] += timed(engines[arm], args.steps, flush)
            for arm in arms:
                row = {"workload": wl, "T": T, "N": N, "P": P, "cano_idx": c, "assign": assign, "arm": arm, "rounds": args.rounds}
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
            emit(dict({"kernel": "skinned-cloud gradient of the flow loss", "workload": wl, "T": T, "N": N, "cano_idx": c},
                      **{f"ms_{k}": v for k, v in kernel_timing(T, N, c).items()}))


if __name__ == "__main__":
    main()
