"""Culling statistics of the default engine (RelaxationEngine(search="auto")) on cfg3_16k at the two states a fit spends
its time in: the headline window of bench.py (warm-up steps, then its timed steps on the same tau schedule) and 600 steps
into a fit (a compressed cosine schedule 5 -> 1, then steps at tau = 1).  For each: the fraction of (warp, 32-target
chunk) blocks the culled search evaluated, the points per step its exact tie path resolved, ms/step (L2 flushed between
steps), and the skinned cloud at the end (caller order, .npy) for scripts/posed_order_potential.py.

    python scripts/gpu_posed_order.py --out OUT.jsonl [--dump DIR] [--profile DIR]

--profile: one extra step under torch.profiler per state, per-kernel CUDA times written to DIR/<state>_kernels.json.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def window(eng, flush, steps, taus):
    import torch
    eng.culling_stats(); eng.flagged_ties()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    loss = None
    for i in range(steps):
        flush.fill_(i & 0xff)
        eng.tau.fill_(taus(i))
        ev[i][0].record()
        loss = eng.step()
        ev[i][1].record()
    torch.cuda.synchronize()
    st = eng.culling_stats()
    return {"ms_per_step": sum(a.elapsed_time(b) for a, b in ev) / steps, "steps": steps,
            "blocks_evaluated_fraction": st[0] / max(st[1], 1) if st else None,
            "flagged_ties_per_step": (eng.flagged_ties() or 0) / steps, "loss": float(loss.item())}


def kernel_times(eng, path):
    import torch
    from torch.profiler import ProfilerActivity, profile
    eng.step(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.step()
        torch.cuda.synchronize()
    rows = sorted(((e.key, e.device_time_total / max(e.count, 1), e.count) for e in prof.key_averages()
                   if e.device_time_total > 0), key=lambda r: -r[1] * r[2])
    out = [{"kernel": k, "us": round(us, 2), "count": c} for k, us, c in rows]
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    return out


def main():
    import numpy as np
    import torch
    from bench import WORKLOADS
    from reart_b200.engine import RelaxationEngine, tau_schedule
    from reart_b200.synth import make_sequence
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg3_16k")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--late", type=int, default=600)
    ap.add_argument("--out", required=True, help="JSON lines are appended here")
    ap.add_argument("--dump", default=None, help="directory for the skinned clouds (.npy)")
    ap.add_argument("--profile", default=None, help="directory for per-kernel times of one step per state")
    args = ap.parse_args()
    T, N, P = WORKLOADS[args.workload]
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    dev = torch.device("cuda")
    eng = RelaxationEngine(torch.from_numpy(seq["cano"]).to(dev), torch.from_numpy(seq["frames"]).to(dev), num_parts=P)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > L2, as in bench.py
    for i in range(args.warmup):
        eng.step(tau_schedule(i, 15000, 5.0, 1.0))
    torch.cuda.synchronize()
    lines = []
    head = window(eng, flush, args.steps, lambda i: tau_schedule(args.warmup + i, 15000, 5.0, 1.0))
    head.update(state="headline", workload=args.workload, after_steps=eng.iteration)
    lines.append(head)
    for d in (args.dump, args.profile):
        if d:
            os.makedirs(d, exist_ok=True)
    if args.dump:
        np.save(os.path.join(args.dump, "skinned_headline.npy"), eng.skinned.float().cpu().numpy())
    if args.profile:
        head["kernels"] = kernel_times(eng, os.path.join(args.profile, "headline_kernels.json"))[:12]
    for i in range(eng.iteration, args.late):
        eng.step(tau_schedule(i, args.late, 5.0, 1.0))
    late = window(eng, flush, args.steps, lambda i: 1.0)
    late.update(state="late", workload=args.workload, after_steps=args.late, tau=1.0)
    lines.append(late)
    if args.dump:
        np.save(os.path.join(args.dump, "skinned_late.npy"), eng.skinned.float().cpu().numpy())
    if args.profile:
        late["kernels"] = kernel_times(eng, os.path.join(args.profile, "late_kernels.json"))[:12]
    eng.release()
    with open(args.out, "a") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
            print(json.dumps({k: v for k, v in ln.items() if k != "kernels"}))


if __name__ == "__main__":
    main()
