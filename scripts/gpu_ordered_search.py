"""Brute-force vs culled-in-caller-order search (RelaxationEngine(search="brute" | "culled")) on the bench workloads:
ms/step under the graph, the fraction of (warp, 32-target chunk) blocks the culled search evaluates, the points per step
its exact tie path resolves, and whether the two runs produced the same losses.  One JSON line per (workload, search).

    python scripts/gpu_ordered_search.py [--workloads cfg3_4k cfg3_16k] [--steps 40] --out OUT.jsonl
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run(workload, search, steps, warmup):
    import torch
    from bench import WORKLOADS
    from reart_b200.engine import RelaxationEngine, tau_schedule
    from reart_b200.synth import make_sequence
    T, N, P = WORKLOADS[workload]
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    dev = torch.device("cuda")
    eng = RelaxationEngine(torch.from_numpy(seq["cano"]).to(dev), torch.from_numpy(seq["frames"]).to(dev), num_parts=P,
                           search=search)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > L2: every step starts cold, as in bench.py
    for i in range(warmup):
        eng.step(tau_schedule(i, 15000, 5.0, 1.0))
    torch.cuda.synchronize()
    eng.culling_stats(); eng.flagged_ties()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    losses = []
    for i in range(steps):
        flush.fill_(i & 0xff)
        eng.tau.fill_(tau_schedule(warmup + i, 15000, 5.0, 1.0))
        ev[i][0].record()
        losses.append(eng.step())
        ev[i][1].record()
    torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in ev]
    out = {"workload": workload, "search": search, "search_culled": eng.search_culled, "T": T, "N": N,
           "ms_per_step": sum(ms) / steps, "ms_min": min(ms), "ms_max": max(ms), "steps": steps, "warmup": warmup,
           "losses": [float(x) for x in losses]}
    st = eng.culling_stats()
    if st is not None:
        out["blocks_evaluated_fraction"] = st[0] / max(st[1], 1)
        out["flagged_ties_per_step"] = eng.flagged_ties() / steps
    eng.release()
    return out


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["cfg3_4k", "cfg3_16k"])
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", required=True, help="JSON lines are appended here")
    args = ap.parse_args()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    props = torch.cuda.get_device_properties(0)
    with open(args.out, "a") as f:
        for wl in args.workloads:
            rows = {s: run(wl, s, args.steps, args.warmup) for s in ("brute", "culled")}
            same = rows["brute"]["losses"] == rows["culled"]["losses"]
            for s, r in rows.items():
                r["losses_equal_to_brute"] = same
                r["gpu"] = props.name
                r["speedup_vs_brute"] = rows["brute"]["ms_per_step"] / r["ms_per_step"]
                line = json.dumps(r)
                print(json.dumps({k: v for k, v in r.items() if k != "losses"}))
                f.write(line + "\n")


if __name__ == "__main__":
    main()
