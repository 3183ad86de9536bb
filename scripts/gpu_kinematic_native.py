"""The kinematic fit of cfg4 (bench.WORKLOADS, synth.kinematic_init) on three iterations, alternated in one process:
KinematicEngine's autograd composition (the default), and native=True with search="brute" / "culled".  Per arm: ms/step
under the CUDA graph (events, 256 MiB L2 flush between steps), our kernels per step (bench.kernels_of_one_step), the fraction
of (warp, 32-target chunk) blocks the culled search evaluates and the points per step its tie path resolves -- early in the
fit and again ~300 steps in -- and whether native brute and native culled produced equal losses.  One JSON line per
(window, arm).

    python scripts/gpu_kinematic_native.py [--steps 40] [--late 300] --out OUT.jsonl
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ARMS = ("autograd", "native_brute", "native_culled")


def make(arm, workload):
    import numpy as np
    import torch
    from bench import WORKLOADS
    from reart_b200.engine import KinematicEngine
    from reart_b200.synth import kinematic_init, make_sequence
    T, N, P = WORKLOADS[workload]
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    dev = torch.device("cuda")
    kw = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else v) for k, v in kinematic_init(seq).items()}
    extra = {} if arm == "autograd" else dict(native=True, search=arm.split("_")[1])
    return KinematicEngine(kw, torch.from_numpy(seq["part"]), torch.from_numpy(seq["cano"]).to(dev),
                           torch.from_numpy(seq["frames"]).to(dev), **extra), (T, N, P)


def timed(eng, steps, flush, losses):
    import torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    out = []
    for i in range(steps):
        flush.fill_(i & 0xff)
        ev[i][0].record()
        out.append(eng.step())
        ev[i][1].record()
    torch.cuda.synchronize()
    losses += [float(x) for x in out]
    return [a.elapsed_time(b) for a, b in ev]


def main():
    import torch
    from bench import kernels_of_one_step
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg4")
    ap.add_argument("--steps", type=int, default=40, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the three arms per window")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--late", type=int, default=300, help="steps into the fit of the second window")
    ap.add_argument("--out", required=True, help="JSON lines are appended here")
    args = ap.parse_args()
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    dev = torch.device("cuda")
    props = torch.cuda.get_device_properties(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > L2: every step starts cold, as in bench.py
    engines, losses, done = {}, {a: [] for a in ARMS}, {a: 0 for a in ARMS}
    for arm in ARMS:
        engines[arm], dims = make(arm, args.workload)
    for arm in ARMS:                                                        # graph capture + warm-up, same steps for all
        for _ in range(args.warmup):
            losses[arm].append(float(engines[arm].step()))
        done[arm] += args.warmup
    kernels = {}
    for arm in ARMS:                                                        # one eager step each: the launch census
        ours, names = kernels_of_one_step(engines[arm])
        kernels[arm] = (ours, sum(names.values()) if names else None)
        losses[arm].append(float(engines[arm]._nat["loss_out"][0]) if arm != "autograd" else float("nan"))
        done[arm] += 1
    with open(args.out, "a") as f:
        for window in ("early", "late"):
            if window == "late":
                for arm in ARMS:                                            # advance every fit to the same step
                    while done[arm] < args.late:
                        losses[arm].append(float(engines[arm].step())); done[arm] += 1
            ms = {a: [] for a in ARMS}
            for arm in ARMS:
                engines[arm].culling_stats(); engines[arm].flagged_ties()
            for _ in range(args.rounds):
                for arm in ARMS:
                    ms[arm] += timed(engines[arm], args.steps, flush, losses[arm])
                    done[arm] += args.steps
            same = losses["native_brute"] == losses["native_culled"]
            for arm in ARMS:
                eng = engines[arm]
                T, N, P = dims
                row = {"workload": args.workload, "window": window, "arm": arm, "T": T, "N": N, "P": P,
                       "step_at_window_end": done[arm], "ms_per_step": sum(ms[arm]) / len(ms[arm]), "ms_min": min(ms[arm]),
                       "ms_max": max(ms[arm]), "timed_steps": len(ms[arm]), "rounds": args.rounds,
                       "our_kernels_per_step": kernels[arm][0], "all_kernels_per_step": kernels[arm][1],
                       "last_loss": losses[arm][-1], "native_brute_and_culled_losses_equal": same, "gpu": props.name}
                st = eng.culling_stats()
                if st is not None:
                    row["blocks_evaluated_fraction"] = st[0] / max(st[1], 1)
                    row["flagged_ties_per_step"] = eng.flagged_ties() / len(ms[arm])
                print(json.dumps(row), flush=True)
                f.write(json.dumps(row) + "\n")
    for eng in engines.values():
        eng.release()


if __name__ == "__main__":
    main()
