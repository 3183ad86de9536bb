"""Time ``checkpoint()`` and ``load_checkpoint()`` of a native RelaxationEngine at a bench workload (default cfg3_16k:
64 frames x 16384 points, 15 parts) after a few steps, and the size of the saved file.  One JSON line to stdout.

    python scripts/gpu_checkpoint_timing.py [--workload cfg3_16k] [--steps 20] [--reps 10]
"""
import argparse
import io
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    import bench
    from reart_b200.engine import RelaxationEngine, tau_schedule
    from reart_b200.synth import make_sequence
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg3_16k", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    T, N, P = bench.WORKLOADS[args.workload]
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    dev = torch.device("cuda")
    eng = RelaxationEngine(torch.from_numpy(seq["cano"]).to(dev), torch.from_numpy(seq["frames"]).to(dev), P, seed=2)
    for i in range(args.steps):
        eng.step(tau_schedule(i, 1000, 5.0, 1.0))
    torch.cuda.synchronize()
    save, load = [], []
    ck = None
    for _ in range(args.reps):
        t0 = time.perf_counter()
        ck = eng.checkpoint()
        save.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        eng.load_checkpoint(ck)                                  # ends in a device synchronise
        load.append((time.perf_counter() - t0) * 1e3)
    buf = io.BytesIO()
    torch.save(ck, buf)
    tensor_bytes = sum(t.numel() * t.element_size() for t in _tensors(ck))
    print(json.dumps(dict(workload=args.workload, T=T, N=N, P=P, native=eng.native, search_culled=eng.search_culled,
                          steps_before=args.steps, reps=args.reps, checkpoint_ms_median=statistics.median(save),
                          checkpoint_ms_min=min(save), load_ms_median=statistics.median(load), load_ms_min=min(load),
                          tensor_bytes=tensor_bytes, file_bytes=len(buf.getvalue()), gpu=torch.cuda.get_device_name())))
    eng.release()


def _tensors(x):
    if torch.is_tensor(x):
        yield x
    elif isinstance(x, dict):
        for v in x.values():
            yield from _tensors(v)
    elif isinstance(x, (list, tuple)):
        for v in x:
            yield from _tensors(v)


if __name__ == "__main__":
    main()
