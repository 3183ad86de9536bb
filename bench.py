"""bench.py -- skinned-Chamfer forward+backward throughput of the reart energy evaluation on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cfg3_16k] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE full optimisation iteration of the relaxation model (run_robot.py:154-221, --model=base,
recon loss): seg MLP -> gumbel weights -> 6D->R -> skin -> bidirectional Chamfer against every observed
frame -> loss -> backward -> (N>1: one NCCL all-reduce of the shared grads) -> Adam, on the synthetic
sequence named by --workload.  Metric: directed point pairs / s = 2*T*N*M per step / time, whole job.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (T frames, N = M points, P parts) -- BASELINE.json configs
    "cfg3_16k": (64, 16384, 15),      # the sequence the north_star quotes its targets on (default)
    "cfg2": (16, 4096, 15),           # nao-shaped relaxation model, recon + flow + assign losses
    "cfg3_4k": (64, 4096, 15),
    "cfg3_64k": (64, 65536, 15),
    "cfg3_256k": (64, 262144, 15),
    "cfg4": (32, 16384, 8),           # sapien-shaped kinematic projection model (KinematicEngine)
    "cfg5": (64, 32768, 15),          # real-scan-shaped sequence; one cano_idx candidate fit per GPU
    "cfg3_16k_8f": (8, 16384, 15),    # one rank's shard of cfg3_16k at 8 GPUs (tuning aid)
    "tiny": (8, 2048, 6),
}
SWEEP = ("cfg2", "cfg3_4k", "cfg3_64k", "cfg3_256k", "cfg4", "cfg5")
METRIC = "skinned_chamfer_fwd_bwd_directed_point_pairs_per_s"
UNIT = "pairs/s"
FLOP_PER_PAIR = 8.0                   # 3 FSUB + 1 FMUL + 2 FFMA (BASELINE.md section 3)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline workload (>= 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3_16k", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the per-config sweep (N=1) / candidate fits (N>1)")
    ap.add_argument("--sustained-s", type=float, default=10.0, help="seconds of back-to-back steps after the timed region (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, skinned cloud, updated parameters; rank 0's shard) "
                         "as DIR/<name>.npy in float32, at most 60 MiB in all, for comparing two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times the CPU port, not the engine)")
    return args


def config_dict(args, T, N, P, world):
    kind = "kinematic projection model" if args.workload == "cfg4" else "relaxation model (base)"
    return {"workload": f"{args.workload}: {kind}, P={P}, synthetic sequence T={T} frames x "
                        f"N=M={N} points, skin + bidirectional Chamfer recon loss fwd+bwd + Adam",
            "T": T, "N": N, "M": N, "P": P, "frames_per_gpu": T // max(world, 1) if args.scaling == "strong" else T,
            "partitioning": f"frames sharded over {world} rank(s), one all-reduce of shared grads per step",
            "l2": "L2 flushed (256 MiB write) between timed steps", "seed": 2}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_throughput(T, N, budget_s=12.0):
    """Time the oracle port (OpenMP, all host cores) on a bounded sample of the workload: `frames` frames of
    N x N bidirectional Chamfer forward + backward.  Returns (pairs_per_s, cores, sample description)."""
    import numpy as np
    import oracle
    from reart_b200.synth import make_sequence
    oracle.build()
    cores = os.cpu_count() or 1
    oracle.set_num_threads(cores)
    seq = make_sequence(T=2, N=N, P=15, seed=2)
    src = np.ascontiguousarray(seq["frames"][0:1]); tgt = np.ascontiguousarray(seq["frames"][1:2])
    t0 = time.perf_counter()
    oracle.chamfer_bidir_fwd_bwd(src, tgt)
    one = time.perf_counter() - t0
    frames = int(max(1, min(T, budget_s / max(one, 1e-6))))
    src = np.repeat(src, frames, axis=0); tgt = np.repeat(tgt, frames, axis=0)
    t0 = time.perf_counter()
    oracle.chamfer_bidir_fwd_bwd(src, tgt)
    dt = time.perf_counter() - t0
    pairs = 2.0 * frames * N * N
    return pairs / dt, oracle.num_threads(), f"{frames} of {T} frames x {N}x{N} points, bidirectional Chamfer fwd+bwd, oracle C port ({dt:.2f} s)"


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The reference's
    own arithmetic lives in absent third-party CUDA packages, so this is the oracle port (kind 'port')."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    T, N, P = WORKLOADS[args.workload]
    steps, warm = max(args.steps, 1), max(args.warmup, 0)
    budget = max(1.0, min(12.0, 150.0 / (steps + warm)))
    vals, cores, sample = [], 1, ""
    for i in range(warm + steps):
        v, cores, sample = cpu_reference_throughput(T, N, budget_s=budget)
        if i >= warm:
            vals.append(v)
    value = sum(vals) / len(vals)
    pairs_per_step = 2.0 * T * N * N
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": pairs_per_step / value * 1e3, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, T, N, P, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    try:        # the reference's own Python loop on the same cores (needs the staged copy baseline/_ref/reart), reported beside it
        line["cpu_baseline_reference_python"] = reference_python_cpu_baseline(T, N, P)
    except Exception as exc:
        line["cpu_baseline_reference_python"] = {"error": f"{type(exc).__name__}: {exc}"}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  The timed region of the default run is < 0.1 s,
    shorter than nvidia-smi's start-up, so the primary source is an in-process NVML thread (the library nvidia-smi
    itself reads) polling every ~4 ms between begin() and end(); an `nvidia-smi -lms 20` subprocess started early is
    the fallback, filtered to the same wall-clock window."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, uuid: str | None = None):
        import threading
        self.samples = []                                  # (wall time, sm MHz, max MHz, watts, reasons tuple)
        self.t0 = self.t1 = None
        self._stop = threading.Event()
        self._thread = None
        self.smi_path, self.smi = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

            def poll():
                while not self._stop.is_set():
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                        try:
                            r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        except Exception:
                            r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.samples.append((time.time(), sm, mx, pw, tuple(k for k, b in bits.items() if r & b)))
                    except Exception:
                        pass
                    time.sleep(0.004)

            self._thread = threading.Thread(target=poll, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None
        try:
            self.smi_path = tempfile.NamedTemporaryFile(suffix=".csv", delete=False).name
            self.smi = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                         "-lms", "20", "-i", str(gpu_index)], stdout=open(self.smi_path, "w"),
                                        stderr=subprocess.DEVNULL)
        except Exception:
            self.smi = None

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def _smi_samples(self):
        import datetime
        out = []
        if self.smi is None:
            return out
        self.smi.terminate()
        try:
            self.smi.wait(timeout=5)
        except Exception:
            self.smi.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.smi_path):
            parts = [q.strip() for q in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                out.append((ts, float(parts[1]), float(parts[2]), float(parts[3]),
                            tuple(n for n, v in zip(names, parts[4:8]) if v.lower().startswith("active"))))
            except ValueError:
                continue
        os.unlink(self.smi_path)
        return out

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=1.0)
        source = "nvml"
        sel = [q for q in self.samples if self.t0 is not None and self.t0 <= q[0] <= (self.t1 or time.time())]
        smi = self._smi_samples()
        if len(sel) < 3:
            sel = [q for q in smi if self.t0 is not None and self.t0 - 0.02 <= q[0] <= (self.t1 or time.time()) + 0.02]
            source = "nvidia-smi"
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": len(sel), "source": source}
        if sel:
            sm = sorted(q[1] for q in sel)
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(q[2] for q in sel),
                       reasons=sorted({r for q in sel for r in q[4]}), power_w_max=max(q[3] for q in sel))
        return out


# ------------------------------------------------------------------------------------------------ GPU arm helpers
def reference_python_cpu_baseline(T, N, P, budget_frames=4, iters=2):
    """The reference's OWN Python path (networks/model.py BaseModel + networks/loss.py recon_loss over utils/chamfer.py,
    with the torch stand-in for the absent chamferdist._C, oracle/ref_harness.py) on the host cores, when a staged copy
    of the reference exists (baseline/_ref/reart, scripts/stage_reference.py).  Bounded sample: `budget_frames` frames of
    the workload, `iters` optimisation iterations (fwd + bwd + Adam).  Returns None when the reference is not staged."""
    staged = os.path.join(ROOT, "baseline", "_ref", "reart")
    if not os.path.isdir(os.path.join(staged, "utils")):
        return None
    import torch
    os.environ["REART_REFERENCE_ROOT"] = staged
    from oracle import ref_harness
    ref_harness.REFERENCE_ROOT = staged
    ref = ref_harness.import_reference()
    from reart_b200.synth import make_sequence
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    Ts = min(T, budget_frames)
    seq = make_sequence(T=Ts, N=N, P=P, seed=2)
    cano = torch.from_numpy(seq["cano"]); frames = torch.from_numpy(seq["frames"])
    torch.manual_seed(2)
    model = ref.model.BaseModel(num_parts=P, pose_len=Ts)
    cd = ref.chamfer.ChamferDistance()
    seg_params = [q for q in model.seg_head.parameters() if q.requires_grad]
    opt = torch.optim.Adam([{"params": [model.proposal_6d, model.proposal_t], "lr": 1e-2},
                            {"params": seg_params, "lr": 1e-3}], lr=1e-3)
    t0 = time.perf_counter()
    for _ in range(iters):
        pc_trans, _, _ = model(cano, tau=5.0)
        loss = ref.loss.recon_loss(pc_trans, frames, chamfer_dist=cd)
        opt.zero_grad(); loss.backward(); opt.step()
    dt = (time.perf_counter() - t0) / iters
    pairs = 2.0 * Ts * N * N
    return {"value": pairs / dt, "unit": UNIT, "cores": cores, "kind": "reference",
            "iters_per_s_sample": 1.0 / dt, "iters_per_s_full_T": (pairs / dt) / (2.0 * T * N * N),
            "sample": f"reference Python loop (BaseModel.forward + recon_loss + backward + Adam, torch stand-in for chamferdist._C), "
                      f"{Ts} of {T} frames x {N}x{N} points, {iters} iterations, {dt:.2f} s/iteration"}


def kernels_of_one_step(engine):
    """Names and counts of the CUDA kernels ONE eager iteration launches (torch profiler / CUPTI); `ours` = those in
    namespace reart.  Returns (ours_count, {name: count}) or (None, {}) when the profiler is unavailable."""
    import torch
    try:
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            engine._run_iteration()
            torch.cuda.synchronize()
        names = {}
        for ev in prof.events():
            if getattr(ev, "device_type", None) is not None and "cuda" in str(ev.device_type).lower():
                n = ev.name.split("(")[0].strip()
                if n.lower().startswith("memcpy") or n.lower().startswith("memset"):
                    continue
                names[n] = names.get(n, 0) + 1
        ours = sum(c for n, c in names.items() if "reart::" in n)
        return (ours if names else None), names
    except Exception:
        return None, {}


def make_engine(workload, ctx, dev, use_graph, scaling, extra_losses=True, cull=False, fuse_producer=False):
    """Synthetic sequence + engine of one named workload.  Returns (engine, host cano, host frames, T_total, N, P, desc)."""
    import numpy as np
    import torch
    from reart_b200.engine import KinematicEngine, RelaxationEngine
    from reart_b200.synth import kinematic_init, make_flow_reference, make_sequence
    T, N, P = WORKLOADS[workload]
    T_total = T if scaling == "strong" else T * ctx.world_size
    seq = make_sequence(T=T_total, N=N, P=P, seed=2)
    cano_h = torch.from_numpy(seq["cano"]).pin_memory()
    frames_h = torch.from_numpy(seq["frames"]).pin_memory()
    desc = "relaxation model (base), recon loss"
    if workload == "cfg4":
        kw = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else v) for k, v in kinematic_init(seq).items()}
        engine = KinematicEngine(kw, torch.from_numpy(seq["part"]), cano_h.to(dev), frames_h.to(dev), ctx=ctx, use_graph=use_graph)
        desc = "kinematic projection model, recon loss"
    elif workload == "cfg2" and extra_losses:
        refs, flows = make_flow_reference(seq, cano_idx=0, n_ref=N // 4)
        from reart_b200.flow_utils import FlowReference
        fr = FlowReference([torch.from_numpy(r).to(dev) for r in refs], [torch.from_numpy(f).to(dev) for f in flows])
        kwargs = {}
        try:
            import inspect
            if "assign" in inspect.signature(RelaxationEngine.__init__).parameters:
                kwargs["assign"] = dict(downsample=4, assign_gap=5, lambda_assign=0.3)
                desc = "relaxation model (base), recon + flow + assign losses"
            else:
                desc = "relaxation model (base), recon + flow losses"
        except Exception:
            pass
        engine = RelaxationEngine(cano_h.to(dev), frames_h.to(dev), num_parts=P, ctx=ctx, use_graph=use_graph, flow_ref=fr,
                                  cano_idx=0, **kwargs)
    else:
        engine = RelaxationEngine(cano_h.to(dev), frames_h.to(dev), num_parts=P, ctx=ctx, use_graph=use_graph, cull=cull,
                                  fuse_producer=fuse_producer)
    return engine, cano_h, frames_h, T_total, N, P, desc


def time_engine_steps(engine, ctx, K, W, flush, n_iter=15000, sampler=None):
    """W untimed + K timed steps, each bracketed by its own CUDA events on the launch stream, L2 flushed in between
    (untimed), max over ranks.  Returns (ms_per_step, wall_s, last loss tensor)."""
    import torch
    from reart_b200.engine import tau_schedule
    dev = flush.device
    for i in range(W):
        engine.step(tau_schedule(i, n_iter, 5.0, 1.0))
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    ctx.barrier(); torch.cuda.synchronize()
    if sampler:
        sampler.begin()
    t0 = time.perf_counter()
    loss = None
    for i in range(K):
        flush.fill_(i & 0xff)
        engine.tau.fill_(tau_schedule(W + i, n_iter, 5.0, 1.0))
        ev[i][0].record()
        loss = engine.step()
        ev[i][1].record()
    torch.cuda.synchronize(); ctx.barrier()
    wall = time.perf_counter() - t0
    if sampler:
        sampler.end()
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    ctx.all_reduce_max_(tmax)
    return float(tmax.item()) / K, wall, loss


DUMP_BYTES = 60 << 20                # under 64 MB with the .npy headers


def dump_outputs(engine, loss, out_dir):
    """What one engine step hands its caller: the loss, the skinned cloud and the parameters after the Adam update, as
    float32 .npy files.  Beyond DUMP_BYTES in all, the skinned cloud keeps a fixed sample of its points (seed 0, sorted
    indices), so that two runs with the same arguments write the same arrays."""
    import numpy as np
    arrays = {"loss": loss.detach().reshape(1), "skinned": engine.skinned}
    arrays.update({"param_" + n: p for n, p in engine.model.named_parameters() if p.requires_grad})
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    sk = arrays["skinned"]
    T, N, _ = sk.shape
    keep = (DUMP_BYTES - sum(a.nbytes for k, a in arrays.items() if k != "skinned")) // (T * 3 * 4)
    if keep < N:
        arrays["skinned"] = sk[:, np.sort(np.random.default_rng(0).choice(N, keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a))


def search_kernel_timing(engine, flush, reps=5):
    """The dominant kernel (chamfer_sym_kernel) alone on this rank's shard: CUDA events on the launch stream, L2 flushed."""
    import torch
    from reart_b200 import _lib
    L = _lib.lib()
    dev = flush.device
    Tl, N = engine.frames.shape[0], engine.cano.shape[0]
    M = engine.frames.shape[1]
    keys_a = torch.empty(Tl * N, dtype=torch.int64, device=dev); keys_b = torch.empty(Tl * M, dtype=torch.int64, device=dev)
    skinned = engine.skinned.detach().contiguous()

    def search():
        _lib.check(L.reart_chamfer_sym_search(_lib.ptr(skinned), _lib.ptr(engine.frames_packed), Tl, N, M,
                                              _lib.ptr(keys_a), _lib.ptr(keys_b), None, 0, _lib.stream_ptr()), "search")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        search()
    k_ms = 0.0
    for i in range(reps):
        flush.fill_(i)
        e0.record(); search(); e1.record(); torch.cuda.synchronize()
        k_ms += e0.elapsed_time(e1)
    return k_ms / reps, 2.0 * Tl * N * M, Tl * (12.0 * (N + M) + 8.0 * (N + M))


def fp32_peak_tf(dev):
    import torch
    props = torch.cuda.get_device_properties(dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sm_max_mhz = float(peaks.get("sm_max_mhz", 1965.0))
    return props.multi_processor_count * 128 * 2 * sm_max_mhz * 1e6 / 1e12, sm_max_mhz, props.multi_processor_count, peaks


def sustained_run(engine, ctx, seconds, ms_per_step_hint, gpu_index, uuid, pairs_per_step, kernel_share, peak_tf, sm_max_mhz):
    """>= `seconds` of back-to-back steps (graph replays, no flush, no host sync inside): what a real 15 000-iteration fit
    sees.  SM clock / power / throttle reasons are sampled during the run (NVML)."""
    import torch
    n = max(50, int(seconds * 1e3 / max(ms_per_step_hint, 1e-3)))
    sampler = ClockSampler(gpu_index, uuid) if ctx.is_main else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier(); torch.cuda.synchronize()
    if sampler:
        sampler.begin()
    e0.record()
    for _ in range(n):
        engine.step()
    e1.record(); torch.cuda.synchronize(); ctx.barrier()
    if sampler:
        sampler.end()
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([e0.elapsed_time(e1) / n], dtype=torch.float64, device=engine.cano.device)
    ctx.all_reduce_max_(ms)
    ms = float(ms.item())
    out = {"seconds": ms * n * 1e-3, "steps": n, "ms_per_step": ms, "value": pairs_per_step / (ms * 1e-3), "unit": UNIT,
           "clocks": clocks, "l2": "no flush between steps (steady state of a fit)"}
    if clocks and clocks.get("sm_mhz"):
        # the step as a whole against the FP32 roofline: all pairs of the step / step time (not the kernel alone)
        tf = FLOP_PER_PAIR * pairs_per_step / ctx.world_size / (ms * 1e-3) / 1e12
        out["step_tflops_per_gpu"] = tf
        out["step_frac_of_peak_at_max_clock"] = tf / peak_tf
        out["step_frac_of_peak_at_observed_clock"] = tf / (peak_tf * clocks["sm_mhz"] / sm_max_mhz)
        out["search_kernel_share_of_step_measured_cold"] = kernel_share
    return out


def culled_entry(workload, ctx, dev, flush, steps, warmup, scaling, brute_loss, brute_ms, late_fit_steps=0):
    """The workload on RelaxationEngine(cull=True): k-d leaf order at set-up, bounds seeded by the previous step's arg-mins,
    bit-identical search results (tests/test_cull_gpu.py); reports ms/step and the fraction of blocks evaluated."""
    import torch
    engine, _, _, T_total, N, P, _ = make_engine(workload, ctx, dev, True, scaling, extra_losses=False, cull=True)
    ms, _, loss = time_engine_steps(engine, ctx, steps, warmup, flush)
    final = float(loss.item())
    engine.culling_stats()
    for _ in range(5):
        engine.step()
    st = engine.culling_stats()
    late = None
    if late_fit_steps:
        # the timed steps above are the first of a fit (tau = 5: every point follows a random part each step, so the seeds
        # are poor).  The same engine further into a fit: a compressed cosine schedule 5 -> 1 over `late_fit_steps` steps,
        # then K more timed steps at the end state.  The brute-force step costs the same at any state.
        from reart_b200.engine import tau_schedule
        done = engine.iteration
        for i in range(done, late_fit_steps):
            engine.step(tau_schedule(i, late_fit_steps, 5.0, 1.0))
        engine.culling_stats()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        for i in range(steps):
            flush.fill_(i & 0xff)
            ev[i][0].record(); l_late = engine.step(1.0); ev[i][1].record()
        torch.cuda.synchronize()
        st2 = engine.culling_stats()
        ms2 = sum(a.elapsed_time(b) for a, b in ev) / steps
        late = {"after_steps": late_fit_steps, "tau": 1.0, "ms_per_step": ms2, "speedup_vs_brute_force_step": brute_ms / ms2,
                "fraction_evaluated": (st2[0] / st2[1]) if st2 and st2[1] else None, "loss": float(l_late.item())}
    engine.release()
    del engine
    torch.cuda.empty_cache()
    pairs = 2.0 * T_total * N * N
    return {"enabled_in_headline": False, "ms_per_step": ms, "value": pairs / (ms * 1e-3), "unit": UNIT, "late_in_a_fit": late,
            "speedup_vs_brute_force_step": brute_ms / ms, "final_loss": final, "final_loss_brute_force": brute_loss,
            "block_pairs_evaluated": st[0] if st else None, "block_pairs_offered": st[1] if st else None,
            "fraction_evaluated": (st[0] / st[1]) if st and st[1] else None,
            "what": "opt-in exact tile culling (csrc/cull.cu, RelaxationEngine(cull=True)): (256-row, 32-target) blocks whose "
                    "bounding-box gap exceeds the upper bounds seeded by the previous step's arg-mins are skipped; search keys "
                    "bit-identical to the brute force on the same clouds (tests/test_cull_gpu.py); the engine reorders both "
                    "clouds into k-d leaves, so float sums associate differently and the losses agree to rounding, not bits"}


def fused_producer_entry(workload, ctx, dev, flush, steps, warmup, scaling, default_loss, default_ms):
    """The workload with the skinning fused into the producer side of the search (RelaxationEngine(fuse_producer=True),
    reart_skinned_chamfer_fwd_bwd_fused): same bits, one launch less; opt-in because it measures slower."""
    import torch
    engine, _, _, T_total, N, P, _ = make_engine(workload, ctx, dev, True, scaling, extra_losses=False, fuse_producer=True)
    ms, _, loss = time_engine_steps(engine, ctx, steps, warmup, flush)
    final = float(loss.item())
    n_ours, _ = kernels_of_one_step(engine)
    engine.release()
    del engine
    torch.cuda.empty_cache()
    return {"enabled_in_headline": False, "ms_per_step": ms, "ms_per_step_default": default_ms, "our_kernels_per_step": n_ours,
            "final_loss": final, "final_loss_default": default_loss, "bit_identical_loss": final == default_loss,
            "what": "skinning fused into the search kernel's prologue (SURVEY N1): every search CTA skins its own 2048 "
                    "canonical points, the first target split also emits the cloud and its x-sorted copy; no skin launch"}


def sweep_entry(workload, ctx, dev, flush, steps, warmup, peak_tf):
    import torch
    engine, _, _, T_total, N, P, desc = make_engine(workload, ctx, dev, True, "strong")
    ms, _, loss = time_engine_steps(engine, ctx, steps, warmup, flush)
    final_loss = float(loss.item())                               # also surfaces any asynchronous error of the steps here
    k_ms, local_pairs, _ = search_kernel_timing(engine, flush, reps=3)
    n_ours, names = kernels_of_one_step(engine)
    pairs = 2.0 * T_total * N * N
    ent = {"workload": workload, "what": desc, "T": T_total, "N": N, "P": P, "steps": steps, "warmup": warmup,
           "ms_per_step": ms, "value": pairs / (ms * 1e-3), "unit": UNIT, "iters_per_s": 1e3 / ms,
           "final_loss": final_loss, "search_kernel_ms": k_ms,
           "search_frac_of_fp32_peak": FLOP_PER_PAIR * local_pairs / (k_ms * 1e-3) / 1e12 / peak_tf,
           "our_kernels_per_step": n_ours,
           "kernels_per_step": {n[:70]: c for n, c in sorted(names.items(), key=lambda kv: -kv[1])}}
    engine.release()
    del engine
    torch.cuda.empty_cache()
    if workload not in ("cfg4", "cfg2"):
        try:
            c = culled_entry(workload, ctx, dev, flush, steps, warmup, "strong", final_loss, ms)
            ent["culled"] = {k: c[k] for k in ("ms_per_step", "value", "speedup_vs_brute_force_step", "fraction_evaluated", "final_loss")}
        except Exception as exc:
            ent["culled"] = {"error": f"{type(exc).__name__}: {exc}"}
    return ent


def candidate_fits(ctx, dev, n_iter=10):
    """cfg5: one `cano_idx` candidate per rank (README.md:60 of the reference), NO communication during the fits, one
    NCCL exchange of the energies at the end (engine.fit_candidates -> all_reduce MIN)."""
    import torch
    from reart_b200.engine import fit_candidates
    from reart_b200.synth import make_sequence
    T, N, P = WORKLOADS["cfg5"]
    seq = make_sequence(T=T, N=N, P=P, seed=2)
    sequence = torch.cat((torch.from_numpy(seq["cano"])[None], torch.from_numpy(seq["frames"])), dim=0).to(dev)
    cands = [int(round(k * T / max(ctx.world_size, 1))) for k in range(ctx.world_size)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier(); torch.cuda.synchronize()
    e0.record()
    best, table = fit_candidates(sequence, cands, P, n_iter, ctx=ctx, criterion="loss", use_graph=True)
    e1.record(); torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    ctx.all_reduce_max_(ms)
    total_pairs = 2.0 * T * N * N * n_iter * len(cands)
    return {"workload": "cfg5", "what": f"{len(cands)} cano_idx candidate fits, one per rank, {n_iter} iterations each (graph capture and "
            "warm-up included in the time), energies exchanged once over NCCL; criterion = final recon loss (the reference's "
            "total_err needs an N x N assignment per frame, infeasible at 32k points for the reference too)",
            "candidates": cands, "best_cano_idx": best, "energies": table, "ms_total": float(ms.item()),
            "value": total_pairs / (float(ms.item()) * 1e-3), "unit": UNIT}


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    from reart_b200 import ops
    from reart_b200.dist import DistContext

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: reart_b200 has no CPU fallback")
    ctx = DistContext.from_env()
    world = ctx.world_size
    assert world == args.gpus or world == 1, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"
    dev = torch.device("cuda", ctx.local_rank)
    torch.cuda.set_device(dev)

    engine, cano_h, frames_h, T_total, N, P, _ = make_engine(args.workload, ctx, dev, not args.no_graph, args.scaling,
                                                             extra_losses=False)
    T = WORKLOADS[args.workload][0]
    lo, hi = engine.frame_range
    frames_local_h = frames_h[lo:hi]
    if getattr(engine, "perm_cano", None) is not None:
        # the engine keeps both clouds in k-d leaf order (a one-time set-up step, like packing): the host copies that the
        # e2e loop streams in every step are put into the same order once
        cano_h = cano_h[engine.perm_cano.cpu()].pin_memory()
        frames_local_h = torch.gather(frames_local_h, 1, engine.perm_frames.cpu()[:, :, None].expand(-1, -1, 3)).pin_memory()
    pairs_per_step = 2.0 * T_total * N * N
    uuid = str(torch.cuda.get_device_properties(dev).uuid)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(ctx.local_rank, uuid) if ctx.is_main else None
    W = max(args.warmup, 3)
    K = args.steps
    ms_per_step, wall_s, loss = time_engine_steps(engine, ctx, K, W, flush, sampler=sampler)
    clocks = sampler.stop() if sampler else None
    value = pairs_per_step / (ms_per_step * 1e-3)
    final_loss = float(loss.item())
    if args.dump_outputs and ctx.is_main:                # before any later section steps the engine again
        dump_outputs(engine, loss, args.dump_outputs)

    # ---- e2e: host buffers in, loss out, every step.  The H2D of step i+1 (pinned host clouds -> staging buffer, copy
    # stream) runs while step i computes; each step then takes its clouds from the staging buffer (D2D), re-packs the
    # observed frames, runs the iteration and reads the loss back (a host sync per step, like the reference loop's print).
    cano_d, frames_d = engine.cano, engine.frames
    h2d = cano_h.numel() * 4 + frames_local_h.numel() * 4
    copy_stream = torch.cuda.Stream()
    stage_c = [torch.empty_like(cano_d) for _ in range(2)]
    stage_f = [torch.empty_like(frames_d) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            stage_c[slot].copy_(cano_h, non_blocking=True)
            stage_f[slot].copy_(frames_local_h, non_blocking=True)
            ready[slot].record(copy_stream)

    K2 = max(3, min(K, 10))
    pinned_loss = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_done = [torch.cuda.Event() for _ in range(2)]

    def e2e_loop(deferred):
        """deferred = False: the loss of step i is on the host before step i+1 is launched (a host sync per step, like the
        reference loop's print) -- the reported e2e.  True: the same copies and the same read-back every step, but the host
        looks at step i's loss only after it has launched step i+1 (what a caller that logs asynchronously gets)."""
        for s_ in range(2):
            consumed[s_].record()
        torch.cuda.synchronize(); ctx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        host_loss = None
        for i in range(K2 + 2):
            if i == 2:                                            # steps 0 and 1 warm both staging slots up (each has its
                flush.fill_(1); torch.cuda.synchronize(); ctx.barrier()   # own captured graph); time steps 2..K2+1
                e0.record()
                prefetch(i & 1)                                   # the first timed step's H2D is inside the timed region
            elif i < 2:
                torch.cuda.synchronize()
                prefetch(i & 1)
            if i >= 2 and i + 1 <= K2 + 1:
                prefetch((i + 1) & 1)                             # next step's clouds: overlaps this step's compute
            torch.cuda.current_stream().wait_event(ready[i & 1])
            # staging buffer -> engine clouds (D2D) -> re-pack -> iteration: ONE graph launch (engine.step(ingest=...))
            lval = engine.step(ingest=(i & 1, stage_c[i & 1], stage_f[i & 1]))
            consumed[i & 1].record()
            if not deferred:
                host_loss = lval.to("cpu", non_blocking=False)         # D2H read of the step's result
            else:
                pinned_loss[i & 1].copy_(lval.reshape(1), non_blocking=True)
                loss_done[i & 1].record()
                if i >= 1:                                             # the previous step's loss, now that this step is in flight
                    loss_done[(i - 1) & 1].synchronize()
                    host_loss = pinned_loss[(i - 1) & 1].clone()
        if deferred:
            loss_done[(K2 + 1) & 1].synchronize()
            host_loss = pinned_loss[(K2 + 1) & 1].clone()
        e1.record(); torch.cuda.synchronize()
        t2 = torch.tensor([e0.elapsed_time(e1) / K2], dtype=torch.float64, device=dev)
        ctx.all_reduce_max_(t2)
        _ = float(host_loss)
        return pairs_per_step / (float(t2.item()) * 1e-3)

    e2e_value = e2e_loop(False)
    e2e_deferred = e2e_loop(True)

    # ---- roofline of the dominant kernel (chamfer_sym_kernel), timed alone with CUDA events on this stream
    Tl = hi - lo
    k_ms, local_pairs, alg_bytes = search_kernel_timing(engine, flush)
    achieved_tf = FLOP_PER_PAIR * local_pairs / (k_ms * 1e-3) / 1e12
    peak_tf, sm_max_mhz, n_sms, peaks = fp32_peak_tf(dev)
    ms_ffma, ops_ffma = ops.fp32_probe(0, iters=2000, device=dev)
    ffma_tf = 2.0 * ops_ffma / (ms_ffma * 1e-3) / 1e12
    roofline = {"bound": "fp32_fma", "kernel": "chamfer_sym_kernel<8,1>", "achieved": achieved_tf, "peak": peak_tf,
                "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                "peak_source": f"SMs({n_sms}) x 128 lanes x 2 x sm_max_mhz({sm_max_mhz:.0f}) from "
                               "MEASURED_PEAKS.json (it carries no FP32 entry; BASELINE.md section 3)",
                "peak_measured_ffma": ffma_tf, "frac_of_measured_ffma": achieved_tf / ffma_tf,
                "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_per_step,
                "flop_per_pair": FLOP_PER_PAIR, "pairs_per_launch": local_pairs,
                "executed_flop_note": "one evaluation per unordered pair feeds both directions: executed FLOP = half the credited",
                "hbm_achieved_gbs": alg_bytes / (k_ms * 1e-3) / 1e9, "hbm_peak_gbs": peaks.get("hbm_gbs"),
                "traffic": None}
    for cand in ("r02_sym_traffic.json", "r01_sym_traffic.json"):
        try:    # dram bytes of the same kernel from a committed `ncu --set full` capture; only for the captured shape
            tr = json.load(open(os.path.join(ROOT, "profiles", cand)))
            if tr.get("workload") == args.workload and tr.get("frames_per_launch") == Tl:
                roofline["traffic"] = tr["dram_bytes_read"] + tr["dram_bytes_write"]
                roofline["traffic_unit"] = "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)"
                roofline["traffic_source"] = f"profiles/{cand} (one ncu --set full capture of this kernel at this shape; not re-measured in this run)"
                roofline["algorithmic_bytes_per_launch"] = alg_bytes
                break
        except Exception:
            pass

    # ---- what one step launches (torch profiler / CUPTI on one eager iteration)
    n_ours, step_kernels = kernels_of_one_step(engine)
    table = 8                                                     # head, skin_fwd_sorted, search, energy cols + rows, skin bwd + reduce, tail
    launches_per_step = n_ours if n_ours else table

    # ---- sustained run
    sustained = None
    if args.sustained_s > 0:
        sustained = sustained_run(engine, ctx, args.sustained_s, ms_per_step, ctx.local_rank, uuid, pairs_per_step,
                                  k_ms / ms_per_step, peak_tf, sm_max_mhz)

    engine.release()
    del engine
    torch.cuda.empty_cache()

    # ---- the same workload with the opt-in exact tile culling (a second engine; the headline above is the brute force)
    culling = None
    if args.workload != "cfg4":
        try:
            culling = culled_entry(args.workload, ctx, dev, flush, K, W, args.scaling, final_loss, ms_per_step,
                                   late_fit_steps=600 if (world == 1 and args.workload == "cfg3_16k" and not args.no_sweep) else 0)
        except Exception as exc:
            culling = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- and with the skinning fused into the producer side of the search (SURVEY N1; opt-in, measured beside the default)
    fused = None
    if args.workload != "cfg4":
        try:
            fused = fused_producer_entry(args.workload, ctx, dev, flush, K, W, args.scaling, final_loss, ms_per_step)
        except Exception as exc:
            fused = {"error": f"{type(exc).__name__}: {exc}"}

    # ---- sweep over the other BASELINE configs (N=1) / candidate fits (N>1)
    sweep = None
    if not args.no_sweep and args.workload == "cfg3_16k":
        sweep = []
        if world == 1:
            for wl in SWEEP:
                big = WORKLOADS[wl][1] >= 262144
                try:     # cfg2 refreshes its assignments every 5 steps: time enough steps to see the steady state
                    sweep.append(sweep_entry(wl, ctx, dev, flush, 2 if big else (25 if wl == "cfg2" else 5), 3, peak_tf))
                except Exception as exc:                          # never lose the headline line to a sweep failure
                    import traceback
                    sweep.append({"workload": wl, "error": f"{type(exc).__name__}: {exc}", "traceback": traceback.format_exc()[-1500:]})
        else:
            try:
                sweep.append(candidate_fits(ctx, dev))
            except Exception as exc:
                sweep.append({"workload": "cfg5", "error": f"{type(exc).__name__}: {exc}"})

    if ctx.is_main:
        cpu = cpu_py = None
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample = cpu_reference_throughput(T, N, budget_s=12.0)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
            try:
                cpu_py = reference_python_cpu_baseline(T, N, P)
            except Exception as exc:
                cpu_py = {"error": f"{type(exc).__name__}: {exc}"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config_dict(args, T_total, N, P, world),
                "iters_per_s": 1e3 / ms_per_step, "wall_s_timed_region": wall_s, "final_loss": final_loss,
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                        "value_deferred_readback": e2e_deferred,
                        "what": "per step: pinned host cano+frames -> H2D (copy stream, overlapping the previous step) -> "
                                "D2D into the engine -> pack -> full iteration (these three: one CUDA-graph launch) -> loss D2H + host sync"},
                "gpu_launches": launches_per_step * K,
                "gpu_launches_per_step": launches_per_step,
                "gpu_launches_source": "torch profiler (CUPTI) on one eager iteration: kernels in namespace reart" if n_ours
                                       else "table (profiler unavailable)",
                "step_kernels": {n[:70]: c for n, c in sorted(step_kernels.items(), key=lambda kv: -kv[1])},
                "cuda_graph": not args.no_graph,
                "roofline": roofline, "culling": culling, "fused_producer": fused, "cpu_baseline": cpu, "cpu_baseline_reference_python": cpu_py,
                "sustained": sustained, "sweep": sweep}
        print(json.dumps(line), flush=True)
    # teardown: captured graphs reference the NCCL communicator; with more than one rank leave through os._exit after
    # a final barrier so a slow communicator teardown can never hold the job
    ctx.barrier()
    if world > 1:
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
