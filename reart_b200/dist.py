"""Frame-sharded data parallelism for the energy evaluation (SURVEY.md section 8e).

The energy is a sum over frames (networks/loss.py:27-28), per-frame parameters are private to their frame
and only the small shared parameters (seg MLP, or axis/moment of the kinematic model) couple the frames.
One process per GPU; frames are split into contiguous blocks; per iteration ONE all-reduce (sum) of a
flat bucket holding the shared-parameter gradients (+ the scalar loss).  Backend: NCCL on GPUs
(NVLink 5 / NVSwitch), gloo on CPU for the tests.  The reference has no distributed code at all.
"""
from __future__ import annotations

import os
from typing import Iterable, List, Tuple

import torch
import torch.distributed as dist


def shard_bounds(total: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous block [lo, hi) of ``total`` frames owned by ``rank`` (sizes differ by at most one)."""
    base, rem = divmod(total, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class DistContext:
    """Thin wrapper over torch.distributed; world_size 1 needs no process group."""

    def __init__(self, rank: int = 0, world_size: int = 1, local_rank: int = 0, backend: str | None = None):
        self.rank, self.world_size, self.local_rank, self.backend = rank, world_size, local_rank, backend

    @classmethod
    def from_env(cls, backend: str | None = None) -> "DistContext":
        ws = int(os.environ.get("WORLD_SIZE", "1"))
        rank = int(os.environ.get("RANK", "0"))
        local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if ws > 1 and not dist.is_initialized():
            if backend is None:
                backend = "nccl" if torch.cuda.is_available() else "gloo"
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29511")
            if backend == "nccl":
                torch.cuda.set_device(local_rank)
                dist.init_process_group(backend, rank=rank, world_size=ws,
                                        device_id=torch.device("cuda", local_rank))
            else:
                dist.init_process_group(backend, rank=rank, world_size=ws)
        return cls(rank, ws, local_rank, backend)

    @property
    def is_main(self) -> bool:
        return self.rank == 0

    def frames(self, total: int) -> Tuple[int, int]:
        return shard_bounds(total, self.world_size, self.rank)

    def barrier(self) -> None:
        if self.world_size > 1:
            dist.barrier()

    def all_reduce_sum_(self, t: torch.Tensor) -> torch.Tensor:
        if self.world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t

    def all_reduce_max_(self, t: torch.Tensor) -> torch.Tensor:
        if self.world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t

    def all_gather_scalar(self, value: float, device=None) -> List[float]:
        if self.world_size == 1:
            return [float(value)]
        t = torch.tensor([float(value)], dtype=torch.float64, device=device or ("cuda" if self.backend == "nccl" else "cpu"))
        out = [torch.zeros_like(t) for _ in range(self.world_size)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def destroy(self) -> None:
        if self.world_size > 1 and dist.is_initialized():
            dist.destroy_process_group()


class GradBucket:
    """One flat buffer for the shared-parameter gradients (+ extra scalars): a single latency-bound
    all-reduce per iteration (~10 KB for the relaxation model) instead of one per tensor."""

    def __init__(self, params: Iterable[torch.nn.Parameter], extra_scalars: int = 1):
        self.params = [p for p in params]
        self.sizes = [p.numel() for p in self.params]
        n = sum(self.sizes) + extra_scalars
        ref = self.params[0]
        self.flat = torch.zeros(n, dtype=torch.float32, device=ref.device)
        self.extra = self.flat[sum(self.sizes):]

    def pack(self) -> None:
        off = 0
        for p, n in zip(self.params, self.sizes):
            if p.grad is None:
                self.flat[off:off + n].zero_()
            else:
                self.flat[off:off + n].copy_(p.grad.reshape(-1))
            off += n

    def unpack(self) -> None:
        off = 0
        for p, n in zip(self.params, self.sizes):
            if p.grad is None:
                p.grad = torch.empty_like(p)
            p.grad.copy_(self.flat[off:off + n].view_as(p))
            off += n

    def all_reduce(self, ctx: DistContext) -> None:
        self.pack()
        if ctx.world_size > 1:
            if getattr(self, "_reducer", None) is None:
                self._reducer = make_small_all_reduce(ctx, self.flat.numel(), self.flat.device)
            self._reducer(self.flat)
        self.unpack()


class OneShotAllReduce:
    """In-place sum of a small float tensor across ranks through ``reart_allreduce_oneshot`` (peer memory over
    NVLink).  Buffers come from torch's symmetric-memory allocator, which also exchanges the peer mappings.
    Raises at construction if symmetric memory is unavailable -- callers fall back to NCCL."""

    def __init__(self, ctx: DistContext, numel: int, device):
        import torch.distributed._symmetric_memory as symm_mem
        from . import _lib
        self._lib = _lib
        self.ctx = ctx
        self.n = int(numel)
        self.n_pad = (self.n + 63) // 64 * 64
        total = 2 * self.n_pad + max(64, ctx.world_size)
        self.buf = symm_mem.empty(total, dtype=torch.float32, device=device)
        self.buf.zero_()
        torch.cuda.synchronize(device)
        hdl = symm_mem.rendezvous(self.buf, dist.group.WORLD)
        self.hdl = hdl
        self.peer_base = torch.tensor([int(p) for p in hdl.buffer_ptrs], dtype=torch.int64, device=device)
        self.epoch = torch.zeros(1, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        ctx.barrier()                                            # every rank's flags are zero before anyone signals

    def __call__(self, flat: torch.Tensor) -> torch.Tensor:
        assert flat.is_contiguous() and flat.dtype == torch.float32 and flat.numel() == self.n
        L = self._lib.lib()
        with torch.cuda.device(flat.device):
            self._lib.check(L.reart_allreduce_oneshot(self._lib.ptr(self.peer_base), self.ctx.rank, self.ctx.world_size,
                                                      self.n, self.n_pad, self._lib.ptr(self.epoch), self._lib.ptr(flat),
                                                      self._lib.stream_ptr()), "reart_allreduce_oneshot")
        return flat


def make_small_all_reduce(ctx: DistContext, numel: int, device):
    """Best available in-place sum for a small bucket: the peer-memory one-shot kernel, else NCCL."""
    if ctx.world_size <= 1:
        return None
    if ctx.backend == "nccl" and os.environ.get("REART_ONESHOT_ALLREDUCE", "1") != "0":
        try:
            return OneShotAllReduce(ctx, numel, device)
        except Exception as exc:                                  # symmetric memory not available on this system
            if ctx.is_main:
                import sys
                print(f"[reart_b200] one-shot all-reduce unavailable ({type(exc).__name__}: {exc}); using NCCL",
                      file=sys.stderr, flush=True)
    return lambda flat: ctx.all_reduce_sum_(flat)


def gather_frames(ctx: DistContext, x: torch.Tensor, total: int) -> torch.Tensor:
    """The complete [total, ...] tensor of a per-frame tensor whose rows [lo, hi) each rank holds (``shard_bounds``), on
    every rank: the uneven shards are padded to the largest one, all-gathered and trimmed.  Collective."""
    if ctx.world_size <= 1:
        return x
    bounds = [shard_bounds(total, ctx.world_size, r) for r in range(ctx.world_size)]
    rows = max(hi - lo for lo, hi in bounds)
    pad = x.new_zeros((rows,) + tuple(x.shape[1:]))
    pad[:x.shape[0]] = x
    out = [torch.empty_like(pad) for _ in bounds]
    dist.all_gather(out, pad)
    return torch.cat([o[:hi - lo] for o, (lo, hi) in zip(out, bounds)])


def flow_pairs_for_rank(T: int, cano_idx: int, lo: int, hi: int):
    """Which consecutive pairs of the COMPLETE sequence (canonical frame inserted at cano_idx, run_robot.py:204-207)
    a rank owning skinned frames [lo, hi) evaluates, and where each side comes from.

    Returns (p0, p1, a_src, b_src): pairs p in [p0, p1) and per pair the source of complete[p] / complete[p+1] as
    ("local", i) (i-th local frame), ("cano",) or ("halo",) (the previous rank's last frame).  A pair belongs to
    the owner of its SECOND frame, or of its first one when the second is the canonical frame; every pair is
    owned exactly once and only a previous-rank halo is ever needed."""
    def src(k):
        if k == cano_idx:
            return ("cano",)
        g = k if k < cano_idx else k - 1
        if lo <= g < hi:
            return ("local", g - lo)
        if g == lo - 1:
            return ("halo",)
        return None

    def frame(k):
        return None if k == cano_idx else (k if k < cano_idx else k - 1)

    pairs, a_src, b_src = [], [], []
    for p in range(T):
        gB, gA = frame(p + 1), frame(p)
        owner_frame = gB if gB is not None else gA
        if owner_frame is not None and lo <= owner_frame < hi:
            pairs.append(p); a_src.append(src(p)); b_src.append(src(p + 1))
    if not pairs:
        return 0, 0, [], []
    assert pairs == list(range(pairs[0], pairs[-1] + 1)) and all(x is not None for x in a_src + b_src)
    return pairs[0], pairs[-1] + 1, a_src, b_src


def flow_window_plan(T: int, cano_idx: int, bounds: List[Tuple[int, int]]) -> List[dict]:
    """The windows and the neighbour-frame exchange of the native kinematic flow step (``reart_kin_flow``), for every rank
    at once: plain host arithmetic on (T skinned frames, cano_idx, shard bounds [(lo, hi)] per rank), so every rank
    computes the same plan.

    Rank r's window is complete indices [j0, j0 + K) with j0 = max(0, j(lo) - 1) and j0 + K - 1 = min(T, j(hi - 1) + 1),
    j(g) the complete index of skinned frame g: its frames and both their neighbours.  Per rank a dict with
      j0, K;  slots: per slot ("local", i) | ("cano",) | ("prev",) (rank r-1's last frame) | ("next",) (rank r+1's first);
      q0, q1: the pairs of the window whose loss the rank counts (``flow_pairs_for_rank``'s, window-relative);
      send_prev / send_next: send the first / last local frame to rank r-1 / r+1;  recv_prev / recv_next: the slot that
      receives rank r-1's last / rank r+1's first frame, or None.
    Frames only travel forward (no gradient comes back): where the canonical frame separates two shards, nothing is sent."""
    def j(g):
        return g if g < cano_idx else g + 1

    plans = []
    for lo, hi in bounds:
        j0, j1 = max(0, j(lo) - 1), min(T, j(hi - 1) + 1)
        slots = []
        for k in range(j0, j1 + 1):
            g = None if k == cano_idx else (k if k < cano_idx else k - 1)
            if g is None:
                slots.append(("cano",))
            elif lo <= g < hi:
                slots.append(("local", g - lo))
            elif g == lo - 1:
                slots.append(("prev",))
            else:
                assert g == hi, (g, lo, hi)
                slots.append(("next",))
        p0, p1, _, _ = flow_pairs_for_rank(T, cano_idx, lo, hi)
        q0, q1 = (p0 - j0, p1 - j0) if p1 > p0 else (0, 0)
        assert 0 <= q0 <= q1 <= len(slots) - 1
        plans.append(dict(j0=j0, K=len(slots), slots=slots, q0=q0, q1=q1,
                          recv_prev=next((s for s, x in enumerate(slots) if x[0] == "prev"), None),
                          recv_next=next((s for s, x in enumerate(slots) if x[0] == "next"), None)))
    for r, pl in enumerate(plans):
        pl["send_prev"] = r > 0 and plans[r - 1]["recv_next"] is not None
        pl["send_next"] = r + 1 < len(plans) and plans[r + 1]["recv_prev"] is not None
    return plans


class _HaloPrev(torch.autograd.Function):
    """Forward: every rank sends its last local skinned frame to the next rank and receives the previous rank's
    (rank 0 receives nothing and gets zeros).  Backward: the gradient of the received frame travels back.
    One frame [N,3] per shard boundary per direction -- the only data-path message of the flow loss."""

    @staticmethod
    def forward(ctx, x_last, rank, world):
        ctx.rank, ctx.world = rank, world
        recv = torch.zeros_like(x_last)
        ops_ = []
        send = x_last.detach().contiguous()
        if rank < world - 1:
            ops_.append(dist.P2POp(dist.isend, send, rank + 1))
        if rank > 0:
            ops_.append(dist.P2POp(dist.irecv, recv, rank - 1))
        if ops_:
            for req in dist.batch_isend_irecv(ops_):
                req.wait()
        return recv

    @staticmethod
    def backward(ctx, g_recv):
        rank, world = ctx.rank, ctx.world
        g_last = torch.zeros_like(g_recv)
        ops_ = []
        g_send = g_recv.contiguous()
        if rank > 0:
            ops_.append(dist.P2POp(dist.isend, g_send, rank - 1))
        if rank < world - 1:
            ops_.append(dist.P2POp(dist.irecv, g_last, rank + 1))
        if ops_:
            for req in dist.batch_isend_irecv(ops_):
                req.wait()
        return g_last, None, None


def halo_from_previous_rank(x_last: torch.Tensor, ctx: DistContext) -> torch.Tensor:
    if ctx.world_size <= 1:
        return torch.zeros_like(x_last)
    return _HaloPrev.apply(x_last, ctx.rank, ctx.world_size)


def select_best_candidate(ctx: DistContext, energy: float, device=None) -> Tuple[int, List[float]]:
    """cano_idx candidate fits are independent runs, one per rank (README.md:60): gather one scalar energy per rank and
    return (rank of the lowest energy, all energies).  The reference's energy is total_err (run_robot.py:306-314); that
    is what ``engine.candidate_energy`` / ``engine.fit_candidates(criterion="total_err")`` compute."""
    energies = ctx.all_gather_scalar(energy, device=device)
    best = min(range(len(energies)), key=lambda i: (energies[i], i))
    return best, energies
