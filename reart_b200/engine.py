"""The optimisation iteration of the reference's run scripts, B200-native.

``RelaxationEngine.step`` is one pass of run_robot.py:154-221 for ``--model=base`` with the recon loss:
seg MLP -> straight-through gumbel weights -> 6D -> R -> fused [skin -> bidirectional Chamfer -> sum -> backward]
-> (multi-GPU: one all-reduce of the shared-parameter gradients) -> Adam.  The steady-state iteration is
captured once in a CUDA graph (NCCL all-reduce included) and replayed, so neither Python nor the ~4 host syncs
per iteration of the reference loop (SURVEY Q20) sit on the critical path.

``KinematicEngine.step`` is the same for ``--model=kinematic`` (fused tree FK instead of the 6D proposals).
Frames are sharded across ranks by ``DistContext``; per-frame parameters stay local to their rank.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F

from . import ops
from .dist import DistContext, GradBucket, make_small_all_reduce
from .model import BaseModel, KinematicModel


class _EngineBase:
    def __init__(self, ctx: Optional[DistContext], use_graph: bool):
        self.ctx = ctx or DistContext()
        self.use_graph = use_graph
        self._graphs = {}
        self.iteration = 0

    # subclasses: _iteration() -> loss tensor (local part), self.optimizer, self.bucket
    def _run_iteration(self):
        src = getattr(self, "_ingest_src", None)
        if src is not None:
            # fresh clouds for this step (a caller streaming data in): device copies + re-pack as part of the iteration,
            # i.e. inside the captured graph -- one launch per step instead of four enqueues in front of it
            cano_src, frames_src = src
            self.cano.copy_(cano_src)
            self.frames.copy_(frames_src)
            ops.pack_cloud(self.frames, out=self.frames_packed)
            if getattr(self, "search_culled", False):
                torch.gather(self.frames, 1, self._search_gather, out=self.frames_search)
                ops.pack_cloud(self.frames_search, out=self.frames_search_packed)
        if getattr(self, "native", False):
            return self._run_iteration_native()
        if getattr(self, "sink", None) is not None:
            return self._run_iteration_sink()
        # set_to_none: AccumulateGrad then adopts the fresh gradient tensors (no zero-fill and no add kernels); inside a
        # captured graph their addresses are stable because they come from the graph's private pool
        self.optimizer.zero_grad(set_to_none=True)
        loss = self._iteration()
        loss.backward()
        if self.ctx.world_size > 1:
            self.bucket.extra[0] = loss.detach()
            self.bucket.all_reduce(self.ctx)
            total = self.bucket.extra[0]
        else:
            total = loss.detach()
        self.optimizer.step()
        return total

    def _run_iteration_sink(self):
        """Relaxation model: the seg-MLP backward writes into a flat bucket that also carries the loss and is
        all-reduced in place from inside the backward (no pack/unpack copies around the collective)."""
        self.optimizer.zero_grad(set_to_none=True)
        loss = self._iteration()
        self.sink.extra[0:1].copy_(loss.detach().reshape(1))
        self.sink.active = True
        try:
            loss.backward()
        finally:
            self.sink.active = False
        total = self.sink.extra[0]
        self.optimizer.step()
        return total

    def _opt_params(self):
        return [p for g in self.optimizer.param_groups for p in g["params"]]

    def _opt_state_tensors(self):
        return [v for st in self.optimizer.state.values() for v in st.values() if torch.is_tensor(v)]

    def _aux_state_tensors(self):
        """Other device state an iteration carries from step to step (restored after a capture's warm-up)."""
        return []

    def _variant(self):
        """Which flavour of the iteration the NEXT step runs (hashable); one CUDA graph is captured per flavour."""
        return None

    def _capture(self, variant):
        """Warm up (allocator, library handles, NCCL communicator, lazily created Adam state), capture one
        iteration, then put parameters, optimiser state and the RNG stream back where they were, so a graph
        run is step-for-step the same optimisation as an eager run (also when a flavour is first needed mid-run)."""
        params = self._opt_params()
        dev = params[0].device
        rng_state = torch.cuda.get_rng_state(dev)
        fresh_state = len(self._opt_state_tensors()) == 0          # torch creates Adam state lazily in the first step
        snapshot = [p.detach().clone() for p in params]
        opt_snapshot = [v.detach().clone() for v in self._opt_state_tensors()]
        aux_snapshot = [v.detach().clone() for v in self._aux_state_tensors()]
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                self._run_iteration()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self.ctx.barrier()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            static_loss = self._run_iteration()
        self._graphs[variant] = (g, static_loss)
        with torch.no_grad():
            for p, q in zip(params, snapshot):
                p.copy_(q)
            if fresh_state:
                for v in self._opt_state_tensors():
                    v.zero_()                                  # step, exp_avg, exp_avg_sq (kept in place)
            else:
                for v, q in zip(self._opt_state_tensors(), opt_snapshot):
                    v.copy_(q)
            for v, q in zip(self._aux_state_tensors(), aux_snapshot):
                v.copy_(q)
        torch.cuda.set_rng_state(rng_state, dev)
        torch.cuda.synchronize()

    def release(self) -> None:
        """Drop the captured graphs.  Must happen before the NCCL process group is destroyed: tearing down a
        communicator that a live CUDA graph still references blocks inside destroy_process_group()."""
        self._graphs = {}
        torch.cuda.synchronize()

    def step(self, tau: Optional[float] = None, ingest=None) -> torch.Tensor:
        """One optimisation iteration; returns the (all-rank) loss as a device tensor -- no host sync.

        ``ingest`` = (slot, cano_src, frames_src): run the step on NEW clouds taken from the device tensors ``cano_src``
        [N,3] / ``frames_src`` [T_local,N,3] (same shapes as the engine's; e.g. staging buffers an H2D copy just filled).
        The copies and the re-pack are part of the captured iteration; ``slot`` (hashable) names the staging buffers, one
        graph is captured per slot, so alternate between a fixed set of them.  Not available with ``cull=True`` (the
        engine keeps its clouds in its own order)."""
        if tau is not None:
            self.tau.fill_(float(tau))
        self.iteration += 1
        variant = self._variant()
        self._cur_variant = variant                            # fixed for this step (warm-up and capture included)
        self._ingest_src = None
        key = variant
        if ingest is not None:
            if getattr(self, "cull", False):
                raise ValueError("ingest is not available with cull=True")
            slot, cano_src, frames_src = ingest
            assert cano_src.shape == self.cano.shape and frames_src.shape == self.frames.shape
            self._ingest_src = (cano_src, frames_src)
            key = (variant, "ingest", slot, cano_src.data_ptr(), frames_src.data_ptr())
        try:
            if not self.use_graph:
                out = self._run_iteration()
                self._after_replay(variant)
                return out
            if key not in self._graphs:
                self._capture(key)
            g, static_loss = self._graphs[key]
            g.replay()
            self._after_replay(variant)
            return static_loss
        finally:
            self._ingest_src = None

    def _after_replay(self, variant):
        pass


# search="auto" runs the culled search from this many points per cloud on (both clouds): the coarse bounds of cull.cu
# start culling there
SEARCH_CULLED_MIN_POINTS = 8192


class RelaxationEngine(_EngineBase):
    """Relaxation model (networks/model.py BaseModel) + recon loss, frame-sharded."""

    def __init__(self, cano: torch.Tensor, frames: torch.Tensor, num_parts: int, ctx: Optional[DistContext] = None,
                 trans_lr: float = 1e-2, seg_lr: float = 1e-3, weight_decay: float = 0.0, use_graph: bool = True,
                 seed: int = 2, flow_ref=None, cano_idx: int = 0, lambda_flow: float = 1.0, robust_flow: bool = False,
                 native: Optional[bool] = None, betas=(0.9, 0.999), eps: float = 1e-8, assign: Optional[dict] = None,
                 cull: Optional[bool] = None, fuse_producer: bool = False, search: str = "auto"):
        """assign: optional dict(downsample=4, assign_gap=5, lambda_assign=0.3, assign_iter=0, mode="add"|"replace")
        enabling the assignment loss (run_robot.py:164-187): from iteration ``assign_iter`` on it is ADDED to the Chamfer
        loss (run_real.py / run_sapien.py) or REPLACES it (run_robot.py's if/else, SURVEY Q12); assignments are refreshed
        on the GPU (``reart_lap``) at ``assign_iter`` and whenever ``i % assign_gap == 0``, inside the captured iteration.
        flow_ref: optional ``flow_utils.FlowReference`` (run_robot.py:78-84) enabling the flow loss of
        run_robot.py:194-213.  Consecutive frames couple across shard boundaries: under frame sharding each rank
        receives one skinned frame per iteration from the previous rank (``dist.halo_from_previous_rank``).
        search: "brute" evaluates every pair; "culled" runs the exact culled search on k-d ordered copies of the clouds
        while everything else stays in the caller's order -- bit-identical to "brute" (native fused iteration only);
        "auto" picks "culled" from ``SEARCH_CULLED_MIN_POINTS`` points per cloud on, where the coarse bounds of cull.cu make
        it faster.  ``cull=True`` (the engine reorders the caller's clouds) and ``fuse_producer=True`` search brute force."""
        super().__init__(ctx, use_graph)
        self.flow_ref, self.cano_idx, self.lambda_flow, self.robust_flow = flow_ref, cano_idx, lambda_flow, robust_flow
        # the flow loss couples consecutive frames: under frame sharding each rank evaluates the pairs whose second
        # frame it owns and receives ONE skinned frame (the previous rank's last) per iteration (dist.py)
        dev = cano.device
        if frames.shape[0] < self.ctx.world_size:
            raise ValueError(f"{frames.shape[0]} frames cannot be sharded over {self.ctx.world_size} ranks: every rank must "
                             "own at least one frame (an empty shard would skip the step's collectives)")
        lo, hi = self.ctx.frames(frames.shape[0])
        self.frame_range = (lo, hi)
        self.total_frames = int(frames.shape[0])
        self.cano = cano.float().contiguous()
        self.frames = frames[lo:hi].float().contiguous()          # local shard of the observed frames
        # cull=True: the engine's own clouds are put into k-d leaf order ONCE here (256-point leaves for the canonical
        # cloud = one warp of the search, 32-point leaves for the observed frames = one target chunk); ``perm_cano`` /
        # ``perm_frames`` map engine order -> caller order (engine.skinned[:, k] is caller point perm_cano[k]).  Every
        # order-dependent float sum then associates differently: the same optimisation, not the same bits.  The default
        # (search="auto") culls without this: only the search runs on k-d ordered copies (search_order_rows / _tgt).
        self.cull = bool(cull) if cull is not None else False
        # fuse_producer: skin inside the search kernel's prologue (reart_skinned_chamfer_fwd_bwd_fused; SURVEY N1).  Bit-identical,
        # one launch less, but measured SLOWER than the separate skin kernel on B200 (profiles/r02_fused_producer.md), so opt-in.
        self.fuse_producer = bool(fuse_producer) and not self.cull
        if self.cull and (flow_ref is not None or native is False):
            raise ValueError("exact tile culling runs on the native fused iteration (recon / assignment losses)")
        self.perm_cano = self.perm_frames = None
        if search not in ("auto", "brute", "culled"):
            raise ValueError("search must be 'auto', 'brute' or 'culled'")
        native_path = (flow_ref is None) if native is None else bool(native)
        can_order = native_path and not self.cull and not self.fuse_producer
        if search == "culled" and not can_order:
            raise ValueError("search='culled' runs on the native fused iteration, without cull=True or fuse_producer=True")
        self.search_culled = can_order and (search == "culled" or (
            search == "auto" and min(self.cano.shape[0], self.frames.shape[1]) >= SEARCH_CULLED_MIN_POINTS))
        cano_orig, frames_orig = self.cano, self.frames
        if self.cull:
            # k-d order refined well below the chunk sizes of the search (256 rows / 32 targets): the chunks stay the same
            # compact sets, and consecutive points become nearest neighbours -- whose arg-mins cull.cu tries as extra seeds
            self.perm_cano = ops.kd_order(self.cano[None], 8)[0]
            self.perm_frames = ops.kd_order(self.frames, 4)
            self.cano = self.cano[self.perm_cano].contiguous()
            self.frames = torch.gather(self.frames, 1, self.perm_frames[:, :, None].expand(-1, -1, 3)).contiguous()
        self.frames_packed = ops.pack_cloud(self.frames)          # constant over the optimisation: packed once
        self.search_order_rows = self.search_order_tgt = None
        if self.search_culled:
            # the culled search's own order, fixed here (256-row blocks = one warp of the search, 32-target chunks); the
            # engine's clouds, outputs and every sum stay in the caller's order.  Any order is exact, a stale one (after
            # step(ingest=...)) only culls less.
            self.search_order_rows = ops.search_order(self.cano[None], 256)[0].int()
            self.search_order_tgt = ops.search_order(self.frames, 32).int()
            self.search_inv_rows = torch.empty_like(self.search_order_rows)
            self.search_inv_rows[self.search_order_rows.long()] = torch.arange(
                self.cano.shape[0], dtype=torch.int32, device=dev)
            self.search_inv_tgt = torch.empty_like(self.search_order_tgt)
            self.search_inv_tgt.scatter_(1, self.search_order_tgt.long(), torch.arange(
                self.frames.shape[1], dtype=torch.int32, device=dev)[None].expand_as(self.search_order_tgt).contiguous())
            self._search_gather = self.search_order_tgt.long()[:, :, None].expand(-1, -1, 3)
            self.frames_search = torch.gather(self.frames, 1, self._search_gather).contiguous()
            self.frames_search_packed = ops.pack_cloud(self.frames_search)
        torch.manual_seed(seed)                                    # identical init + gumbel draws on every rank
        torch.cuda.manual_seed_all(seed)
        self.model = BaseModel(num_parts=num_parts, pose_len=hi - lo).to(dev)
        self.tau = torch.ones((), device=dev)
        seg_params = [p for p in self.model.seg_head.parameters() if p.requires_grad]
        self.optimizer = torch.optim.Adam(
            [{"params": [self.model.proposal_6d, self.model.proposal_t], "lr": trans_lr},
             {"params": seg_params, "lr": seg_lr}], lr=1e-3, weight_decay=weight_decay, capturable=use_graph, fused=True)
        self.bucket = None
        H = self.model.seg_head.model[0].weight.shape[0]
        reducer = make_small_all_reduce(self.ctx, 4 * H + num_parts * H + 1, dev)
        self.sink = ops.GradSink(H, num_parts, dev, extra_scalars=1, reducer=reducer)
        self.model.seg_head.grad_sink = self.sink
        self.pairs_per_step_local = 2 * (hi - lo) * self.cano.shape[0] * self.frames.shape[1]
        # recon-only iterations run on the fused head / energy / tail kernels with the library's own Adam (8 launches per
        # step, no autograd); extra losses on the skinned cloud (flow) keep the autograd composition
        self.assign = None
        if assign is not None:
            from .assign import AssignLoss
            cfg = dict(assign)
            self.assign_iter = int(cfg.pop("assign_iter", 0))
            self.assign_mode = cfg.pop("mode", "add")
            if self.assign_mode not in ("add", "replace"):
                raise ValueError("assign mode must be 'add' (run_real/run_sapien) or 'replace' (run_robot)")
            if self.cull:
                # sample the clouds in the CALLER's order (FPS starts at the caller's point 0, like the reference's
                # kernel), then express the samples in engine order
                from .assign import farthest_point_sample
                n_fps = self.cano.shape[0] // int(cfg.get("downsample", 4))
                inv_c = torch.empty_like(self.perm_cano); inv_c[self.perm_cano] = torch.arange(len(inv_c), device=dev)
                inv_f = torch.empty_like(self.perm_frames)
                inv_f.scatter_(1, self.perm_frames, torch.arange(inv_f.shape[1], device=dev)[None].expand_as(inv_f))
                cfg["src_idx"] = inv_c[farthest_point_sample(cano_orig[None], n_fps)[0]]
                cfg["tgt_idx"] = torch.gather(inv_f, 1, farthest_point_sample(frames_orig, n_fps))
            self.assign = AssignLoss(self.cano, self.frames, **cfg)
        self.native = (flow_ref is None) if native is None else bool(native)
        if self.native:
            if flow_ref is not None:
                raise ValueError("the native fused iteration covers the recon loss only; pass native=False with a flow loss")
            self._init_native(trans_lr, seg_lr, weight_decay, betas, eps)

    # ------------------------------------------------------------------------------------------ native fused iteration
    def _init_native(self, trans_lr, seg_lr, weight_decay, betas, eps):
        import ctypes
        from . import _lib
        L = _lib.lib()
        dev = self.cano.device
        m = self.model
        T, P = m.proposal_6d.shape[0], m.num_parts
        N, M = self.cano.shape[0], self.frames.shape[1]
        conv0, conv2 = m.seg_head.model[0], m.seg_head.model[2]
        H = conv0.weight.shape[0]
        nseg = 4 * H + P * H
        f32 = dict(dtype=torch.float32, device=dev)
        b = self._nat = {}
        b["expo"] = torch.empty(N, P, **f32)
        b["W"], b["ysoft"] = torch.empty(N, P, **f32), torch.empty(N, P, **f32)
        b["hot"] = torch.empty(N, 2, **f32)                      # the one non-zero of every row of W: (part bits, value)
        b["R"] = torch.empty(T, P, 3, 3, **f32)
        b["skinned"] = torch.empty(T, N, 3, **f32)
        b["loss64"] = torch.zeros(1, dtype=torch.float64, device=dev)
        b["gW"] = torch.empty(N, P, **f32)
        b["gpose"] = torch.empty(T * P * 12, **f32)
        b["gR"], b["gtr"] = b["gpose"][:T * P * 9], b["gpose"][T * P * 9:]
        b["ws_bytes"] = int(L.reart_energy_workspace_bytes(T, N, M))
        b["ws"] = _lib.workspace(b["ws_bytes"], dev)
        b["tail_ws"] = _lib.workspace(int(L.reart_relax_tail_workspace_bytes(N, H, P)), dev)
        for k, ref in (("seg", None), ("d6", m.proposal_6d), ("tr", m.proposal_t)):
            shape = (nseg,) if ref is None else tuple(ref.shape)
            b["m_" + k], b["v_" + k] = torch.zeros(shape, **f32), torch.zeros(shape, **f32)
        b["step"] = torch.zeros(1, **f32)
        b["tickets"] = torch.zeros(int(L.reart_relax_tail_ticket_words(N)), dtype=torch.int32, device=dev)
        b["bucket"] = torch.zeros(nseg + 1, **f32)
        b["loss_out"] = torch.zeros(1, **f32)
        b["dims"] = (T, N, M, P, H)
        if self.cull or self.search_culled:                      # arg-mins carried from step to step (-1: none yet)
            b["nn_rows"] = torch.full((T, N), -1, dtype=torch.int32, device=dev)
            b["nn_cols"] = torch.full((T, M), -1, dtype=torch.int32, device=dev)
            # evaluated / offered (warp, chunk) pairs; ordered search: + points resolved by the exact tie path
            b["cull_stats"] = torch.zeros(3 if self.search_culled else 2, dtype=torch.int64, device=dev)
        red = self.sink.reducer if self.sink is not None else None
        self.model.seg_head.grad_sink = None                     # the autograd sink is not used on this path
        oneshot = red if (red is not None and hasattr(red, "peer_base")) else None
        b["nccl"] = red is not None and oneshot is None
        a = _lib.RelaxTailArgs()
        p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
        a.cano, a.w0, a.b0, a.w2 = p(self.cano), p(conv0.weight), p(conv0.bias), p(conv2.weight)
        a.ysoft, a.tau, a.gW = p(b["ysoft"]), p(self.tau), p(b["gW"])
        a.d6, a.tr, a.gR, a.gtr = p(m.proposal_6d), p(m.proposal_t), p(b["gR"]), p(b["gtr"])
        a.m_seg, a.v_seg, a.m_d6, a.v_d6, a.m_tr, a.v_tr = (p(b[k]) for k in ("m_seg", "v_seg", "m_d6", "v_d6", "m_tr", "v_tr"))
        a.step = p(b["step"])
        a.lr_pose, a.lr_seg, a.beta1, a.beta2, a.eps, a.weight_decay = trans_lr, seg_lr, betas[0], betas[1], eps, weight_decay
        a.partials, a.tickets, a.loss_local = p(b["tail_ws"]), p(b["tickets"]), p(b["loss64"])
        a.bucket, a.loss_out = p(b["bucket"]), p(b["loss_out"])
        a.rank, a.world = (self.ctx.rank, self.ctx.world_size) if oneshot is not None else (0, 1)
        if oneshot is not None:
            assert oneshot.n == nseg + 1
            a.peer_base, a.epoch, a.n_pad = p(oneshot.peer_base), p(oneshot.epoch), oneshot.n_pad
        a.phase = 0
        a.N, a.H, a.P, a.T = N, H, P, T
        b["args"] = a
        b["keep"] = (conv0, conv2, oneshot)
        assert self.tau.dtype == torch.float32 and conv0.weight.is_contiguous() and conv2.weight.is_contiguous()

    def _opt_params(self):
        if self.native:
            m = self.model
            return [m.proposal_6d, m.proposal_t] + [q for q in m.seg_head.parameters() if q.requires_grad]
        return super()._opt_params()

    def _opt_state_tensors(self):
        if self.native:
            return [self._nat[k] for k in ("m_seg", "v_seg", "m_d6", "v_d6", "m_tr", "v_tr", "step")]
        return super()._opt_state_tensors()

    def _aux_state_tensors(self):
        aux = [self.assign.col4row, self.assign.dual_u] if self.assign is not None else []
        if self.native and (self.cull or self.search_culled):
            aux += [self._nat["nn_rows"], self._nat["nn_cols"], self._nat["cull_stats"]]
        return aux

    # ------------------------------------------------------------------------------------------ iteration flavours
    def _phase(self):
        """(use_chamfer, use_assign, refresh) of the iteration that is about to run (self.iteration is 1-based)."""
        if self.assign is None:
            return True, False, False
        i = self.iteration - 1
        if i < self.assign_iter:
            return True, False, False
        return self.assign_mode == "add", True, self.assign.due(i, self.assign_iter)

    def _variant(self):
        return self._phase()

    def _after_replay(self, variant):
        if variant[2]:
            self.assign.have_assignment = True

    def _step_phase(self):
        return getattr(self, "_cur_variant", None) or self._phase()

    def _energy_call(self, L, b, T, N, M, P, gW, gR, gtr, g_skinned, compute_grad):
        """The fused energy evaluation of this step: brute-force search, or the exact culled one seeded by the previous
        step's arg-mins (bit-identical results)."""
        from ._lib import check, ptr, stream_ptr
        m = self.model
        if self.search_culled:
            check(L.reart_skinned_chamfer_fwd_bwd_ordered(
                ptr(self.cano), ptr(b["W"]), ptr(b["R"]), ptr(m.proposal_t), ptr(self.frames), ptr(self.frames_search),
                ptr(self.frames_search_packed), T, N, M, P, ptr(self.search_order_rows), ptr(self.search_inv_rows),
                ptr(self.search_order_tgt), ptr(self.search_inv_tgt), ptr(b["skinned"]), ptr(b["loss64"]), ptr(gW), ptr(gR),
                ptr(gtr), ptr(g_skinned), compute_grad, None, None, None, None, ptr(b["nn_rows"]), ptr(b["nn_cols"]),
                ptr(b["cull_stats"]), ptr(b["ws"]), b["ws_bytes"], stream_ptr()), "reart_skinned_chamfer_fwd_bwd_ordered")
        elif self.cull:
            check(L.reart_skinned_chamfer_fwd_bwd_culled(
                ptr(self.cano), ptr(b["W"]), ptr(b["R"]), ptr(m.proposal_t), ptr(self.frames), ptr(self.frames_packed), T, N, M, P,
                ptr(b["skinned"]), ptr(b["loss64"]), ptr(gW), ptr(gR), ptr(gtr), ptr(g_skinned), compute_grad, None, None, None,
                None, ptr(b["nn_rows"]), ptr(b["nn_cols"]), ptr(b["cull_stats"]), ptr(b["ws"]), b["ws_bytes"], stream_ptr()),
                "reart_skinned_chamfer_fwd_bwd_culled")
        elif not self.fuse_producer:
            check(L.reart_skinned_chamfer_fwd_bwd(
                ptr(self.cano), ptr(b["W"]), ptr(b["R"]), ptr(m.proposal_t), ptr(self.frames), ptr(self.frames_packed), T, N, M, P,
                ptr(b["skinned"]), ptr(b["loss64"]), ptr(gW), ptr(gR), ptr(gtr), ptr(g_skinned), compute_grad, ptr(b["ws"]),
                b["ws_bytes"], stream_ptr()), "reart_skinned_chamfer_fwd_bwd")
        else:
            # skinning fused into the producer side of the search (the weights are one-hot: the head wrote them in compact form)
            check(L.reart_skinned_chamfer_fwd_bwd_fused(
                ptr(self.cano), ptr(b["hot"]), ptr(b["W"]), ptr(b["R"]), ptr(m.proposal_t), ptr(self.frames), ptr(self.frames_packed),
                T, N, M, P, ptr(b["skinned"]), ptr(b["loss64"]), ptr(gW), ptr(gR), ptr(gtr), ptr(g_skinned), compute_grad, ptr(b["ws"]),
                b["ws_bytes"], stream_ptr()), "reart_skinned_chamfer_fwd_bwd_fused")

    def culling_stats(self):
        """(evaluated, offered) (warp, 32-target chunk) pairs since the last call; resets the counters.  Host sync."""
        if not (self.native and (self.cull or self.search_culled)):
            return None
        ev, off = (int(x) for x in self._nat["cull_stats"][:2].tolist())
        self._nat["cull_stats"][:2].zero_()
        return ev, off

    def flagged_ties(self):
        """Points the culled search saw reach their minimum in two of its chunks, resolved by the exact tie path, since
        the last call (resets the counter; None unless search is culled).  Host sync."""
        if not self.search_culled:
            return None
        n = int(self._nat["cull_stats"][2])
        self._nat["cull_stats"][2].zero_()
        return n

    def _run_iteration_native(self):
        """head -> [memset, skin (x-sorted copy), search, energy columns, energy rows, skin backward, reduce] -> tail."""
        import ctypes
        from . import _lib
        from ._lib import check, ptr, stream_ptr
        L = _lib.lib()
        b = self._nat
        T, N, M, P, H = b["dims"]
        m = self.model
        conv0, conv2 = m.seg_head.model[0], m.seg_head.model[2]
        use_chamfer, use_assign, refresh = self._step_phase()
        b["expo"].exponential_()                                  # the same RNG draw F.gumbel_softmax makes
        with torch.cuda.device(self.cano.device):
            check(L.reart_relax_head(ptr(self.cano), ptr(conv0.weight), ptr(conv0.bias), ptr(conv2.weight), ptr(b["expo"]),
                                     ptr(self.perm_cano), ptr(self.tau), ptr(m.proposal_6d), N, H, P, T, None, ptr(b["W"]), ptr(b["ysoft"]),
                                     ptr(b["R"]), ptr(b["hot"]), stream_ptr()), "reart_relax_head")
            if not use_assign:
                self._energy_call(L, b, T, N, M, P, b["gW"], b["gR"], b["gtr"], None, 1)
            else:
                if "gs" not in b:
                    b["gs"] = torch.zeros(T, N, 3, dtype=torch.float32, device=self.cano.device)
                    b["bwd_ws_bytes"] = int(L.reart_skin_bwd_workspace_bytes(T, N, P))
                    b["bwd_ws"] = _lib.workspace(b["bwd_ws_bytes"], self.cano.device)
                if use_chamfer:                                   # Chamfer energy and its gradient w.r.t. the skinned cloud
                    self._energy_call(L, b, T, N, M, P, None, None, None, b["gs"], 0)
                else:                                             # run_robot.py:164-192: the assignment loss REPLACES Chamfer
                    check(L.reart_skin_fwd(ptr(self.cano), ptr(b["W"]), ptr(b["R"]), ptr(m.proposal_t), T, N, P, ptr(b["skinned"]),
                                           stream_ptr()), "reart_skin_fwd")
                    b["gs"].zero_()
                    b["loss64"].zero_()
                if refresh:
                    self.assign.refresh(b["skinned"])
                self.assign.add_loss_and_grad(b["skinned"], b["gs"], b["loss64"], accumulate=True)
                check(L.reart_skin_bwd(ptr(self.cano), ptr(b["W"]), ptr(b["R"]), ptr(m.proposal_t), ptr(b["gs"]), T, N, P,
                                       ptr(b["gW"]), ptr(b["gR"]), ptr(b["gtr"]), ptr(b["bwd_ws"]), b["bwd_ws_bytes"], stream_ptr()),
                      "reart_skin_bwd")
            a = b["args"]
            if not b["nccl"]:
                check(L.reart_relax_tail(ctypes.byref(a), stream_ptr()), "reart_relax_tail")
            else:                                                 # no peer memory: gradients -> bucket, NCCL, Adam
                a.phase = 1
                check(L.reart_relax_tail(ctypes.byref(a), stream_ptr()), "reart_relax_tail")
                self.ctx.all_reduce_sum_(b["bucket"])
                a.phase = 2
                check(L.reart_relax_tail(ctypes.byref(a), stream_ptr()), "reart_relax_tail")
        self.skinned = b["skinned"]
        return b["loss_out"][0]

    def _iteration(self):
        use_chamfer, use_assign, refresh = self._step_phase()
        seg, weight = self.model.weights(self.cano, tau=self.tau)
        R, tr = self.model.pose()
        if use_chamfer:
            loss, skinned = ops.skinned_chamfer_loss(self.cano, weight, R, tr, self.frames, self.frames_packed,
                                                     unit_grad=True)
        else:
            skinned = ops.skin(self.cano, weight, R, tr)
            loss = skinned.new_zeros(())
        if use_assign:
            if refresh:
                self.assign.refresh(skinned)
            loss = loss + self.assign.loss(skinned)
        if self.flow_ref is not None:
            loss = loss + self.lambda_flow * self._flow_term(skinned)
        self.skinned = skinned.detach()                         # keep the cloud, not the autograd graph
        return loss

    def _flow_term(self, pc_trans_list):
        """run_robot.py:194-209: k=3 blended anchor flow (no grad, ONE launch for all pairs) vs predicted flow."""
        from .flow_utils import blend_anchor_motion_batched
        from .loss import flow_loss
        c = self.cano_idx
        if self.ctx.world_size == 1:
            complete = torch.cat((pc_trans_list[:c], self.cano[None], pc_trans_list[c:]), dim=0)
            with torch.no_grad():
                target_flow, mask = blend_anchor_motion_batched(complete[:-1].detach().contiguous(), self.flow_ref)
            pred_flow = complete[1:] - complete[:-1]
            return flow_loss(target_flow, pred_flow, flow_mask_list=mask, robust=self.robust_flow)
        # frame-sharded: own pairs [p0, p1), sides taken from local frames, the canonical cloud or the halo frame
        from .dist import flow_pairs_for_rank, halo_from_previous_rank
        lo, hi = self.frame_range
        halo = halo_from_previous_rank(pc_trans_list[-1], self.ctx)          # every rank takes part, even with no pairs
        # the halo's backward is a matched send/recv: tie it into every rank's loss (weight 0) so it always runs,
        # also on ranks that do not consume their halo (rank 0) or own no pair
        anchor = halo.sum() * 0.0
        p0, p1, a_src, b_src = flow_pairs_for_rank(self.total_frames, c, lo, hi)
        if p1 <= p0:
            return anchor

        def pick(src):
            return self.cano if src[0] == "cano" else (halo if src[0] == "halo" else pc_trans_list[src[1]])

        A = torch.stack([pick(x) for x in a_src])
        Bm = torch.stack([pick(x) for x in b_src])
        with torch.no_grad():
            sub = self.flow_ref.slice(p0, p1)
            target_flow, mask = blend_anchor_motion_batched(A.detach().contiguous(), sub)
        return flow_loss(target_flow, Bm - A, flow_mask_list=mask, robust=self.robust_flow) + anchor


class KinematicEngine(_EngineBase):
    """Projection model (networks/model.py KinematicModel) + recon loss, frame-sharded.
    axis/moment are shared (all-reduced); theta/distance/root pose are per frame."""

    def __init__(self, model_kwargs: dict, seg_part: torch.Tensor, cano: torch.Tensor, frames: torch.Tensor,
                 ctx: Optional[DistContext] = None, lr: float = 1e-2, weight_decay: float = 0.0,
                 use_graph: bool = True):
        super().__init__(ctx, use_graph)
        from .knn_module import KNN
        dev = cano.device
        if frames.shape[0] < self.ctx.world_size:
            raise ValueError(f"{frames.shape[0]} frames cannot be sharded over {self.ctx.world_size} ranks")
        lo, hi = self.ctx.frames(frames.shape[0])
        self.frame_range = (lo, hi)
        self.cano = cano.float().contiguous()
        self.frames = frames[lo:hi].float().contiguous()
        self.frames_packed = ops.pack_cloud(self.frames)
        kw = dict(model_kwargs)
        for k in ("theta_list", "distance_list", "root_trans"):
            if k in kw:
                kw[k] = kw[k][lo:hi].clone()
        self.model = KinematicModel(pose_len=hi - lo, seg_part=seg_part, cano_pc=self.cano,
                                    knn=KNN(k=1, transpose_mode=True), **kw).to(dev)
        self.tau = torch.ones((), device=dev)
        params = [p for p in self.model.parameters() if p.requires_grad]
        self.optimizer = torch.optim.Adam(params, lr=lr, weight_decay=weight_decay, capturable=use_graph, fused=True)
        self.bucket = GradBucket([self.model.axis_list, self.model.moment_list], extra_scalars=1)
        with torch.no_grad():                                       # constant label transfer (SURVEY Q27)
            self.weight = F.one_hot(self.model._labels(self.model.cano_pc), num_classes=self.model.num_parts).float()
        self.pairs_per_step_local = 2 * (hi - lo) * self.cano.shape[0] * self.frames.shape[1]

    def _iteration(self):
        trans = self.model.transforms()
        loss, skinned = ops.skinned_chamfer_loss(self.cano, self.weight, trans[:, :, :3, :3].contiguous(),
                                                 trans[:, :, :3, 3].contiguous(), self.frames, self.frames_packed,
                                                 unit_grad=True)
        self.skinned = skinned.detach()
        return loss


def tau_schedule(i: int, n_iter: int, start_tau: float, end_tau: float) -> float:
    """utils/model_utils.py:33-37 as run_robot.py:86,157 uses it (cur_iter = i + 1)."""
    return end_tau + (start_tau - end_tau) * (math.cos(math.pi * (i + 1) / n_iter) + 1.0) * 0.5


def fit_relaxation(cano: torch.Tensor, frames: torch.Tensor, num_parts: int, n_iter: int, ctx: Optional[DistContext] = None,
                   start_tau: float = 5.0, end_tau: float = 1.0, log_every: int = 0, **engine_kwargs):
    """The relaxation optimisation of run_robot.py:153-221 (recon loss, cosine tau schedule :86,157) on the engine.
    Returns (engine, losses) where ``losses`` holds the all-rank loss every ``log_every`` iterations (0: only the
    last) -- reading it is the only host sync."""
    eng = RelaxationEngine(cano, frames, num_parts, ctx=ctx, **engine_kwargs)
    losses = []
    loss = None
    for i in range(n_iter):
        loss = eng.step(tau_schedule(i, n_iter, start_tau, end_tau))
        if log_every and (i % log_every == 0):
            losses.append(float(loss))
    if loss is not None:
        losses.append(float(loss))
    return eng, losses


@torch.no_grad()
def candidate_energy(engine: "RelaxationEngine", cano_idx: int, merge_thr: float = 3e-2, merge_it: int = 2,
                     cano_dist_thr: float = 1e-2, lambda_joint: float = 100.0) -> float:
    """The reference's model-selection energy of a finished relaxation fit (run_robot.py:224-240, 306-314):
    ``total_err = 100 * ass_err + screw_err + group_err`` after the snapshot tail (denoise -> merging_wrapper ->
    mst_wrapper -> extract_kinematic) has turned the soft segmentation into a kinematic tree."""
    from .chamfer import ChamferDistance
    from .knn_module import KNN
    from .model_utils import compute_ass_err, compute_group_temporal_err, compute_pc_transform
    from .structure import (compute_screw_cost, denoise_seg_label, extract_kinematic, merging_wrapper, mst_wrapper)
    cano, frames = engine.cano, engine.frames
    _, seg_part, trans_list = engine.model(cano)
    cd, knn = ChamferDistance(), KNN(k=1, transpose_mode=True)
    seg_part = denoise_seg_label(seg_part, cano, knn, min_num=20)
    if len(torch.unique(seg_part)) > 1:
        seg_part = merging_wrapper(seg_part, trans_list, cano, cd, merge_thr, n_it=merge_it)
    conn = mst_wrapper(seg_part, trans_list, cano, cd, verbose=False, num_fps=20, cano_dist_thr=cano_dist_thr,
                       joint_cost_weight=lambda_joint)
    seg_part, trans_list, conn = extract_kinematic(seg_part, trans_list, conn)
    pred = compute_pc_transform(cano, trans_list, seg_part)
    ass_err = 100.0 * compute_ass_err(pred, frames, use_nproc=True)
    screw_err = compute_screw_cost(trans_list, conn)
    complete = torch.cat((pred[:cano_idx], cano[None], pred[cano_idx:]), dim=0)
    group_err = compute_group_temporal_err(complete, seg_part)
    return float(ass_err + screw_err + group_err)


def fit_candidates(sequence: torch.Tensor, candidates, num_parts: int, n_iter: int, ctx: Optional[DistContext] = None,
                   criterion: str = "total_err", **kwargs):
    """``cano_idx`` model selection (README.md:60 of the reference: fit every candidate canonical frame, keep the
    lowest energy).  The fits are independent runs: with G ranks, rank r fits candidates r, r+G, ... on its own GPU
    with NO communication; one exchange of the final energies picks the winner.  ``sequence`` [T+1,N,3] is the
    complete sequence; candidate c uses frame c as the canonical cloud and the others as observations.

    ``criterion="total_err"`` (default) is the reference's selection energy, ``100 * ass_err + screw_err + group_err``
    (run_robot.py:306-314), evaluated by ``candidate_energy`` after each fit; a fit whose structure stage cannot be
    built (degenerate collapse, SURVEY Q21: the reference crashes there) gets energy +inf.  ``criterion="loss"`` keeps
    the final training loss instead -- NOT the reference's criterion (it favours over-segmented fits); it exists for
    clouds too large for the N x N assignment inside ``ass_err`` (which the reference cannot run either).
    Returns (best_cano_idx, {cano_idx: energy}) on every rank."""
    if criterion not in ("total_err", "loss"):
        raise ValueError("criterion must be 'total_err' or 'loss'")
    ctx = ctx or DistContext()
    mine = {}
    for k, c in enumerate(candidates):
        if k % ctx.world_size != ctx.rank:
            continue
        cano = sequence[c]
        frames = torch.cat((sequence[:c], sequence[c + 1:]), dim=0)
        eng, losses = fit_relaxation(cano, frames, num_parts, n_iter, ctx=DistContext(), **kwargs)   # local, unsharded
        if criterion == "loss":
            mine[int(c)] = losses[-1]
        else:
            try:
                mine[int(c)] = candidate_energy(eng, int(c))
            except (ValueError, AssertionError, RuntimeError, IndexError):
                mine[int(c)] = float("inf")
        eng.release()
    # one exchange of len(candidates) scalars: every rank fills in the energies it computed (+inf elsewhere), MIN-reduce
    dev = sequence.device if (sequence.is_cuda and ctx.backend != "gloo") else torch.device("cpu")
    vec = torch.full((len(candidates),), float("inf"), dtype=torch.float64, device=dev)
    for k, c in enumerate(candidates):
        if int(c) in mine:
            vec[k] = mine[int(c)]
    if ctx.world_size > 1:
        import torch.distributed as dist
        dist.all_reduce(vec, op=dist.ReduceOp.MIN)
    table = {int(c): float(vec[k]) for k, c in enumerate(candidates)}
    best = min(table.items(), key=lambda kv: (kv[1], kv[0]))[0]
    return best, table
