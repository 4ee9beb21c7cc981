"""Fused PairSampling training step (train_eval_Gowalla.py:109-139 of the reference), resident on the GPU:

    sampler -> propagation x2 (two streams) -> pair scores -> BPR loss + dscore -> gradient scatter
    -> backward x2 -> Adam || dropout masks of the NEXT step (eager steps draw their masks first instead)

over persistent HBM buffers, with no host synchronisation (the reference has 55 per step) and, for the
full-size batches, replayed from ONE captured CUDA graph whose train-row cursor and dropout-stream
counter live in device memory.  The reference's semantics are kept: two full propagations with
independent dropout per step, gradients of both summed, Adam with L2 weight decay on all parameters.
"""
from __future__ import annotations

import os

import torch

from . import ops
from .data import Interactions
from .graph import BipartiteGraph
from .propagation import Propagation


class FusedTrainer:
    CALLS_PER_STEP = 2          # dropout call indices consumed per step (pos and neg propagation)

    def __init__(self, model, inter: Interactions, graph: BipartiteGraph, batch_size: int, optim, sample_seed: int,
                 use_cuda_graph: bool = True, two_streams: bool = True, split_dense_backward: bool = False):
        self.model, self.inter, self.g = model, inter, graph
        self.B = int(batch_size)
        self.optim = optim
        self.sample_seed = int(sample_seed)
        self.use_cuda_graph = use_cuda_graph
        self.two_streams = two_streams
        # False: one fused dX+dW+da kernel per stage (shares the tile loads; measured best: 1.22 ms/step at Gowalla shape).
        # True: dX on the chain, dW/da deferred to a third stream (1.24 ms/step: ~40% more dense work for a shorter chain).
        self.split_dense_backward = split_dense_backward
        if split_dense_backward and getattr(model, "embedSize", 64) != 64:
            raise NotImplementedError("the split dense backward (NGACF_SPLIT_DENSE_BWD=1) is built for embedSize 64 only")
        # captured steps: masks of step t+1 are generated next to Adam of step t (NGACF_PREFETCH_MASKS=0: at the head of the step)
        self.prefetch_masks = os.environ.get("NGACF_PREFETCH_MASKS", "1") != "0"
        # NGACF_STAGGER=1: the neg propagation starts one kernel after the pos one.  That paid while the dense kernels were long
        # FFMA kernels (1.44 -> 1.34 ms/step); with the tensor-core kernels both pipelines starting together is faster
        # (in-box A/B: 0.995 -> 0.983 ms/step), so it is off by default
        self.stagger = os.environ.get("NGACF_STAGGER", "0") == "1"
        dev = graph.device
        self.dev = dev
        self.props = [Propagation(graph, model.stages), Propagation(graph, model.stages)]      # pos / neg
        for p in self.props:
            p._bwd_buffers()
        # The loss reads the last stage's output at the batch rows only (SPUIGACF.py:49-52): that stage's aggregation and its
        # backward are computed for the rows / edges that matter (exact -- everything skipped is a zero).  NGACF_PRUNE=0
        # (or prune_last_stage=False) runs the full last stage, for A/B measurements and the parity tests of both paths.
        self.prune_last_stage = os.environ.get("NGACF_PRUNE", "1") != "0" and self.props[0].can_prune()
        self.active = [ops.ActiveRows(graph) for _ in self.props] if self.prune_last_stage else [None, None]
        if inter.host["pool"].shape[0] - int(torch.diff(inter.train_ptr).max().item() if inter.train_ptr.numel() > 1 else 0) < 1:
            # the reference's random.sample(negative_items, 1) raises for such a user (loadGowalla.py:76)
            raise ValueError("a user's train items cover the whole item pool: no negative to sample")
        i64 = dict(dtype=torch.int64, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        self.users = torch.zeros(self.B, **i64)
        self.pos = torch.zeros(self.B, **i64)
        self.neg = torch.zeros(self.B, **i64)
        self.sc_pos = torch.zeros(self.B, **f32)
        self.sc_neg = torch.zeros(self.B, **f32)
        self.dpos = torch.zeros(self.B, **f32)
        self.dneg = torch.zeros(self.B, **f32)
        self.loss = torch.zeros((), **f32)
        self.total = torch.zeros((), dtype=torch.float64, device=dev)
        self.row_dev = torch.zeros(2, **i64)       # {train-row cursor, epoch} of the captured step
        self.call_dev = torch.zeros(1, **i64)      # dropout call counter (two calls per step)
        self.side = torch.cuda.Stream(device=dev) if two_streams else None
        self.grad_stream = torch.cuda.Stream(device=dev) if two_streams else None      # deferred dW/da kernels
        self._graph = None
        self._graph_update = None
        self._setup_params()

    # ------------------------------------------------------------------------------------------
    def _setup_params(self):
        m = self.model
        self.params = [m.uEmbd.weight, m.iEmbd.weight] + m._flat_stage_params()
        for p in self.params:
            if p.grad is None or not p.grad.is_contiguous():
                p.grad = torch.zeros_like(p)
        stage_params = m.gat.stage_parameters()
        self.wtabs = [ops.pointer_table([p.detach() for p in st]) for st in stage_params]
        self.gtabs = [ops.pointer_table([p.grad for p in st]) for st in stage_params]
        # Adam state lives in the optimizer (torch.optim.Adam's keys), so checkpoints stay interchangeable
        self.hyper = self._read_hyper()
        rows, step0 = [], 0
        for p in self.params:
            st = self.optim.state[p]
            if len(st) == 0:
                st["step"] = torch.tensor(0.0)
                st["exp_avg"] = torch.zeros_like(p)
                st["exp_avg_sq"] = torch.zeros_like(p)
            step0 = int(float(st["step"]))
            rows.append([p.data_ptr(), p.grad.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), p.numel()])
        self.adam_tab = torch.tensor(rows, dtype=torch.int64).to(self.dev)
        self.adam_total = sum(p.numel() for p in self.params)
        self.adam_state = torch.tensor([float(step0), 0.0, 0.0, 0.0], dtype=torch.float64, device=self.dev)
        self._ptr_key = tuple(tuple(r[:4]) for r in rows)

    def _read_hyper(self):
        group = self.optim.param_groups[0]
        return dict(lr=float(group["lr"]), b1=float(group["betas"][0]), b2=float(group["betas"][1]), eps=float(group["eps"]),
                    wd=float(group["weight_decay"]))

    # hooks overridden by dist.ReplicaTrainer ------------------------------------------------------
    def _row_offset(self):
        return 0

    def _row_stride(self):
        return self.B

    def _dropout_seed(self, seed):
        return seed

    def _reduce_grads(self):
        pass

    def _collective_between(self):
        return False

    def _replay(self):
        self._graph.replay()
        if self._graph_update is not None:
            self._reduce_grads()
            self._graph_update.replay()

    def _sync_optimizer_state(self):
        step = float(self.adam_state[0].item())
        for p in self.params:
            self.optim.state[p]["step"] = torch.tensor(step)
            torch.autograd.graph.increment_version(p)

    # ------------------------------------------------------------------------------------------
    def _validate(self):
        """Pointer tables (and a captured graph) are only valid while params/grads/Adam state stay in place."""
        rows = []
        for p in self.params:
            st = self.optim.state.get(p, {})
            if p.grad is None or len(st) == 0:
                rows = None
                break
            rows.append([p.data_ptr(), p.grad.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()])
        if rows is None or tuple(tuple(r) for r in rows) != tuple(tuple(r) for r in self._ptr_key):
            self._setup_params()
            self._graph = None
        hyper = self._read_hyper()
        if hyper != self.hyper:
            # lr / betas / eps / weight_decay are kernel arguments baked into the captured step: an LR scheduler (or a manual
            # change of optim.param_groups between epochs) must invalidate the graph, not be ignored
            self.hyper = hyper
            self._graph = None

    def _step_body(self, b: int, epoch: int, droprate: float, seed: int, row0: int, call0: int, dev_counters: bool, part: str = "all"):
        m, g = self.model, self.g
        uE, iE = m.uEmbd.weight.detach(), m.iEmbd.weight.detach()
        rd = self.row_dev if dev_counters else None
        cd = self.call_dev if dev_counters else None
        row0 = row0 + (self._row_offset() if dev_counters else 0)
        ops.sample_pairs(self.inter, row0, row0 + b, self.sample_seed, 0 if dev_counters else epoch, self.users, self.pos, self.neg, rd)
        cur = torch.cuda.current_stream()
        items = (self.pos, self.neg)
        scores = (self.sc_pos, self.sc_neg)
        # active rows of propagation k: stamped with its dropout call index (unique per propagation, so never cleared)
        act = [self.active[k].at(call0 + k, cd) if self.prune_last_stage else None for k in (0, 1)]

        def mark(k):
            if act[k] is not None:
                act[k].mark(self.users[:b], items[k][:b])

        side = self.side

        def fwd(k, hook=None):
            if dev_counters and self.prefetch_masks:
                self.props[k].use_dropout_buffers(droprate)
            else:
                self.props[k].set_dropout(droprate, seed, call0 + k, None, cd)
            mark(k)
            Z = self.props[k].forward(uE, iE, self.wtabs, hook, active=act[k])
            ops.score_pairs(Z, g.U, self.users[:b], items[k][:b], scores[k][:b])
        # captured steps find their dropout masks ready: they were generated at the end of the previous replay (or by
        # _prime_masks before the first one), next to Adam instead of at the head of the critical path
        premask = dev_counters and self.prefetch_masks
        self._mask_args = (droprate, seed) if premask else None
        if side is not None:
            # two pipelines on two streams; optionally (self.stagger) the neg propagation starts one kernel after the pos one
            ev = torch.cuda.Event()
            side.wait_stream(cur)

            def start_side():
                ev.record(cur)
            if premask:
                self.props[0].use_dropout_buffers(droprate)
                self.props[1].use_dropout_buffers(droprate)
            else:
                # masks of the side propagation do not depend on anything: issue them first
                with torch.cuda.stream(side):
                    self.props[1].set_dropout(droprate, seed, call0 + 1, None, cd)
                self.props[0].set_dropout(droprate, seed, call0, None, cd)
            if not self.stagger:
                ev.record(cur)
            mark(0)
            Z0 = self.props[0].forward(uE, iE, self.wtabs, start_side if self.stagger else None, active=act[0])
            ops.score_pairs(Z0, g.U, self.users[:b], items[0][:b], scores[0][:b])
            with torch.cuda.stream(side):
                side.wait_event(ev)
                mark(1)
                Z1 = self.props[1].forward(uE, iE, self.wtabs, active=act[1])
                ops.score_pairs(Z1, g.U, self.users[:b], items[1][:b], scores[1][:b])
            cur.wait_stream(side)
        else:
            fwd(0)
            fwd(1)
        ops.bpr_loss(self.sc_pos[:b], self.sc_neg[:b], 1.0, self.loss, self.dpos[:b], self.dneg[:b])
        dsc = (self.dpos, self.dneg)

        def scatter(k):
            G = self.props[k].grad_in()
            if act[k] is None:
                G.zero_()          # pruned: the scatter writes exactly the active rows, nothing else of G is read
            ops.score_pairs_bwd(self.props[k].Z[-1], g.U, self.users[:b], items[k][:b], dsc[k][:b], G)
        dU, dI = m.uEmbd.weight.grad, m.iEmbd.weight.grad
        if side is not None:
            # both backward passes run concurrently, one kernel apart; the only shared state is the gradient buffers, written by
            # stage k's transform_bwd: pos writes, neg accumulates after it (event per stage)
            S = len(self.props[0].stages)
            evs = [torch.cuda.Event() for _ in range(S)]
            ev_go = torch.cuda.Event()
            gs = self.grad_stream

            def defer(stream):
                # the weight-gradient kernel of a stage is needed by Adam only: run it on the gradient stream as soon as `stream`
                # has produced dh/dS of that stage (pos before neg per stage = program order on the single gradient stream)
                def launch(k, fn):
                    e = torch.cuda.Event()
                    e.record(stream)
                    gs.wait_event(e)
                    with torch.cuda.stream(gs):
                        fn()
                return launch
            side.wait_stream(cur)
            gs.wait_stream(cur)
            with torch.cuda.stream(side):
                scatter(1)
            scatter(0)
            split = self.split_dense_backward
            if not self.stagger:
                ev_go.record(cur)
            self.props[0].backward(self.props[0].grad_in(), uE, iE, self.wtabs, self.gtabs, dU, dI, False,
                                   after_first_kernel=(lambda: ev_go.record(cur)) if self.stagger else None, after_grads=lambda k: evs[k].record(cur),
                                   dw_launcher=defer(cur) if split else None, active=act[0])
            with torch.cuda.stream(side):
                side.wait_event(ev_go)
                self.props[1].backward(self.props[1].grad_in(), uE, iE, self.wtabs, self.gtabs, dU, dI, True,
                                       before_grads=lambda k: side.wait_event(evs[k]), dw_launcher=defer(side) if split else None, active=act[1])
            cur.wait_stream(side)
            cur.wait_stream(gs)
        else:
            scatter(0)
            scatter(1)
            inline = (lambda k, fn: fn()) if self.split_dense_backward else None
            self.props[0].backward(self.props[0].grad_in(), uE, iE, self.wtabs, self.gtabs, dU, dI, False, dw_launcher=inline, active=act[0])
            self.props[1].backward(self.props[1].grad_in(), uE, iE, self.wtabs, self.gtabs, dU, dI, True, dw_launcher=inline, active=act[1])
        if part == "compute":
            return
        self._reduce_grads()
        self._step_update(dev_counters)

    def _step_update(self, dev_counters: bool):
        h = self.hyper
        margs = getattr(self, "_mask_args", None) if dev_counters else None
        mask_stream = self.side if self.side is not None else None
        if margs is not None and mask_stream is not None:
            # next step's masks (call counter + 2) on the side stream, concurrently with Adam; every reader of the current masks
            # (the backward kernels) is already ordered before this point
            cur = torch.cuda.current_stream()
            mask_stream.wait_stream(cur)
            with torch.cuda.stream(mask_stream):
                ops.counter_add(self.call_dev, self.CALLS_PER_STEP)
                self._generate_masks(*margs)
        ops.adam_step_dev(self.adam_tab, len(self.params), self.adam_total, h["lr"], h["b1"], h["b2"], h["eps"], h["wd"], self.adam_state)
        # epoch loss accumulator + train-row cursor in one launch of ours (no eager-torch kernels inside the captured step)
        ops.step_counters(self.total, self.loss, self.row_dev if dev_counters else None, self._row_stride())
        if dev_counters:
            if margs is None:
                ops.counter_add(self.call_dev, self.CALLS_PER_STEP)
            elif mask_stream is None:
                ops.counter_add(self.call_dev, self.CALLS_PER_STEP)
                self._generate_masks(*margs)
            else:
                torch.cuda.current_stream().wait_stream(mask_stream)

    def _generate_masks(self, droprate, seed):
        """masks of both propagations for the step whose first call index is the current value of call_dev"""
        for k in (0, 1):
            self.props[k].set_dropout(droprate, seed, k, None, self.call_dev)

    def _prime_masks(self, droprate, seed):
        """before the first replay of a captured step: the masks that step will read"""
        if self.prefetch_masks:
            self._generate_masks(droprate, seed)

    # ------------------------------------------------------------------------------------------
    def launches_per_step(self, droprate: float) -> int:
        """Number of OUR kernels launched per step (bench.py's gpu_launches claim)."""
        S = len(self.props[0].stages)
        per_prop_fwd = (1 if droprate > 0 else 0) + 2 * S + 1              # masks (one launch), transform+aggregate, score
        per_prop_bwd = 1 + S * (1 + 2 + (4 if self.split_dense_backward else 2))   # scatter, prep + 2 edge passes + dense backward
        marks = 6 if self.prune_last_stage else 0                           # mark_active + plan + active-user rows kernel per propagation
        return 1 + marks + 2 * (per_prop_fwd + per_prop_bwd) + 1 + 2 + 2     # sampler, ..., loss, adam(2), counters(2)

    def train_epoch(self, epoch: int = 0, max_steps=None) -> float:
        """Returns sum(batch-mean loss)/len(train_df) (train_eval_Gowalla.py:139,144)."""
        m = self.model
        m.train()
        self._validate()
        droprate = m.droprate if m.droprate > 0 else 0.0
        seed = self._dropout_seed(m._seed())
        n = len(self.inter)
        stride = self._row_stride()
        n_batches = n // stride + 1
        if max_steps is not None:
            n_batches = min(n_batches, max_steps)
        self.total.zero_()
        n_full = min(n // stride, n_batches)
        if self.use_cuda_graph and n_full > 0:
            if self._graph is None or self._graph_key != (droprate, seed):
                self._capture(droprate, seed)
            self.row_dev.copy_(torch.tensor([0, epoch], dtype=torch.int64), non_blocking=False)
            self.call_dev.fill_(m._call)
            self._prime_masks(droprate, seed)
            for _ in range(n_full):
                self._replay()
            m._call += self.CALLS_PER_STEP * n_full
        else:
            for bi in range(n_full):
                self._step_body(self.B, epoch, droprate, seed, bi * stride + self._row_offset(), m._call, False)
                m._call += self.CALLS_PER_STEP
        if n_batches > n_full:         # tail step (len % stride rows), eager; a rank may get fewer rows or none
            lo = min(n, n_full * stride + self._row_offset())
            hi = min(n, lo + self.B)
            if n - n_full * stride > 0:
                if hi > lo:
                    self._step_body(hi - lo, epoch, droprate, seed, lo, m._call, False)
                else:
                    self._empty_step()
                m._call += self.CALLS_PER_STEP
        self._sync_optimizer_state()
        return self._epoch_loss(n)

    def _epoch_loss(self, n):
        return float(self.total.item()) / n

    def _empty_step(self):
        """A replica whose slice of the tail step is empty still joins the gradient all-reduce and the update."""
        for p in self.params:
            p.grad.zero_()
        self._reduce_grads()
        h = self.hyper
        ops.adam_step_dev(self.adam_tab, len(self.params), self.adam_total, h["lr"], h["b1"], h["b2"], h["eps"], h["wd"], self.adam_state)

    def _capture(self, droprate, seed):
        epoch = 0
        # warm-up on a side stream (allocations, lazy module state), restoring everything it touched
        snap = [p.detach().clone() for p in self.params]
        opt_snap = [(self.optim.state[p]["exp_avg"].clone(), self.optim.state[p]["exp_avg_sq"].clone()) for p in self.params]
        adam_snap, total_snap = self.adam_state.clone(), self.total.clone()
        row_snap, call_snap = self.row_dev.clone(), self.call_dev.clone()
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._step_body(self.B, epoch, droprate, seed, 0, 0, True)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize(self.dev)
        graph = torch.cuda.CUDAGraph()
        self._graph_update = None
        if self._collective_between():
            # the NCCL all-reduce of the gradients stays OUTSIDE the captured graphs (capturing it deadlocked on
            # the B200 box): graph 1 = everything up to the gradients, eager all-reduce, graph 2 = Adam + counters
            with torch.cuda.graph(graph):
                self._step_body(self.B, epoch, droprate, seed, 0, 0, True, part="compute")
            self._graph_update = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph_update):
                self._step_update(True)
        else:
            with torch.cuda.graph(graph):
                self._step_body(self.B, epoch, droprate, seed, 0, 0, True)
        with torch.no_grad():
            for p, sp, (a, b) in zip(self.params, snap, opt_snap):
                p.copy_(sp)
                self.optim.state[p]["exp_avg"].copy_(a)
                self.optim.state[p]["exp_avg_sq"].copy_(b)
            self.adam_state.copy_(adam_snap)
            self.total.copy_(total_snap)
            self.row_dev.copy_(row_snap)
            self.call_dev.copy_(call_snap)
        self._graph, self._graph_key = graph, (droprate, seed)

    # ------------------------------------------------------------------------------------------
    # step-level driver used by bench.py
    # ------------------------------------------------------------------------------------------
    def run_steps(self, n_steps: int, host_rows=None, read_loss: bool = False):
        """n_steps full-batch steps through the captured graph, wrapping around the train rows.
        host_rows: pinned int32 host tensor of the train rows' users -- the batch's rows are copied H2D every
        step (end-to-end mode); read_loss: D2H read of the step loss every step (the reference's .item())."""
        m = self.model
        m.train()
        self._validate()
        droprate = m.droprate if m.droprate > 0 else 0.0
        seed = self._dropout_seed(m._seed())
        n = len(self.inter)
        stride = self._row_stride()
        if n < stride:
            raise ValueError("fewer train rows than one step consumes")
        if self._graph is None or self._graph_key != (droprate, seed):
            self._capture(droprate, seed)
        if not hasattr(self, "_cursor"):
            self._cursor = 0
        self.row_dev.copy_(torch.tensor([self._cursor, 0], dtype=torch.int64))
        self.call_dev.fill_(m._call)
        self._prime_masks(droprate, seed)
        losses = []
        for _ in range(n_steps):
            if self._cursor + stride > n:
                self._cursor = 0
                self.row_dev.zero_()
            if host_rows is not None:
                lo = self._cursor + self._row_offset()
                self.inter.train_rows_user[lo:lo + self.B].copy_(host_rows[lo:lo + self.B], non_blocking=True)
            self._replay()
            self._cursor += stride
            if read_loss:
                losses.append(float(self.loss.item()))
        m._call += self.CALLS_PER_STEP * n_steps
        return losses

    def units_per_step(self) -> int:
        return 2 * self.g.E          # propagated edges: two full-graph propagations per step

    def parallelism(self) -> str:
        return "single GPU"

    def working_set_bytes(self) -> int:
        N, E = self.g.N, self.g.E
        per_prop = 4 * N * 256 + 4 * N * 256 + 8 * E * 4 + 2 * (N * 8 + E)    # h,Z x2 stages; G x2, Ghat, dh; ds_store; masks
        return 2 * per_prop + 7 * sum(p.numel() for p in self.params) * 4 + self.g.structure_bytes()

    def profile_kernels(self, n_steps: int = 3):
        """Per-kernel CUDA-event durations of n eager single-stream steps: [(entry point, args, ms)].
        Parameters/optimizer state are restored afterwards."""
        from . import _lib
        m = self.model
        droprate = m.droprate if m.droprate > 0 else 0.0
        snap = [p.detach().clone() for p in self.params]
        opt_snap = [(self.optim.state[p]["exp_avg"].clone(), self.optim.state[p]["exp_avg_sq"].clone()) for p in self.params]
        adam_snap, total_snap = self.adam_state.clone(), self.total.clone()
        side, self.side = self.side, None
        # batches from the middle of the train rows: the first rows belong to the heaviest users (one user can fill a whole
        # batch there), which is not what a typical step looks like
        row0 = max(0, (len(self.inter) // 2 // self.B) * self.B - n_steps * self.B)
        self._step_body(self.B, 0, droprate, m._seed(), row0, 0, False)     # warm
        torch.cuda.synchronize(self.dev)
        _lib.PROFILE = []
        try:
            for k in range(n_steps):
                self._step_body(self.B, 0, droprate, self._dropout_seed(m._seed()), row0 + (k + 1) * self.B, self.CALLS_PER_STEP * (k + 1), False)
            torch.cuda.synchronize(self.dev)
            out = [(name, args, e0.elapsed_time(e1)) for name, args, e0, e1 in _lib.PROFILE]
        finally:
            _lib.PROFILE = None
            self.side = side
        with torch.no_grad():
            for p, sp, (a, b) in zip(self.params, snap, opt_snap):
                p.copy_(sp)
                self.optim.state[p]["exp_avg"].copy_(a)
                self.optim.state[p]["exp_avg_sq"].copy_(b)
            self.adam_state.copy_(adam_snap)
            self.total.copy_(total_snap)
        return out
