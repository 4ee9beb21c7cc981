"""Full-graph SpUIGAT propagation on the GPU: forward (SPUIGACF.py:30-39,207-215,340-400) and the
closed-form backward (SURVEY.md 3.4) over persistent HBM buffers, plus the autograd bridge used by the
drop-in ``SPUIGACF.forward``.

Layout in HBM per propagation (N = U+I nodes, users first; a row is 64 fp32 = 256 B at embedSize 64; at embedSize 128 the
embedding tables, the last stage's h/Z and the backward buffers of that stage are 128 wide, masks of the first stage 2 words):
  stage k:  h_k (N,64)  transformed features      s_k (N,H)  rank-1 logit scalars (p|q)
            Z_k (N,64)  pre-ELU stage output       norm_k (N,H) attention row/col sums (R|C)
            featmask_k uint64[N], edgemask_k uint8[E]   dropout keep bits (only when dropout is on)
  backward: G (N,64) x2 ping-pong, Ghat (N,64), dh (N,64), dN/dS (N,8), ds_store (E,8)
The stage input is never materialised: stage 0 reads the embedding tables in place, stage k>0 reads
Z_{k-1} and applies ELU + dropout on load.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch

from . import ops
from .graph import BipartiteGraph
from .ops import STAGES


class Propagation:
    def __init__(self, graph: BipartiteGraph, stages=STAGES):
        """stages: (heads, width per head) per stage.  Stage k writes H*DH columns; the first stage reads the embedding tables, whose
        width is the last stage's output width (SPUIGACF's out_att maps back to embedSize), every later stage the previous output."""
        self.g = graph
        self.stages = tuple(stages)
        self.w_out = [H * DH for H, DH in self.stages]
        self.w_in = [self.w_out[-1]] + self.w_out[:-1]
        for w in self.w_out + self.w_in:
            ops.check_width(w)
        self.w_max = max(self.w_out)
        dev, N, E = graph.device, graph.N, graph.E
        f32 = dict(dtype=torch.float32, device=dev)
        self.h = [torch.empty((N, w), **f32) for w in self.w_out]
        self.Z = [torch.zeros((N, w), **f32) for w in self.w_out]        # zeros: rows a pruned last stage skips stay finite
        self.s = [torch.empty((N, H), **f32) for H, _ in self.stages]
        self.norm = [torch.zeros((N, H), **f32) for H, _ in self.stages]
        self.featmask: List[Optional[torch.Tensor]] = [None] * len(self.stages)
        self.edgemask: List[Optional[torch.Tensor]] = [None] * len(self.stages)
        self._own_masks = None
        self.scale = 1.0
        self.scratch, self.counter = (torch.empty(max(graph.S, 1) * (self.w_max + 8), **f32),
                                      torch.zeros(max(graph.L, 1), dtype=torch.int32, device=dev))
        self._bwd = None

    # ------------------------------------------------------------------------------------------
    def _mask_buffers(self):
        if self._own_masks is None:
            dev = self.g.device
            self._own_masks = ([torch.empty(self.g.N * (w // 64), dtype=torch.int64, device=dev) for w in self.w_in],
                               [torch.empty(max(self.g.E, 1), dtype=torch.uint8, device=dev) for _ in self.stages])
        return self._own_masks

    def set_dropout(self, droprate: float, seed: int = 0, call: int = 0, injected=None, call_dev=None):
        """droprate 0 -> no masks.  injected = dict(feat=[uint64/int64 [N]]*S, edge=[uint8 [E]]*S) device tensors
        (parity tests inject masks captured from the reference); else Philox(seed, call)."""
        S = len(self.stages)
        if droprate <= 0.0:
            self.featmask, self.edgemask, self.scale = [None] * S, [None] * S, 1.0
            return
        self.scale = 1.0 / (1.0 - droprate)
        if injected is not None:
            self.featmask = [m.contiguous() for m in injected["feat"]]
            self.edgemask = [m.contiguous() for m in injected["edge"]]
            return
        fm, em = self._mask_buffers()
        ops.dropout_masks(fm, em, [H for H, _ in self.stages], self.g.N, self.g.E, seed, call, droprate, call_dev, widths=self.w_in)
        self.featmask, self.edgemask = list(fm), [m[:self.g.E] for m in em]

    def use_dropout_buffers(self, droprate: float):
        """Point the kernels at the own mask buffers WITHOUT generating masks: the trainer's captured step generates the masks of
        step t+1 at the end of step t (overlapping Adam), so the next replay finds them ready."""
        S = len(self.stages)
        if droprate <= 0.0:
            self.featmask, self.edgemask, self.scale = [None] * S, [None] * S, 1.0
            return
        self.scale = 1.0 / (1.0 - droprate)
        fm, em = self._mask_buffers()
        self.featmask, self.edgemask = list(fm), [m[:self.g.E] for m in em]

    # ------------------------------------------------------------------------------------------
    def can_prune(self) -> bool:
        """The pruned last stage (ops.ActiveRows) exists for a single-head, 64-wide output stage, which every model of the family
        has at embedSize 64 (at 128 the full last stage runs)."""
        return self.stages[-1][0] == 1 and self.w_out[-1] == 64

    def forward(self, uEmbd: torch.Tensor, iEmbd: torch.Tensor, wtabs: Sequence[torch.Tensor], after_first_kernel=None,
                active=None) -> torch.Tensor:
        """after_first_kernel: optional callback run right after the first (dense) kernel was enqueued -- the trainer uses it to
        start the OTHER propagation one kernel later, so that its dense kernels overlap this one's gather kernels.
        active (ops.ActiveRows): the caller reads the returned Z at the marked rows only (the batch rows of a training step,
        SPUIGACF.py:49-52) -- the last stage's aggregation is then computed for those rows alone; every other row of Z[-1] /
        norm[-1] keeps stale data."""
        g = self.g
        Xu, Xi, act = uEmbd, iEmbd, 0
        last = len(self.stages) - 1
        for k, (H, _) in enumerate(self.stages):
            ops.transform_fwd(Xu, Xi, act, self.featmask[k], self.scale, wtabs[k], H, g.U, g.I, self.h[k], self.s[k],
                              d_in=self.w_in[k], d_out=self.w_out[k])
            if k == 0 and after_first_kernel is not None:
                after_first_kernel()
            if active is not None and k == last:
                ops.aggregate_fwd_active(g, self.scratch, self.counter, self.h[k], self.s[k], H, self.edgemask[k], self.scale,
                                         self.Z[k], self.norm[k], active)
            else:
                ops.aggregate_fwd(g, self.scratch, self.counter, self.h[k], self.s[k], H, self.edgemask[k], self.scale,
                                  self.Z[k], self.norm[k], width=self.w_out[k])
            Xu, Xi, act = self.Z[k], self.Z[k][g.U:], 1
        return self.Z[-1]

    # ------------------------------------------------------------------------------------------
    def _bwd_buffers(self):
        if self._bwd is None:
            dev, N, E = self.g.device, self.g.N, self.g.E
            f32 = dict(dtype=torch.float32, device=dev)
            S = len(self.stages)
            D = self.w_max        # G / Ghat / dh hold the widest stage; narrower stages use the leading N*w floats (_rows)
            ws = max(ops.transform_bwd_workspace_bytes(self.g.U, self.g.I, a, b) for a, b in zip(self.w_in, self.w_out))
            # G / Ghat / dN start as zeros: the pruned output stage leaves the rows of inactive nodes untouched (stale, finite)
            self._bwd = dict(G=[torch.zeros((N, D), **f32), torch.zeros((N, D), **f32)], Ghat=torch.zeros((N, D), **f32),
                             dh=torch.empty((N, D), **f32), dN=torch.zeros((N, 8), **f32), dS=torch.empty((N, 8), **f32),
                             ds=torch.empty(max(E, 1) * 8, **f32),
                             ws=torch.empty(ws // 4, **f32),
                             # split mode: per-stage dh/dS (the deferred dW kernel of stage k reads them while stage k-1 is running)
                             dh_k=[torch.empty((N, D), **f32) for _ in range(S)], dS_k=[torch.empty((N, 8), **f32) for _ in range(S)],
                             ws_k=[torch.empty(ops.transform_bwd_dw_workspace_bytes(self.g.U, self.g.I) // 4 + 16, **f32) for _ in range(S)])
        return self._bwd

    def _rows(self, buf, w):
        """(N, w) view of the leading N*w floats of a (N, w_max) buffer (the buffer itself when w == w_max)"""
        return buf if w == buf.shape[1] else buf.view(-1)[:self.g.N * w].view(self.g.N, w)

    def grad_in(self) -> torch.Tensor:
        """(N, width of the last stage) buffer the caller fills with dL/dZ_last (zero-filled by the caller as needed)."""
        return self._rows(self._bwd_buffers()["G"][0], self.w_out[-1])

    def backward(self, G_last: torch.Tensor, uEmbd, iEmbd, wtabs, gtabs, dU, dI, accumulate: bool, after_first_kernel=None,
                 before_grads=None, after_grads=None, dw_launcher=None, active=None):
        """G_last = dL/dZ_last (N,64).  Writes (accumulate=False) or adds (True) every parameter gradient:
        embedding grads into dU/dI, attention grads through the pointer tables gtabs[k].
        before_grads(k)/after_grads(k) bracket the only kernels that touch the shared gradient buffers (stage k's
        transform_bwd), so two propagations can run their backward passes on two streams.
        dw_launcher(k, fn): split mode -- only dX stays on this chain; fn (the dW/da kernel of stage k, needed by the optimizer
        only) is handed to the caller, which runs it on another stream once this stream reached the current point.
        active (ops.ActiveRows): G_last is defined on the marked rows only and is zero elsewhere (forward ran with the same
        `active`): the last stage's backward is the pruned pass."""
        g = self.g
        b = self._bwd_buffers()
        G = G_last
        last = len(self.stages) - 1
        wide = self.w_max != 64
        if wide and (dw_launcher is not None or active is not None):
            raise NotImplementedError("the split dense backward and the pruned output stage are built for 64-wide stages only")
        for k in range(last, -1, -1):
            H, _ = self.stages[k]
            w, w_in = self.w_out[k], self.w_in[k]
            pruned = active is not None and k == last
            if pruned:
                ops.stage_bwd_prep_active(g, G, self.Z[k], self.h[k], self.norm[k], H, b["Ghat"], b["dN"], active)
            else:
                Ghat = self._rows(b["Ghat"], w)
                ops.stage_bwd_prep(G, self.Z[k], self.h[k], self.norm[k], H, Ghat, b["dN"], width=w)
            if k == last and after_first_kernel is not None:
                after_first_kernel()
            dh, dS = (b["dh_k"][k], b["dS_k"][k]) if dw_launcher is not None else (b["dh"], b["dS"])
            for mode in (0, 1):
                if pruned:
                    ops.stage_bwd_edges_active(mode, g, self.scratch, self.counter, G, b["Ghat"], b["dN"], self.h[k], self.s[k], H,
                                               self.edgemask[k], self.scale, wtabs[k], b["ds"], dh, dS, active)
                else:
                    dh = self._rows(dh, w)
                    ops.stage_bwd_edges(mode, g, self.scratch, self.counter, G, self._rows(b["Ghat"], w), b["dN"], self.h[k], self.s[k], H,
                                        self.edgemask[k], self.scale, wtabs[k], b["ds"], dh, dS, width=w)
            if dw_launcher is not None:
                Xu, Xi, act = (self.Z[k - 1], self.Z[k - 1][g.U:], 1) if k > 0 else (uEmbd, iEmbd, 0)
                dw_launcher(k, lambda k=k, H=H, dh=dh, dS=dS, Xu=Xu, Xi=Xi, act=act: ops.transform_bwd_dw(
                    dh, dS, Xu, Xi, act, self.featmask[k], self.scale, wtabs[k], gtabs[k], H, g.U, g.I, int(accumulate), b["ws_k"][k]))
                if before_grads is not None:
                    before_grads(k)
                if k > 0:
                    Gprev = b["G"][1] if G is not b["G"][1] else b["G"][0]
                    ops.transform_bwd_dx(dh, Xu, Xi, 1, self.featmask[k], self.scale, wtabs[k], H, g.U, g.I, Gprev, Gprev[g.U:], 0)
                    G = Gprev
                else:
                    ops.transform_bwd_dx(dh, None, None, 0, self.featmask[k], self.scale, wtabs[k], H, g.U, g.I, dU, dI, int(accumulate))
                if after_grads is not None:
                    after_grads(k)
                continue
            if before_grads is not None:
                before_grads(k)
            dh = self._rows(b["dh"], w)
            if k > 0:
                Gprev = b["G"][1] if G.data_ptr() != b["G"][1].data_ptr() else b["G"][0]
                Gprev = self._rows(Gprev, w_in)
                ops.transform_bwd(dh, b["dS"], self.h[k], self.Z[k - 1], self.Z[k - 1][g.U:], 1, self.featmask[k], self.scale,
                                  wtabs[k], gtabs[k], H, g.U, g.I, Gprev, Gprev[g.U:], 0, int(accumulate), b["ws"], d_in=w_in, d_out=w)
                G = Gprev
            else:
                ops.transform_bwd(dh, b["dS"], self.h[k], uEmbd, iEmbd, 0, self.featmask[k], self.scale, wtabs[k], gtabs[k],
                                  H, g.U, g.I, dU, dI, int(accumulate), int(accumulate), b["ws"], d_in=w_in, d_out=w)
            if after_grads is not None:
                after_grads(k)


# ------------------------------------------------------------------------------------------------
# autograd bridge (generic path: model(u, i, adj) -> scores, loss.backward())
# ------------------------------------------------------------------------------------------------


def stage_param_lists(stage_params, stages=STAGES):
    """flat [Wu heads | Wi heads | a heads] per stage -> list of lists."""
    out, i = [], 0
    for H, _ in stages:
        out.append(list(stage_params[i:i + 3 * H]))
        i += 3 * H
    return out


class PropagateFn(torch.autograd.Function):
    """Z_last = propagate(uEmbd, iEmbd, attention params).  Fresh buffers per call (the two forwards of a
    PairSampling step are alive together until loss.backward)."""

    @staticmethod
    def forward(ctx, graph, droprate, seed, call, injected, stages, uEmbd, iEmbd, *stage_params):
        prop = Propagation(graph, stages)
        prop.set_dropout(droprate, seed, call, injected)
        per_stage = stage_param_lists([p.detach() for p in stage_params], stages)
        ctx.stages = stages
        wtabs = [ops.pointer_table(ps) for ps in per_stage]
        Z = prop.forward(uEmbd.detach(), iEmbd.detach(), wtabs)
        ctx.prop, ctx.wtabs = prop, wtabs
        ctx.shapes = [p.shape for p in stage_params]
        ctx.uEmbd, ctx.iEmbd = uEmbd.detach(), iEmbd.detach()
        return Z

    @staticmethod
    def backward(ctx, G):
        prop = ctx.prop
        G = G.contiguous()
        dU = torch.empty_like(ctx.uEmbd)
        dI = torch.empty_like(ctx.iEmbd)
        grads = [torch.empty(s, dtype=torch.float32, device=G.device) for s in ctx.shapes]
        gtabs = [ops.pointer_table(gs) for gs in stage_param_lists(grads, ctx.stages)]
        prop.backward(G, ctx.uEmbd, ctx.iEmbd, ctx.wtabs, gtabs, dU, dI, accumulate=False)
        ctx.prop = None
        return (None, None, None, None, None, None, dU, dI, *grads)


class ScoreFn(torch.autograd.Function):
    """score_b = ELU(Z[u_b]) . ELU(Z[U+i_b])  (SPUIGACF.py:49-52)."""

    @staticmethod
    def forward(ctx, Z, U, users, items):
        users = users.to(torch.int64).contiguous()
        items = items.to(torch.int64).contiguous()
        out = torch.empty(users.numel(), dtype=torch.float32, device=Z.device)
        ops.score_pairs(Z, U, users, items, out)
        ctx.save_for_backward(Z, users, items)
        ctx.U = U
        return out

    @staticmethod
    def backward(ctx, dscore):
        Z, users, items = ctx.saved_tensors
        G = torch.zeros_like(Z)
        ops.score_pairs_bwd(Z, ctx.U, users, items, dscore.contiguous().float(), G)
        return G, None, None, None


class BPRLossFn(torch.autograd.Function):
    """-log(sigmoid(pos-neg)).mean()  (BPRLoss.py:8-9), stable form."""

    @staticmethod
    def forward(ctx, pos, neg):
        pos = pos.contiguous()
        neg = neg.contiguous()
        loss = torch.empty((), dtype=torch.float32, device=pos.device)
        dpos = torch.empty_like(pos)
        dneg = torch.empty_like(neg)
        ops.bpr_loss(pos, neg, 1.0, loss, dpos, dneg)
        ctx.save_for_backward(dpos, dneg)
        return loss

    @staticmethod
    def backward(ctx, gl):
        dpos, dneg = ctx.saved_tensors
        return dpos * gl, dneg * gl
