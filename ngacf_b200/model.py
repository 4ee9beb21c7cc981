"""Drop-in ``SPUIGACF`` (graphattention/SPUIGACF.py:5-52) backed by the sm_100a kernels.

Same constructor, same parameter names/shapes (so reference checkpoints load and vice-versa,
run_Gowalla.py:127-131,142-143), same ``forward(userIdx, itemIdx, mask) -> scores[B]`` contract:
every training-mode call runs a full-graph propagation with fresh dropout (SPUIGACF.py:41-52); in
eval mode the propagated features are cached until a parameter changes, because the reference's AllNeg
loop calls the model once per 64x2048 score tile (train_eval_Gowalla.py:300-326).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib, ops
from .graph import BipartiteGraph
from .propagation import PropagateFn, Propagation, ScoreFn

ALPHA = 0.2


class SpUIGraphAttentionLayer(nn.Module):
    """Parameter container with the reference's names and init (SPUIGACF.py:263-282).  The compute of
    all heads of a stage is batched inside the CUDA kernels, so a single layer has no forward here."""

    def __init__(self, in_dim, out_dim, dropout, alpha, concat=True):
        super().__init__()
        self.in_dim, self.out_dim, self.alpha, self.concat, self.p = in_dim, out_dim, alpha, concat, dropout
        self.W_u = nn.Parameter(torch.zeros(size=(in_dim, out_dim)))
        nn.init.xavier_normal_(self.W_u.data, gain=1.414)
        self.W_i = nn.Parameter(torch.zeros(size=(in_dim, out_dim)))
        nn.init.xavier_normal_(self.W_i.data, gain=1.414)
        self.a = nn.Parameter(torch.zeros(size=(1, 2 * out_dim)))
        nn.init.xavier_normal_(self.a.data, gain=1.414)

    def forward(self, *args, **kwargs):
        raise NotImplementedError("heads are evaluated batched by SPUIGACF.forward (ngacf_transform_fwd/ngacf_aggregate_fwd)")

    def __repr__(self):
        return self.__class__.__name__ + " (" + str(self.in_dim) + " -> " + str(self.out_dim) + ")"


class SpUIGAT(nn.Module):
    """attention_0..7 (embedSize->8, concat) + out_att (64->embedSize)  (SPUIGACF.py:187-205)."""

    def __init__(self, nfeat, nhid, nclass, dropout, alpha, nheads):
        super().__init__()
        self.dropout = dropout
        self.nheads = nheads
        for k in range(nheads):
            self.add_module("attention_{}".format(k), SpUIGraphAttentionLayer(nfeat, nhid, dropout, alpha, True))
        self.out_att = SpUIGraphAttentionLayer(nhid * nheads, nclass, dropout, alpha, False)

    @property
    def attentions(self):
        return [getattr(self, "attention_{}".format(k)) for k in range(self.nheads)]

    def stage_parameters(self):
        """[[W_u x8, W_i x8, a x8], [W_u, W_i, a]] -- the wtab order of include/ngacf_b200.h."""
        att = self.attentions
        return [[l.W_u for l in att] + [l.W_i for l in att] + [l.a for l in att],
                [self.out_att.W_u, self.out_att.W_i, self.out_att.a]]


class SPUIMultiGAT(nn.Module):
    """attention1_0..7 (embedSize->8), attention2_0..7 (64->8, concat) + out_att (64->embedSize): the 3-stage variant
    (SPUIGACF.py:217-256).  attention2 reads the 64-wide concatenation of attention1; at embedSize 64 its in_dim is nfeat."""

    def __init__(self, nfeat, nhid, nclass, dropout, alpha, nheads):
        super().__init__()
        self.dropout = dropout
        self.nheads = nheads
        # the reference constructs all attentions1 layers, then all attentions2 layers, then registers them (same RNG order)
        a1 = [SpUIGraphAttentionLayer(nfeat, nhid, dropout, alpha, True) for _ in range(nheads)]
        a2 = [SpUIGraphAttentionLayer(nhid * nheads, nhid, dropout, alpha, True) for _ in range(nheads)]
        for k, l in enumerate(a1):
            self.add_module("attention1_{}".format(k), l)
        for k, l in enumerate(a2):
            self.add_module("attention2_{}".format(k), l)
        self.out_att = SpUIGraphAttentionLayer(nhid * nheads, nclass, dropout, alpha, False)

    def stage_parameters(self):
        out = []
        for tag in ("attention1_", "attention2_"):
            att = [getattr(self, tag + str(k)) for k in range(self.nheads)]
            out.append([l.W_u for l in att] + [l.W_i for l in att] + [l.a for l in att])
        out.append([self.out_att.W_u, self.out_att.W_i, self.out_att.a])
        return out


class SPUIGACF(nn.Module):
    """embedSize 64 or 128 (ops.WIDTHS); anything else raises ValueError."""
    GAT = SpUIGAT
    HEAD_STAGES = 1               # 8-head stages in front of out_att

    def __init__(self, userNum, itemNum, embedSize, layers, droprate, useCuda=True):
        super().__init__()
        ops.check_width(embedSize)
        self.useCuda = useCuda
        self.embedSize = int(embedSize)
        self.userNum, self.itemNum, self.droprate = int(userNum), int(itemNum), float(droprate)
        self.stages = ops.spuigacf_stages(embedSize, self.HEAD_STAGES)
        self.uEmbd = nn.Embedding(userNum, embedSize)
        self.iEmbd = nn.Embedding(itemNum, embedSize)
        # `layers` is accepted and ignored exactly as in the reference (SPUIGACF.py:7 is its only use)
        self.gat = self.GAT(nfeat=embedSize, nhid=8, nclass=embedSize, dropout=droprate, nheads=8, alpha=ALPHA)
        self._extra_modules(embedSize, layers)      # subclasses create their modules HERE: the reference's RNG order (init after all modules)
        nn.init.normal_(self.uEmbd.weight, std=0.01)
        nn.init.normal_(self.iEmbd.weight, std=0.01)
        self.drop_seed = None       # Philox key of the dropout streams; defaults to torch.initial_seed()
        self._call = 0              # one dropout stream per forward call
        self._graph_key, self._graph = None, None
        self._eval_key, self._eval_Z = None, None
        self.injected_masks = None  # parity tests: dict(feat=[...], edge=[...]) consumed by the next call

    def _extra_modules(self, embedSize, layers):
        pass

    # ------------------------------------------------------------------------------------------
    def graph_for(self, mask: torch.Tensor) -> BipartiteGraph:
        if isinstance(mask, BipartiteGraph):
            return mask
        m = mask.squeeze(0) if mask.dim() == 3 else mask
        key = (m.data_ptr(), tuple(m.shape), m._version, str(m.device))
        if key != self._graph_key:
            self._graph = BipartiteGraph(m, self.userNum, self.itemNum)
            self._graph_key = key
            self._eval_key = None
        return self._graph

    def _flat_stage_params(self):
        return [p for stage in self.gat.stage_parameters() for p in stage]

    def _seed(self):
        if self.drop_seed is None:
            self.drop_seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
        return self.drop_seed

    def propagate(self, mask) -> torch.Tensor:
        """Pre-ELU output Z (N,embedSize) of the last stage; final features are ELU(Z)."""
        dev = self.uEmbd.weight.device
        if dev.type != "cuda":
            raise _lib.NgacfError("SPUIGACF runs on CUDA only (sm_100a kernels, no CPU fallback); call .cuda() first")
        graph = self.graph_for(mask)
        params = self._flat_stage_params()
        training = self.training and self.droprate > 0
        if not self.training:
            # eval mode: no autograd graph (the reference detaches every eval score, train_eval_Gowalla.py:334)
            key = tuple(p._version for p in [self.uEmbd.weight, self.iEmbd.weight] + params) + (id(graph), self.training)
            if key != self._eval_key:
                prop = getattr(self, "_eval_prop", None)
                if prop is None or prop.g is not graph:        # buffers are reused across evaluations of the same graph
                    prop = Propagation(graph, self.stages)
                    prop.set_dropout(0.0)
                ptrs = tuple(p.data_ptr() for p in params)
                if getattr(self, "_wtab_key", None) != ptrs:   # pointer tables only change when parameters move
                    self._wtabs = [ops.pointer_table([p.detach() for p in st]) for st in self.gat.stage_parameters()]
                    self._wtab_key = ptrs
                self._eval_Z = prop.forward(self.uEmbd.weight.detach(), self.iEmbd.weight.detach(), self._wtabs)
                self._eval_prop = prop
                self._eval_key = key
            return self._eval_Z
        call = self._call
        self._call += 1
        injected, self.injected_masks = self.injected_masks, None
        return PropagateFn.apply(graph, self.droprate if training else 0.0, self._seed(), call, injected, self.stages,
                                 self.uEmbd.weight, self.iEmbd.weight, *params)

    def forward(self, userIdx, itemIdx, mask):
        Z = self.propagate(mask)
        return ScoreFn.apply(Z, self.userNum, userIdx.to(Z.device), itemIdx.to(Z.device))


class SPUIMultiGACF(SPUIGACF):
    """3-stage variant (SPUIGACF.py:54-101): two 8-head stages, then out_att.  Same kernels, one more entry in the stage list."""
    GAT = SPUIMultiGAT
    HEAD_STAGES = 2
