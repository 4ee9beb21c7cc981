"""One process per GPU over torch.distributed (NCCL over NVLink/NVSwitch on the B200 box, gloo in CPU tests).

Two multi-GPU modes, both replacing the reference's single-process thread-per-GPU ``parallel.py``
(DataParallelModel / DataParallelCriterion2, SURVEY.md 2.4):

* ``ReplicaTrainer`` -- the reference's own ``--parallel True`` semantics (train_eval_Gowalla.py:97-104,137;
  SURVEY.md 5.8): every GPU runs the full-graph propagation with its own dropout stream and scores a
  different ``batch_size`` slice of the train rows, so a step consumes ``batch_size * world`` rows; the
  gradient is the SUM of the per-GPU mean-loss gradients (``loss.backward(ones(ndev))``).  Instead of
  broadcasting 18 MB of parameters before every forward and reduce-adding gradients to GPU 0
  (parallel.py:19,127-130), the replicas stay bit-identical: one NCCL all-reduce of the flat 18 MB gradient
  buffer per step and the same Adam update everywhere.  Weak scaling.  ``NegSamplingReplicaTrainer`` does the
  same for the NegSampling step (one propagation per GPU, the 1 + K items of its own rows).
* ``ShardedTrainer`` / ``ShardedNegSamplingTrainer`` -- the propagation(s) of one step partitioned by user range
  over the GPUs (below): the single-GPU step on the same batch.  Strong scaling.
* ``shard_eval_users`` / ``allreduce_sums`` -- AllNeg evaluation shards the test users over the ranks;
  only 16 metric sums (and optionally the top-20 lists) are merged; SampledNeg evaluation shards the test
  rows and merges its two sums.

The host-side pieces (row slicing, user sharding, flat-gradient all-reduce, metric merge) are plain
functions so that the world_size-2 gloo tests in tests/test_dist_cpu.py exercise them without a GPU.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import ops
from .negsampling import NegSamplingTrainer
from .train import FusedTrainer


def world_info():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def rank_rows(cursor: int, batch: int, rank: int, world: int, n_rows: int):
    """Train rows [lo,hi) of `rank` for the step starting at global `cursor` (a step consumes batch*world rows,
    train_eval_Gowalla.py:104).  Rows past n_rows are clipped (tail step)."""
    lo = min(n_rows, cursor + rank * batch)
    hi = min(n_rows, lo + batch)
    return lo, hi


def shard_range(n: int, rank: int, world: int):
    """Contiguous, balanced [lo,hi) split of n items."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def flat_views(params):
    """One contiguous gradient buffer with a view per parameter (a single all-reduce per step)."""
    total = sum(p.numel() for p in params)
    flat = torch.zeros(total, dtype=params[0].dtype, device=params[0].device)
    views, off = [], 0
    for p in params:
        views.append(flat[off:off + p.numel()].view_as(p))
        off += p.numel()
    return flat, views


def allreduce_sums(t: torch.Tensor):
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def shard_eval_users(eval_users: torch.Tensor, rank: int, world: int) -> torch.Tensor:
    lo, hi = shard_range(int(eval_users.numel()), rank, world)
    return eval_users[lo:hi].contiguous()


def require_width_64(model):
    """The multi-GPU trainers (partial-row kernels, batch-row exchange) are built for embedSize 64 only."""
    if getattr(model, "embedSize", 64) != 64:
        raise ValueError("multi-GPU training is built for embedSize 64 only (got %d); train embedSize %d on one GPU"
                         % (model.embedSize, model.embedSize))


class _ReplicaHooks:
    """The hooks of FusedTrainer._step_body / train_epoch that make a trainer one data-parallel replica: rank r scores the rows
    [r*B, (r+1)*B) of every step of batch*world rows with its own dropout stream, and the flat gradient is summed over the ranks
    between the two captured graphs.  Mixed in before a FusedTrainer subclass; self.rank / self.world are set before its __init__."""

    def _setup_params(self):
        m = self.model
        params = [m.uEmbd.weight, m.iEmbd.weight] + m._flat_stage_params()
        self.flat_grad, views = flat_views(params)
        for p, v in zip(params, views):
            p.grad = v
        super()._setup_params()

    # hooks used by FusedTrainer._step_body ---------------------------------------------------------
    def _row_offset(self):
        return self.rank * self.B

    def _row_stride(self):
        return self.B * self.world

    def _dropout_seed(self, seed):
        return (seed ^ (0x9E3779B97F4A7C15 * (self.rank + 1))) & 0xFFFFFFFFFFFFFFFF if self.world > 1 else seed

    def _reduce_grads(self):
        if self.world > 1:
            dist.all_reduce(self.flat_grad, op=dist.ReduceOp.SUM)      # sum of per-GPU mean-loss gradients

    def _collective_between(self):
        return self.world > 1

    def _epoch_loss(self, n):
        t = self.total.clone()
        allreduce_sums(t)          # the reference adds the per-GPU losses (loss.sum(), train_eval_Gowalla.py:139)
        return float(t.item()) / n


class ReplicaTrainer(_ReplicaHooks, FusedTrainer):
    """Data-parallel replicas of the fused PairSampling step (see module docstring)."""

    def __init__(self, model, inter, graph, batch_size, optim, sample_seed, use_cuda_graph=True, two_streams=True):
        require_width_64(model)
        self.rank, self.world = world_info()
        super().__init__(model, inter, graph, batch_size, optim, sample_seed, use_cuda_graph, two_streams)
        self.weak = True

    def units_per_step(self):
        return 2 * self.g.E * self.world

    def parallelism(self):
        return "dp%d replicas (reference --parallel semantics): batch %d x %d rows/step, one NCCL all-reduce of %.1f MB grads" % (
            self.world, self.B, self.world, self.flat_grad.numel() * 4 / 2 ** 20)


class NegSamplingReplicaTrainer(_ReplicaHooks, NegSamplingTrainer):
    """Data-parallel replicas of the NegSampling step: every GPU propagates the whole graph once with its own dropout stream and
    scores the 1 + K items of its own batch_size train rows; the gradients are summed (the reference's --parallel True in
    train_neg_sample).  The tail step of len % (batch*world) rows is trained, a rank without rows joins with a zero gradient."""

    def __init__(self, model, inter, graph, batch_size, optim, sample_seed, K=4, use_cuda_graph=True):
        require_width_64(model)
        self.rank, self.world = world_info()
        super().__init__(model, inter, graph, batch_size, optim, sample_seed, K=K, use_cuda_graph=use_cuda_graph)
        self.weak = True

    def units_per_step(self):
        return self.g.E * self.world

    def parallelism(self):
        return "dp%d NegSampling replicas (reference --parallel semantics): batch %d x %d rows/step, one NCCL all-reduce of %.1f MB grads" % (
            self.world, self.B, self.world, self.flat_grad.numel() * 4 / 2 ** 20)


# ------------------------------------------------------------------------------------------------
# north-star partition (SURVEY.md 8e): users and their edge rows range-partitioned over the GPUs, item rows OWNED by range;
# per stage the item rows are all-gathered and the item-side partial sums reduce-scattered
# ------------------------------------------------------------------------------------------------
class ShardPlan:
    """Host-side description of the partition (numpy only -- the world_size-2 gloo tests exercise it on the CPU).

    users : contiguous ranges balanced by EDGE count (rank r owns users [ub[r], ub[r+1]) and their CSR rows, which are the
            contiguous global edge ids [eb[r], eb[r+1]) -- so the Philox dropout streams, keyed by global edge id, are those of
            the single-GPU run);
    items : contiguous equal ranges of `chunk` = ceil(I / world) rows (the NCCL all-gather / reduce-scatter need equal counts);
            item-side buffers carry I_pad = chunk * world rows, the tail rows stay zero."""

    def __init__(self, edge_u, edge_i, U: int, I: int, world: int):
        import numpy as np
        key = np.unique(np.asarray(edge_u, np.int64) * np.int64(I) + np.asarray(edge_i, np.int64))     # global coalesce (host, once)
        self.eu, self.ei = key // I, key % I
        rowptr = np.zeros(U + 1, np.int64)
        np.add.at(rowptr, self.eu + 1, 1)
        self.rowptr = np.cumsum(rowptr)
        self.U, self.I, self.E, self.world = int(U), int(I), int(key.shape[0]), int(world)
        ub = [int(np.searchsorted(self.rowptr, (self.E * r) // world, side="left")) for r in range(world)] + [U]
        ub[0] = 0
        for r in range(1, world + 1):              # monotone even when one user holds more than E/world edges
            ub[r] = max(ub[r], ub[r - 1])
        self.ub = ub
        self.eb = [int(self.rowptr[b]) for b in ub]
        self.chunk = -(-I // world)
        self.I_pad = self.chunk * world

    def users(self, rank):
        return self.ub[rank], self.ub[rank + 1]

    def items(self, rank):
        lo = min(self.I, rank * self.chunk)
        return lo, min(self.I, lo + self.chunk)

    def edges(self, rank):
        return self.eb[rank], self.eb[rank + 1]

    def local_edges(self, rank):
        lo, hi = self.edges(rank)
        return self.eu[lo:hi], self.ei[lo:hi]


class Topology:
    """Two-level decomposition of a step over `world` GPUs.

    A PairSampling step is two independent propagations (pos, neg: train_eval_Gowalla.py:131-132).  With an even world size the
    GPUs form two groups of G = world/2: group q runs propagation q, user-range partitioned over its G ranks -- the per-stage
    exchanges then involve G ranks instead of `world`, carry one propagation instead of two, and at world = 2 disappear
    altogether (only the batch rows and the gradients cross NVLink).  With an odd world size (or NGACF_DIST_PROP_PARALLEL=0)
    every rank runs both propagations over the world-wide partition.

      scope "sub"  : the ranks that partition one propagation        (all-gather / reduce-scatter of item rows)
      scope "pair" : the ranks holding the SAME row ranges in the two groups (sum of the pos and neg embedding gradients)
      scope "world": everyone                                         (batch rows, attention-parameter gradients)"""

    def __init__(self, rank: int, world: int, prop_parallel=None):
        import os
        if prop_parallel is None:
            prop_parallel = os.environ.get("NGACF_DIST_PROP_PARALLEL", "1") != "0"
        self.rank, self.world = int(rank), int(world)
        self.prop_parallel = bool(prop_parallel) and world % 2 == 0 and world >= 2
        self.G = world // 2 if self.prop_parallel else world       # ranks per partition
        self.props = [rank // self.G] if self.prop_parallel else [0, 1]
        self.sub_rank = rank % self.G

    def members(self, scope, rank=None):
        r = self.rank if rank is None else rank
        if scope == "world":
            return list(range(self.world))
        if scope == "sub":
            base = (r // self.G) * self.G
            return list(range(base, base + self.G))
        if scope == "pair":
            return [r % self.G, r % self.G + self.G] if self.prop_parallel else [r]
        raise KeyError(scope)

    def rank_in(self, scope, rank=None):
        r = self.rank if rank is None else rank
        return self.members(scope, r).index(r)


class NcclTransport:
    """In-place collectives over torch.distributed (NCCL over NVLink / NVSwitch on the box; gloo in the CPU tests, where the two
    tensor collectives gloo lacks are expressed through all_gather / all_reduce)."""

    def __init__(self, topo: Topology = None):
        import os
        self.rank, self.world = world_info()
        self.gloo = dist.is_initialized() and dist.get_backend() == "gloo"
        self.coalesce = os.environ.get("NGACF_DIST_COALESCE", "1") != "0"
        self.topo = topo if topo is not None else Topology(self.rank, self.world)
        self._groups = {"world": None}
        if self.world > 1 and self.topo.prop_parallel:
            # every rank creates every group, in the same order
            G = self.topo.G
            for q in range(2):
                pg = dist.new_group(list(range(q * G, (q + 1) * G)))
                if self.rank // G == q:
                    self._groups["sub"] = pg
            for r in range(G):
                pg = dist.new_group([r, r + G])
                if self.rank % G == r:
                    self._groups["pair"] = pg
        else:
            self._groups["sub"] = None
            self._groups["pair"] = None

    def _coalesced(self, dev, group):
        """one NCCL group launch for the calls issued inside (ncclGroupStart/End): a collective point of the step exchanges
        several arrays (h | s, Ghat | dN, ...); issued one by one they cost one launch latency each"""
        import contextlib
        cm = getattr(dist, "_coalescing_manager", None)
        if self.gloo or cm is None or not self.coalesce:
            return contextlib.nullcontext()
        return cm(group=group, device=dev)

    def all_gather_rows(self, tensors, chunk, scope="sub"):
        """every tensor is (n*chunk, w): the rows [r*chunk,(r+1)*chunk) of rank-in-scope r are valid and are sent to the scope"""
        members = self.topo.members(scope)
        if len(members) == 1 or not tensors:
            return
        r, pg = self.topo.rank_in(scope), self._groups[scope]
        if self.gloo:
            for t in tensors:
                own = t[r * chunk:(r + 1) * chunk]
                parts = [torch.empty_like(own) for _ in members]
                dist.all_gather(parts, own.contiguous(), group=pg)
                for q, part in enumerate(parts):
                    t[q * chunk:(q + 1) * chunk].copy_(part)
            return
        with self._coalesced(tensors[0].device, pg):
            for t in tensors:
                dist.all_gather_into_tensor(t, t[r * chunk:(r + 1) * chunk], group=pg)

    def reduce_scatter_rows(self, tensors, chunk, scope="sub"):
        """every tensor is (n*chunk, w) of per-rank partial sums: afterwards the rows of rank-in-scope r hold the scope's sum"""
        members = self.topo.members(scope)
        if len(members) == 1 or not tensors:
            return
        r, pg = self.topo.rank_in(scope), self._groups[scope]
        if self.gloo:
            for t in tensors:
                dist.all_reduce(t, group=pg)
            return
        with self._coalesced(tensors[0].device, pg):
            for t in tensors:
                dist.reduce_scatter_tensor(t[r * chunk:(r + 1) * chunk], t, group=pg)

    def all_reduce(self, tensors, scope="world"):
        if len(self.topo.members(scope)) == 1 or not tensors:
            return
        pg = self._groups[scope]
        with self._coalesced(tensors[0].device, pg):
            for t in tensors:
                dist.all_reduce(t, group=pg)


class LocalCluster:
    """All ranks of the partition inside ONE process on one device: the trainers' plans are executed phase by phase and the
    collectives are applied directly to the ranks' buffers (sums in rank order).  This is how the sharded step is checked
    against the single-GPU step in the 1-GPU test suite (tests/test_gpu_parity.py) -- the NCCL run only swaps the transport."""

    def __init__(self, trainers):
        self.trainers = trainers

    @staticmethod
    def apply(kind, per_rank, chunk):
        """per_rank: the tensor lists of the members of ONE scope instance, in rank-in-scope order"""
        world = len(per_rank)
        if world == 1 or not per_rank[0]:
            return
        for j in range(len(per_rank[0])):
            ts = [per_rank[r][j] for r in range(world)]
            if kind == "ag":
                for d in range(world):
                    for q in range(world):
                        if d != q:
                            ts[d][q * chunk:(q + 1) * chunk].copy_(ts[q][q * chunk:(q + 1) * chunk])
            elif kind == "rs":
                sums = []
                for q in range(world):
                    acc = ts[0][q * chunk:(q + 1) * chunk].clone()
                    for d in range(1, world):
                        acc += ts[d][q * chunk:(q + 1) * chunk]
                    sums.append(acc)
                for q in range(world):
                    ts[q][q * chunk:(q + 1) * chunk].copy_(sums[q])
            else:
                acc = ts[0].clone()
                for d in range(1, world):
                    acc += ts[d]
                for d in range(world):
                    ts[d].copy_(acc)

    def _collective(self, phase):
        """phase: the same collective entry of every rank's plan; applied per scope instance"""
        _, _, kind, _, scope = phase[0]
        topo = self.trainers[0].topo
        done = set()
        for r in range(len(self.trainers)):
            members = tuple(topo.members(scope, r))
            if members in done:
                continue
            done.add(members)
            self.apply(kind, [phase[m][3] for m in members], self.trainers[0].plan.chunk)

    def run_steps(self, n_steps, read_loss=False):
        losses = []
        plans = None
        for tr in self.trainers:
            tr.model.train()
            tr._prepare_run()
        for _ in range(n_steps):
            for tr in self.trainers:
                tr._begin_step()
            if plans is None:
                plans = [tr._plan(*tr._mode()) for tr in self.trainers]
            for phase in zip(*plans):
                if phase[0][0] == "k":
                    for tr, (_, name, fn) in zip(self.trainers, phase):
                        with torch.cuda.device(tr.dev):
                            fn()
                else:
                    self._collective(phase)
            for tr in self.trainers:
                tr._end_step()
            if read_loss:
                losses.append(float(self.trainers[0].loss.item()))
        for tr in self.trainers:
            tr.model._call += tr.CALLS_PER_STEP * n_steps
        return losses

    def gather_state(self):
        """state_dict of the whole model assembled from the owners' rows (attention parameters from rank 0)"""
        sd = {k: v.detach().clone() for k, v in self.trainers[0].model.state_dict().items()}
        for tr in self.trainers[:self.trainers[0].topo.G]:        # the first partition holds every row once
            sd["uEmbd.weight"][tr.u_lo:tr.u_hi] = tr.model.uEmbd.weight.detach()[tr.u_lo:tr.u_hi]
            sd["iEmbd.weight"][tr.i_lo:tr.i_hi] = tr.model.iEmbd.weight.detach()[tr.i_lo:tr.i_hi]
        return sd

    def gather_grads(self):
        """{name: gradient} assembled the same way (after a step: embedding rows from their owners, attention grads summed)"""
        t0 = self.trainers[0]
        out = {"uEmbd.weight": torch.zeros_like(t0.model.uEmbd.weight), "iEmbd.weight": torch.zeros_like(t0.model.iEmbd.weight)}
        for tr in self.trainers[:t0.topo.G]:
            out["uEmbd.weight"][tr.u_lo:tr.u_hi] = tr.model.uEmbd.weight.grad[tr.u_lo:tr.u_hi]
            out["iEmbd.weight"][tr.i_lo:tr.i_hi] = tr.model.iEmbd.weight.grad[tr.i_lo:tr.i_hi]
        for name, p in t0.model.named_parameters():
            if name not in out:
                out[name] = p.grad.detach().clone()
        return out


class ShardedTrainer:
    """PairSampling step with the propagation partitioned by user range, one process per GPU (the reference's single-process
    DataParallelModel / DataParallelCriterion2, parallel.py:94-130,165-196 and train_eval_Gowalla.py:97-104,137, recompute the
    whole graph on every GPU).  Same maths as the single-GPU step on the same batch (strong scaling):

      stage forward : dense transform of the OWN users and the OWN items -> all-gather of the item rows (h | s) -> user rows
                      complete locally, item rows as partial sums over the own users' edges -> reduce-scatter to the item
                      owners -> finalize of the own item rows;
      pair scores   : every rank samples the same batch; the batch's rows are summed into a compact table by one all-reduce
                      (a row has one owner), scores / loss / dscore are computed redundantly, the gradient rows land on owners;
      stage backward: all-gather of the own items' Ghat | dN -> user pass (complete) + item pass (partial) over the local
                      edges -> reduce-scatter of dh | dS to the item owners -> dense backward of the own rows;
      update        : one all-reduce of the 17 K attention-parameter gradients (embedding gradients never leave their owner);
                      Adam on the own user rows, the own item rows and the (replicated) attention parameters.

    The pos and the neg propagation run on two streams between the collectives and share every collective call.  The whole
    step -- kernels and NCCL calls -- is captured in ONE CUDA graph; if the capture of the collectives is refused, the compute
    phases are captured separately and the collectives run eagerly between them (the round-1 structure)."""

    CALLS_PER_STEP = 2          # dropout call indices per step = propagations per step (pos, neg)
    PRUNABLE = True             # the output stage may be pruned to the batch rows when a rank holds a whole propagation (G == 1)
    PROP_PARALLEL = None        # layout of Topology (None: NGACF_DIST_PROP_PARALLEL decides)

    def __init__(self, model, inter, edge_u, edge_i, batch_size, optim, sample_seed, use_cuda_graph=True, transport=None, rank=None, world=None,
                 plan=None, prop_parallel=None):
        from .graph import BipartiteGraph
        from .propagation import Propagation
        require_width_64(model)
        if prop_parallel is None:
            prop_parallel = self.PROP_PARALLEL
        if transport is None:
            r0, w0 = world_info()
            self.topo = Topology(r0, w0, prop_parallel)
            transport = NcclTransport(self.topo)
        else:
            self.topo = Topology(rank, world, prop_parallel)
        self.transport = transport
        self.rank, self.world = self.topo.rank, self.topo.world
        self.model, self.inter, self.B, self.optim = model, inter, int(batch_size), optim
        self.sample_seed = int(sample_seed)
        self.use_cuda_graph = use_cuda_graph
        dev = model.uEmbd.weight.device
        self.dev = dev
        U, I = model.userNum, model.itemNum
        self.plan = plan if plan is not None else ShardPlan(edge_u, edge_i, U, I, self.topo.G)
        P = self.plan
        if P.world != self.topo.G:
            raise ValueError("the ShardPlan partitions over %d ranks, the topology needs %d" % (P.world, self.topo.G))
        sr = self.topo.sub_rank
        self.U, self.I = U, I
        self.u_lo, self.u_hi = P.users(sr)
        self.i_lo, self.i_hi = P.items(sr)
        self.e_lo, self.e_hi = P.edges(sr)
        eu, ei = P.local_edges(sr)
        import numpy as np
        with torch.cuda.device(dev):
            self.g = BipartiteGraph(torch.from_numpy(np.stack([eu, ei])).to(dev), U, I, check_users=False)
        g = self.g
        self.stages = tuple(model.stages)
        S = len(self.stages)
        N_alloc = U + P.I_pad                       # item-side rows padded to world * chunk (the pad rows stay zero)
        f32 = dict(dtype=torch.float32, device=dev)
        i64 = dict(dtype=torch.int64, device=dev)

        def rows(w):
            return torch.zeros((N_alloc, w), **f32)
        self.props = []
        for _ in range(self.CALLS_PER_STEP):       # one propagation per dropout call: pos / neg
            p = Propagation.__new__(Propagation)
            p.g, p.stages = g, self.stages
            p.h = [rows(ops.D) for _ in self.stages]
            p.Z = [rows(ops.D) for _ in self.stages]
            p.s = [rows(H) for H, _ in self.stages]
            p.norm = [rows(H) for H, _ in self.stages]
            p.scratch = torch.empty(max(g.S, 1) * 72, **f32)
            p.counter = torch.zeros(max(g.L, 1), dtype=torch.int32, device=dev)
            p.G = [rows(ops.D), rows(ops.D)]
            p.Ghat, p.dh = rows(ops.D), rows(ops.D)
            p.dN = [rows(H) for H, _ in self.stages]      # one (N,H) array per stage width (the kernels index them as (N,H))
            p.dS = [rows(H) for H, _ in self.stages]
            p.ds = torch.empty(max(g.E, 1) * 8, **f32)
            p.ws = torch.empty(ops.transform_bwd_workspace_bytes(U, I) // 4, **f32)
            p.ZS = rows(ops.D)                             # scoring table: the batch's rows at their global positions
            p.fm = [torch.zeros(N_alloc, **i64) for _ in self.stages]
            p.em = [torch.zeros(max(P.E, 1), dtype=torch.uint8, device=dev) for _ in self.stages]      # indexed by GLOBAL edge id
            p.featmask, p.edgemask, p.scale = [None] * S, [None] * S, 1.0
            self.props.append(p)
        self._batch_buffers(f32, i64)
        self.loss = torch.zeros((), **f32)
        self.total = torch.zeros((), dtype=torch.float64, device=dev)
        self.row_dev = torch.zeros(2, **i64)
        self.call_dev = torch.zeros(1, **i64)
        self.side = torch.cuda.Stream(device=dev)
        # G == 1 (world 2, propagation-parallel): the propagation is whole on this rank -- no partial sums, and the output stage is
        # pruned to the batch rows exactly as in the single-GPU trainer (csrc/pruned_stage.cu)
        import os
        self.complete = self.topo.G == 1
        self.prune = self.complete and self.PRUNABLE and os.environ.get("NGACF_PRUNE", "1") != "0" and self.stages[-1][0] == 1
        self.active = {q: ops.ActiveRows(g) for q in self.topo.props} if self.prune else {}
        # parameters: embedding gradients stay with the owner of the row; the attention parameters are replicated and their
        # gradients (partial sums over the own rows) are summed by one small all-reduce
        m = model
        self.small = m._flat_stage_params()
        self.flat_small, views = flat_views(self.small)
        for p_, v in zip(self.small, views):
            p_.grad = v
        for p_ in (m.uEmbd.weight, m.iEmbd.weight):
            if p_.grad is None:
                p_.grad = torch.zeros_like(p_)
        stage_params = m.gat.stage_parameters()
        self.wtabs = [ops.pointer_table([q.detach() for q in st]) for st in stage_params]
        self.gtabs = [ops.pointer_table([q.grad for q in st]) for st in stage_params]
        group = optim.param_groups[0]
        self.hyper = dict(lr=float(group["lr"]), b1=float(group["betas"][0]), b2=float(group["betas"][1]), eps=float(group["eps"]),
                          wd=float(group["weight_decay"]))
        self.params = [m.uEmbd.weight, m.iEmbd.weight] + self.small
        for p_ in self.params:
            st = optim.state[p_]
            if len(st) == 0:
                st["step"], st["exp_avg"], st["exp_avg_sq"] = torch.tensor(0.0), torch.zeros_like(p_), torch.zeros_like(p_)
        # Adam table: row slices of the embedding tables (own rows only) + the attention parameters
        entries = []

        def entry(p_, lo=None, hi=None):
            st = optim.state[p_]
            sl = slice(lo, hi)
            return (p_.detach()[sl], p_.grad[sl], st["exp_avg"][sl], st["exp_avg_sq"][sl])
        if self.u_hi > self.u_lo:
            entries.append(entry(m.uEmbd.weight, self.u_lo, self.u_hi))
        if self.i_hi > self.i_lo:
            entries.append(entry(m.iEmbd.weight, self.i_lo, self.i_hi))
        entries += [entry(q) for q in self.small]
        self._adam_entries = entries
        self.adam_tab = torch.tensor([[a.data_ptr(), b.data_ptr(), c.data_ptr(), d.data_ptr(), a.numel()] for a, b, c, d in entries],
                                     dtype=torch.int64).to(dev)
        self.adam_total = sum(a.numel() for a, _, _, _ in entries)
        self.adam_state = torch.tensor([float(optim.state[self.params[0]]["step"]), 0.0, 0.0, 0.0], dtype=torch.float64, device=dev)
        self._graph = None
        self._segments = None
        self._key = None
        self._cursor = 0
        self.capture_mode = None

    # ------------------------------------------------------------------------------------------
    # the PairSampling-specific parts of the step (ShardedNegSamplingTrainer overrides them)
    def _batch_buffers(self, f32, i64):
        self.Zb = torch.zeros((2, 2 * self.B, ops.D), **f32)           # compact batch rows of both propagations (one all-reduce)
        self.users, self.pos, self.neg = torch.zeros(self.B, **i64), torch.zeros(self.B, **i64), torch.zeros(self.B, **i64)
        self.sc_all = torch.zeros((2, self.B), **f32)          # pair scores of both propagations (exchanged as scores when G == 1)
        self.sc = [self.sc_all[0], self.sc_all[1]]
        self.dsc = [torch.zeros(self.B, **f32), torch.zeros(self.B, **f32)]

    def _mine(self):
        """the propagations this rank runs: [0, 1], or [q] in the propagation-parallel layout"""
        return list(self.topo.props)

    def _sample(self):
        ops.sample_pairs(self.inter, 0, self.B, self.sample_seed, 0, self.users, self.pos, self.neg, self.row_dev)
        if self.prune:      # active rows of propagation q: stamped with its dropout call index (as in train.FusedTrainer)
            for q in self._mine():
                self.active[q].at(q, self.call_dev).mark(self.users, (self.pos, self.neg)[q])

    def _output_rows(self, q, Z):
        """end of the last stage of propagation q (Z: its output rows, complete for the own rows)"""
        item = (self.pos, self.neg)[q]
        if self.complete:      # every row is local: score the own propagation's pairs here, exchange SCORES instead of rows
            ops.score_pairs(Z, self.U, self.users, item, self.sc[q])
        else:
            ops.batch_rows_gather(Z, self.U, self.users, item, (self.u_lo, self.u_hi), (self.i_lo, self.i_hi), self.Zb[q])

    def _loss_phases(self, both, zero_own):
        """the phases from the exchange of the batch rows (or scores) to the gradient rows G of the last stage"""
        U, S, mine = self.U, len(self.stages), self._mine()
        items = (self.pos, self.neg)
        plan = []
        if self.complete:
            other = 1 - mine[0]
            plan.append(("k", "zero the other propagation's scores", lambda: ops.memset_zero(self.sc[other])))
            plan.append(("c", "all-reduce pair scores", "ar", [self.sc_all], "world"))
        else:
            if len(mine) == 1:
                other = 1 - mine[0]
                plan.append(("k", "zero the other propagation's batch rows", lambda: ops.memset_zero(self.Zb[other])))
            plan.append(("c", "all-reduce batch rows", "ar", [self.Zb], "world"))

        def score(q):
            p = self.props[q]
            ops.batch_rows_scatter(self.Zb[q], U, self.users, items[q], p.ZS)
            ops.score_pairs(p.ZS, U, self.users, items[q], self.sc[q])

        def loss_and_scatter():
            if not self.complete:
                both(score, [0, 1])()           # every rank scores both propagations' pairs (the loss needs both)
            ops.bpr_loss(self.sc[0], self.sc[1], 1.0, self.loss, self.dsc[0], self.dsc[1])

            def scatter(q):
                p = self.props[q]
                G = p.G[0]
                if not self.prune:      # pruned: the scatter writes exactly the active rows, nothing else of G is read
                    zero_own(G)
                # rows of other owners are written and never read
                ops.score_pairs_bwd(p.Z[S - 1] if self.complete else p.ZS, U, self.users, items[q], self.dsc[q], G)
            both(scatter)()
            ops.memset_zero(self.flat_small)        # attention-parameter gradients are accumulated by every dense backward
        plan.append(("k", "scores+loss+scatter", loss_and_scatter))
        return plan

    # ------------------------------------------------------------------------------------------
    def _items_view(self, t):
        return t[self.U:]                        # (I_pad, w): the item rows of a per-node buffer

    def _mode(self):
        m = self.model
        return (m.droprate if m.droprate > 0 else 0.0), m._seed()

    def _plan(self, droprate, seed):
        """[("k", name, fn) | ("c", name, kind, tensors)]: compute phases (kernels of both propagations on two streams) and
        collectives ("ag" / "rs" over the item rows, "ar")."""
        m, P, g = self.model, self.plan, self.g
        U, I, B = self.U, self.I, self.B
        ulo, uhi, ilo, ihi = self.u_lo, self.u_hi, self.i_lo, self.i_hi
        nu, ni = uhi - ulo, ihi - ilo
        uE, iE = m.uEmbd.weight.detach(), m.iEmbd.weight.detach()
        dU, dI = m.uEmbd.weight.grad, m.iEmbd.weight.grad
        side = self.side
        S = len(self.stages)
        heads = [H for H, _ in self.stages]
        scale = 1.0 / (1.0 - droprate) if droprate > 0 else 1.0
        plan = []

        mine = self._mine()

        def both(fn, props=None):
            """fn(q) for each propagation of this rank: the first on the current stream, the second on the side stream"""
            qs = mine if props is None else props

            def run():
                if len(qs) == 1:
                    fn(qs[0])
                    return
                cur = torch.cuda.current_stream()
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    fn(qs[1])
                fn(qs[0])
                cur.wait_stream(side)
            return run

        complete, prune = self.complete, self.prune
        plan.append(("k", "sample", self._sample))

        def masks(k):
            p = self.props[k]
            if droprate <= 0:
                p.featmask, p.edgemask, p.scale = [None] * S, [None] * S, 1.0
                return
            p.scale = scale
            ops.dropout_masks_ranges(p.fm, p.em, heads, ((ulo, uhi), (U + ilo, U + ihi)), (self.e_lo, self.e_hi), seed, k, droprate, self.call_dev)
            p.featmask = list(p.fm)
            p.edgemask = [e[self.e_lo:] for e in p.em]          # local edge id + e_lo = global edge id
        for k in range(len(self.props)):
            masks(k) if droprate <= 0 else None
        if droprate > 0:
            plan.append(("k", "masks", both(masks)))

        for k, (H, _) in enumerate(self.stages):
            act = 0 if k == 0 else 1

            def transform(q, k=k, H=H, act=act):
                p = self.props[q]
                Xu = uE if k == 0 else p.Z[k - 1]
                Xi = iE if k == 0 else p.Z[k - 1][U:]
                fm = p.featmask[k]
                if nu:
                    ops.transform_fwd(Xu[ulo:uhi], None, act, None if fm is None else fm[ulo:], p.scale, self.wtabs[k], H, nu, 0,
                                      p.h[k][ulo:uhi], p.s[k][ulo:uhi])
                if ni:
                    ops.transform_fwd(None, Xi[ilo:ihi], act, None if fm is None else fm[U + ilo:], p.scale, self.wtabs[k], H, 0, ni,
                                      p.h[k][U + ilo:U + ihi], p.s[k][U + ilo:U + ihi])
            plan.append(("k", "transform%d" % k, both(transform)))
            plan.append(("c", "all-gather h|s items, stage %d" % k, "ag",
                         [self._items_view(t) for q in mine for t in (self.props[q].h[k], self.props[q].s[k])], "sub"))

            def aggregate(q, k=k, H=H):
                p = self.props[q]
                if prune and k == S - 1:
                    ops.aggregate_fwd_active(g, p.scratch, p.counter, p.h[k], p.s[k], H, p.edgemask[k], p.scale, p.Z[k], p.norm[k], self.active[q])
                else:
                    ops.aggregate_fwd(g, p.scratch, p.counter, p.h[k], p.s[k], H, p.edgemask[k], p.scale, p.Z[k], p.norm[k],
                                      partial_from=-1 if complete else g.T_users)
            plan.append(("k", "aggregate%d" % k, both(aggregate)))
            plan.append(("c", "reduce-scatter Z|norm items, stage %d" % k, "rs",
                         [self._items_view(t) for q in mine for t in (self.props[q].Z[k], self.props[q].norm[k])], "sub"))

            def finalize(q, k=k, H=H):
                p = self.props[q]
                if ni and not complete:
                    ops.aggregate_finalize(p.Z[k][U + ilo:U + ihi], p.h[k][U + ilo:U + ihi], p.norm[k][U + ilo:U + ihi], H)
                if k == S - 1:
                    self._output_rows(q, p.Z[k])
            plan.append(("k", "finalize%d" % k, both(finalize)))

        def zero_own(G):
            if nu:
                ops.memset_zero(G[ulo:uhi])
            if ni:
                ops.memset_zero(G[U + ilo:U + ihi])
        plan += self._loss_phases(both, zero_own)

        evs = [torch.cuda.Event() for _ in range(S)]
        for k in range(S - 1, -1, -1):
            H, _ = self.stages[k]
            Gi = (S - 1 - k) % 2                  # G ping-pong: stage S-1 reads G[0]

            def prep(q, k=k, H=H, Gi=Gi):
                p = self.props[q]
                G = p.G[Gi]
                if prune and k == S - 1:
                    ops.stage_bwd_prep_active(g, G, p.Z[k], p.h[k], p.norm[k], H, p.Ghat, p.dN[k], self.active[q])
                    return
                if nu:
                    ops.stage_bwd_prep(G[ulo:uhi], p.Z[k][ulo:uhi], p.h[k][ulo:uhi], p.norm[k][ulo:uhi], H, p.Ghat[ulo:uhi], p.dN[k][ulo:uhi])
                if ni:
                    ops.stage_bwd_prep(G[U + ilo:U + ihi], p.Z[k][U + ilo:U + ihi], p.h[k][U + ilo:U + ihi], p.norm[k][U + ilo:U + ihi], H,
                                       p.Ghat[U + ilo:U + ihi], p.dN[k][U + ilo:U + ihi])
            plan.append(("k", "prep%d" % k, both(prep)))
            plan.append(("c", "all-gather Ghat|dN items, stage %d" % k, "ag",
                         [self._items_view(t) for q in mine for t in (self.props[q].Ghat, self.props[q].dN[k])], "sub"))

            def edges(q, k=k, H=H, Gi=Gi):
                p = self.props[q]
                for mode in (0, 1):
                    if prune and k == S - 1:
                        ops.stage_bwd_edges_active(mode, g, p.scratch, p.counter, p.G[Gi], p.Ghat, p.dN[k], p.h[k], p.s[k], H, p.edgemask[k],
                                                   p.scale, self.wtabs[k], p.ds, p.dh, p.dS[k], self.active[q])
                    else:
                        ops.stage_bwd_edges(mode, g, p.scratch, p.counter, p.G[Gi], p.Ghat, p.dN[k], p.h[k], p.s[k], H, p.edgemask[k], p.scale,
                                            self.wtabs[k], p.ds, p.dh, p.dS[k], partial=0 if complete else mode)
            plan.append(("k", "edges%d" % k, both(edges)))
            plan.append(("c", "reduce-scatter dh|dS items, stage %d" % k, "rs",
                         [self._items_view(t) for q in mine for t in (self.props[q].dh, self.props[q].dS[k])], "sub"))

            def dense(k=k, H=H, Gi=Gi):
                cur = torch.cuda.current_stream()

                def fin(q):
                    p = self.props[q]
                    if ni and not complete:
                        ops.stage_bwd_finalize(p.dh[U + ilo:U + ihi], p.dS[k][U + ilo:U + ihi], p.G[Gi][U + ilo:U + ihi], self.wtabs[k], H, 1)

                def tb(q):
                    # weight gradients always ACCUMULATE into the (zero-filled) flat buffer: a rank may own no rows of a side
                    p = self.props[q]
                    Gprev = p.G[1 - Gi]
                    acc = int(mine.index(q) > 0)       # the first propagation of this rank writes the embedding gradients
                    fm = p.featmask[k]
                    fu = None if fm is None else fm[ulo:]
                    fi = None if fm is None else fm[U + ilo:]
                    if k > 0:
                        Zp = p.Z[k - 1]
                        if nu:
                            ops.transform_bwd(p.dh[ulo:uhi], p.dS[k][ulo:uhi], None, Zp[ulo:uhi], None, 1, fu, p.scale, self.wtabs[k], self.gtabs[k], H,
                                              nu, 0, Gprev[ulo:uhi], None, 0, 1, p.ws)
                        if ni:
                            ops.transform_bwd(p.dh[U + ilo:U + ihi], p.dS[k][U + ilo:U + ihi], None, None, Zp[U + ilo:U + ihi], 1, fi, p.scale,
                                              self.wtabs[k], self.gtabs[k], H, 0, ni, None, Gprev[U + ilo:U + ihi], 0, 1, p.ws)
                    else:
                        if nu:
                            ops.transform_bwd(p.dh[ulo:uhi], p.dS[k][ulo:uhi], None, uE[ulo:uhi], None, 0, fu, p.scale, self.wtabs[k], self.gtabs[k], H,
                                              nu, 0, dU[ulo:uhi], None, acc, 1, p.ws)
                        if ni:
                            ops.transform_bwd(p.dh[U + ilo:U + ihi], p.dS[k][U + ilo:U + ihi], None, None, iE[ilo:ihi], 0, fi, p.scale, self.wtabs[k],
                                              self.gtabs[k], H, 0, ni, None, dI[ilo:ihi], acc, 1, p.ws)
                if len(mine) == 1:
                    fin(mine[0])
                    tb(mine[0])
                    return
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    fin(1)
                fin(0)
                tb(0)
                evs[k].record(cur)                # the gradient buffers: pos first, neg accumulates after it
                with torch.cuda.stream(side):
                    side.wait_event(evs[k])
                    tb(1)
                cur.wait_stream(side)
            plan.append(("k", "dense-bwd%d" % k, dense))

        if self.topo.prop_parallel:
            # the two groups hold the pos and the neg contribution to the SAME embedding rows: summed between counterparts
            pair = [t for t in (dU[ulo:uhi] if nu else None, dI[ilo:ihi] if ni else None) if t is not None]
            plan.append(("c", "all-reduce pos+neg embedding gradients of the own rows (pair)", "ar", pair, "pair"))
        plan.append(("c", "all-reduce attention-parameter grads", "ar", [self.flat_small], "world"))

        def update():
            h = self.hyper
            ops.adam_step_dev(self.adam_tab, len(self._adam_entries), self.adam_total, h["lr"], h["b1"], h["b2"], h["eps"], h["wd"], self.adam_state)
            ops.step_counters(self.total, self.loss, self.row_dev, B)
            ops.counter_add(self.call_dev, self.CALLS_PER_STEP)
        plan.append(("k", "adam", update))
        return plan

    # ------------------------------------------------------------------------------------------
    def _run_eager(self, plan):
        for ph in plan:
            if ph[0] == "k":
                ph[2]()
            else:
                self._collective(ph[2], ph[3], ph[4])

    def _collective(self, kind, tensors, scope):
        t = self.transport
        if kind == "ag":
            t.all_gather_rows(tensors, self.plan.chunk, scope)
        elif kind == "rs":
            t.reduce_scatter_rows(tensors, self.plan.chunk, scope)
        else:
            t.all_reduce(tensors, scope)

    def _snapshot(self):
        st = self.optim.state
        return ([p.detach().clone() for p in self.params], [(st[p]["exp_avg"].clone(), st[p]["exp_avg_sq"].clone()) for p in self.params],
                [t.clone() for t in (self.adam_state, self.total, self.row_dev, self.call_dev)])

    def _restore(self, snap):
        ps, opt, misc = snap
        with torch.no_grad():
            for p, sp, (a, b) in zip(self.params, ps, opt):
                p.copy_(sp)
                self.optim.state[p]["exp_avg"].copy_(a)
                self.optim.state[p]["exp_avg_sq"].copy_(b)
            for t, v in zip((self.adam_state, self.total, self.row_dev, self.call_dev), misc):
                t.copy_(v)

    def _compile(self, droprate, seed):
        """Capture the step.  NGACF_DIST_CAPTURE = full (default: kernels AND collectives in one CUDA graph), segments (compute
        phases captured, collectives eager between them) or eager."""
        import os
        plan = self._plan(droprate, seed)
        self._plan_cache = plan
        self._key = (droprate, seed)
        self._graph, self._segments = None, None
        want = os.environ.get("NGACF_DIST_CAPTURE", "full") if self.use_cuda_graph else "eager"
        self.capture_mode = "eager"
        if want == "eager":
            return
        snap = self._snapshot()
        s = torch.cuda.Stream(device=self.dev)           # warm-up (communicators, lazy state) off the default stream
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._run_eager(plan)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize(self.dev)
        if want == "full":
            try:
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr, capture_error_mode="thread_local"):
                    self._run_eager(plan)
                self._graph = gr
                self.capture_mode = "one CUDA graph (kernels + NCCL)"
            except Exception as e:       # noqa: BLE001  -- the collectives' capture was refused: fall back to segments
                import sys
                print("[ngacf_b200.dist] whole-step capture failed (%s: %s); capturing compute segments only" % (type(e).__name__, e),
                      file=sys.stderr, flush=True)
                torch.cuda.synchronize(self.dev)
                want = "segments"
        if want == "segments":
            segs, cur = [], []
            for ph in plan + [("c", "end", None, None, None)]:
                if ph[0] == "k":
                    cur.append(ph[2])
                    continue
                if cur:
                    gr = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gr):
                        for fn in cur:
                            fn()
                    segs.append(gr.replay)
                    cur = []
                if ph[2] is not None:
                    segs.append(lambda kind=ph[2], ts=ph[3], sc=ph[4]: self._collective(kind, ts, sc))
            self._segments = segs
            self.capture_mode = "CUDA-graph segments, eager collectives"
        self._restore(snap)

    def _prepare_run(self):
        self.row_dev.copy_(torch.tensor([self._cursor, 0], dtype=torch.int64))
        self.call_dev.fill_(self.model._call)

    def release(self):
        """drop the captured graph(s) (they hold NCCL work): call before dist.destroy_process_group()"""
        torch.cuda.synchronize(self.dev)
        self._graph, self._segments, self._key = None, None, None

    def _begin_step(self):
        if self._cursor + self.B > len(self.inter):
            self._cursor = 0
            self.row_dev.zero_()

    def _end_step(self):
        self._cursor += self.B

    def _replay(self):
        if self._graph is not None:
            self._graph.replay()
        elif self._segments is not None:
            for f in self._segments:
                f()
        else:
            self._run_eager(self._plan_cache)

    def run_steps(self, n_steps, host_rows=None, read_loss=False):
        m = self.model
        m.train()
        droprate, seed = self._mode()
        if self._key != (droprate, seed):
            self._compile(droprate, seed)
        self._prepare_run()
        losses = []
        for _ in range(n_steps):
            self._begin_step()
            if host_rows is not None:
                lo = self._cursor
                self.inter.train_rows_user[lo:lo + self.B].copy_(host_rows[lo:lo + self.B], non_blocking=True)
            self._replay()
            self._end_step()
            if read_loss:
                losses.append(float(self.loss.item()))
        m._call += self.CALLS_PER_STEP * n_steps
        return losses

    def train_epoch(self, epoch: int = 0, max_steps=None) -> float:
        """Full batches of one epoch (the tail batch of len % batch rows is dropped in the sharded mode); returns
        sum(batch-mean loss) / len(train_df) like train_bpr (train_eval_Gowalla.py:139,144).  The embedding tables are
        re-assembled on every rank afterwards."""
        n = len(self.inter)
        n_full = n // self.B
        if max_steps is not None:
            n_full = min(n_full, max_steps)
        self.total.zero_()
        self._cursor = 0
        self.row_dev.copy_(torch.tensor([0, epoch], dtype=torch.int64))
        self.run_steps(n_full)
        self.sync_embeddings()
        return float(self.total.item()) / n

    def sync_embeddings(self):
        """every rank ends up with the full, updated embedding tables (rows travel from their owner); once per epoch"""
        if self.world == 1 or not isinstance(self.transport, NcclTransport):
            return
        m, P = self.model, self.plan
        with torch.no_grad():
            for r in range(self.topo.G):          # the ranks of the first partition hold every row once
                for w, (lo, hi) in ((m.uEmbd.weight, P.users(r)), (m.iEmbd.weight, P.items(r))):
                    if hi > lo:        # parameters and Adam moments: rank 0's checkpoint is then the whole model + optimizer
                        st = self.optim.state[w]
                        for t in (w.data, st["exp_avg"], st["exp_avg_sq"]):
                            dist.broadcast(t[lo:hi], src=r)
        step = float(self.adam_state[0].item())
        for p in self.params:
            self.optim.state[p]["step"] = torch.tensor(step)

    # ------------------------------------------------------------------------------------------
    def profile_phases(self, n_steps=5):
        """CUDA-event time of every phase of the step (eager, phases back to back): [(kind, name, ms)] averaged over n_steps.
        State is restored afterwards."""
        droprate, seed = self._mode()
        plan = self._plan(droprate, seed)
        snap = self._snapshot()
        self._run_eager(plan)
        torch.cuda.synchronize(self.dev)
        evs = []
        for _ in range(n_steps):
            row = []
            for ph in plan:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                if ph[0] == "k":
                    ph[2]()
                else:
                    self._collective(ph[2], ph[3], ph[4])
                e1.record()
                row.append((e0, e1))
            evs.append(row)
        torch.cuda.synchronize(self.dev)
        out = []
        for j, ph in enumerate(plan):
            ms = sum(evs[i][j][0].elapsed_time(evs[i][j][1]) for i in range(n_steps)) / n_steps
            nbytes = sum(t.numel() * t.element_size() for t in ph[3]) if ph[0] == "c" else 0
            out.append(dict(kind="collective" if ph[0] == "c" else "compute", name=ph[1], ms=ms, bytes=nbytes,
                            ranks=len(self.topo.members(ph[4])) if ph[0] == "c" else 1))
        self._restore(snap)
        return out

    def launches_per_step(self, droprate):
        S = len(self.stages)
        per_prop = (1 if droprate > 0 else 0) + S * (2 + 1 + 1) + 1 + 2 + 1 + S * (2 + 2 + 1 + 4)
        return 1 + 2 * per_prop + 1 + 2 + 2

    def units_per_step(self):
        return len(self.props) * self.plan.E           # strong scaling: the same global step on every world size

    def _layout(self):
        return ("2 groups of %d GPUs (group q runs propagation q)" % self.topo.G) if self.topo.prop_parallel else "both propagations on every GPU"

    def parallelism(self):
        return ("%d GPUs: %s; users range-partitioned over %d ranks by edge count (rank %d: users [%d,%d), %d of %d edges), item rows owned by "
                "range (%d per rank); per stage: all-gather of the item rows, reduce-scatter of the item partials; %s" % (
                    self.world, self._layout(), self.topo.G, self.rank, self.u_lo, self.u_hi, self.e_hi - self.e_lo, self.plan.E, self.plan.chunk,
                    self.capture_mode))

    def working_set_bytes(self):
        N = self.U + self.plan.I_pad
        return len(self.props) * (9 * N * 256 + 8 * (self.e_hi - self.e_lo) * 4) + 7 * self.adam_total * 4

    def profile_kernels(self, n_steps=3):
        return []


class ShardedNegSamplingTrainer(ShardedTrainer):
    """NegSampling step (negsampling.NegSamplingTrainer) with its ONE propagation partitioned by user range over all `world` ranks
    (one group, G = world: no propagation-parallel layout, no sub-groups).  Same maths as the single-GPU step on the same batch:

      batch         : every rank samples the same b train rows x (1 positive + K negatives), column-major (column j = pairs
                      [j*b, (j+1)*b));
      stages        : as in ShardedTrainer, for one propagation (dropout call offset 0, one call index per step);
      pair scores   : the (K+1)*b pairs' rows are gathered into a compact table (a user row appears K+1 times; every copy is
                      the same row) and summed by one all-reduce; scores, BCE and dscore are computed redundantly, and the
                      gradient rows are scattered one column at a time (accumulating), as on one GPU;
      backward and update as in ShardedTrainer.

    As in the PairSampling partition, the tail batch of len % batch rows is dropped."""

    CALLS_PER_STEP = 1
    PRUNABLE = False            # a pruned NegSampling output stage is not built
    PROP_PARALLEL = False       # one propagation: one group of `world` ranks

    def __init__(self, model, inter, edge_u, edge_i, batch_size, optim, sample_seed, K=4, use_cuda_graph=True, transport=None, rank=None,
                 world=None, plan=None):
        self.K = int(K)
        if inter.min_negatives() < self.K:      # random.sample(negative_items, K) raises in the reference (loadGowalla.py:82)
            raise ValueError("a user has fewer than K=%d negatives (item pool minus the user's positives)" % self.K)
        super().__init__(model, inter, edge_u, edge_i, batch_size, optim, sample_seed, use_cuda_graph=use_cuda_graph, transport=transport,
                         rank=rank, world=world, plan=plan)

    def _batch_buffers(self, f32, i64):
        n = self.B * (self.K + 1)
        self.pu, self.pi = torch.zeros(n, **i64), torch.zeros(n, **i64)
        self.Zb = torch.zeros((2 * n, ops.D), **f32)          # compact rows of the n users, then of the n items
        self.sc, self.dsc = torch.zeros(n, **f32), torch.zeros(n, **f32)

    def _mine(self):
        return [0]

    def _sample(self):
        it = self.inter
        ops.sample_negs(it, it.train_rows_user, it.train_rows_item, 0, self.B, self.sample_seed, 0, self.K, ops.NEG_TAG_TRAIN, self.pu, self.pi,
                        self.row_dev, col_stride=self.B)

    def _output_rows(self, q, Z):
        ops.batch_rows_gather(Z, self.U, self.pu, self.pi, (self.u_lo, self.u_hi), (self.i_lo, self.i_hi), self.Zb)

    def _loss_phases(self, both, zero_own):
        U, b, p = self.U, self.B, self.props[0]

        def loss_and_scatter():
            ops.batch_rows_scatter(self.Zb, U, self.pu, self.pi, p.ZS)
            ops.score_pairs(p.ZS, U, self.pu, self.pi, self.sc)
            ops.bce_logits_loss(self.sc, -b, self.loss, self.dsc)
            G = p.G[0]
            zero_own(G)
            # one column of b pairs at a time, accumulating (negsampling.NegSamplingTrainer._step_body); rows of other owners are
            # written and never read
            for j in range(self.K + 1):
                sl = slice(j * b, (j + 1) * b)
                ops.score_pairs_bwd(p.ZS, U, self.pu[sl], self.pi[sl], self.dsc[sl], G, accumulate=j > 0)
            ops.memset_zero(self.flat_small)        # attention-parameter gradients are accumulated by every dense backward
        return [("c", "all-reduce batch rows", "ar", [self.Zb], "world"),
                ("k", "scores+loss+scatter", loss_and_scatter)]

    def launches_per_step(self, droprate):
        S = len(self.stages)
        fwd = (1 if droprate > 0 else 0) + S * (2 + 1 + 1) + 1            # masks, per stage transform x2 + aggregate + finalize, gather
        loss = 2 + 1 + 2 + (self.K + 1) + 1                                # rows scatter + scores, BCE, zero G x2, scatter per column, zero grads
        return 1 + fwd + loss + S * (2 + 2 + 1 + 4) + 2 + 2               # sampler, ..., backward per stage, adam(2), counters(2)

    def _layout(self):
        return "one propagation over all GPUs"
