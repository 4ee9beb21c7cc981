"""PairSampling training epoch and AllNeg evaluation with the reference's call signatures
(train_eval_Gowalla.py:90 `train_bpr`, :274 `eval_neg_all` of cleverer123/NGACF), on the B200 path.

Both accept either the reference's pandas structures (train_df rows + train_pos_neg with python sets,
data/loadGowalla.py:63-92) or an ``ngacf_b200.data.Interactions`` object in their place; the sets are
converted once into CSR arrays in HBM and never consulted again.
"""
from __future__ import annotations

import os
import time

import numpy as np
import torch

from ngacf_b200 import ops
from ngacf_b200.data import Interactions
from ngacf_b200.evaluate import AllNegEvaluator

_INTER_CACHE = {}          # key -> (source objects, Interactions); the sources are kept alive so an id() can never be recycled
_INTER_CACHE_MAX = 8


def _cached_interactions(key, sources, build):
    """id()-keyed cache that (a) holds the source objects, so a garbage-collected frame cannot hand its id to a new one,
    (b) re-checks identity on every hit and (c) is bounded (oldest entry evicted; its device arrays are freed with it)."""
    hit = _INTER_CACHE.get(key)
    if hit is not None and all(a is b for a, b in zip(hit[0], sources)):
        return hit[1]
    while len(_INTER_CACHE) >= _INTER_CACHE_MAX:
        _INTER_CACHE.pop(next(iter(_INTER_CACHE)))
    inter = build()
    _INTER_CACHE[key] = (tuple(sources), inter)
    return inter


def _unwrap(model):
    return model.module if hasattr(model, "module") else model


def _interactions(model, train_df, pos_neg, test_df=None):
    """Interactions for the reference's pandas structures -- converted once per object identity."""
    for cand in (train_df, pos_neg, test_df):
        if isinstance(cand, Interactions):
            return cand
    m = _unwrap(model)
    return _cached_interactions((id(train_df), id(pos_neg), id(test_df)), (train_df, pos_neg, test_df),
                                lambda: Interactions.from_reference_frames(m.userNum, m.itemNum, train_df, pos_neg, test_df,
                                                                           device=m.uEmbd.weight.device))


def _device_adj(model, adj):
    m = _unwrap(model)
    cached = getattr(m, "_adj_cache", None)
    if cached is not None and cached[0] is adj:
        return cached[1]
    dev = m.uEmbd.weight.device
    t = torch.as_tensor(adj, dtype=torch.int64).to(dev)        # torch.LongTensor(adj).cuda(), train_eval_Gowalla.py:106
    m._adj_cache = (adj, t)
    return t


def _plain_gat_model(m):
    """True for the models whose final features ARE the SpUIGAT propagation (what the captured steps and the evaluators use)."""
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    return type(m) in (SPUIGACF, SPUIMultiGACF)


def _require_plain(m, what):
    if not _plain_gat_model(m):
        raise NotImplementedError("%s ranks on the 64-wide SpUIGAT features of SPUIGACF / SPUIMultiGACF; %s scores through "
                                  "model(userIdx, itemIdx, adj) only" % (what, type(m).__name__))


def _fused_ok(m, optim, lossfn, loss_type=None):
    from ngacf_b200.loss import BPRLoss
    from ngacf_b200.optim import FusedAdam
    loss_type = BPRLoss if loss_type is None else loss_type
    # exact types: a subclass with more layers behind the propagation (SPUIGAGPCF) must not be trained as its base class
    if not _plain_gat_model(m) or not isinstance(lossfn, loss_type) or len(optim.param_groups) != 1:
        return False
    if loss_type is torch.nn.BCEWithLogitsLoss and (lossfn.reduction != "mean" or lossfn.weight is not None or lossfn.pos_weight is not None):
        return False
    if not isinstance(optim, (torch.optim.Adam, FusedAdam)) or isinstance(optim, torch.optim.AdamW):
        return False
    g = optim.param_groups[0]
    if g.get("amsgrad") or g.get("maximize") or g.get("decoupled_weight_decay"):
        return False
    return {id(p) for p in g["params"]} == {id(p) for p in m.parameters()}


def train_bpr(model, batch_size, train_df, train_pos_neg, adj, optim, lossfn, is_parallel, epoch=0, sample_seed=None, fused=None,
              max_steps=None):
    """One epoch over train_df in file order (train_eval_Gowalla.py:108-115): per batch, one (u,pos,neg)
    triple per train row from the GPU sampler, two full propagations with independent dropout, BPR,
    backward, optimizer step.  Returns sum(batch-mean loss) / len(train_df) like the reference (:139,144).
    `epoch`/`sample_seed` select the sampler's Philox stream (the reference's sampler is unseeded)."""
    m = _unwrap(model)
    model.train()
    inter = _interactions(model, train_df, train_pos_neg)
    dev = m.uEmbd.weight.device
    if sample_seed is None:
        sample_seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
    if is_parallel and _world() > 1:
        return _train_bpr_parallel(m, batch_size, inter, adj, optim, lossfn, epoch, sample_seed, max_steps)
    # --parallel True in a single process: the reference scatters over torch.cuda.device_count() GPUs in one process
    # (parallel.py); here the multi-GPU modes are one process per GPU (torchrun), so a lone process is the one-GPU step
    adj_t = _device_adj(model, adj)
    graph = m.graph_for(adj_t)
    if fused is None:
        fused = os.environ.get("NGACF_FUSED", "1") != "0"
    if fused and _fused_ok(m, optim, lossfn):
        # whole step on the GPU (sampler .. Adam), CUDA-graph replayed; same maths as the generic loop below
        from ngacf_b200.train import FusedTrainer
        tr = getattr(m, "_trainer", None)
        key = (id(inter), id(graph), int(batch_size), id(optim), int(sample_seed))
        if tr is None or tr.key != key:
            tr = FusedTrainer(m, inter, graph, batch_size, optim, sample_seed,
                              split_dense_backward=os.environ.get("NGACF_SPLIT_DENSE_BWD", "0") == "1")
            tr.key = key
            m._trainer = tr
        return tr.train_epoch(epoch, max_steps)
    n = len(inter)
    n_batches = n // batch_size + 1
    if max_steps is not None:
        n_batches = min(n_batches, max_steps)
    users = torch.empty(batch_size, dtype=torch.int64, device=dev)
    pos = torch.empty_like(users)
    neg = torch.empty_like(users)
    total = torch.zeros((), dtype=torch.float64, device=dev)
    for batch_id in range(n_batches):
        lo, hi = batch_id * batch_size, min(n, (batch_id + 1) * batch_size)
        if hi <= lo:
            continue        # len(train_df) % batch_size == 0: the reference's empty batch yields a NaN mean; skipped
        b = hi - lo
        ops.sample_pairs(inter, lo, hi, sample_seed, epoch, users, pos, neg)
        optim.zero_grad()
        pos_scores = model(users[:b], pos[:b], graph)
        neg_scores = model(users[:b], neg[:b], graph)
        loss = lossfn(pos_scores, neg_scores)
        loss.backward()
        optim.step()
        total += loss.detach().double()
        if batch_id % 60 == 0:
            print("-----------The timeStamp of training batch {:03d}/{}".format(batch_id, n_batches) + " is: "
                  + time.strftime("%H: %M: %S", time.gmtime(time.time())))
    return float(total.item()) / n


def _world():
    import torch.distributed as dist
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def _train_bpr_parallel(m, batch_size, inter, adj, optim, lossfn, epoch, sample_seed, max_steps):
    """--parallel True under torchrun (one process per GPU).  NGACF_PARALLEL_MODE:
      shard   (default) users range-partitioned, item rows all-gathered / reduce-scattered per stage (ngacf_b200.dist.ShardedTrainer):
              the SAME step as one GPU on the same batch, split over the GPUs (the tail batch of len % batch rows is dropped);
      replica the reference's own --parallel semantics (parallel.py, train_eval_Gowalla.py:97-104,137): every GPU propagates the
              whole graph and scores its own batch_size rows, gradients are summed (ngacf_b200.dist.ReplicaTrainer)."""
    from ngacf_b200.dist import ReplicaTrainer, ShardedTrainer
    if not _fused_ok(m, optim, lossfn):
        raise NotImplementedError("--parallel True needs the fused step: SPUIGACF + BPRLoss + a single-group Adam over model.parameters()")
    mode = os.environ.get("NGACF_PARALLEL_MODE", "shard")
    tr = getattr(m, "_parallel_trainer", None)
    key = (mode, id(inter), id(adj), int(batch_size), id(optim), int(sample_seed))
    if tr is None or tr.key != key:
        if mode == "replica":
            tr = ReplicaTrainer(m, inter, m.graph_for(_device_adj(m, adj)), batch_size, optim, sample_seed)
        else:
            idx = np.asarray(adj.cpu() if torch.is_tensor(adj) else adj).reshape(2, -1)
            tr = ShardedTrainer(m, inter, idx[0], idx[1], batch_size, optim, sample_seed)
        tr.key = key
        m._parallel_trainer = tr
    return tr.train_epoch(epoch, max_steps)


def eval_neg_all(model, batch_size, test_df, test_pos_neg, adj, itemNum, is_parallel, mode="auto"):
    """Full-ranking evaluation: every test user against every candidate item (item_pool minus the user's
    train items), top-20, precision/recall/ndcg/hit_ratio @ [1,5,10,20] averaged with the reference's
    divisor (train_eval_Gowalla.py:283).  Returns the reference's result dict (:277-278,354)."""
    m = _unwrap(model)
    model.eval()
    _require_plain(m, "eval_neg_all")
    inter = _interactions(model, None, test_pos_neg, test_df)
    adj_t = _device_adj(model, adj)
    with torch.no_grad():
        Z = m.propagate(adj_t)
        ev = getattr(m, "_evaluator", None)
        world = _world() if is_parallel else 1
        if ev is None or ev.inter is not inter or ev.mode != mode or getattr(ev, "world", 1) != world:
            users = None
            if world > 1:       # users sharded over the ranks; only the 16 metric sums are merged (AllNegEvaluator.metrics)
                import torch.distributed as dist
                from ngacf_b200.dist import shard_eval_users
                users = shard_eval_users(inter.eval_users, dist.get_rank(), world)
            ev = AllNegEvaluator(inter, mode, users=users)
            ev.world = world
            m._evaluator = ev
        return ev(Z)


def eval_full_ranking(model, test_df, test_pos_neg, adj, ks, is_parallel, mode="auto", novelty_weight=0.0, mmr_lambda=None):
    """Full-ranking metrics at the cut-offs `ks` (up to 8 of 1..100) with the standard definitions: precision, recall, NDCG with the
    ideal DCG of min(|test|, k) hits, hit ratio and MRR, averaged over the users with train and test items
    (ngacf_b200.cutoff_eval).  Returns FullRankingEvaluator.metrics()'s dict.  is_parallel under torchrun: the users are sharded over
    the ranks and the sums merged, as in eval_neg_all.  novelty_weight w != 0: the metrics of the novelty-weighted lists
    (FullRankingEvaluator(novelty_weight=w)), from an evaluator cached per weight next to the plain one.  mmr_lambda lam: the metrics
    of the MMR-diversified lists (FullRankingEvaluator(mmr_lambda=lam)), from an evaluator cached per (weight, lam)."""
    from ngacf_b200.cutoff_eval import FullRankingEvaluator, check_ks, check_mmr_lambda, check_novelty_weight
    m = _unwrap(model)
    model.eval()
    _require_plain(m, "eval_full_ranking")
    ks = check_ks(ks)
    w = check_novelty_weight(novelty_weight)
    lam = None if mmr_lambda is None else check_mmr_lambda(mmr_lambda)
    inter = _interactions(model, None, test_pos_neg, test_df)
    adj_t = _device_adj(model, adj)
    with torch.no_grad():
        Z = m.propagate(adj_t)
        ev = _full_evaluator(m, w, lam)
        world = _world() if is_parallel else 1
        if ev is None or ev.inter is not inter or ev.mode != mode or ev.ks != ks or getattr(ev, "world", 1) != world:
            users = None
            if world > 1:
                import torch.distributed as dist
                from ngacf_b200.dist import shard_eval_users
                users = shard_eval_users(inter.eval_users, dist.get_rank(), world)
            ev = FullRankingEvaluator(inter, ks, mode, users=users, novelty_weight=w, mmr_lambda=lam)
            ev.world = world
            if lam is not None:
                m.__dict__.setdefault("_mmr_evaluators", {})[(w, lam)] = ev
            elif w == 0.0:
                m._full_evaluator = ev
            else:
                m.__dict__.setdefault("_novelty_evaluators", {})[w] = ev
        return ev(Z)


def _full_evaluator(m, w, lam=None):
    """the evaluator eval_full_ranking cached for novelty weight w (0: the plain one) and MMR lambda lam (None: no re-ranking), or
    None"""
    if lam is not None:
        return m.__dict__.get("_mmr_evaluators", {}).get((w, lam))
    if w == 0.0:
        return getattr(m, "_full_evaluator", None)
    return m.__dict__.get("_novelty_evaluators", {}).get(w)


def _cached_evaluator(model, novelty_weight, mmr_lambda, what):
    from ngacf_b200.cutoff_eval import check_mmr_lambda, check_novelty_weight
    lam = None if mmr_lambda is None else check_mmr_lambda(mmr_lambda)
    ev = _full_evaluator(_unwrap(model), check_novelty_weight(novelty_weight), lam)
    if ev is None or ev.source is None:
        raise RuntimeError("%s: call eval_full_ranking first (with the same novelty_weight and mmr_lambda); it ranks the lists these "
                           "reports read" % what)
    return ev


def diversity_report(model, novelty_weight=0.0, mmr_lambda=None):
    """The intra-list diversity (FullRankingEvaluator.diversity_metrics()) of the lists the preceding eval_full_ranking call with the
    same novelty_weight and mmr_lambda ranked, from the evaluator it cached: no second propagation or ranking.  Under torchrun every
    rank calls it (the sums are all-reduced)."""
    return _cached_evaluator(model, novelty_weight, mmr_lambda, "diversity_report").diversity_metrics()


def list_reports(model, beyond=True, groups=None, novelty_weight=0.0, mmr_lambda=None):
    """The beyond-accuracy metrics (coverage, Gini of the item exposure, novelty, ARP) and the metrics per user-activity group
    (NGCF section 4.3.2) of the lists the preceding eval_full_ranking call ranked, from the evaluator it cached: no second
    propagation or ranking.  Returns {"beyond": FullRankingEvaluator.list_metrics() or None, "groups":
    FullRankingEvaluator.group_metrics(groups) or None}.  novelty_weight: read the lists of the eval_full_ranking call with that
    weight (and mmr_lambda: of the MMR-diversified lists).  Under torchrun every rank calls it (the counts and sums are
    all-reduced)."""
    ev = _cached_evaluator(model, novelty_weight, mmr_lambda, "list_reports")
    return {"beyond": ev.list_metrics() if beyond else None, "groups": ev.group_metrics(groups) if groups else None}


# ------------------------------------------------------------------------------------------------
# NegSampling training / SampledNeg evaluation (the reference CLI's default modes, SURVEY 8f-3)
# ------------------------------------------------------------------------------------------------
def _neg_interactions(model, pos_neg, train_df=None, test_df=None):
    for cand in (train_df, pos_neg, test_df):
        if isinstance(cand, Interactions):
            return cand
    m = _unwrap(model)
    return _cached_interactions(("neg", id(pos_neg), id(train_df), id(test_df)), (pos_neg, train_df, test_df),
                                lambda: Interactions.from_negsampling_frames(m.userNum, m.itemNum, pos_neg, train_df, test_df,
                                                                             device=m.uEmbd.weight.device))


def train_neg_sample(model, batch_size, train_df, train_pos_neg, adj, optim, lossfn, is_parallel, epoch=0, sample_seed=None, fused=None,
                     max_steps=None):
    """One epoch of train_neg_sample (train_eval_Gowalla.py:36-88): per train row 1 positive + 4 sampled negatives, ONE propagation per
    batch, BCEWithLogitsLoss on the B*5 scores, backward, optimizer step.  Returns sum(batch-mean loss) / len(train_df) (:84,88).
    train_pos_neg = positives_negtives(rt) (or an ngacf_b200.data.Interactions); `epoch`/`sample_seed` select the sampler's stream."""
    m = _unwrap(model)
    model.train()
    inter = _neg_interactions(model, train_pos_neg, train_df=train_df)
    dev = m.uEmbd.weight.device
    if sample_seed is None:
        sample_seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
    if is_parallel and _world() > 1:
        return _train_neg_parallel(m, batch_size, inter, adj, optim, lossfn, epoch, sample_seed, max_steps)
    # a lone --parallel True process runs the one-GPU step (see train_bpr)
    graph = m.graph_for(_device_adj(model, adj))
    if fused is None:
        fused = os.environ.get("NGACF_FUSED", "1") != "0"
    K = 4
    if fused and _fused_ok(m, optim, lossfn, loss_type=torch.nn.BCEWithLogitsLoss):
        from ngacf_b200.negsampling import NegSamplingTrainer
        tr = getattr(m, "_neg_trainer", None)
        key = (id(inter), id(graph), int(batch_size), id(optim), int(sample_seed))
        if tr is None or tr.key != key:
            tr = NegSamplingTrainer(m, inter, graph, batch_size, optim, sample_seed, K=K)
            tr.key = key
            m._neg_trainer = tr
        return tr.train_epoch(epoch, max_steps)
    n = len(inter)
    n_batches = n // batch_size + 1
    if max_steps is not None:
        n_batches = min(n_batches, max_steps)
    pu = torch.empty(batch_size * (K + 1), dtype=torch.int64, device=dev)
    pi = torch.empty_like(pu)
    labels = torch.zeros(batch_size, K + 1, device=dev)
    labels[:, 0] = 1
    total = torch.zeros((), dtype=torch.float64, device=dev)
    for batch_id in range(n_batches):
        lo, hi = batch_id * batch_size, min(n, (batch_id + 1) * batch_size)
        if hi <= lo:
            continue
        nb = (hi - lo) * (K + 1)
        ops.sample_negs(inter, inter.train_rows_user, inter.train_rows_item, lo, hi, sample_seed, epoch, K, ops.NEG_TAG_TRAIN, pu, pi)
        optim.zero_grad()
        predictions = model(pu[:nb], pi[:nb], graph)
        loss = lossfn(predictions, labels[:hi - lo].reshape(-1))
        loss.backward()
        optim.step()
        total += loss.detach().double()
    return float(total.item()) / n


def _train_neg_parallel(m, batch_size, inter, adj, optim, lossfn, epoch, sample_seed, max_steps):
    """--parallel True under torchrun for NegSampling, NGACF_PARALLEL_MODE as in _train_bpr_parallel:
      shard   (default) the one propagation user-range partitioned over all GPUs (ngacf_b200.dist.ShardedNegSamplingTrainer): the SAME
              step as one GPU on the same batch, split over the GPUs (the tail batch of len % batch rows is dropped);
      replica the reference's semantics: every GPU propagates the whole graph and scores the 1 + 4 items of its own batch_size rows,
              gradients are summed (ngacf_b200.dist.NegSamplingReplicaTrainer)."""
    from ngacf_b200.dist import NegSamplingReplicaTrainer, ShardedNegSamplingTrainer
    if not _fused_ok(m, optim, lossfn, loss_type=torch.nn.BCEWithLogitsLoss):
        raise NotImplementedError("--parallel True needs the fused step: SPUIGACF + BCEWithLogitsLoss (mean) + a single-group Adam over "
                                  "model.parameters()")
    mode = os.environ.get("NGACF_PARALLEL_MODE", "shard")
    tr = getattr(m, "_neg_parallel_trainer", None)
    key = (mode, id(inter), id(adj), int(batch_size), id(optim), int(sample_seed))
    if tr is None or tr.key != key:
        if mode == "replica":
            tr = NegSamplingReplicaTrainer(m, inter, m.graph_for(_device_adj(m, adj)), batch_size, optim, sample_seed)
        else:
            idx = np.asarray(adj.cpu() if torch.is_tensor(adj) else adj).reshape(2, -1)
            tr = ShardedNegSamplingTrainer(m, inter, idx[0], idx[1], batch_size, optim, sample_seed)
        tr.key = key
        m._neg_parallel_trainer = tr
    return tr.train_epoch(epoch, max_steps)


def eval_neg_sample(model, batch_size, test_df, test_pos_neg, adj, top_k, is_parallel, seed=0):
    """eval_neg_sample (train_eval_Gowalla.py:193-257): per test row 1 positive + 99 sampled negatives, HR@top_k and NDCG@top_k
    averaged over the test rows.  All rows are scored against one propagation.  Returns (HR, NDCG).
    is_parallel under torchrun: every rank evaluates its shard of the test rows, the two metric sums are merged, and every rank
    returns the same (HR, NDCG)."""
    m = _unwrap(model)
    model.eval()
    _require_plain(m, "eval_neg_sample")
    inter = _neg_interactions(model, test_pos_neg, test_df=test_df)
    adj_t = _device_adj(model, adj)
    from ngacf_b200.negsampling import SampledNegEvaluator
    world = _world() if is_parallel else 1
    rows = None
    if world > 1:
        import torch.distributed as dist
        from ngacf_b200.dist import shard_range
        rows = shard_range(inter.n_test_rows, dist.get_rank(), world)
    with torch.no_grad():
        Z = m.propagate(adj_t)
        ev = getattr(m, "_neg_evaluator", None)
        if ev is None or ev.inter is not inter or ev.top_k != int(top_k) or ev.seed != int(seed) or ev.rows != (rows or (0, inter.n_test_rows)):
            ev = SampledNegEvaluator(inter, top_k, 99, seed, rows=rows)
            m._neg_evaluator = ev
        if world == 1:
            return ev(Z)
        from ngacf_b200.dist import allreduce_sums
        sums = allreduce_sums(ev.metric_sums(Z))
        hr, nd = (sums / max(inter.n_test_rows, 1)).tolist()
        return hr, nd
