"""NegSampling training and SampledNeg evaluation (SURVEY 8f-3) -- the reference CLI's default modes
(run_Gowalla.py:179-180; train_neg_sample / eval_neg_sample, train_eval_Gowalla.py:36-88,193-270):

  train step : per train row (user, item): 1 positive + K=4 sampled negatives -> ONE propagation -> B*(K+1) pair scores ->
               BCE-with-logits against [1,0,0,0,0] -> backward -> Adam
  evaluation : per test row: 1 positive + 99 sampled negatives -> scores on one propagation -> HR@k / NDCG@k of the positive

Everything but the sampler, the loss and the rank metric (csrc/neg_sampling.cu) is the PairSampling machinery: the step is
captured in one CUDA graph with device-resident row / epoch / dropout counters (train.FusedTrainer)."""
from __future__ import annotations

import torch

from . import ops
from .data import Interactions
from .graph import BipartiteGraph
from .train import FusedTrainer


class NegSamplingTrainer(FusedTrainer):
    CALLS_PER_STEP = 1          # one propagation, one dropout call index per step

    def __init__(self, model, inter: Interactions, graph: BipartiteGraph, batch_size: int, optim, sample_seed: int, K: int = 4,
                 use_cuda_graph: bool = True):
        super().__init__(model, inter, graph, batch_size, optim, sample_seed, use_cuda_graph=use_cuda_graph, two_streams=False)
        self.K = int(K)
        if inter.min_negatives() < self.K:      # random.sample(negative_items, K) raises in the reference (loadGowalla.py:82)
            raise ValueError("a user has fewer than K=%d negatives (item pool minus the user's positives)" % self.K)
        n = self.B * (self.K + 1)
        i64, f32 = dict(dtype=torch.int64, device=self.dev), dict(dtype=torch.float32, device=self.dev)
        self.pu, self.pi = torch.zeros(n, **i64), torch.zeros(n, **i64)
        self.sc, self.dsc = torch.zeros(n, **f32), torch.zeros(n, **f32)

    # one step: sampler -> masks -> propagation -> scores -> BCE -> scatter -> backward -> Adam
    def _step_body(self, b: int, epoch: int, droprate: float, seed: int, row0: int, call0: int, dev_counters: bool, part: str = "all"):
        m, g, it = self.model, self.g, self.inter
        uE, iE = m.uEmbd.weight.detach(), m.iEmbd.weight.detach()
        rd = self.row_dev if dev_counters else None
        cd = self.call_dev if dev_counters else None
        row0 = row0 + (self._row_offset() if dev_counters else 0)
        n = b * (self.K + 1)
        # column-major pairs: column j (0 = positives, 1..K = negatives) is the contiguous slice [j*b, (j+1)*b)
        ops.sample_negs(it, it.train_rows_user, it.train_rows_item, row0, row0 + b, self.sample_seed, 0 if dev_counters else epoch, self.K,
                        ops.NEG_TAG_TRAIN, self.pu, self.pi, rd, col_stride=b)
        premask = dev_counters and self.prefetch_masks
        self._mask_args = (droprate, seed) if premask else None
        prop = self.props[0]
        if premask:
            prop.use_dropout_buffers(droprate)
        else:
            prop.set_dropout(droprate, seed, call0, None, cd)
        Z = prop.forward(uE, iE, self.wtabs)
        ops.score_pairs(Z, g.U, self.pu[:n], self.pi[:n], self.sc[:n])
        ops.bce_logits_loss(self.sc[:n], -b, self.loss, self.dsc[:n])
        G = prop.grad_in()
        G.zero_()
        # the scatter's cost grows with the square of the pairs per call: one column of b pairs at a time, accumulating
        for j in range(self.K + 1):
            sl = slice(j * b, (j + 1) * b)
            ops.score_pairs_bwd(prop.Z[-1], g.U, self.pu[sl], self.pi[sl], self.dsc[sl], G, accumulate=j > 0)
        inline = (lambda k, fn: fn()) if self.split_dense_backward else None
        prop.backward(G, uE, iE, self.wtabs, self.gtabs, m.uEmbd.weight.grad, m.iEmbd.weight.grad, False, dw_launcher=inline)
        if part == "compute":
            return
        self._reduce_grads()
        self._step_update(dev_counters)

    def _generate_masks(self, droprate, seed):
        self.props[0].set_dropout(droprate, seed, 0, None, self.call_dev)

    def launches_per_step(self, droprate: float) -> int:
        S = len(self.props[0].stages)
        fwd = (1 if droprate > 0 else 0) + 2 * S + 1                  # masks, transform+aggregate per stage, pair scores
        bwd = (self.K + 1) + S * (1 + 2 + (4 if self.split_dense_backward else 2))   # scatter per column; prep + 2 edge passes + dense backward per stage
        return 1 + fwd + 1 + bwd + 2 + 2                               # sampler, ..., loss, ..., adam(2), counters(2)

    def units_per_step(self) -> int:
        return self.g.E             # propagated edges: ONE full-graph propagation per step

    def parallelism(self) -> str:
        return "single GPU"


class SampledNegEvaluator:
    """eval_neg_sample (train_eval_Gowalla.py:193-257): HR@top_k / NDCG@top_k over 1 positive + K sampled negatives per test row,
    all rows scored against ONE propagation (the reference re-propagates for every batch of batch_size//8 rows).

    rows = (lo, hi) evaluates the test rows [lo, hi) only (one rank's shard): the sampler is keyed by the test row, so a shard draws
    exactly the negatives of the whole evaluation, and the metric sums of the shards add up to those of the whole."""

    def __init__(self, inter: Interactions, top_k: int = 10, K: int = 99, seed: int = 0, rows=None):
        self.inter, self.top_k, self.K, self.seed = inter, int(top_k), int(K), int(seed)
        if inter.n_test_rows and inter.min_negatives() < self.K:      # loadGowalla.py:103
            raise ValueError("a user has fewer than K=%d negatives (item pool minus the user's positives)" % self.K)
        self.rows = (0, inter.n_test_rows) if rows is None else (int(rows[0]), int(rows[1]))
        if not 0 <= self.rows[0] <= self.rows[1] <= inter.n_test_rows:
            raise ValueError("test rows [%d, %d) outside [0, %d)" % (self.rows + (inter.n_test_rows,)))
        n = (self.rows[1] - self.rows[0]) * (self.K + 1)
        dev = inter.device
        self.pu = torch.zeros(n, dtype=torch.int64, device=dev)
        self.pi = torch.zeros(n, dtype=torch.int64, device=dev)
        self.sc = torch.zeros(n, dtype=torch.float32, device=dev)
        self.sums = torch.zeros(2, dtype=torch.float64, device=dev)

    def metric_sums(self, Z: torch.Tensor) -> torch.Tensor:
        """float64[2] on the device: the sums of HR@top_k and NDCG@top_k over the evaluated rows"""
        it = self.inter
        lo, hi = self.rows
        self.sums.zero_()
        if hi > lo:
            ops.sample_negs(it, it.test_rows_user, it.test_rows_item, lo, hi, self.seed, 0, self.K, ops.NEG_TAG_EVAL, self.pu, self.pi)
            ops.score_pairs(Z, it.U, self.pu, self.pi, self.sc)
            ops.rank_metrics(self.sc, self.K + 1, self.top_k, self.sums)
        return self.sums

    def __call__(self, Z: torch.Tensor):
        """Z: pre-ELU output of the last stage (model.propagate in eval mode).  Returns (HR, NDCG) as python floats, averaged over
        all test rows (a shard's sums divided by the total count: add the shards' results to get the whole)."""
        rows = self.inter.n_test_rows
        if rows == 0:
            return 0.0, 0.0
        hr, nd = (self.metric_sums(Z) / rows).tolist()
        return hr, nd
