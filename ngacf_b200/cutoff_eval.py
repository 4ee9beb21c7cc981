"""Full-ranking metrics at any cut-offs up to 100 (csrc/cutoff_metrics.cu), with the definitions published work on graph
collaborative filtering uses (NGCF, LightGCN), so that the numbers can be compared with the literature.

For an evaluated user with test items T, a ranked list L (item_pool minus the user's train items, score descending, then item id
ascending) and a cut-off k, with h = the number of the first k entries of L that are in T:
    precision@k = h / k                       recall@k = h / |T|                 hit_ratio@k = 1 if h > 0 else 0
    mrr@k       = 1 / (r + 1) for the first hit at rank r < k, else 0
    ndcg@k      = DCG / IDCG, DCG = sum over hits at rank r < k of 1 / log2(r + 2), IDCG = the same sum over ranks r < min(|T|, k)
Every value is fp64.  The evaluated users are the users with at least one train and one test item (inter.eval_users, the AllNeg
set), and the means divide by their number.  This differs from the reference-format metrics of AllNegEvaluator, which divide by the
users with train data (users without test items count as zeros) and normalise NDCG by the DCG of the sorted top-20 hit list itself
(a user with 30 test items and one hit at rank 1 scores NDCG@20 = 1); neither is the standard definition.

Where the lists come from: for max(ks) <= 20 at width 64 the tcgen05 AllNeg scorer's top-20 lists (its flagged rows re-ranked
exactly; the ids equal the exact path's for every user), otherwise ngacf_recommend_topk with K = max(ks)."""
from __future__ import annotations

import numbers

import torch

from . import _lib, ops
from .data import Interactions
from .evaluate import K as ALLNEG_K, AllNegEvaluator

MAX_K = 100
MAX_KS = 8
METRICS = ("precision", "recall", "ndcg", "hit_ratio", "mrr")
MODES = ("auto", "tc", "exact")


def check_ks(ks):
    """-> the cut-offs sorted, without duplicates; ValueError unless they are 1 .. 8 integers in 1..100"""
    ks = list(ks)
    if any(isinstance(k, bool) or not isinstance(k, numbers.Integral) for k in ks):
        raise ValueError("cut-offs must be integers, got %r" % (ks,))
    ks = sorted({int(k) for k in ks})
    if not ks or len(ks) > MAX_KS:
        raise ValueError("between 1 and %d distinct cut-offs are supported, got %d" % (MAX_KS, len(ks)))
    if ks[0] < 1 or ks[-1] > MAX_K:
        raise ValueError("cut-offs must lie in 1..%d, got %r" % (MAX_K, ks))
    return ks


def parse_ks(text: str):
    """'20,50,100' -> [20, 50, 100] (sorted, distinct); ValueError for anything else"""
    try:
        ks = [int(x) for x in str(text).split(",")]
    except ValueError:
        raise ValueError("cut-offs must be a comma-separated list of integers, got %r" % text) from None
    return check_ks(ks)


class FullRankingEvaluator:
    def __init__(self, inter: Interactions, ks, mode: str = "auto", users=None):
        """ks: cut-offs (1..8 integers in 1..100).  mode: 'auto' (the tcgen05 AllNeg lists when they are long enough and the features
        64-wide, otherwise the exact ranking lists), 'tc' (the tcgen05 lists only) or 'exact' (always the ranking lists).
        users: int32 device tensor of the users this rank evaluates (default: inter.eval_users)."""
        self.ks = check_ks(ks)
        if mode not in MODES:
            raise ValueError("mode must be one of %s, got %r" % ("/".join(MODES), mode))
        self.K = self.ks[-1]
        if mode == "tc" and self.K > ALLNEG_K:
            raise _lib.NgacfError("the tcgen05 AllNeg scorer ranks top-%d lists; cut-off %d needs mode='exact' or 'auto'" % (ALLNEG_K, self.K))
        self.inter = inter
        self.mode = mode
        self.users = inter.eval_users if users is None else users.to(torch.int32).contiguous()
        dev = inter.device
        n = self.users.numel()
        nc = len(METRICS) * len(self.ks)
        self._allneg = AllNegEvaluator(inter, mode, self.users) if mode != "exact" and self.K <= ALLNEG_K else None
        self._ids = torch.empty((max(n, 1), self.K), dtype=torch.int32, device=dev)
        self._scores = torch.empty((max(n, 1), self.K), dtype=torch.float32, device=dev)
        self._list_ws = None
        self._rows = torch.zeros((n, nc), dtype=torch.float64, device=dev)
        self._sums = torch.zeros(nc + 1, dtype=torch.float64, device=dev)      # the metric sums, then the number of users
        self._metric_ws = torch.empty(ops.cutoff_metrics_workspace_bytes(n, len(self.ks)), dtype=torch.uint8, device=dev)
        self.F = None
        self.source = None

    def rank(self, Z: torch.Tensor):
        """Z: pre-ELU last-stage output (N, 64) or (N, 128).  Ranks the lists of self.users."""
        width = Z.shape[-1]
        if self._allneg is not None and self._allneg._use_tc(width):
            self._allneg.rank(Z)
            self.source = "tc"
            return
        it = self.inter
        if self.F is None or self.F.shape != Z.shape:
            self.F = torch.empty_like(Z)
            n = self.users.numel()
            self._list_ws = torch.empty(ops.recommend_topk_workspace_bytes(width, it.I, n, self.K), dtype=torch.uint8, device=Z.device)
        ops.final_features(Z, self.F)
        ops.recommend_topk(self.F, it.U, it.I, self.users, self.K, it.train_ptr, it.train_items, it.in_pool, self._ids, self._scores,
                           self._list_ws)
        self.source = "list"

    @property
    def top_ids(self):
        """(n_users, L) int32 lists of the last rank(), -1 padded: L = 20 from the tcgen05 source, max(ks) otherwise"""
        if self.source is None:
            raise RuntimeError("FullRankingEvaluator: call rank(Z) first")
        return self._allneg.top_ids if self.source == "tc" else self._ids

    def _compute(self):
        top = self.top_ids
        n = self.users.numel()
        ops.cutoff_metrics(top, self.users, self.inter, self.ks, self._sums[:-1], self._rows if n else None, self._metric_ws)
        self._sums[-1] = float(n)

    def per_user(self):
        """(n_users, 5 * len(ks)) float64: row j is self.users[j]'s values, metric-major ([precision at each cut-off | recall | ndcg |
        hit_ratio | mrr]); this rank's users only"""
        self._compute()
        return self._rows

    def metrics(self):
        """{"ks": [...], "precision", "recall", "ndcg", "hit_ratio", "mrr": float64 arrays of len(ks), "n_users": int}: means over the
        evaluated users of every rank (sums and user counts all-reduced when sharded; every rank returns the same dict)"""
        from .dist import allreduce_sums
        self._compute()
        allreduce_sums(self._sums)
        s = self._sums.cpu().numpy()
        n = int(round(s[-1]))
        means = s[:-1] / max(n, 1)
        nk = len(self.ks)
        out = {"ks": list(self.ks)}
        for q, name in enumerate(METRICS):
            out[name] = means[q * nk:(q + 1) * nk].copy()
        out["n_users"] = n
        return out

    def __call__(self, Z):
        self.rank(Z)
        return self.metrics()
