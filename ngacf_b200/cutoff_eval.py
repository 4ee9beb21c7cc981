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
exactly; the ids equal the exact path's for every user), otherwise ngacf_recommend_topk with K = max(ks).

Beyond-accuracy metrics of the same lists (list_metrics(), csrc/list_stats.cu).  An entry of a list is valid when its id lies in
[0, I) (-1 pads).  Item statistics come from the train split only: d_i = the number of distinct users with item i among their train
items, n_tr = inter.n_train_users.
    exposure c_k(i) = the number of evaluated users whose first k entries contain item i (integers, all-reduced when sharded)
    coverage@k      = |{i in pool : c_k(i) > 0}| / |pool|                          (pool = inter.pool)
    gini@k          = sum_j (2 j - n - 1) c_(j) / (n sum c) over the pool items' c_k sorted ascending as c_(1..n), n = |pool|
                      (0 when sum c = 0); numerator and denominator exact in int64, one fp64 division
    novelty@k       = per user, the mean over the valid entries among the first k of nov(i) = -log2((d_i + 1) / (n_tr + 1))
    arp@k           = per user, the mean of d_i over the same entries (average recommended popularity)
The per-user sums run in rank order in fp64 and are divided once by the number of valid entries (0 when there is none); novelty and
arp are then averaged over the evaluated users with the divisor of metrics().  nov and d are fp64 item tables built once per
Interactions on the host.

User-activity groups (group_metrics(G), the interaction sparsity levels of NGCF section 4.3.2): every user of inter.eval_users,
sorted by (train degree, user id) ascending; with C_j the train degree summed over the users before user j and T the total, user j
is in group min(G - 1, floor(G C_j / T)) (int64), G in 1..8.  The groups therefore hold about T / G train interactions each; one
user with a very large degree can leave a group empty.  Per group: the number of evaluated users, their min / max train degree, their
train interactions and the means over the group's users of the five metrics above and of novelty / arp at each cut-off.

Novelty-weighted lists (novelty_weight=w, any finite float): the lists rank by s(u, i) + off(i) with off(i) = float32(w * nov(i))
(the fp64 product rounded once), the sum rounded to fp32 (ngacf_recommend_topk_offset).  Up to terms equal for every item this is
s(u, i) - w log2(d_i + 1): a positive w moves popular items down, in the units of novelty@k.  The lists always come from the exact
ranking (the tcgen05 scorer has no offsets), and every report above reads them unchanged.

Intra-list diversity (diversity_metrics(), csrc/diversity.cu) of the same lists, with sim(x, y) the cosine of the items' final
features as the similar-item lists compute it (x the entry of lower rank) and v_1..v_m the valid entries among the first k:
    ild@k = sum over b = 2..m of (sum over a < b of (1 - sim(v_a, v_b))) / (m (m - 1) / 2), 0 when m < 2
summed in fp64, a ascending inside b ascending, one division; averaged over the evaluated users with the divisor of metrics().

MMR-diversified lists (mmr_lambda=lam in [0, 1]): rank() first ranks N = mmr_candidates candidates exactly (with the novelty offsets
when novelty_weight is set), then picks K = max(ks) of them greedily by lam * rel(c) - (1 - lam) * max similarity to the picks so
far, rel being the candidate score min-max normalised over the row (ngacf_mmr_rerank).  lam = 1 gives the exact lists; every report
above reads the re-ranked lists unchanged."""
from __future__ import annotations

import math
import numbers

import numpy as np
import torch

from . import _lib, ops
from .data import Interactions
from .evaluate import K as ALLNEG_K, AllNegEvaluator

MAX_K = 100
MAX_KS = 8
METRICS = ("precision", "recall", "ndcg", "hit_ratio", "mrr")
LIST_VALUES = ("novelty", "arp")
MAX_GROUPS = 8
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


def check_groups(G):
    """-> G as an int; ValueError unless it is an integer in 1..8"""
    if isinstance(G, bool) or not isinstance(G, numbers.Integral) or not 1 <= int(G) <= MAX_GROUPS:
        raise ValueError("the number of user groups must be an integer in 1..%d, got %r" % (MAX_GROUPS, G))
    return int(G)


def item_degrees(inter: Interactions):
    """d_i: the number of distinct users with item i among their train items, int64[I] (host)"""
    return np.bincount(inter.host["train_items"], minlength=inter.I).astype(np.int64)


def item_tables(inter: Interactions):
    """float64 (2, I) device tables [nov | d] with nov(i) = -log2((d_i + 1) / (n_tr + 1)); built once per Interactions"""
    t = inter.__dict__.get("_list_item_tables")
    if t is None:
        d = item_degrees(inter).astype(np.float64)
        nov = -np.log2((d + 1.0) / (inter.n_train_users + 1.0))
        t = torch.from_numpy(np.stack([nov, d])).to(inter.device)
        inter._list_item_tables = t
    return t


def check_novelty_weight(w):
    """-> w as a float; ValueError unless it is a finite real number"""
    if isinstance(w, bool) or not isinstance(w, numbers.Real) or not math.isfinite(float(w)):
        raise ValueError("the novelty weight must be a finite number, got %r" % (w,))
    return float(w)


def novelty_offsets(inter: Interactions, w):
    """float32[I] device offsets off(i) = float32(w * nov(i)) of the novelty-weighted lists (fp64 product, rounded once); built once
    per Interactions and weight"""
    w = check_novelty_weight(w)
    cache = inter.__dict__.setdefault("_novelty_offsets", {})
    off = cache.get(w)
    if off is None:
        off = (w * item_tables(inter)[0]).to(torch.float32).contiguous()
        cache[w] = off
    return off


def check_mmr_lambda(lam):
    """-> lam as a float; ValueError unless it is a real number in [0, 1]"""
    if isinstance(lam, bool) or not isinstance(lam, numbers.Real) or not 0.0 <= float(lam) <= 1.0:
        raise ValueError("the MMR lambda must be a number in [0, 1], got %r" % (lam,))
    return float(lam)


def check_mmr_candidates(n, K):
    """-> n as an int; ValueError unless it is an integer in K..100"""
    if isinstance(n, bool) or not isinstance(n, numbers.Integral) or not K <= int(n) <= MAX_K:
        raise ValueError("the MMR candidates must be an integer in %d..%d (the list length .. 100), got %r" % (K, MAX_K, n))
    return int(n)


def coverage_gini(counts, pool=None):
    """counts: (n_ks, I) exposure counts, pool: item ids (None: counts holds the pool's columns already) -> (coverage, gini) float64
    arrays of n_ks (definitions above)"""
    c = np.asarray(counts) if pool is None else np.asarray(counts)[:, np.asarray(pool, np.int64)]
    n = c.shape[1]
    coverage = (c > 0).sum(1) / max(n, 1)
    w = 2 * np.arange(1, n + 1, dtype=np.int64) - n - 1
    num = np.sort(c, axis=1).astype(np.int64) @ w
    den = n * c.sum(1, dtype=np.int64)
    gini = np.where(den > 0, num / np.maximum(den, 1), 0.0)
    return coverage, gini


def split_groups(users, degrees, G):
    """users, train degrees (host arrays) -> (users, degrees, group) sorted by (degree, user id) ascending, group[j] =
    min(G - 1, floor(G C_j / T)) with C_j the degrees before j and T their total (int64)"""
    G = check_groups(G)
    users = np.asarray(users, np.int64)
    degrees = np.asarray(degrees, np.int64)
    order = np.lexsort((users, degrees))
    users, degrees = users[order], degrees[order]
    C = np.cumsum(degrees) - degrees
    T = int(degrees.sum())
    group = np.minimum(G - 1, (G * C) // max(T, 1))
    return users, degrees, group


def user_groups(inter: Interactions, G):
    """the activity groups of every user of inter.eval_users (split_groups over their train degrees)"""
    users = inter.eval_users.cpu().numpy().astype(np.int64)
    return split_groups(users, np.diff(inter.host["train_ptr"])[users], G)


class FullRankingEvaluator:
    def __init__(self, inter: Interactions, ks, mode: str = "auto", users=None, novelty_weight=0.0, mmr_lambda=None, mmr_candidates=100):
        """ks: cut-offs (1..8 integers in 1..100).  mode: 'auto' (the tcgen05 AllNeg lists when they are long enough and the features
        64-wide, otherwise the exact ranking lists), 'tc' (the tcgen05 lists only) or 'exact' (always the ranking lists).
        users: int32 device tensor of the users this rank evaluates (default: inter.eval_users).  novelty_weight: w of the
        novelty-weighted lists (module docstring); non-zero always ranks exactly at K = max(ks), so mode='tc' refuses it.
        mmr_lambda: lam of the MMR-diversified lists (module docstring), re-ranked from the exact top mmr_candidates (max(ks)..100);
        None: no re-ranking.  mode='tc' refuses it too."""
        self.ks = check_ks(ks)
        if mode not in MODES:
            raise ValueError("mode must be one of %s, got %r" % ("/".join(MODES), mode))
        self.K = self.ks[-1]
        if mode == "tc" and self.K > ALLNEG_K:
            raise _lib.NgacfError("the tcgen05 AllNeg scorer ranks top-%d lists; cut-off %d needs mode='exact' or 'auto'" % (ALLNEG_K, self.K))
        self.novelty_weight = check_novelty_weight(novelty_weight)
        if mode == "tc" and self.novelty_weight != 0.0:
            raise _lib.NgacfError("the tcgen05 AllNeg scorer has no score offsets; novelty_weight=%r needs mode='exact' or 'auto'"
                                  % self.novelty_weight)
        self.mmr_lambda = None if mmr_lambda is None else check_mmr_lambda(mmr_lambda)
        self.mmr_candidates = check_mmr_candidates(mmr_candidates, self.K)
        if mode == "tc" and self.mmr_lambda is not None:
            raise _lib.NgacfError("the tcgen05 AllNeg scorer has no MMR re-ranking; mmr_lambda=%r needs mode='exact' or 'auto'"
                                  % self.mmr_lambda)
        self.inter = inter
        self.mode = mode
        self._offset = novelty_offsets(inter, self.novelty_weight) if self.novelty_weight != 0.0 else None
        self.users = inter.eval_users if users is None else users.to(torch.int32).contiguous()
        dev = inter.device
        n = self.users.numel()
        nc = len(METRICS) * len(self.ks)
        use_tc = mode != "exact" and self.K <= ALLNEG_K and self._offset is None and self.mmr_lambda is None
        self._allneg = AllNegEvaluator(inter, mode, self.users) if use_tc else None
        self._ids = torch.empty((max(n, 1), self.K), dtype=torch.int32, device=dev)
        self._scores = torch.empty((max(n, 1), self.K), dtype=torch.float32, device=dev)
        self._list_ws = None
        if self.mmr_lambda is not None:      # the candidate lists the re-ranking reads
            self._cand_ids = torch.empty((max(n, 1), self.mmr_candidates), dtype=torch.int32, device=dev)
            self._cand_scores = torch.empty((max(n, 1), self.mmr_candidates), dtype=torch.float32, device=dev)
        self._div_rows = None
        self._rows = torch.zeros((n, nc), dtype=torch.float64, device=dev)
        self._sums = torch.zeros(nc + 1, dtype=torch.float64, device=dev)      # the metric sums, then the number of users
        self._metric_ws = torch.empty(ops.cutoff_metrics_workspace_bytes(n, len(self.ks)), dtype=torch.uint8, device=dev)
        self.F = None
        self.source = None
        self._tables = None            # list_metrics / group_metrics state, built on first use
        self._groups = {}

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
            K = self.K if self.mmr_lambda is None else self.mmr_candidates
            self._list_ws = torch.empty(ops.recommend_topk_workspace_bytes(width, it.I, n, K), dtype=torch.uint8, device=Z.device)
        ops.final_features(Z, self.F)
        if self.mmr_lambda is None:
            ops.recommend_topk(self.F, it.U, it.I, self.users, self.K, it.train_ptr, it.train_items, it.in_pool, self._ids, self._scores,
                               self._list_ws, self._offset)
            self.source = "list"
            return
        n = self.users.numel()
        ops.recommend_topk(self.F, it.U, it.I, self.users, self.mmr_candidates, it.train_ptr, it.train_items, it.in_pool,
                           self._cand_ids, self._cand_scores, self._list_ws, self._offset)
        if n:
            ops.mmr_rerank(self.F, it.U, it.I, self._cand_ids[:n], self._cand_scores[:n], self.K, self.mmr_lambda, self._ids, self._scores)
        self.source = "mmr"

    @property
    def top_ids(self):
        """(n_users, L) int32 lists of the last rank(), -1 padded: L = 20 from the tcgen05 source, max(ks) otherwise (the exact
        ranking, source "list", or its MMR re-ranking, source "mmr")"""
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

    # ---- beyond-accuracy metrics and user-activity groups over the lists of the last rank() ----
    def _list_setup(self):
        if self._tables is not None:
            return
        it, dev = self.inter, self.inter.device
        n, nk = self.users.numel(), len(self.ks)
        self._tables = item_tables(it)
        self._counts = torch.zeros((nk, it.I), dtype=torch.int32, device=dev)
        self._list_rows = torch.zeros((n, len(LIST_VALUES) * nk), dtype=torch.float64, device=dev)
        self._gsums = torch.zeros(MAX_GROUPS * (len(METRICS) + len(LIST_VALUES)) * nk + MAX_GROUPS, dtype=torch.float64, device=dev)
        self._gs_ws = torch.empty(ops.group_sums_workspace_bytes(n, len(METRICS) * nk, MAX_GROUPS), dtype=torch.uint8, device=dev)
        self._one_group = torch.zeros(max(n, 1), dtype=torch.int32, device=dev)

    def _list_stats(self, counts: bool):
        self._list_setup()
        n = self.users.numel()
        ops.list_stats(self.top_ids[:n], self.inter.I, self.ks, self._tables, self._counts if counts else None,
                       self._list_rows if n else None)

    def list_metrics(self):
        """{"ks", "coverage", "gini", "novelty", "arp": float64 arrays of len(ks), "n_users", "n_items"}: exposure over the lists of
        every rank (counts all-reduced when sharded; every rank returns the same dict); n_items = |pool|"""
        from .dist import allreduce_sums
        self._list_stats(True)
        n, nk = self.users.numel(), len(self.ks)
        nc = len(LIST_VALUES) * nk
        buf = self._gsums[:nc + 1]
        ops.group_sums(self._list_rows, self._one_group[:n], 1, buf[:nc].view(1, nc), self._gs_ws)
        buf[-1] = float(n)
        allreduce_sums(buf)
        allreduce_sums(self._counts)
        s = buf.cpu().numpy()
        coverage, gini = coverage_gini(self._counts.index_select(1, self.inter.pool).cpu().numpy())
        n_all = int(round(s[-1]))
        means = s[:-1] / max(n_all, 1)
        out = {"ks": list(self.ks), "coverage": coverage, "gini": gini}
        for q, name in enumerate(LIST_VALUES):
            out[name] = means[q * nk:(q + 1) * nk].copy()
        out["n_users"] = n_all
        out["n_items"] = int(self.inter.pool.numel())
        return out

    def _group_setup(self, G):
        st = self._groups.get(G)
        if st is not None:
            return st
        it = self.inter
        mine = self.users.cpu().numpy().astype(np.int64)
        users, deg, group = user_groups(it, G)
        if not np.isin(mine, users).all():
            raise ValueError("group_metrics: the evaluator's users must be evaluation users (users with train and test items)")
        lookup = np.full(it.U, -1, np.int32)
        lookup[users] = group
        ev_groups = torch.from_numpy(lookup).to(it.device)[self.users.long()].to(torch.int32).contiguous()
        n_users = np.bincount(lookup[mine], minlength=G).astype(np.float64)
        degree = np.zeros((G, 2), np.int64)
        inter_sum = np.zeros(G, np.int64)
        for g in range(G):
            d = deg[group == g]
            if d.size:
                degree[g] = (d.min(), d.max())
                inter_sum[g] = d.sum()
        st = dict(lookup=torch.from_numpy(lookup).to(it.device), rows=ev_groups,
                  n_users=torch.from_numpy(n_users).to(it.device), degree=degree, interactions=inter_sum)
        self._groups[G] = st
        return st

    def group_metrics(self, G=4):
        """{"ks", "groups", "n_users", "degree", "interactions", "precision", "recall", "ndcg", "hit_ratio", "mrr", "novelty", "arp"}:
        the user-activity groups (module docstring).  n_users (G,): the evaluated users of each group (all-reduced when sharded);
        degree (G, 2): their min / max train degree; interactions (G,): their train interactions (both over inter.eval_users);
        the metrics: (G, len(ks)) float64 means over each group's users, zeros for an empty group.  ValueError unless G is in 1..8
        and the evaluator's users are evaluation users."""
        from .dist import allreduce_sums
        G = check_groups(G)
        st = self._group_setup(G)
        self._list_setup()
        self._compute()
        self._list_stats(False)
        n, nk = self.users.numel(), len(self.ks)
        na, nl = len(METRICS) * nk, len(LIST_VALUES) * nk
        buf = self._gsums[:G * (na + nl) + G]
        ops.group_sums(self._rows, st["rows"], G, buf[:G * na].view(G, na), self._gs_ws)
        ops.group_sums(self._list_rows, st["rows"], G, buf[G * na:G * (na + nl)].view(G, nl), self._gs_ws)
        buf[G * (na + nl):].copy_(st["n_users"])
        allreduce_sums(buf)
        s = buf.cpu().numpy()
        counts = np.rint(s[G * (na + nl):]).astype(np.int64)
        div = np.maximum(counts, 1)[:, None].astype(np.float64)
        acc = s[:G * na].reshape(G, na) / div
        lst = s[G * na:G * (na + nl)].reshape(G, nl) / div
        out = {"ks": list(self.ks), "groups": G, "n_users": counts, "degree": st["degree"].copy(),
               "interactions": st["interactions"].copy()}
        for q, name in enumerate(METRICS):
            out[name] = acc[:, q * nk:(q + 1) * nk].copy()
        for q, name in enumerate(LIST_VALUES):
            out[name] = lst[:, q * nk:(q + 1) * nk].copy()
        return out

    # ---- intra-list diversity over the lists of the last rank() ----
    def diversity_metrics(self):
        """{"ks", "ild": float64 array of len(ks), "n_users"}: the mean intra-list diversity (module docstring) over the evaluated
        users of every rank (sums all-reduced when sharded; every rank returns the same dict), from the final features rank()
        computed"""
        from .dist import allreduce_sums
        top = self.top_ids
        self._list_setup()
        it = self.inter
        n, nk = self.users.numel(), len(self.ks)
        if self._div_rows is None:
            self._div_rows = torch.zeros((n, nk), dtype=torch.float64, device=it.device)
        F = self._allneg.F if self.source == "tc" else self.F
        if n:
            ops.list_diversity(F, it.U, it.I, top[:n], self.ks, self._div_rows)
        buf = self._gsums[:nk + 1]
        ops.group_sums(self._div_rows, self._one_group[:n], 1, buf[:nk].view(1, nk), self._gs_ws)
        buf[-1] = float(n)
        allreduce_sums(buf)
        s = buf.cpu().numpy()
        n_all = int(round(s[-1]))
        return {"ks": list(self.ks), "ild": s[:nk] / max(n_all, 1), "n_users": n_all}
