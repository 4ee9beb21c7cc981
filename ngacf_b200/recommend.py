"""Top-K lists from a trained SPUIGACF / SPUIMultiGACF (csrc/recommend.cu): items for users (ngacf_recommend_topk), items like
an item (ngacf_similar_items_topk), users for an item (ngacf_audience_topk) and users like a user (ngacf_similar_users_topk).

User lists are the AllNeg ranking's: exact fp32 scores with the specified summation tree, candidates = item pool minus the excluded
items, order = score descending, then item id ascending (the reference's ranklist_by_heapq).  Similar-item lists rank by the cosine
of the items' final features (the same tree for the dot products and the norms), candidates = item pool minus the query item, same
order.  Audience lists rank users by the same score as the user lists (the same bits for each (user, item) pair), candidates = user
pool minus the users the exclusion rule leaves out for that item; similar-user lists are the similar-item lists over the users'
features.  K is 1 .. 100.

Diversified user lists (diversified()) re-rank the top `candidates` of the user lists by maximal marginal relevance against the
cosine of the items' final features (ngacf_mmr_rerank); list_diversity() scores any item lists by their intra-list diversity
(ngacf_list_diversity).  Both are defined in ngacf_b200.cutoff_eval."""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .data import Interactions
from .graph import BipartiteGraph

MAX_K = 100
EXCLUDE = ("train", "all", "none")


class Recommender:
    """Ranks items for users of `model` propagated over `adj` (the (2,E) user-item index tensor the model trains on, or a
    BipartiteGraph).  exclude: "train" (the user's train items, the AllNeg candidate rule), "all" (train and test items) or
    "none"; `inter` (ngacf_b200.data.Interactions) supplies the excluded items and restricts the candidates to its item pool.
    Without `inter` every item is a candidate and only exclude="none" is accepted.  The user-side lists (audience, similar_users)
    take the users with any train or test item of `inter` as candidates, every user without it."""

    def __init__(self, model, adj, inter: Interactions = None, exclude: str = "train"):
        from .model import SPUIGACF, SPUIMultiGACF
        if type(model) not in (SPUIGACF, SPUIMultiGACF):
            raise NotImplementedError("Recommender ranks the SpUIGAT features of SPUIGACF / SPUIMultiGACF; %s is not supported"
                                      % type(model).__name__)
        if exclude not in EXCLUDE:
            raise ValueError("exclude must be one of %s, got %r" % ("/".join(EXCLUDE), exclude))
        if inter is None and exclude != "none":
            raise ValueError("exclude=%r needs the interactions (inter=...); without them only exclude='none' is possible" % exclude)
        self.model = model
        self.U, self.I = int(model.userNum), int(model.itemNum)
        dev = model.uEmbd.weight.device
        if inter is not None and (inter.U != self.U or inter.I != self.I):
            raise ValueError("interactions are %d x %d, the model %d x %d" % (inter.U, inter.I, self.U, self.I))
        self.adj = adj if isinstance(adj, BipartiteGraph) else torch.as_tensor(adj, dtype=torch.int64).to(dev)
        self.exclude = exclude
        self.excl_ptr = self.excl_items = self.in_pool = None
        self.inter = inter
        self._user_side = None
        if inter is not None:
            self.in_pool = inter.in_pool
            if exclude == "train":
                self.excl_ptr, self.excl_items = inter.train_ptr, inter.train_items
            elif exclude == "all":          # the union CSR of train and test items, sorted per user (Interactions.csr)
                to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(torch.int32).to(dev)
                self.excl_ptr, self.excl_items = to_dev(inter.host["all_ptr"]), to_dev(inter.host["all_items"])
        self.F = None
        self.refresh()

    def refresh(self):
        """Propagates again (eval mode: no dropout) and keeps the final features; call after more training."""
        m = self.model
        was_training = m.training
        m.eval()
        try:
            with torch.no_grad():
                Z = m.propagate(self.adj)
                if self.F is None or self.F.shape != Z.shape:
                    self.F = torch.empty_like(Z)
                ops.final_features(Z, self.F)
        finally:
            m.train(was_training)

    def _ids(self, ids, bound, what):
        """integer ids in [0, bound) -> int32 tensor on the features' device; ValueError otherwise (before any launch)"""
        if torch.is_tensor(ids):
            if ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool:
                raise ValueError("%ss must be integer ids, got %s" % (what, ids.dtype))
            t = ids
        else:
            a = np.asarray(ids)
            if a.size and not np.issubdtype(a.dtype, np.integer):
                raise ValueError("%ss must be integer ids, got %s" % (what, a.dtype))
            t = torch.from_numpy(a.astype(np.int64, copy=False).reshape(a.shape))
        if t.dim() != 1:
            raise ValueError("%ss must be one-dimensional, got shape %s" % (what, tuple(t.shape)))
        if t.numel() and (int(t.min()) < 0 or int(t.max()) >= bound):
            raise ValueError("%s ids must lie in [0, %d)" % (what, bound))
        return t.to(device=self.F.device, dtype=torch.int32).contiguous()

    @staticmethod
    def _k(K):
        if isinstance(K, bool) or not isinstance(K, (int, np.integer)) or not 1 <= int(K) <= MAX_K:
            raise ValueError("K must be an integer in 1..%d, got %r" % (MAX_K, K))
        return int(K)

    def _rank(self, q, K, n_cand, ws_bytes, rank):
        """(n, K) outputs for the int32 queries q, a workspace of ws_bytes(width, n_cand, n, K) bytes and rank(q, K, ids, scores, ws)
        -> (ids int32, scores float32)"""
        n = q.numel()
        dev = self.F.device
        ids = torch.empty((n, K), dtype=torch.int32, device=dev)
        scores = torch.empty((n, K), dtype=torch.float32, device=dev)
        if n:
            ws = torch.empty(ws_bytes(self.F.shape[-1], n_cand, n, K), dtype=torch.uint8, device=dev)
            rank(q, K, ids, scores, ws)
        return ids, scores

    def _lists(self, q, K, n_cand, ws_bytes, rank):
        """_rank with int64 ids"""
        ids, scores = self._rank(q, K, n_cand, ws_bytes, rank)
        return ids.long(), scores

    def _user_lists(self, users, K, novelty_weight):
        """the user lists of __call__ for a checked K -> (ids int32 (n, K), scores float32 (n, K)); the weight is checked before any
        feature is read"""
        from .cutoff_eval import check_novelty_weight, novelty_offsets
        w = check_novelty_weight(novelty_weight)
        if w != 0.0 and self.inter is None:
            raise ValueError("novelty_weight needs the interactions (inter=...): the item novelty comes from their train split")
        off = novelty_offsets(self.inter, w) if w != 0.0 else None
        u = self._ids(users, self.U, "user")
        return self._rank(u, K, self.I, ops.recommend_topk_workspace_bytes, lambda q, K, ids, scores, ws: ops.recommend_topk(
            self.F, self.U, self.I, q, K, self.excl_ptr, self.excl_items, self.in_pool, ids, scores, ws, off))

    def user_candidates(self):
        """-> (excl_ptr, excl_users, user_pool): the candidate inputs of ngacf_audience_topk / ngacf_similar_users_topk that audience()
        and similar_users() pass, for callers of ops.audience_topk / ops.similar_users_topk.  excl_ptr[I+1] / excl_users (int32, users
        ascending per item) is `exclude` transposed, None for "none" or without `inter`; user_pool (uint8[U]) marks the users with a
        train or test item, None without `inter`.  Built on the host from `inter` on first use and kept on the device."""
        if self._user_side is None:
            ptr = users = pool = None
            if self.inter is not None:
                h = self.inter.host
                dev = self.F.device
                to_dev = lambda a, dt=torch.int32: torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(dev)
                pool = to_dev(np.diff(h["all_ptr"]) > 0, torch.uint8)
                if self.exclude != "none":
                    p, items = (h["train_ptr"], h["train_items"]) if self.exclude == "train" else (h["all_ptr"], h["all_items"])
                    owner = np.repeat(np.arange(self.U, dtype=np.int64), np.diff(p))
                    order = np.argsort(items, kind="stable")         # by item; users stay ascending within an item
                    ptr = to_dev(np.concatenate([[0], np.cumsum(np.bincount(items, minlength=self.I))]))
                    users = to_dev(owner[order])
            self._user_side = (ptr, users, pool)
        return self._user_side

    def __call__(self, users, K: int = 20, novelty_weight=0.0):
        """-> (ids int64 (n, K), scores float32 (n, K)) on the GPU; rows with fewer than K candidates end in id -1 / score 0.0.
        novelty_weight w != 0: novelty-weighted lists, ranked (and scored) by s(u, i) + float32(w * nov(i)) with the item novelty of
        the train split of `inter` (ngacf_b200.cutoff_eval.novelty_offsets); a positive w moves popular items down.  w = 0 is the
        plain ranking."""
        ids, scores = self._user_lists(users, self._k(K), novelty_weight)
        return ids.long(), scores

    def diversified(self, users, K: int = 20, mmr_lambda=0.5, candidates: int = 100, novelty_weight=0.0):
        """-> (ids int64 (n, K), scores float32 (n, K)) on the GPU: MMR-diversified lists.  Each user's top `candidates` (K..100) of
        __call__(users, candidates, novelty_weight) (the same exclusion, pool and scores) are re-ranked greedily by mmr_lambda *
        rel(c) - (1 - mmr_lambda) * (max cosine similarity to the items picked so far), rel being the score min-max normalised over
        the candidates (ngacf_b200.cutoff_eval).  Rows hold the picks in pick order with their scores (so the scores are not
        sorted), padded with id -1 / score 0.0.  mmr_lambda = 1 gives __call__(users, K, novelty_weight)."""
        from .cutoff_eval import check_mmr_candidates, check_mmr_lambda
        K = self._k(K)
        lam = check_mmr_lambda(mmr_lambda)
        N = check_mmr_candidates(candidates, K)
        cand_ids, cand_scores = self._user_lists(users, N, novelty_weight)
        n = cand_ids.shape[0]
        ids = torch.empty((n, K), dtype=torch.int32, device=self.F.device)
        scores = torch.empty((n, K), dtype=torch.float32, device=self.F.device)
        if n:
            ops.mmr_rerank(self.F, self.U, self.I, cand_ids, cand_scores, K, lam, ids, scores)
        return ids.long(), scores

    def list_diversity(self, ids, ks):
        """ids: (n, L) item lists (L 1..100, integer ids; entries outside [0, I), such as -1 padding, are skipped), ks: cut-offs
        (1..8 integers in 1..L) -> float64 (n, len(ks)) on the GPU: each row's intra-list diversity at each cut-off
        (ngacf_b200.cutoff_eval) from the final features of the last refresh()"""
        from .cutoff_eval import check_ks
        ks = check_ks(ks)
        t = ids if torch.is_tensor(ids) else torch.from_numpy(np.asarray(ids))
        if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError("item lists must hold integer ids, got %s" % t.dtype)
        if t.dim() != 2 or not 1 <= t.shape[1] <= MAX_K:
            raise ValueError("item lists must be (n, L) with L in 1..%d, got shape %s" % (MAX_K, tuple(t.shape)))
        if ks[-1] > t.shape[1]:
            raise ValueError("cut-off %d is longer than the lists (%d entries)" % (ks[-1], t.shape[1]))
        lo, hi = np.iinfo(np.int32).min, np.iinfo(np.int32).max
        t = t.to(device=self.F.device, dtype=torch.int64).clamp(lo, hi).to(torch.int32).contiguous()
        rows = torch.zeros((t.shape[0], len(ks)), dtype=torch.float64, device=self.F.device)
        if t.shape[0]:
            ops.list_diversity(self.F, self.U, self.I, t, ks, rows)
        return rows

    def similar_items(self, items, K: int = 20):
        """-> (ids int64 (n, K), scores float32 (n, K)) on the GPU: for each query item the K items of highest cosine similarity of the
        final features of the last refresh(), the query itself left out, candidates restricted to the item pool when the Recommender
        has `inter` (`exclude` does not apply); rows with fewer than K candidates end in id -1 / score 0.0"""
        K = self._k(K)
        q = self._ids(items, self.I, "item")
        return self._lists(q, K, self.I, ops.similar_items_topk_workspace_bytes, lambda q, K, ids, scores, ws: ops.similar_items_topk(
            self.F, self.U, self.I, q, K, self.in_pool, ids, scores, ws))

    def audience(self, items, K: int = 20):
        """-> (ids int64 (n, K), scores float32 (n, K)) on the GPU: for each query item the K users of highest score (the score of the
        user lists, the same bits for each (user, item) pair) from the final features of the last refresh().  `exclude` applies
        transposed: "train" leaves out the users with the item in train, "all" also those with it in test.  Candidates are the users
        with any train or test item when the Recommender has `inter`, otherwise every user; rows with fewer than K candidates end in
        id -1 / score 0.0"""
        K = self._k(K)
        q = self._ids(items, self.I, "item")
        excl_ptr, excl_users, pool = self.user_candidates()
        return self._lists(q, K, self.U, ops.audience_topk_workspace_bytes, lambda q, K, ids, scores, ws: ops.audience_topk(
            self.F, self.U, self.I, q, K, excl_ptr, excl_users, pool, ids, scores, ws))

    def similar_users(self, users, K: int = 20):
        """-> (ids int64 (n, K), scores float32 (n, K)) on the GPU: for each query user the K users of highest cosine similarity of the
        final features of the last refresh(), the query itself left out; candidates as for audience(), `exclude` does not apply; rows
        with fewer than K candidates end in id -1 / score 0.0"""
        K = self._k(K)
        q = self._ids(users, self.U, "user")
        pool = self.user_candidates()[2]
        return self._lists(q, K, self.U, ops.similar_users_topk_workspace_bytes, lambda q, K, ids, scores, ws: ops.similar_users_topk(
            self.F, self.U, self.I, q, K, pool, ids, scores, ws))


def recommend(model, adj, users, K: int = 20, inter: Interactions = None, exclude: str = "train"):
    """One-shot Recommender(model, adj, inter, exclude)(users, K)."""
    return Recommender(model, adj, inter, exclude)(users, K)
