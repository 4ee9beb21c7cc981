"""AllNeg evaluation on the GPU (train_eval_Gowalla.py:274-354 + :356-429 of the reference):
one propagation, fused user x item scoring + masking + top-20 per user, hit lists and metric sums on
the device.  Only top-K lists / 16 sums ever leave the GPU."""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .data import Interactions

KS = [1, 5, 10, 20]
K = 20


class AllNegEvaluator:
    def __init__(self, inter: Interactions, mode: str = "auto", users=None):
        """mode: 'exact' (fp32 CUDA cores, bit-reproducible), 'tc' (tcgen05 + exact re-score), 'auto' = tc when available.
        users: int32 device tensor of the users this rank evaluates (default: every evaluable user)."""
        self.inter = inter
        self.mode = mode
        self.users = inter.eval_users if users is None else users.to(torch.int32).contiguous()
        dev = inter.device
        n = self.users.numel()
        self._top_ids = torch.empty((max(n, 1), K), dtype=torch.int32, device=dev)
        self._top_scores = torch.empty((max(n, 1), K), dtype=torch.float32, device=dev)
        self.hits = torch.empty((max(n, 1), K), dtype=torch.uint8, device=dev)
        self.sums = torch.zeros(16, dtype=torch.float64, device=dev)
        self.metric_ws = torch.empty(max(n, 1) * 16, dtype=torch.float64, device=dev)
        self.F = None
        self._tc_ws = None
        self.fallback = torch.zeros(max(n, 1) + 1, dtype=torch.int32, device=dev)      # flag per user + number of flagged users
        self._pending_fallback = False

    def _use_tc(self, width: int = 64):
        from . import _lib
        if self.mode == "exact":
            return False
        if width != 64:
            # the tcgen05 scorer is built for 64-wide features; 'auto' ranks wider ones on the exact path
            if self.mode == "tc":
                raise _lib.NgacfError("ngacf_score_topk_tc is built for 64-wide features (got %d); use mode='exact' or 'auto'" % width)
            return False
        have = hasattr(_lib.load(), "ngacf_score_topk_tc")
        if self.mode == "tc" and not have:
            raise _lib.NgacfError("ngacf_score_topk_tc is not built")
        return have

    def rank(self, Z: torch.Tensor):
        """Z: pre-ELU last-stage output (N,64) or (N,128).  Fills top_ids/top_scores for inter.eval_users."""
        it = self.inter
        if self.F is None or self.F.shape != Z.shape:
            self.F = torch.empty_like(Z)
        ops.final_features(Z, self.F)
        n = self.users.numel()
        if n == 0:
            return
        if self._use_tc(Z.shape[-1]):
            # the workspace also carries the allowed-column matrix of (users, train set, pool): built by the first call, reused while
            # this evaluator's users tensor and the interactions' arrays are the same objects at the same version
            key = (self.users.data_ptr(), self.users._version, it.train_ptr.data_ptr(), it.train_ptr._version, it.train_items.data_ptr(),
                   it.train_items._version, it.in_pool.data_ptr(), it.in_pool._version)
            if self._tc_ws is None:
                self._tc_ws = torch.empty(ops.score_topk_tc_workspace_bytes(it.I, n), dtype=torch.uint8, device=Z.device)
                self._mask_key = None
            ops.score_topk_tc(self.F, it.U, it.I, self.users, it, self._top_ids, self._top_scores, self.fallback, self._tc_ws,
                              reuse_mask=self._mask_key == key)
            self._mask_key = key
            # rows whose error guard failed are recomputed exactly -- checked in metrics() / resolve(), together with the read-back of
            # the result, so that ranking itself never synchronises with the host
            self._pending_fallback = True
            self.n_fallback = 0
        else:
            ops.score_topk_exact(self.F, it.U, it.I, self.users, it, self._top_ids, self._top_scores)
            self.n_fallback = 0

    @property
    def top_ids(self):
        """(n_users, 20) int32, -1 padded; reading it finishes a pending rank() (see resolve)"""
        self.resolve()
        return self._top_ids

    @property
    def top_scores(self):
        self.resolve()
        return self._top_scores

    def resolve(self):
        """Finish rank(): recompute the flagged rows through the exact entry point (one 4-byte read-back; normally zero rows).
        Returns True if rows were replaced."""
        if not self._pending_fallback:
            return False
        self._pending_fallback = False
        n = self.users.numel()
        it = self.inter
        self.n_fallback = int(self.fallback[n].item())
        if self.n_fallback == 0:
            return False
        bad = torch.nonzero(self.fallback[:n]).flatten()
        users = self.users[bad].contiguous()
        ids = torch.empty((bad.numel(), K), dtype=torch.int32, device=self.F.device)
        sc = torch.empty((bad.numel(), K), dtype=torch.float32, device=self.F.device)
        ops.score_topk_exact_split(self.F, it.U, it.I, users, it, ids, sc)
        self._top_ids[bad] = ids
        self._top_scores[bad] = sc
        return True

    def metrics(self):
        """dict in the reference's format (train_eval_Gowalla.py:277-278,354)."""
        it = self.inter
        ops.eval_metrics(self._top_ids, self.users, it, self.hits, self.sums, self.metric_ws)      # queued behind rank(): no host sync yet
        if self.resolve():
            ops.eval_metrics(self._top_ids, self.users, it, self.hits, self.sums, self.metric_ws)
        from .dist import allreduce_sums
        allreduce_sums(self.sums)                                   # multi-GPU: users are sharded, only 16 sums are merged
        s = self.sums.cpu().numpy() / max(it.n_train_users, 1)      # divisor = users with train data (:283)
        return {"precision": s[0:4].copy(), "recall": s[4:8].copy(), "ndcg": s[8:12].copy(), "hit_ratio": s[12:16].copy(), "auc": 0.0}

    def __call__(self, Z):
        self.rank(Z)
        return self.metrics()
