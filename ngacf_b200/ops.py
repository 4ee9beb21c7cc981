"""Thin tensor-level wrappers over the C-ABI (include/ngacf_b200.h).  Each function only validates
devices/dtypes, passes raw pointers + the current CUDA stream, and never allocates or synchronises
(so everything here can be captured in a CUDA graph).  No CPU path exists."""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from .graph import BipartiteGraph

STAGES = ((8, 8), (1, 64))   # SPUIGACF: eight 64->8 heads, then out_att 64->64 (SPUIGACF.py:17-22,191-205)
D = 64
WIDTHS = (64, 128)           # embedSize values the kernels are built for; the `_w` entry points carry widths other than 64


def spuigacf_stages(embed: int, n_head_stages: int = 1):
    """Stage list (heads, width per head) of SPUIGACF (n_head_stages = 1) / SPUIMultiGACF (2) at embedSize `embed`: every head
    stage writes 8 x 8 = 64 columns, out_att writes `embed`.  The input width of the first stage is `embed` (the embedding tables)."""
    check_width(embed)
    return ((8, 8),) * n_head_stages + ((1, int(embed)),)


def check_width(embed: int):
    if int(embed) not in WIDTHS:
        raise ValueError("embedSize %r is not supported: the sm_100a kernels are built for embedSize %s"
                         % (embed, " and ".join(str(w) for w in WIDTHS)))


def _p(t):
    return None if t is None else t.data_ptr()


def _s():
    return torch.cuda.current_stream().cuda_stream


def _f32(t, name):
    if t.dtype != torch.float32 or not t.is_contiguous():
        raise _lib.NgacfError("%s must be a contiguous float32 tensor" % name)
    _lib.require_cuda(t)


def pointer_table(tensors):
    """Device array of raw pointers (wtab / gtab of the header)."""
    dev = tensors[0].device
    for t in tensors:
        _f32(t, "table entry")
    return torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64).to(dev, non_blocking=False)


def feature_mask(out, seed, call, stage, droprate, call_dev=None):
    _lib.call("ngacf_feature_mask", _p(out), out.numel(), int(seed), int(call) & 0xFFFFFFFF, _p(call_dev), int(stage), float(droprate), _s())


def edge_mask(out, H, seed, call, stage, droprate, call_dev=None):
    _lib.call("ngacf_edge_mask", _p(out), out.numel(), int(H), int(seed), int(call) & 0xFFFFFFFF, _p(call_dev), int(stage), float(droprate), _s())


def counter_add(counter, delta):
    _lib.call("ngacf_counter_add", _p(counter), int(delta), _s())


def dropout_masks(feats, edges, heads, N, E, seed, call, droprate, call_dev=None, widths=None):
    """every stage's feature + edge mask of one propagation in a single launch (same bits as feature_mask/edge_mask per stage);
    widths: per-stage input widths (feature masks of width/64 words per row), None = all 64"""
    S = len(heads)
    fa = (ctypes.c_void_p * S)(*[f.data_ptr() for f in feats])
    ea = (ctypes.c_void_p * S)(*[e.data_ptr() for e in edges])
    ha = (ctypes.c_int32 * S)(*[int(h) for h in heads])
    if widths is None or all(int(w) == 64 for w in widths):
        _lib.call("ngacf_dropout_masks", fa, ea, ha, S, int(N), int(E), int(seed), int(call) & 0xFFFFFFFF, _p(call_dev), float(droprate), _s())
        return
    wa = (ctypes.c_int32 * S)(*[int(w) for w in widths])
    _lib.call("ngacf_dropout_masks_w", fa, ea, ha, wa, S, int(N), int(E), int(seed), int(call) & 0xFFFFFFFF, _p(call_dev), float(droprate), _s())


def dropout_masks_ranges(feats, edges, heads, node_ranges, edge_range, seed, call, droprate, call_dev=None):
    """masks of the node ranges [(a0,b0),(a1,b1)] and the edge range (e0,e1) only, written at their global positions"""
    S = len(heads)
    fa = (ctypes.c_void_p * S)(*[f.data_ptr() for f in feats])
    ea = (ctypes.c_void_p * S)(*[e.data_ptr() for e in edges])
    ha = (ctypes.c_int32 * S)(*[int(h) for h in heads])
    (a0, b0), (a1, b1) = node_ranges
    _lib.call("ngacf_dropout_masks_ranges", fa, ea, ha, S, int(a0), int(b0), int(a1), int(b1), int(edge_range[0]), int(edge_range[1]), int(seed),
              int(call) & 0xFFFFFFFF, _p(call_dev), float(droprate), _s())


def batch_rows_gather(Z, U, users, items, u_range, i_range, Zb):
    _lib.call("ngacf_batch_rows_gather", _p(Z), int(U), _p(users), _p(items), users.numel(), int(u_range[0]), int(u_range[1]), int(i_range[0]),
              int(i_range[1]), _p(Zb), _s())


def batch_rows_scatter(Zb, U, users, items, Z):
    _lib.call("ngacf_batch_rows_scatter", _p(Zb), int(U), _p(users), _p(items), users.numel(), _p(Z), _s())


def memset_zero(t):
    _lib.call("ngacf_memset_zero", _p(t), t.numel() * t.element_size(), _s())


def transform_fwd(Xu, Xi, apply_elu, featmask, scale, wtab, H, U, I, h, s, d_in=64, d_out=64):
    if d_in == 64 and d_out == 64:
        _lib.call("ngacf_transform_fwd", _p(Xu), _p(Xi), int(apply_elu), _p(featmask), float(scale), _p(wtab), H, U, I, _p(h), _p(s), _s())
    else:
        _lib.call("ngacf_transform_fwd_w", _p(Xu), _p(Xi), int(apply_elu), _p(featmask), float(scale), _p(wtab), H, int(d_in), int(d_out), U, I,
                  _p(h), _p(s), _s())


def aggregate_fwd(g: BipartiteGraph, scratch, counter, h, s, H, edgemask, scale, Z, norm, partial_from=-1, width=64):
    if width == 64:
        _lib.call("ngacf_aggregate_fwd", _p(g.tasks), g.T, _p(g.adj_ptr), _p(g.adj_idx), _p(g.adj_eid), _p(g.long_first_slot),
                  _p(counter), _p(scratch), _p(h), _p(s), H, _p(edgemask), float(scale), _p(Z), _p(norm), int(partial_from), _s())
    else:
        _lib.call("ngacf_aggregate_fwd_w", _p(g.tasks), g.T, _p(g.adj_ptr), _p(g.adj_idx), _p(g.adj_eid), _p(g.long_first_slot),
                  _p(counter), _p(scratch), _p(h), _p(s), H, int(width), _p(edgemask), float(scale), _p(Z), _p(norm), int(partial_from), _s())


class ActiveRows:
    """Rows a pruned output stage computes (csrc/pruned_stage.cu): stamp int32[N] (a node is active iff stamp[node] == val
    (+ *val_dev)), the compacted list of their tasks and one activity bit per adjacency position."""

    def __init__(self, g: BipartiteGraph, val=0, val_dev=None):
        dev = g.device
        self.g = g
        self.stamp = torch.full((g.N,), -1, dtype=torch.int32, device=dev)
        self.task_list = torch.empty(max(g.T, 1), dtype=torch.int32, device=dev)
        self.task_count = torch.zeros(2, dtype=torch.int32, device=dev)      # {user tasks, item tasks}
        self.edge_bits = torch.zeros((2 * g.E + 31) // 32 + 1, dtype=torch.int32, device=dev)
        self.val, self.val_dev = int(val), val_dev

    def at(self, val, val_dev=None):
        self.val, self.val_dev = int(val) & 0x7FFFFFFF, val_dev
        return self

    def mark(self, users, items):
        """stamps the batch rows and builds the task list / activity bits for them"""
        g = self.g
        _lib.call("ngacf_mark_active", _p(self.stamp), _p(users), _p(items), users.numel(), g.U, self.val, _p(self.val_dev),
                  _p(self.task_count), _s())
        _lib.call("ngacf_active_plan", _p(self.stamp), self.val, _p(self.val_dev), _p(g.tasks), g.T, g.T_users, _p(g.adj_idx), 2 * g.E,
                  _p(self.task_list), _p(self.task_count), _p(self.edge_bits), _s())


def aggregate_fwd_active(g: BipartiteGraph, scratch, counter, h, s, H, edgemask, scale, Z, norm, act: ActiveRows):
    _lib.call("ngacf_aggregate_fwd_active", _p(g.tasks), g.T, _p(act.task_list), _p(act.task_count), _p(g.adj_ptr), _p(g.adj_idx),
              _p(g.adj_eid), _p(g.long_first_slot), _p(counter), _p(scratch), _p(h), _p(s), H, _p(edgemask), float(scale), _p(Z),
              _p(norm), _s())


def stage_bwd_prep_active(g: BipartiteGraph, G, Z, h, norm, H, Ghat, dN, act: ActiveRows):
    _lib.call("ngacf_stage_bwd_prep_active", _p(g.tasks), g.T, _p(act.task_list), _p(act.task_count), _p(G), _p(Z), _p(h), _p(norm), H,
              _p(Ghat), _p(dN), _s())


def stage_bwd_edges_active(mode, g: BipartiteGraph, scratch, counter, G, Ghat, dN, h, s, H, edgemask, scale, wtab, ds_store, dh, dS, act: ActiveRows):
    t0, t1 = (0, g.T_users) if mode == 0 else (g.T_users, g.T)
    _lib.call("ngacf_stage_bwd_edges_active", mode, _p(g.tasks), t0, t1, _p(act.task_list), _p(act.task_count), _p(g.adj_ptr), _p(g.adj_idx), _p(g.adj_eid),
              _p(g.long_first_slot), _p(counter), _p(scratch), _p(G), _p(Ghat), _p(dN), _p(h), _p(s), H, _p(edgemask),
              float(scale), _p(wtab), g.U, _p(act.stamp), act.val, _p(act.val_dev), _p(act.edge_bits), _p(ds_store), _p(dh), _p(dS), _s())


def step_counters(total, loss, row_dev, row_stride):
    _lib.call("ngacf_step_counters", _p(total), _p(loss), _p(row_dev), int(row_stride), _s())


def aggregate_finalize(Z, h, norm, H):
    _lib.call("ngacf_aggregate_finalize", _p(Z), _p(h), _p(norm), H, Z.shape[0], _s())


def stage_bwd_finalize(dh, dS, G, wtab, H, item_side):
    _lib.call("ngacf_stage_bwd_finalize", _p(dh), _p(dS), _p(G), _p(wtab), H, int(item_side), dh.shape[0], _s())


def bpr_loss_owned(pos, neg, gscale, loss, dpos, dneg, users, u_lo, u_hi):
    _lib.call("ngacf_bpr_loss_owned", _p(pos), _p(neg), pos.numel(), float(gscale), _p(loss), _p(dpos), _p(dneg), _p(users), int(u_lo),
              int(u_hi), _s())


def score_pairs(Z, U, users, items, out):
    """the row width is Z's (64 or 128)"""
    if Z.shape[-1] == 64:
        _lib.call("ngacf_score_pairs", _p(Z), U, _p(users), _p(items), users.numel(), _p(out), _s())
    else:
        _lib.call("ngacf_score_pairs_w", _p(Z), int(Z.shape[-1]), U, _p(users), _p(items), users.numel(), _p(out), _s())


def score_pairs_bwd(Z, U, users, items, dscore, G, accumulate=False):
    if Z.shape[-1] == 64:
        _lib.call("ngacf_score_pairs_bwd", _p(Z), U, _p(users), _p(items), _p(dscore), users.numel(), _p(G), int(accumulate), _s())
    else:
        _lib.call("ngacf_score_pairs_bwd_w", _p(Z), int(Z.shape[-1]), U, _p(users), _p(items), _p(dscore), users.numel(), _p(G),
                  int(accumulate), _s())


def final_features(Z, F):
    if Z.shape[-1] == 64:
        _lib.call("ngacf_final_features", _p(Z), Z.shape[0], _p(F), _s())
    else:
        _lib.call("ngacf_final_features_w", _p(Z), Z.shape[0], int(Z.shape[-1]), _p(F), _s())


def bpr_loss(pos, neg, gscale, loss, dpos, dneg):
    _lib.call("ngacf_bpr_loss", _p(pos), _p(neg), pos.numel(), float(gscale), _p(loss), _p(dpos), _p(dneg), _s())


def stage_bwd_prep(G, Z, h, norm, H, Ghat, dN, width=64):
    if width == 64:
        _lib.call("ngacf_stage_bwd_prep", _p(G), _p(Z), _p(h), _p(norm), H, G.shape[0], _p(Ghat), _p(dN), _s())
    else:
        _lib.call("ngacf_stage_bwd_prep_w", _p(G), _p(Z), _p(h), _p(norm), H, int(width), G.shape[0], _p(Ghat), _p(dN), _s())


def stage_bwd_edges(mode, g: BipartiteGraph, scratch, counter, G, Ghat, dN, h, s, H, edgemask, scale, wtab, ds_store, dh, dS, partial=0,
                    width=64):
    t0, t1 = (0, g.T_users) if mode == 0 else (g.T_users, g.T)
    if width == 64:
        _lib.call("ngacf_stage_bwd_edges", mode, _p(g.tasks), t0, t1, _p(g.adj_ptr), _p(g.adj_idx), _p(g.adj_eid),
                  _p(g.long_first_slot), _p(counter), _p(scratch), _p(G), _p(Ghat), _p(dN), _p(h), _p(s), H, _p(edgemask),
                  float(scale), _p(wtab), g.U, _p(ds_store), _p(dh), _p(dS), int(partial), _s())
    else:
        _lib.call("ngacf_stage_bwd_edges_w", mode, _p(g.tasks), t0, t1, _p(g.adj_ptr), _p(g.adj_idx), _p(g.adj_eid),
                  _p(g.long_first_slot), _p(counter), _p(scratch), _p(G), _p(Ghat), _p(dN), _p(h), _p(s), H, int(width), _p(edgemask),
                  float(scale), _p(wtab), g.U, _p(ds_store), _p(dh), _p(dS), int(partial), _s())


def transform_bwd_workspace_bytes(U, I, d_in=64, d_out=64):
    if d_in == 64 and d_out == 64:
        return int(_lib.load().ngacf_transform_bwd_workspace_bytes(U, I))
    return int(_lib.load().ngacf_transform_bwd_workspace_bytes_w(int(d_in), int(d_out), U, I))


def transform_bwd(dh, dS, h, Xu, Xi, apply_elu, featmask, scale, wtab, gtab, H, U, I, dXu, dXi, accumulate_dx, accumulate_dw, ws,
                  d_in=64, d_out=64):
    if d_in == 64 and d_out == 64:
        _lib.call("ngacf_transform_bwd", _p(dh), _p(dS), _p(h), _p(Xu), _p(Xi), int(apply_elu), _p(featmask), float(scale), _p(wtab),
                  _p(gtab), H, U, I, _p(dXu), _p(dXi), int(accumulate_dx), int(accumulate_dw), _p(ws), ws.numel() * ws.element_size(), _s())
    else:
        _lib.call("ngacf_transform_bwd_w", _p(dh), _p(dS), _p(h), _p(Xu), _p(Xi), int(apply_elu), _p(featmask), float(scale), _p(wtab),
                  _p(gtab), H, int(d_in), int(d_out), U, I, _p(dXu), _p(dXi), int(accumulate_dx), int(accumulate_dw), _p(ws),
                  ws.numel() * ws.element_size(), _s())


def transform_bwd_dx(dh, Xu, Xi, apply_elu, featmask, scale, wtab, H, U, I, dXu, dXi, accumulate):
    _lib.call("ngacf_transform_bwd_dx", _p(dh), _p(Xu), _p(Xi), int(apply_elu), _p(featmask), float(scale), _p(wtab), H, U, I, _p(dXu), _p(dXi),
              int(accumulate), _s())


def transform_bwd_dw_workspace_bytes(U, I):
    return int(_lib.load().ngacf_transform_bwd_dw_workspace_bytes(U, I))


def transform_bwd_dw(dh, dS, Xu, Xi, apply_elu, featmask, scale, wtab, gtab, H, U, I, accumulate, ws):
    _lib.call("ngacf_transform_bwd_dw", _p(dh), _p(dS), _p(Xu), _p(Xi), int(apply_elu), _p(featmask), float(scale), _p(wtab), _p(gtab), H, U, I,
              int(accumulate), _p(ws), ws.numel() * ws.element_size(), _s())


def adam_step(tab, n_tensors, total_numel, lr, beta1, beta2, eps, weight_decay, step):
    _lib.call("ngacf_adam_step", _p(tab), n_tensors, total_numel, lr, beta1, beta2, eps, weight_decay, int(step), _s())


def adam_step_dev(tab, n_tensors, total_numel, lr, beta1, beta2, eps, weight_decay, state):
    _lib.call("ngacf_adam_step_dev", _p(tab), n_tensors, total_numel, lr, beta1, beta2, eps, weight_decay, _p(state), _s())


def sample_pairs(inter, row_begin, row_end, seed, epoch, users, pos, neg, row_dev=None):
    _lib.call("ngacf_sample_pairs", _p(inter.train_rows_user), _p(inter.train_ptr), _p(inter.train_items), _p(inter.train_rank),
              _p(inter.pool), inter.pool.numel(), int(row_begin), int(row_end), _p(row_dev), int(seed), int(epoch), _p(users), _p(pos),
              _p(neg), _s())


def score_topk_exact(F, U, I, users, inter, top_ids, top_scores):
    """the row width is F's (64 or 128)"""
    if F.shape[-1] == 64:
        _lib.call("ngacf_score_topk_exact", _p(F), U, I, _p(users), users.numel(), _p(inter.train_ptr), _p(inter.train_items),
                  _p(inter.in_pool), _p(top_ids), _p(top_scores), _s())
    else:
        _lib.call("ngacf_score_topk_exact_w", _p(F), int(F.shape[-1]), U, I, _p(users), users.numel(), _p(inter.train_ptr),
                  _p(inter.train_items), _p(inter.in_pool), _p(top_ids), _p(top_scores), _s())


def score_topk_exact_split(F, U, I, users, inter, top_ids, top_scores):
    """score_topk_exact for few users: item range split over CTAs (workspace allocated here: this is the rare fallback path)"""
    n = users.numel()
    ws = torch.empty(int(_lib.load().ngacf_score_topk_exact_split_workspace_bytes(I, n)), dtype=torch.uint8, device=F.device)
    if F.shape[-1] == 64:
        _lib.call("ngacf_score_topk_exact_split", _p(F), U, I, _p(users), n, _p(inter.train_ptr), _p(inter.train_items),
                  _p(inter.in_pool), _p(top_ids), _p(top_scores), _p(ws), ws.numel(), _s())
    else:
        _lib.call("ngacf_score_topk_exact_split_w", _p(F), int(F.shape[-1]), U, I, _p(users), n, _p(inter.train_ptr), _p(inter.train_items),
                  _p(inter.in_pool), _p(top_ids), _p(top_scores), _p(ws), ws.numel(), _s())


def score_topk_tc_workspace_bytes(I, n_users):
    return int(_lib.load().ngacf_score_topk_tc_workspace_bytes(I, n_users))


def score_topk_tc(F, U, I, users, inter, top_ids, top_scores, fallback, ws, reuse_mask=False):
    """reuse_mask: `ws` already holds the allowed-column matrix of (users, inter) from an earlier call (include/ngacf_b200.h)"""
    _lib.call("ngacf_score_topk_tc", _p(F), U, I, _p(users), users.numel(), _p(inter.train_ptr), _p(inter.train_items),
              _p(inter.in_pool), _p(top_ids), _p(top_scores), _p(fallback), int(bool(reuse_mask)), _p(ws), ws.numel() * ws.element_size(), _s())


def recommend_topk_workspace_bytes(width, I, n_users, K):
    return int(_lib.load().ngacf_recommend_topk_workspace_bytes(int(width), int(I), int(n_users), int(K)))


def recommend_topk(F, U, I, users, K, excl_ptr, excl_items, in_pool, top_ids, top_scores, ws):
    """top-K lists of `users` (int32) from final features F (U+I, 64 or 128); excl_ptr/excl_items (CSR over users) and in_pool may be
    None; ws: uint8 tensor of recommend_topk_workspace_bytes(...) bytes (may be empty)"""
    _lib.call("ngacf_recommend_topk", _p(F), int(F.shape[-1]), int(U), int(I), _p(users), users.numel(), int(K), _p(excl_ptr),
              _p(excl_items), _p(in_pool), _p(top_ids), _p(top_scores), _p(ws) if ws.numel() else None, ws.numel(), _s())


def similar_items_topk_workspace_bytes(width, I, n_items, K):
    return int(_lib.load().ngacf_similar_items_topk_workspace_bytes(int(width), int(I), int(n_items), int(K)))


def similar_items_topk(F, U, I, items, K, in_pool, top_ids, top_scores, ws):
    """top-K cosine-similar items of the query `items` (int32) from final features F (U+I, 64 or 128), the query itself left out;
    in_pool may be None; ws: uint8 tensor of similar_items_topk_workspace_bytes(...) bytes"""
    _lib.call("ngacf_similar_items_topk", _p(F), int(F.shape[-1]), int(U), int(I), _p(items), items.numel(), int(K), _p(in_pool),
              _p(top_ids), _p(top_scores), _p(ws) if ws.numel() else None, ws.numel(), _s())


def audience_topk_workspace_bytes(width, U, n_items, K):
    return int(_lib.load().ngacf_audience_topk_workspace_bytes(int(width), int(U), int(n_items), int(K)))


def audience_topk(F, U, I, items, K, excl_ptr, excl_users, user_pool, top_ids, top_scores, ws):
    """top-K users of the query `items` (int32) from final features F (U+I, 64 or 128); excl_ptr/excl_users (CSR over items) and
    user_pool may be None; ws: uint8 tensor of audience_topk_workspace_bytes(...) bytes (may be empty)"""
    _lib.call("ngacf_audience_topk", _p(F), int(F.shape[-1]), int(U), int(I), _p(items), items.numel(), int(K), _p(excl_ptr),
              _p(excl_users), _p(user_pool), _p(top_ids), _p(top_scores), _p(ws) if ws.numel() else None, ws.numel(), _s())


def similar_users_topk_workspace_bytes(width, U, n_users, K):
    return int(_lib.load().ngacf_similar_users_topk_workspace_bytes(int(width), int(U), int(n_users), int(K)))


def similar_users_topk(F, U, I, users, K, user_pool, top_ids, top_scores, ws):
    """top-K cosine-similar users of the query `users` (int32) from final features F (U+I, 64 or 128), the query itself left out;
    user_pool may be None; ws: uint8 tensor of similar_users_topk_workspace_bytes(...) bytes"""
    _lib.call("ngacf_similar_users_topk", _p(F), int(F.shape[-1]), int(U), int(I), _p(users), users.numel(), int(K), _p(user_pool),
              _p(top_ids), _p(top_scores), _p(ws) if ws.numel() else None, ws.numel(), _s())


def eval_metrics(top_ids, users, inter, hits, sums, ws):
    _lib.call("ngacf_eval_metrics", _p(top_ids), _p(users), users.numel(), _p(inter.test_ptr), _p(inter.test_items), _p(hits),
              _p(sums), _p(ws), ws.numel() * ws.element_size(), _s())


NEG_TAG_TRAIN, NEG_TAG_EVAL = 0x4E54, 0x4E45


def sample_negs(inter, rows_user, rows_item, row_begin, row_end, seed, epoch, K, tag, users, items, row_dev=None, col_stride=0):
    """K distinct negatives per (user, positive) row: users/items int64[(row_end-row_begin)*(K+1)], column 0 = the positive.
    col_stride = 0: row-major (n, K+1); > 0: column-major, element (row b, column j) at j*col_stride + b."""
    _lib.call("ngacf_sample_negs", _p(rows_user), _p(rows_item), _p(inter.all_ptr), _p(inter.all_rank), _p(inter.pool), int(inter.pool.numel()),
              int(row_begin), int(row_end), _p(row_dev), int(seed), int(epoch), int(K), int(tag), int(col_stride), _p(users), _p(items), _s())


def bce_logits_loss(scores, group, loss, dscore=None):
    """group > 0: every group-th score is a positive (row-major pairs); group < 0: the first -group scores are the positives"""
    _lib.call("ngacf_bce_logits_loss", _p(scores), scores.numel(), int(group), _p(loss), _p(dscore), _s())


def rank_metrics(scores, group, top_k, sums):
    _lib.call("ngacf_rank_metrics", _p(scores), scores.numel() // int(group), int(group), int(top_k), _p(sums), _s())


def spmm_sym(g: BipartiteGraph, scratch, counter, val, diag, X, Y):
    """Y = diag (.) X + A_val X  (symmetric Laplacian on the unified adjacency; SPUIGAGPCF's GPLayer)"""
    _lib.call("ngacf_spmm_sym", _p(g.tasks), g.T, _p(g.adj_ptr), _p(g.adj_idx), _p(g.adj_eid), _p(g.long_first_slot), _p(counter), _p(scratch),
              _p(val), _p(diag), _p(X), _p(Y), _s())


# SpGraphAttentionLayer (csrc/spgat.cu); `graph` is a spgat.HomoGraph
def node_logits(h, wtab, H, N, p, q):
    _lib.call("ngacf_node_logits", _p(h), _p(wtab), int(H), int(N), _p(p), _p(q), _s())


def node_logits_bwd(h, dP, dQ, H, N, partials):
    _lib.call("ngacf_node_logits_bwd", _p(h), _p(dP), _p(dQ), int(H), int(N), _p(partials), partials.shape[0], _s())


def spgat_aggregate_fwd(graph, scratch, counter, h, p, q, H, emask, scale, Z, norm):
    g = graph.g
    _lib.call("ngacf_spgat_aggregate_fwd", _p(g.tasks), g.T, _p(g.adj_ptr), _p(g.adj_idx), _p(g.long_first_slot), _p(counter), _p(scratch), _p(h),
              _p(p), _p(q), int(H), _p(emask), float(scale), int(graph.self_loops), graph.n_adj, _p(Z), _p(norm), _s())


def spgat_bwd(graph, scratch, counter, G, Z, norm, h, p, q, H, emask, scale, wtab, Ghat, pairs, dP, dQ, dh):
    g = graph.g
    _lib.call("ngacf_spgat_bwd", _p(g.tasks), g.T, _p(g.adj_ptr), _p(g.adj_idx), _p(graph.rev), _p(g.long_first_slot), _p(counter), _p(scratch),
              _p(G), _p(Z), _p(norm), _p(h), _p(p), _p(q), int(H), _p(emask), float(scale), int(graph.self_loops), graph.n_adj, _p(wtab),
              _p(Ghat), _p(pairs), _p(dP), _p(dQ), _p(dh), _s())
