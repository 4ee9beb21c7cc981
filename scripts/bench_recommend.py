"""Top-K recommendation lists (ngacf_recommend_topk) at Gowalla shape, with the exact AllNeg top-20 as the baseline.

The features are the propagated features of a seeded model after 20 fused training steps, not random ones: the tie rate and the
score distribution decide how often the candidate buffers are compacted.  Grid: width 64 / 128, K 20 / 100, users 1 / 256 / every
AllNeg evaluation user (train items excluded, the item pool as candidates).  Baselines in the same process:
ngacf_score_topk_exact(_w) at K = 20 for all users, its `_split` variant for 1 and 256 users, and the tcgen05 scorer at width 64
(AllNegEvaluator mode "tc": final features + scoring + re-score of flagged rows).  CUDA events, warm-up, median of 5 windows of
>= 0.5 s each; the card's name and power limit are read in the same run.

--similar measures the similar-item lists (ngacf_similar_items_topk) from the same features instead: 1 / 256 / every item as queries,
K 20 / 100, the item pool as candidates, with the all-users recommend pass (K 20 / 100) of the same process as the yardstick (an
all-items call ranks I queries where the user pass ranks the eval users, so `ratio_to_scaled_recommend` divides by that pass times
I / eval users) and the norm kernel's own time from a torch.profiler capture of the 1-item calls.

--audience and --similar-users measure the user-side lists (ngacf_audience_topk with the train users excluded, ngacf_similar_users_topk)
from the same features: 1 / 256 / every item (audience) or every user (similar users) as queries, K 20 / 100, the users with any train
or test item as candidates.  `ratio_per_query_row` is (ms / queries) over (ms / eval users) of the all-users recommend pass at the
same K, measured in the same process: an all-items audience pass does the same U x I products as that pass.

    python scripts/bench_recommend.py [--workload gowalla] [--out profiles/recommend_bench.json]
    python scripts/bench_recommend.py --similar [--out profiles/similar_bench.json]
    python scripts/bench_recommend.py --audience --similar-users [--out profiles/user_lists_bench.json]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload shapes and hyper-parameters of the flagship benchmark)
from scripts.bench_width import card, median_block_ms  # noqa: E402


def bench_similar(F, U, I, inter, all_users, d):
    from ngacf_b200 import ops
    dev = F.device
    all_items = torch.arange(I, dtype=torch.int32, device=dev)
    item_sets = {"1": all_items[:1], "256": all_items[:256], "all": all_items}
    res = dict(similar_ms={}, recommend_all_users_ms={}, ratio_to_scaled_recommend={})
    for K in (20, 100):
        lists = {}
        for name, q in item_sets.items():
            n = q.numel()
            ids = torch.empty((n, K), dtype=torch.int32, device=dev)
            sc = torch.empty((n, K), dtype=torch.float32, device=dev)
            ws = torch.empty(ops.similar_items_topk_workspace_bytes(d, I, n, K), dtype=torch.uint8, device=dev)
            call = lambda: ops.similar_items_topk(F, U, I, q, K, inter.in_pool, ids, sc, ws)
            call()
            lists[name] = (ids, sc)
            res["similar_ms"]["K%d_items_%s" % (K, name)] = median_block_ms(call, 3 if name == "all" else 20)
        for name in ("1", "256"):        # a row does not depend on the other queries or on the item slicing
            n = item_sets[name].numel()
            assert torch.equal(lists[name][0], lists["all"][0][:n]) and torch.equal(lists[name][1], lists["all"][1][:n]), (d, K, name)
        n = all_users.numel()
        ids = torch.empty((n, K), dtype=torch.int32, device=dev)
        sc = torch.empty((n, K), dtype=torch.float32, device=dev)
        ws = torch.empty(ops.recommend_topk_workspace_bytes(d, I, n, K), dtype=torch.uint8, device=dev)
        call = lambda: ops.recommend_topk(F, U, I, all_users, K, inter.train_ptr, inter.train_items, inter.in_pool, ids, sc, ws)
        call()
        rms = res["recommend_all_users_ms"]["K%d" % K] = median_block_ms(call, 3)
        res["ratio_to_scaled_recommend"]["K%d" % K] = res["similar_ms"]["K%d_items_all" % K] / (rms * I / n)
    # the norm kernel alone: device time per call from a profiler capture of 50 one-item calls (a separate pass, not timed above)
    q = item_sets["1"]
    ids = torch.empty((1, 20), dtype=torch.int32, device=dev)
    sc = torch.empty((1, 20), dtype=torch.float32, device=dev)
    ws = torch.empty(ops.similar_items_topk_workspace_bytes(d, I, 1, 20), dtype=torch.uint8, device=dev)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(50):
            ops.similar_items_topk(F, U, I, q, 20, inter.in_pool, ids, sc, ws)
        torch.cuda.synchronize()
    per_kernel = {}
    for e in prof.key_averages():
        for kname in ("item_rnorm_kernel", "recommend_topk_kernel", "recommend_merge_kernel"):
            if kname in e.key:
                per_kernel[kname] = per_kernel.get(kname, 0.0) + getattr(e, "self_device_time_total", 0.0) / 1000.0 / 50
    res["items_1_K20_kernel_ms_profiled"] = per_kernel
    return res


def bench_user_side(rec, F, U, I, inter, all_users, d, kinds):
    from ngacf_b200 import ops
    dev = F.device
    excl_ptr, excl_users, pool = rec.user_candidates()       # rec excludes "train": the item -> users CSR of the train pairs
    # kind -> (workspace bytes, ranking call, query sets)
    plans = dict(audience=(ops.audience_topk_workspace_bytes,
                           lambda q, K, ids, sc, ws: ops.audience_topk(F, U, I, q, K, excl_ptr, excl_users, pool, ids, sc, ws), I),
                 similar_users=(ops.similar_users_topk_workspace_bytes,
                                lambda q, K, ids, sc, ws: ops.similar_users_topk(F, U, I, q, K, pool, ids, sc, ws), U))
    plans = {k: (wb, run, {"1": torch.arange(1, dtype=torch.int32, device=dev), "256": torch.arange(256, dtype=torch.int32, device=dev),
                           "all": torch.arange(n_all, dtype=torch.int32, device=dev)}) for k, (wb, run, n_all) in plans.items() if k in kinds}
    res = dict(recommend_all_users_ms={})
    for kind in kinds:
        res[kind] = dict(queries_all=plans[kind][2]["all"].numel(), list_ms={}, ratio_per_query_row={})
    for K in (20, 100):
        for kind in kinds:
            ws_bytes, run, sets = plans[kind]
            lists = {}
            for name, q in sets.items():
                n = q.numel()
                ids = torch.empty((n, K), dtype=torch.int32, device=dev)
                sc = torch.empty((n, K), dtype=torch.float32, device=dev)
                ws = torch.empty(ws_bytes(d, U, n, K), dtype=torch.uint8, device=dev)
                call = lambda: run(q, K, ids, sc, ws)
                call()
                lists[name] = (ids, sc)
                res[kind]["list_ms"]["K%d_queries_%s" % (K, name)] = median_block_ms(call, 3 if name == "all" else 20)
            for name in ("1", "256"):    # a row does not depend on the other queries or on the user slicing
                n = sets[name].numel()
                assert torch.equal(lists[name][0], lists["all"][0][:n]) and torch.equal(lists[name][1], lists["all"][1][:n]), (kind, d, K)
        n = all_users.numel()
        ids = torch.empty((n, K), dtype=torch.int32, device=dev)
        sc = torch.empty((n, K), dtype=torch.float32, device=dev)
        ws = torch.empty(ops.recommend_topk_workspace_bytes(d, I, n, K), dtype=torch.uint8, device=dev)
        call = lambda: ops.recommend_topk(F, U, I, all_users, K, inter.train_ptr, inter.train_items, inter.in_pool, ids, sc, ws)
        call()
        rms = res["recommend_all_users_ms"]["K%d" % K] = median_block_ms(call, 3)
        for kind in kinds:
            for name, q in plans[kind][2].items():
                key = "K%d_queries_%s" % (K, name)
                res[kind]["ratio_per_query_row"][key] = (res[kind]["list_ms"][key] / q.numel()) / (rms / n)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="gowalla")
    ap.add_argument("--out", default=None)
    ap.add_argument("--similar", action="store_true", help="measure the similar-item lists instead of the user lists")
    ap.add_argument("--audience", action="store_true", help="measure the audience lists instead of the user lists")
    ap.add_argument("--similar-users", action="store_true", help="measure the similar-user lists instead of the user lists")
    args = ap.parse_args()
    from ngacf_b200 import ops
    from ngacf_b200.data import Interactions
    from ngacf_b200.evaluate import AllNegEvaluator
    from ngacf_b200.graph import BipartiteGraph
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.optim import FusedAdam
    from ngacf_b200.recommend import Recommender
    from ngacf_b200.train import FusedTrainer
    dev = torch.device("cuda:0")
    U, I, u, i, tu, ti, su, si = bench.make_data(args.workload)
    graph = BipartiteGraph(torch.from_numpy(np.stack([u, i])).to(dev), U, I)
    inter = Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)
    H = bench.HYPER
    ev_users = inter.eval_users
    user_sets = {"1": ev_users[:1].contiguous(), "256": ev_users[:256].contiguous(), "all": ev_users}
    out = dict(card=card(), workload=args.workload, U=U, I=I, E=graph.E, eval_users=int(ev_users.numel()), widths={})
    for d in (64, 128):
        torch.manual_seed(2019)
        model = SPUIGACF(U, I, d, [64, 64], H["droprate"]).to(dev)
        tr = FusedTrainer(model, inter, graph, H["batch"], FusedAdam(model.parameters(), lr=H["lr"], weight_decay=H["weight_decay"]),
                          sample_seed=0)
        tr.run_steps(20)
        rec = Recommender(model, graph, inter, "train")
        F = rec.F
        if args.similar:
            out["widths"][str(d)] = bench_similar(F, U, I, inter, user_sets["all"], d)
            del tr, model, rec
            torch.cuda.synchronize()
            continue
        kinds = [k for k, on in (("audience", args.audience), ("similar_users", args.similar_users)) if on]
        if kinds:
            out["widths"][str(d)] = bench_user_side(rec, F, U, I, inter, user_sets["all"], d, kinds)
            del tr, model, rec
            torch.cuda.synchronize()
            continue
        res = dict(recommend_ms={}, baseline_ms={})
        for K in (20, 100):
            for name, us in user_sets.items():
                n = us.numel()
                ids = torch.empty((n, K), dtype=torch.int32, device=dev)
                sc = torch.empty((n, K), dtype=torch.float32, device=dev)
                ws = torch.empty(ops.recommend_topk_workspace_bytes(d, I, n, K), dtype=torch.uint8, device=dev)
                call = lambda: ops.recommend_topk(F, U, I, us, K, inter.train_ptr, inter.train_items, inter.in_pool, ids, sc, ws)
                call()
                if K == 20:      # the lists are the exact AllNeg path's, bit for bit
                    ref_i, ref_s = torch.empty_like(ids), torch.empty_like(sc)
                    ops.score_topk_exact(F, U, I, us, inter, ref_i, ref_s)
                    assert torch.equal(ids, ref_i) and torch.equal(sc.view(torch.int32), ref_s.view(torch.int32)), (d, name)
                res["recommend_ms"]["K%d_users_%s" % (K, name)] = median_block_ms(call, 3 if name == "all" else 20)
        for name, us in user_sets.items():
            n = us.numel()
            ids = torch.empty((n, 20), dtype=torch.int32, device=dev)
            sc = torch.empty((n, 20), dtype=torch.float32, device=dev)
            if name == "all":
                fn, key = (lambda: ops.score_topk_exact(F, U, I, us, inter, ids, sc)), "exact_K20_users_all"
            else:
                fn, key = (lambda: ops.score_topk_exact_split(F, U, I, us, inter, ids, sc)), "exact_split_K20_users_%s" % name
            fn()
            res["baseline_ms"][key] = median_block_ms(fn, 3 if name == "all" else 20)
        if d == 64:
            model.eval()
            Z = model.propagate(graph).clone()
            ev = AllNegEvaluator(inter, "tc")
            ev.rank(Z)
            ev.resolve()
            res["baseline_ms"]["tc_allneg_K20_users_all"] = median_block_ms(lambda: (ev.rank(Z), ev.resolve()), 3)
        allk = res["baseline_ms"]["exact_K20_users_all"]
        res["ratio_to_exact_all_users"] = {k: v / allk for k, v in res["recommend_ms"].items() if k.endswith("_all")}
        out["widths"][str(d)] = res
        del tr, model, rec
        torch.cuda.synchronize()
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
