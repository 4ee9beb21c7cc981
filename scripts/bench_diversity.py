"""Intra-list diversity (ngacf_list_diversity) and MMR re-ranking (ngacf_mmr_rerank) at Gowalla shape.

The features are those of a seeded SPUIGACF after 20 fused training steps, as in bench_novelty_ranking.py, at widths 64 and 128.
Timed (CUDA events, warm-up, median of 5 windows of >= 0.5 s): ngacf_list_diversity alone over the lists of every evaluation user at
K_list 20 (ks [10, 20]) and 100 (ks [20, 50, 100]); ngacf_mmr_rerank alone from N = 100 candidates to K 20 / 100 for the first 1 /
256 evaluation users and all of them; FullRankingEvaluator(ks=[20, 50, 100]) rank + metrics plain and with mmr_lambda=0.5,
alternating window by window; Recommender.diversified next to the plain K = 100 call for 1 user, alternating.  It also records
recall@20, coverage@20, novelty@20 and ILD@20 of the MMR lists for lambda in {1, 0.9, 0.7, 0.5, 0.3}.  The card's name and power
limit are read in the same run.

    python scripts/bench_diversity.py [--workload gowalla] [--out profiles/diversity_bench.json]
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
from scripts.bench_novelty_ranking import alternating_ms  # noqa: E402
from scripts.bench_width import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="gowalla")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from ngacf_b200 import ops
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    from ngacf_b200.data import Interactions
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
    n_all = int(ev_users.numel())
    out = dict(card=card(), workload=args.workload, U=U, I=I, E=graph.E, eval_users=n_all, widths={})
    for d in (64, 128):
        torch.manual_seed(2019)
        model = SPUIGACF(U, I, d, [64, 64], H["droprate"]).to(dev)
        tr = FusedTrainer(model, inter, graph, H["batch"], FusedAdam(model.parameters(), lr=H["lr"], weight_decay=H["weight_decay"]),
                          sample_seed=0)
        tr.run_steps(20)
        rec = Recommender(model, graph, inter, "train")
        F = rec.F
        res = dict(ild_ms={}, mmr_ms={}, evaluator_ms={}, diversified_1user_ms={}, tradeoff={})
        # candidate lists of every evaluation user, N = 100 (the ranking is not timed here)
        cand_ids = torch.empty((n_all, 100), dtype=torch.int32, device=dev)
        cand_sc = torch.empty((n_all, 100), dtype=torch.float32, device=dev)
        ws = torch.empty(ops.recommend_topk_workspace_bytes(d, I, n_all, 100), dtype=torch.uint8, device=dev)
        ops.recommend_topk(F, U, I, ev_users, 100, inter.train_ptr, inter.train_items, inter.in_pool, cand_ids, cand_sc, ws)
        for K_list, ks in ((20, [10, 20]), (100, [20, 50, 100])):
            lists = cand_ids[:, :K_list].contiguous()
            rows = torch.empty((n_all, len(ks)), dtype=torch.float64, device=dev)
            fn = lambda: ops.list_diversity(F, U, I, lists, ks, rows)
            fn()
            res["ild_ms"]["K_list%d_all_users" % K_list] = alternating_ms({"ild": fn}, 5)["ild"]
        for K in (20, 100):
            for name, n in (("1", 1), ("256", 256), ("all", n_all)):
                oi = torch.empty((n, K), dtype=torch.int32, device=dev)
                os_ = torch.empty((n, K), dtype=torch.float32, device=dev)
                ci, cs = cand_ids[:n].contiguous(), cand_sc[:n].contiguous()
                fn = lambda: ops.mmr_rerank(F, U, I, ci, cs, K, 0.5, oi, os_)
                fn()
                res["mmr_ms"]["N100_K%d_users_%s" % (K, name)] = alternating_ms({"mmr": fn}, 5 if name == "all" else 50)["mmr"]
        model.eval()
        with torch.no_grad():
            Z = model.propagate(graph).clone()
        evs = {"plain": FullRankingEvaluator(inter, [20, 50, 100]), "mmr_0.5": FullRankingEvaluator(inter, [20, 50, 100], mmr_lambda=0.5)}
        for ev in evs.values():
            ev(Z)
        res["evaluator_ms"] = alternating_ms({k: (lambda ev=ev: ev(Z)) for k, ev in evs.items()}, 3)
        one = ev_users[:1].cpu().numpy()
        res["diversified_1user_ms"] = alternating_ms({"plain_K100": lambda: rec(one, 100), "diversified_K100_N100": lambda: rec.diversified(one, 100, 0.5, 100),
                                                      "diversified_K20_N100": lambda: rec.diversified(one, 20, 0.5, 100)}, 20)
        for lam in (1.0, 0.9, 0.7, 0.5, 0.3):
            ev = FullRankingEvaluator(inter, [20], mmr_lambda=lam)
            m = ev(Z)
            lm = ev.list_metrics()
            dm = ev.diversity_metrics()
            res["tradeoff"][str(lam)] = dict(recall=float(m["recall"][0]), ndcg=float(m["ndcg"][0]), coverage=float(lm["coverage"][0]),
                                             gini=float(lm["gini"][0]), novelty=float(lm["novelty"][0]), ild=float(dm["ild"][0]))
        out["widths"][str(d)] = res
        del tr, model, rec, evs
        torch.cuda.synchronize()
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
