"""Novelty-weighted top-K lists (ngacf_recommend_topk_offset) next to the plain lists (ngacf_recommend_topk) at Gowalla shape.

The features are the propagated features of a seeded SPUIGACF after 20 fused training steps, as in bench_recommend.py, at widths
64 and 128; the offsets are novelty_offsets(inter, 1.0).  Grid: K 20 / 100, the first 1 / 256 evaluation users and every evaluation
user.  The offset and the plain call alternate window by window in one process (CUDA events, warm-up, 5 windows of >= 0.5 s each,
the median per call), so that both see the same clocks.  Also FullRankingEvaluator(ks=[20, 50, 100]) with novelty_weight=1.0 next to
the plain evaluator, ranking and metrics per call.  The card's name and power limit are read in the same run.

    python scripts/bench_novelty_ranking.py [--workload gowalla] [--out profiles/novelty_bench.json]
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
from scripts.bench_width import card  # noqa: E402


def alternating_ms(fns, per_block, min_s=0.5, blocks=5):
    """fns: {name: fn}; each fn runs one unit.  Window w runs every fn for >= min_s in turn; -> {name: median ms per unit}"""
    res = {k: [] for k in fns}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(blocks):
        for k, fn in fns.items():
            n, ms = 0, 0.0
            while ms < 1000 * min_s:
                e0.record()
                for _ in range(per_block):
                    fn()
                e1.record()
                e1.synchronize()
                ms += e0.elapsed_time(e1)
                n += per_block
            res[k].append(ms / n)
    return {k: float(np.median(v)) for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="gowalla")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from ngacf_b200 import ops
    from ngacf_b200.cutoff_eval import FullRankingEvaluator, novelty_offsets
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
    user_sets = {"1": ev_users[:1].contiguous(), "256": ev_users[:256].contiguous(), "all": ev_users}
    off = novelty_offsets(inter, 1.0)
    out = dict(card=card(), workload=args.workload, U=U, I=I, E=graph.E, eval_users=int(ev_users.numel()), novelty_weight=1.0,
               widths={})
    for d in (64, 128):
        torch.manual_seed(2019)
        model = SPUIGACF(U, I, d, [64, 64], H["droprate"]).to(dev)
        tr = FusedTrainer(model, inter, graph, H["batch"], FusedAdam(model.parameters(), lr=H["lr"], weight_decay=H["weight_decay"]),
                          sample_seed=0)
        tr.run_steps(20)
        rec = Recommender(model, graph, inter, "train")
        F = rec.F
        res = dict(lists_ms={}, ratio={}, evaluator_ms={})
        for K in (20, 100):
            for name, us in user_sets.items():
                n = us.numel()
                ids = torch.empty((n, K), dtype=torch.int32, device=dev)
                sc = torch.empty((n, K), dtype=torch.float32, device=dev)
                ws = torch.empty(ops.recommend_topk_workspace_bytes(d, I, n, K), dtype=torch.uint8, device=dev)
                calls = {
                    "plain": lambda: ops.recommend_topk(F, U, I, us, K, inter.train_ptr, inter.train_items, inter.in_pool, ids, sc, ws),
                    "offset": lambda: ops.recommend_topk(F, U, I, us, K, inter.train_ptr, inter.train_items, inter.in_pool, ids, sc, ws,
                                                         off),
                }
                for fn in calls.values():
                    fn()
                ms = alternating_ms(calls, 3 if name == "all" else 20)
                key = "K%d_users_%s" % (K, name)
                res["lists_ms"][key] = ms
                res["ratio"][key] = ms["offset"] / ms["plain"]
        model.eval()
        with torch.no_grad():
            Z = model.propagate(graph).clone()
        evs = {"plain": FullRankingEvaluator(inter, [20, 50, 100]), "novelty_1.0": FullRankingEvaluator(inter, [20, 50, 100], novelty_weight=1.0)}
        for ev in evs.values():
            ev(Z)
        res["evaluator_ms"] = alternating_ms({k: (lambda ev=ev: ev(Z)) for k, ev in evs.items()}, 3)
        res["evaluator_metrics"] = {k: {m: (v.tolist() if hasattr(v, "tolist") else v) for m, v in ev.metrics().items()}
                                    for k, ev in evs.items()}
        res["evaluator_list_metrics"] = {k: {m: (v.tolist() if hasattr(v, "tolist") else v) for m, v in ev.list_metrics().items()}
                                         for k, ev in evs.items()}
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
