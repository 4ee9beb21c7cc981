"""Full-ranking metrics at several cut-offs (ngacf_b200.cutoff_eval.FullRankingEvaluator) at Gowalla shape, against today's AllNeg
evaluation (AllNegEvaluator: reference-format metrics at 1/5/10/20) as the yardstick.

The features are the propagated features of a seeded SPUIGACF after 20 fused training steps, as in bench_recommend.py.  Per width
(64 / 128), every evaluation user, ms per call (rank + metrics, which ends in the host read-back of the sums):
  allneg          AllNegEvaluator(inter, "auto") (tcgen05 at 64, exact at 128)
  ks_10_20        FullRankingEvaluator ks = [10, 20]: the tcgen05 lists at 64, the ranking lists (K = 20) at 128
  ks_20_50_100    FullRankingEvaluator ks = [20, 50, 100]: the ranking lists (ngacf_recommend_topk, K = 100)
  metrics_kernel  ngacf_cutoff_metrics alone on the K = 100 lists of every evaluation user, ks = [20, 50, 100] and 8 cut-offs
CUDA events, warm-up, median of 5 windows of >= 0.5 s; the card's name and power limit are read in the same run.

    python scripts/bench_cutoff_eval.py [--workload gowalla] [--out profiles/cutoff_eval_bench.json]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="gowalla")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from ngacf_b200 import ops
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    from ngacf_b200.data import Interactions
    from ngacf_b200.evaluate import AllNegEvaluator
    from ngacf_b200.graph import BipartiteGraph
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.optim import FusedAdam
    from ngacf_b200.train import FusedTrainer
    dev = torch.device("cuda:0")
    U, I, u, i, tu, ti, su, si = bench.make_data(args.workload)
    graph = BipartiteGraph(torch.from_numpy(np.stack([u, i])).to(dev), U, I)
    inter = Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)
    H = bench.HYPER
    users = inter.eval_users
    out = dict(card=card(), workload=args.workload, U=U, I=I, E=graph.E, eval_users=int(users.numel()), widths={})
    for d in (64, 128):
        torch.manual_seed(2019)
        model = SPUIGACF(U, I, d, [64, 64], H["droprate"]).to(dev)
        tr = FusedTrainer(model, inter, graph, H["batch"], FusedAdam(model.parameters(), lr=H["lr"], weight_decay=H["weight_decay"]),
                          sample_seed=0)
        tr.run_steps(20)
        model.eval()
        with torch.no_grad():
            Z = model.propagate(graph).clone()
        res = dict(ms={}, source={}, metrics={})
        ae = AllNegEvaluator(inter, "auto")
        ae(Z)
        res["ms"]["allneg"] = median_block_ms(lambda: ae(Z), 3)
        for name, ks in (("ks_10_20", [10, 20]), ("ks_20_50_100", [20, 50, 100])):
            ev = FullRankingEvaluator(inter, ks)
            m = ev(Z)
            res["source"][name] = ev.source
            res["metrics"][name] = {k: (v.tolist() if hasattr(v, "tolist") else v) for k, v in m.items()}
            res["ms"][name] = median_block_ms(lambda: ev(Z), 3)
        # the metrics kernel alone over the K = 100 lists of the last evaluator
        n = users.numel()
        for name, ks in (("metrics_kernel_3ks", [20, 50, 100]), ("metrics_kernel_8ks", [1, 5, 10, 20, 30, 50, 75, 100])):
            sums = torch.empty(5 * len(ks), dtype=torch.float64, device=dev)
            ws = torch.empty(ops.cutoff_metrics_workspace_bytes(n, len(ks)), dtype=torch.uint8, device=dev)
            call = lambda: ops.cutoff_metrics(ev.top_ids, users, inter, ks, sums, None, ws)
            call()
            res["ms"][name] = median_block_ms(call, 200)
        res["ratio_to_allneg"] = {k: v / res["ms"]["allneg"] for k, v in res["ms"].items() if k != "allneg"}
        out["widths"][str(d)] = res
        del tr, model, ae, ev
        torch.cuda.synchronize()
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
