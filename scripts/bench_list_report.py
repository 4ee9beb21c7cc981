"""Beyond-accuracy metrics and user-activity groups (FullRankingEvaluator.list_metrics / group_metrics) at Gowalla shape, next to the
full-ranking metrics they accompany.

The features are the propagated features of a seeded 64-wide SPUIGACF after 20 fused training steps, as in bench_cutoff_eval.py.
Every evaluation user; per cut-off set (ks = [10, 20]: the tcgen05 AllNeg lists; ks = [20, 50, 100]: ngacf_recommend_topk lists,
K = 100), ms per call over the lists of one rank():
  rank_and_metrics  ev(Z): ranking + metrics(), for scale
  metrics           metrics() alone (metrics kernel + read-back of the sums)
  list_metrics      list_metrics() (exposure counts and novelty / arp rows, G = 1 sums, read-back, coverage and Gini on the host)
  group_metrics_4   group_metrics(4) (metrics kernel, novelty / arp rows, two group sums, read-back)
  list_stats_kernel ngacf_list_stats alone, counts and both tables
  group_sums_kernel ngacf_group_sums alone over the (n, 5 len(ks)) metric rows, G = 4
  host_coverage_gini the rest of list_metrics: the pool's counts gathered and read back, coverage and Gini in numpy
CUDA events, warm-up, median of 5 windows of >= 0.5 s; the card's name and power limit are read in the same run.

    python scripts/bench_list_report.py [--workload gowalla] [--out profiles/list_report_bench.json]
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
    from ngacf_b200.cutoff_eval import FullRankingEvaluator, coverage_gini
    from ngacf_b200.data import Interactions
    from ngacf_b200.graph import BipartiteGraph
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.optim import FusedAdam
    from ngacf_b200.train import FusedTrainer
    dev = torch.device("cuda:0")
    U, I, u, i, tu, ti, su, si = bench.make_data(args.workload)
    graph = BipartiteGraph(torch.from_numpy(np.stack([u, i])).to(dev), U, I)
    inter = Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)
    H = bench.HYPER
    n = int(inter.eval_users.numel())
    out = dict(card=card(), workload=args.workload, U=U, I=I, E=graph.E, eval_users=n, width=64, cases={})
    torch.manual_seed(2019)
    model = SPUIGACF(U, I, 64, [64, 64], H["droprate"]).to(dev)
    tr = FusedTrainer(model, inter, graph, H["batch"], FusedAdam(model.parameters(), lr=H["lr"], weight_decay=H["weight_decay"]),
                      sample_seed=0)
    tr.run_steps(20)
    model.eval()
    with torch.no_grad():
        Z = model.propagate(graph).clone()
    for name, ks in (("ks_10_20", [10, 20]), ("ks_20_50_100", [20, 50, 100])):
        ev = FullRankingEvaluator(inter, ks)
        ev(Z)
        b, g = ev.list_metrics(), ev.group_metrics(4)
        plain = lambda d: {k: (v.tolist() if hasattr(v, "tolist") else v) for k, v in d.items()}
        res = dict(source=ev.source, list_length=int(ev.top_ids.shape[1]), list_metrics=plain(b), group_metrics=plain(g), ms={})
        res["ms"]["rank_and_metrics"] = median_block_ms(lambda: ev(Z), 3)
        res["ms"]["metrics"] = median_block_ms(ev.metrics, 20)
        res["ms"]["list_metrics"] = median_block_ms(ev.list_metrics, 20)
        res["ms"]["group_metrics_4"] = median_block_ms(lambda: ev.group_metrics(4), 20)
        top = ev.top_ids[:n]
        counts = torch.empty((len(ks), I), dtype=torch.int32, device=dev)
        rows = torch.empty((n, 2 * len(ks)), dtype=torch.float64, device=dev)
        tables = ev._tables
        call = lambda: ops.list_stats(top, I, ks, tables, counts, rows)
        call()
        res["ms"]["list_stats_kernel"] = median_block_ms(call, 200)
        acc = ev.per_user()
        grp = ev._groups[4]["rows"]
        sums = torch.empty((4, acc.shape[1]), dtype=torch.float64, device=dev)
        ws = torch.empty(ops.group_sums_workspace_bytes(n, acc.shape[1], 4), dtype=torch.uint8, device=dev)
        call = lambda: ops.group_sums(acc, grp, 4, sums, ws)
        call()
        res["ms"]["group_sums_kernel"] = median_block_ms(call, 200)
        res["ms"]["host_coverage_gini"] = median_block_ms(lambda: coverage_gini(ev._counts.index_select(1, inter.pool).cpu().numpy()), 5)
        out["cases"][name] = res
        del ev
        torch.cuda.synchronize()
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
