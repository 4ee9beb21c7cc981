"""embedSize 64 vs 128 on one GPU at Gowalla shape: fused PairSampling ms/step and propagated edges/s, AllNeg evaluation ms.

Both widths run in the same process and are timed alternately (CUDA events, warm-up, median of repeated blocks of >= 0.5 s, the
DESIGN.md section 7 protocol).  AllNeg runs the exact scorer at both widths and the tcgen05 scorer at 64 (it is built for 64 only).
--profile adds a torch.profiler kernel split of the d=128 step, taken in a run of its own after the timed part.

    python scripts/bench_width.py [--workload gowalla] [--rounds 3] [--profile] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload shapes and hyper-parameters of the flagship benchmark)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def median_block_ms(fn, per_block, min_s=0.5, blocks=5):
    """fn() runs one unit; a block = per_block units; returns the median ms per unit over `blocks` blocks of >= min_s each"""
    res = []
    for _ in range(blocks):
        n, ms = 0, 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        while ms < 1000 * min_s:
            e0.record()
            for _ in range(per_block):
                fn()
            e1.record()
            e1.synchronize()
            ms += e0.elapsed_time(e1)
            n += per_block
        res.append(ms / n)
    return float(np.median(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="gowalla")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
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
    setups = {}
    for d in (64, 128):
        torch.manual_seed(2019)
        model = SPUIGACF(U, I, d, [64, 64], H["droprate"]).to(dev)
        optim = FusedAdam(model.parameters(), lr=H["lr"], weight_decay=H["weight_decay"])
        tr = FusedTrainer(model, inter, graph, H["batch"], optim, sample_seed=0)
        tr.run_steps(10)                                      # capture + warm-up
        model.eval()
        Z = model.propagate(graph).clone()
        model.train()
        evs = {m: AllNegEvaluator(inter, m) for m in (("exact", "tc") if d == 64 else ("exact",))}
        for ev in evs.values():
            ev.rank(Z)
            ev.resolve()
        setups[d] = (tr, Z, evs)
    torch.cuda.synchronize()
    res = {d: dict(step_ms=[], eval_ms={m: [] for m in setups[d][2]}) for d in setups}
    for _ in range(args.rounds):                              # the two widths alternate
        for d, (tr, Z, evs) in setups.items():
            res[d]["step_ms"].append(median_block_ms(lambda: tr.run_steps(20), 1) / 20)
            for m, ev in evs.items():
                res[d]["eval_ms"][m].append(median_block_ms(lambda: (ev.rank(Z), ev.resolve()), 3))
    out = dict(card=card(), workload=args.workload, U=U, I=I, E=graph.E, batch=H["batch"], droprate=H["droprate"], widths={})
    for d in setups:
        step = float(np.median(res[d]["step_ms"]))
        out["widths"][str(d)] = dict(step_ms=step, step_ms_rounds=res[d]["step_ms"], gedges_per_s=2 * graph.E / (step * 1e-3) / 1e9,
                                     allneg_ms={m: float(np.median(v)) for m, v in res[d]["eval_ms"].items()},
                                     allneg_ms_rounds=res[d]["eval_ms"], pruned_last_stage=setups[d][0].prune_last_stage)
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        tr = setups[128][0]
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            tr.run_steps(20)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" or getattr(e, "self_device_time_total", 0) > 0:
                kern[e.key] = kern.get(e.key, 0.0) + getattr(e, "self_device_time_total", 0.0) / 1000.0 / 20
        tot = sum(kern.values())
        out["profile_128_ms_per_step"] = {k: round(v, 4) for k, v in sorted(kern.items(), key=lambda kv: -kv[1])[:25]}
        out["profile_128_total_ms_per_step"] = tot
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
