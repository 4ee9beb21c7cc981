"""Times the NegSampling step (sampler + one propagation, dropout 0.2 + BCE on 1 + 4 items per row + backward + Adam) on one GPU and
over N GPUs.  Launched by torchrun; bench.py's shapes, hyper-parameters and synthetic data:

  world 1 : `single` (negsampling.NegSamplingTrainer);
  world N : `shard` (dist.ShardedNegSamplingTrainer: the same step, one propagation partitioned over the N GPUs) and `replica`
            (dist.NegSamplingReplicaTrainer: N propagations of batch rows each, gradients summed).

Every mode: captured steps, warm-up, then blocks of at least 0.5 s timed with CUDA events (max over the ranks), median block.  Rank 0
prints one JSON line per (shape, mode) -- ms/step, propagated edges/s, the partition's per-phase profile with collective bytes, and the
device name and power limit read in the same run -- and appends it to --out if given.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29515 \
        scripts/bench_neg_parallel.py --shapes gowalla sweep-10m --out profiles/negpar_n2.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import HYPER, SHAPES, make_data  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--shapes", nargs="+", default=["gowalla", "sweep-10m"], choices=sorted(SHAPES))
ap.add_argument("--warmup", type=int, default=20)
ap.add_argument("--blocks", type=int, default=5)
ap.add_argument("--out", default=None)
args = ap.parse_args()

rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
if not torch.cuda.is_available():
    raise SystemExit("bench_neg_parallel.py needs CUDA devices")
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)

from ngacf_b200.data import Interactions  # noqa: E402
from ngacf_b200.dist import NegSamplingReplicaTrainer, ShardedNegSamplingTrainer  # noqa: E402
from ngacf_b200.graph import BipartiteGraph  # noqa: E402
from ngacf_b200.model import SPUIGACF  # noqa: E402
from ngacf_b200.negsampling import NegSamplingTrainer  # noqa: E402
from ngacf_b200.optim import FusedAdam  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", str(local)],
                       capture_output=True, text=True)
    name, _, limit = q.stdout.strip().partition(",")
    return dict(device=name.strip() or torch.cuda.get_device_name(dev), power_limit_w=float(limit) if limit.strip() else None)


def sync():
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x):
    if world == 1:
        return x
    t = torch.tensor([float(x)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed(tr, k):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    tr.run_steps(k)
    e1.record()
    sync()
    return max_over_ranks(e0.elapsed_time(e1))


def measure(tr):
    tr.run_steps(args.warmup)
    probe = timed(tr, 10) / 10
    k = int(max_over_ranks(max(10, int(np.ceil(500.0 / max(probe, 1e-3))))))      # steps of a block of at least 0.5 s
    blocks = [timed(tr, k) / k for _ in range(args.blocks)]
    return statistics.median(blocks), blocks, k


info = device_info()
B = HYPER["batch"]
for shape in args.shapes:
    U, I, u, i, tu, ti, su, si = make_data(shape)
    modes = ["single"] if world == 1 else ["shard", "replica"]
    for mode in modes:
        torch.manual_seed(2019)
        model = SPUIGACF(U, I, 64, [64, 64], HYPER["droprate"]).to(dev)
        optim = FusedAdam(model.parameters(), lr=HYPER["lr"], weight_decay=HYPER["weight_decay"])
        inter = Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)
        if mode == "shard":
            tr = ShardedNegSamplingTrainer(model, inter, u, i, B, optim, sample_seed=0)
        else:
            graph = BipartiteGraph(torch.from_numpy(np.stack([u, i])).to(dev), U, I)
            cls = NegSamplingTrainer if mode == "single" else NegSamplingReplicaTrainer
            tr = cls(model, inter, graph, B, optim, sample_seed=0)
        ms, blocks, k = measure(tr)
        units = tr.units_per_step()
        rec = dict(shape=shape, U=U, I=I, E=int(len(u)), mode=mode, world=world, batch=B, droprate=HYPER["droprate"],
                   rows_per_step=B * (world if mode == "replica" else 1), ms_per_step=ms, blocks_ms_per_step=blocks, steps_per_block=k,
                   propagated_edges_per_s=units / (ms / 1000.0), parallelism=tr.parallelism(), **info)
        if mode == "shard":
            rec["capture_mode"] = tr.capture_mode
            rec["phases"] = tr.profile_phases()
            rec["collective_bytes_per_step"] = sum(p["bytes"] for p in rec["phases"] if p["kind"] == "collective")
            rec["collective_ms_per_step_eager"] = sum(p["ms"] for p in rec["phases"] if p["kind"] == "collective")
            tr.release()
        if rank == 0:
            line = json.dumps(rec)
            print(line, flush=True)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "a") as f:
                    f.write(line + "\n")
        del tr, model, optim, inter
        torch.cuda.empty_cache()
sync()
sys.stdout.flush()
os._exit(0)       # no destroy_process_group: tearing NCCL down after captured collectives hung on the box
