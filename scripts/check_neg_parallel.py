"""torchrun check (N GPUs) of the multi-GPU NegSampling step, NGACF_PARALLEL_MODE = shard (default) or replica:

  shard   : ngacf_b200.dist.ShardedNegSamplingTrainer over NCCL == the single-GPU NegSampling step on every rank (same batches, same
            Philox dropout streams; losses to 1e-4, weights to 5e-3); the tables are identical on all ranks after sync_embeddings();
  replica : ngacf_b200.dist.NegSamplingReplicaTrainer; the replicas stay bit-identical and the step losses are finite.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 scripts/check_neg_parallel.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ngacf_b200 import hostdata  # noqa: E402
from ngacf_b200.data import Interactions  # noqa: E402
from ngacf_b200.dist import NegSamplingReplicaTrainer, ShardedNegSamplingTrainer  # noqa: E402
from ngacf_b200.model import SPUIGACF  # noqa: E402
from ngacf_b200.negsampling import NegSamplingTrainer  # noqa: E402
from ngacf_b200.optim import FusedAdam  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
mode = os.environ.get("NGACF_PARALLEL_MODE", "shard")


def say(*a):
    print("[rank %d]" % rank, *a, flush=True)


U, I, E, B = 3000, 5001, 200000, 1024
drop = float(os.environ.get("NGACF_DROP", "0.2"))
u, i = hostdata.synth_bipartite(U, I, E, 2)
(tu, ti), (su, si) = hostdata.split_per_user(u, i, U, 3)
torch.manual_seed(7)
ref = SPUIGACF(U, I, 64, [64, 64], drop)
with torch.no_grad():
    ref.uEmbd.weight.mul_(10.0)
    ref.iEmbd.weight.mul_(10.0)
sd = {k: v.clone() for k, v in ref.state_dict().items()}


def make():
    m = SPUIGACF(U, I, 64, [64, 64], drop)
    m.load_state_dict(sd)
    m = m.to(dev).train()
    m.drop_seed, m._call = 99, 0
    return m, Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)


model, inter = make()
optim = FusedAdam(model.parameters(), lr=0.01, weight_decay=1e-6)
steps = 6
if mode == "replica":
    g = model.graph_for(torch.from_numpy(np.stack([u, i])).to(dev))
    tr = NegSamplingReplicaTrainer(model, inter, g, B, optim, sample_seed=5)
    losses = tr.run_steps(steps, read_loss=True)
    capture = "one CUDA graph per part, gradient all-reduce between them" if tr._graph_update is not None else "one CUDA graph"
else:
    tr = ShardedNegSamplingTrainer(model, inter, u, i, B, optim, sample_seed=5)
    say("users [%d,%d) items [%d,%d) edges [%d,%d)" % (tr.u_lo, tr.u_hi, tr.i_lo, tr.i_hi, tr.e_lo, tr.e_hi))
    losses = tr.run_steps(steps, read_loss=True)
    tr.sync_embeddings()
    capture = tr.capture_mode
torch.cuda.synchronize()
say("mode %s, capture mode: %s, losses %s" % (mode, capture, ["%.6f" % x for x in losses]))
flat = torch.cat([q.detach().reshape(-1) for q in model.parameters()])
mx, mn_ = flat.clone(), flat.clone()
dist.all_reduce(mx, op=dist.ReduceOp.MAX)
dist.all_reduce(mn_, op=dist.ReduceOp.MIN)
same = bool(torch.equal(mx, mn_))
if mode == "replica":
    ok = same and bool(np.isfinite(losses).all())
    say("replica check: world=%d ok=%s | replicas bit-identical: %s" % (world, ok, same))
else:
    # single-GPU reference on every rank (cheap at this size)
    m1, it1 = make()
    g1 = m1.graph_for(torch.from_numpy(np.stack([u, i])).to(dev))
    t1 = NegSamplingTrainer(m1, it1, g1, B, FusedAdam(m1.parameters(), lr=0.01, weight_decay=1e-6), sample_seed=5)
    ref_losses = t1.run_steps(steps, read_loss=True)
    worst = 0.0
    for (k, a), (_, b) in zip(model.state_dict().items(), m1.state_dict().items()):
        a, b = a.double(), b.double()
        worst = max(worst, float((a - b).abs().max() / (b.abs().max() + 1e-30)))
    loss_err = float(np.max(np.abs(np.array(losses) - np.array(ref_losses)) / np.abs(ref_losses)))
    ok = loss_err < 1e-4 and worst < 5e-3 and same
    say("sharded NegSampling check: world=%d ok=%s | losses vs 1-GPU max rel %.2e | worst param rel err %.2e | tables identical on all "
        "ranks after sync: %s" % (world, ok, loss_err, worst, same))
    tr.release()
dist.barrier()
say("leaving")
sys.stdout.flush()
os._exit(0 if ok else 1)       # no destroy_process_group: tearing NCCL down after captured collectives hung on the box
