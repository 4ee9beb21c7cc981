"""Multi-GPU NegSampling training and sharded SampledNeg evaluation (ngacf_b200/dist.py, train_eval_Gowalla.py).

On one GPU: the user-range partition of the NegSampling step (every rank in this process, ngacf_b200.dist.LocalCluster) equals the
single-GPU step; two data-parallel replicas run through the real torch.distributed path (two processes on the same GPU, gloo) and
equal the summed single-GPU gradients; the shards of the SampledNeg evaluation add up to the whole; the CLI's default modes with
--parallel True in one process equal --parallel False.  Without a GPU: the host logic (one-group topology, replica row ranges, test
row shards)."""
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import port

DEV = "cuda:0"


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _graph(U, I, E, seed):
    from ngacf_b200 import hostdata
    u, i = hostdata.synth_bipartite(U, I, E, seed)
    (tu, ti), (su, si) = hostdata.split_per_user(u, i, U, 1)
    return u, i, tu, ti, su, si


def _state(cls_name, U, I, droprate, seed=3):
    from ngacf_b200 import model as M
    torch.manual_seed(seed)
    ref = getattr(M, cls_name)(U, I, 64, [64, 64], droprate)
    with torch.no_grad():
        ref.uEmbd.weight.mul_(10.0)
        ref.iEmbd.weight.mul_(10.0)
    return {k: v.clone() for k, v in ref.state_dict().items()}


def _model(cls_name, U, I, droprate, sd, dev=DEV):
    from ngacf_b200 import model as M
    m = getattr(M, cls_name)(U, I, 64, [64, 64], droprate)
    m.load_state_dict(sd)
    m = m.to(dev).train()
    m.drop_seed, m._call = 77, 0
    return m


def _single(cls_name, data, sd, droprate, batch, dev=DEV):
    from ngacf_b200.data import Interactions
    from ngacf_b200.negsampling import NegSamplingTrainer
    from ngacf_b200.optim import FusedAdam
    U, I, (u, i, tu, ti, su, si) = data
    m = _model(cls_name, U, I, droprate, sd, dev)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)
    g = m.graph_for(torch.from_numpy(np.stack([u, i])).to(dev))
    tr = NegSamplingTrainer(m, dit, g, batch, FusedAdam(m.parameters(), lr=0.01, weight_decay=1e-6), sample_seed=5)
    return m, tr


# ------------------------------------------------------------------------------------------------
# CPU: host logic
# ------------------------------------------------------------------------------------------------
def test_neg_partition_is_one_group_of_world_ranks(monkeypatch):
    """One propagation per step: the NegSampling partition never takes the propagation-parallel layout, whatever
    NGACF_DIST_PROP_PARALLEL says: G = world, the sub scope is everyone, no pair scope; the ShardPlan covers every edge once."""
    from ngacf_b200.dist import ShardedNegSamplingTrainer, ShardedTrainer, ShardPlan, Topology
    monkeypatch.setenv("NGACF_DIST_PROP_PARALLEL", "1")
    assert ShardedNegSamplingTrainer.CALLS_PER_STEP == 1 and ShardedTrainer.CALLS_PER_STEP == 2
    assert not ShardedNegSamplingTrainer.PRUNABLE
    U, I, E = 300, 501, 9000
    u, i = port.synth_bipartite(U, I, E, 6)
    for world in (1, 2, 3, 4, 8):
        for r in range(world):
            t = Topology(r, world, ShardedNegSamplingTrainer.PROP_PARALLEL)
            assert not t.prop_parallel and t.G == world and t.sub_rank == r
            assert t.members("sub") == list(range(world)) and t.members("world") == list(range(world)) and t.members("pair") == [r]
        assert Topology(0, world, ShardedTrainer.PROP_PARALLEL).prop_parallel == (world % 2 == 0)      # PairSampling keeps its default
        P = ShardPlan(u, i, U, I, Topology(0, world, False).G)
        assert P.world == world and P.eb[0] == 0 and P.eb[-1] == P.E and P.ub[-1] == U
        assert sum(P.edges(r)[1] - P.edges(r)[0] for r in range(world)) == P.E


def test_neg_replica_row_ranges():
    """Replica r of a NegSampling step scores the rows [s*B*w + r*B, +B); the steps tile the train rows, and the tail step's slices
    (as FusedTrainer.train_epoch cuts them) cover the remaining rows exactly once, a rank past the end getting none."""
    from ngacf_b200.dist import NegSamplingReplicaTrainer, _ReplicaHooks, rank_rows
    assert issubclass(NegSamplingReplicaTrainer, _ReplicaHooks)
    for world, B, n in ((2, 64, 1000), (3, 50, 1000), (2, 300, 1450), (4, 7, 30)):
        stride = None
        seen = np.zeros(n, np.int32)
        seeds = set()
        n_full = None
        for r in range(world):
            h = types.SimpleNamespace(rank=r, world=world, B=B)
            off, stride = _ReplicaHooks._row_offset(h), _ReplicaHooks._row_stride(h)
            assert off == r * B and stride == B * world
            seeds.add(_ReplicaHooks._dropout_seed(h, 12345))
            n_full = n // stride
            for s in range(n_full):
                lo, hi = rank_rows(s * stride, B, r, world, n)
                assert (lo, hi) == (s * stride + off, s * stride + off + B)
                seen[lo:hi] += 1
            lo = min(n, n_full * stride + off)       # tail step
            hi = min(n, lo + B)
            seen[lo:hi] += 1
        assert (seen == 1).all()
        assert len(seeds) == world                       # every replica draws its own dropout stream
    assert _ReplicaHooks._dropout_seed(types.SimpleNamespace(rank=0, world=1, B=1), 12345) == 12345


def test_sampled_neg_test_row_shards_cpu():
    """The test rows' shards cover [0, n) once; the sampler is keyed by row, so the shards' negatives are those of the whole run
    and their metric sums add up to the whole (oracle sampler and metric)."""
    from ngacf_b200.dist import shard_range
    U, I, E = 120, 600, 3000
    u, i = port.synth_bipartite(U, I, E, 4)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 5)
    it = port.build_interactions(U, I, tu, ti, su, si)
    ap = port.AllPositives(it)
    hu, hi = np.asarray(su, np.int64), np.asarray(si, np.int64)         # the test rows (user, positive item)
    n = hu.shape[0]
    K, seed, tag = 99, 17, 2
    eu, ei = port.sample_negs(it, ap, hu, hi, 0, n, seed, 0, K, tag)
    rng = np.random.default_rng(0)
    sc = rng.standard_normal(eu.shape).astype(np.float32)
    hr, nd = port.rank_metrics(sc, 10)
    for world in (1, 2, 3, 4, 7):
        parts = [shard_range(n, r, world) for r in range(world)]
        assert parts[0][0] == 0 and parts[-1][1] == n and all(parts[k][1] == parts[k + 1][0] for k in range(world - 1))
        shr = snd = 0.0
        for lo, hi_ in parts:
            su_, si_ = port.sample_negs(it, ap, hu, hi, lo, hi_, seed, 0, K, tag)
            assert np.array_equal(su_, eu[lo:hi_]) and np.array_equal(si_, ei[lo:hi_])
            if hi_ > lo:
                a, b = port.rank_metrics(sc[lo:hi_], 10)
                shr += a * (hi_ - lo)
                snd += b * (hi_ - lo)
        assert abs(shr / n - hr) < 1e-12 and abs(snd / n - nd) < 1e-12


# ------------------------------------------------------------------------------------------------
# GPU: the partition, checked in one process
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("world,droprate,cls_name", [(2, 0.0, "SPUIGACF"), (2, 0.2, "SPUIGACF"), (3, 0.2, "SPUIGACF"), (4, 0.0, "SPUIGACF"),
                                                     (4, 0.2, "SPUIGACF"), (3, 0.2, "SPUIMultiGACF")])
def test_sharded_negsampling_equals_single_gpu(world, droprate, cls_name):
    """The NegSampling step with its one propagation user-range partitioned over `world` ranks: the same sampled batch, the loss
    within 2e-6 and EVERY gradient within 2e-5 (relative) of the single-GPU step on the same rows and dropout streams; three more
    Adam steps follow the single-GPU losses (1e-4) and weights (5e-3; 3e-2 for the three-stage model, see below).  I = 2501 is not a multiple of any world size."""
    from ngacf_b200.data import Interactions
    from ngacf_b200.dist import LocalCluster, ShardedNegSamplingTrainer, ShardPlan
    from ngacf_b200.optim import FusedAdam
    U, I, E, batch = 1500, 2501, 60000, 512
    g6 = _graph(U, I, E, 5)
    u, i, tu, ti, su, si = g6
    data = (U, I, g6)
    sd = _state(cls_name, U, I, droprate)
    model, tr = _single(cls_name, data, sd, droprate, batch)
    tr._step_body(batch, 0, droprate, model._seed(), 0, 0, False, part="compute")
    ref_pu, ref_pi = tr.pu.clone(), tr.pi.clone()
    ref_loss = float(tr.loss.item())
    ref_grads = {n: p.grad.detach().cpu().numpy().copy() for n, p in model.named_parameters()}
    model2, tr2 = _single(cls_name, data, sd, droprate, batch)
    ref_losses = tr2.run_steps(4, read_loss=True)

    plan = ShardPlan(u, i, U, I, world)
    trainers = []
    for r in range(world):
        mr = _model(cls_name, U, I, droprate, sd)
        dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
        opt = FusedAdam(mr.parameters(), lr=0.01, weight_decay=1e-6)
        trainers.append(ShardedNegSamplingTrainer(mr, dit, u, i, batch, opt, sample_seed=5, use_cuda_graph=False, transport=object(), rank=r,
                                                  world=world, plan=plan))
    assert all(t.topo.G == world and not t.topo.prop_parallel and len(t.props) == 1 for t in trainers)
    cluster = LocalCluster(trainers)
    losses = cluster.run_steps(1, read_loss=True)
    for t in trainers:
        assert torch.equal(t.pu, ref_pu) and torch.equal(t.pi, ref_pi)
    assert abs(losses[0] - ref_loss) <= 2e-6 * abs(ref_loss)
    got = cluster.gather_grads()
    for n_, gref in ref_grads.items():
        assert rel_err(got[n_].cpu().numpy(), gref) < 2e-5, n_
    assert trainers[0].model._call == 1
    losses += cluster.run_steps(3, read_loss=True)
    assert rel_err(np.array(losses), np.array(ref_losses)) < 1e-4
    sd_ref = {k: v.detach().cpu().numpy() for k, v in model2.state_dict().items()}
    sd_got = cluster.gather_state()
    # Adam moves an element by ~lr * sign(grad + wd * w) whenever that sum exceeds eps: where it lies within the last-bit difference
    # of the two summation orders, one flip moves the element by up to 2 lr.  The three-stage model has more such elements (measured
    # on a B200: 1.7e-2 on iEmbd after four steps, with every first-step gradient within 2e-5)
    tol = 5e-3 if cls_name == "SPUIGACF" else 3e-2
    for k in sd_ref:
        assert rel_err(sd_got[k].cpu().numpy(), sd_ref[k]) < tol, k


# ------------------------------------------------------------------------------------------------
# GPU: replicas through torch.distributed (two processes on the same GPU, gloo)
# ------------------------------------------------------------------------------------------------
R_U, R_I, R_E, R_DROP = 600, 2000, 24000, 0.2


def _replica_case():
    data = _graph(R_U, R_I, R_E, 2)
    n = len(data[2])
    # a batch whose epoch ends in a tail step that rank 1 has no rows of (FusedTrainer._empty_step)
    B = next(b for b in range(200, 1000) if n // (2 * b) >= 2 and 0 < n % (2 * b) < b)
    return data, B, _state("SPUIGACF", R_U, R_I, R_DROP, seed=9)


def _replica_worker(rank, world, port_no, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port_no)
    os.environ["NGACF_PARALLEL_MODE"] = "replica"
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import train_eval_Gowalla as T
    from ngacf_b200.data import Interactions
    from ngacf_b200.dist import NegSamplingReplicaTrainer
    from ngacf_b200.optim import FusedAdam
    (u, i, tu, ti, su, si), B, sd = _replica_case()
    m = _model("SPUIGACF", R_U, R_I, R_DROP, sd)
    dit = Interactions.from_arrays(R_U, R_I, tu, ti, su, si, device=DEV)
    adj = torch.from_numpy(np.stack([u, i]))
    optim = FusedAdam(m.parameters(), lr=0.01, weight_decay=1e-6)
    loss = T.train_neg_sample(m, B, dit, dit, adj, optim, torch.nn.BCEWithLogitsLoss(), True, epoch=0, sample_seed=5)
    tr = m._neg_parallel_trainer
    assert isinstance(tr, NegSamplingReplicaTrainer) and tr._graph_update is not None      # captured, all-reduce between the graphs
    hr_nd = T.eval_neg_sample(m, 512, dit, dit, adj, 10, True, seed=3)
    torch.save(dict(loss=loss, hr_nd=hr_nd, call=m._call, parallelism=tr.parallelism(),
                    sd={k: v.detach().cpu().clone() for k, v in m.state_dict().items()}), out + str(rank))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_neg_replicas_two_processes(tmp_path):
    """train_neg_sample(..., is_parallel=True) with NGACF_PARALLEL_MODE=replica in two processes: one captured epoch (full steps
    through the graphs, the gradient all-reduce between them, a tail step in which rank 1 has no rows).  The two ranks end
    bit-identical; loss and weights equal a reference that sums both ranks' single-GPU gradients per step and takes one Adam step;
    eval_neg_sample(..., is_parallel=True) returns the single-process (HR, NDCG) on both ranks."""
    import train_eval_Gowalla as T
    from ngacf_b200.data import Interactions
    from ngacf_b200.dist import _ReplicaHooks
    out = str(tmp_path / "r")
    mp.spawn(_replica_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    res = [torch.load(out + str(r), weights_only=False) for r in range(2)]
    for k in res[0]["sd"]:
        assert torch.equal(res[0]["sd"][k], res[1]["sd"][k]), k
    assert res[0]["loss"] == res[1]["loss"] and "NegSampling" in res[0]["parallelism"]

    (u, i, tu, ti, su, si), B, sd = _replica_case()
    data = (R_U, R_I, (u, i, tu, ti, su, si))
    model, tr = _single("SPUIGACF", data, sd, R_DROP, B)
    tr.use_cuda_graph = False
    n = len(tr.inter)
    stride, n_full = 2 * B, n // (2 * B)
    seeds = [_ReplicaHooks._dropout_seed(types.SimpleNamespace(rank=r, world=2, B=B), model._seed()) for r in range(2)]
    total = 0.0
    for s in range(n_full + 1):
        acc = [torch.zeros_like(p) for p in tr.params]
        for r in range(2):
            lo = min(n, s * stride + r * B)
            b = min(n, lo + B) - lo
            if b == 0:
                continue
            tr._step_body(b, 0, R_DROP, seeds[r], lo, s, False, part="compute")
            total += float(tr.loss.item())
            for a, p in zip(acc, tr.params):
                a += p.grad
        with torch.no_grad():
            for a, p in zip(acc, tr.params):
                p.grad.copy_(a)
        tr.optim.step()
    assert res[0]["call"] == n_full + 1
    assert abs(res[0]["loss"] - total / n) <= 1e-4 * abs(total / n)
    for k, v in model.state_dict().items():
        assert rel_err(res[0]["sd"][k].numpy(), v.cpu().numpy()) < 5e-3, k
    # evaluation: the single-process result on the ranks' weights
    m1 = _model("SPUIGACF", R_U, R_I, R_DROP, res[0]["sd"])
    dit = Interactions.from_arrays(R_U, R_I, tu, ti, su, si, device=DEV)
    hr, nd = T.eval_neg_sample(m1, 512, dit, dit, torch.from_numpy(np.stack([u, i])), 10, False, seed=3)
    for r in range(2):
        assert res[r]["hr_nd"][0] == hr and abs(res[r]["hr_nd"][1] - nd) < 1e-12


# ------------------------------------------------------------------------------------------------
# GPU: sharded SampledNeg evaluation in one process; the CLI
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sampled_neg_shards_add_up():
    """SampledNegEvaluator over the test-row shards of world 1..4: the negatives are those of the whole evaluation, and the shards'
    metric sums (and results) add up to the unsharded ones (HR exactly, NDCG to 1e-12)."""
    from ngacf_b200.data import Interactions
    from ngacf_b200.dist import shard_range
    from ngacf_b200.negsampling import SampledNegEvaluator
    U, I, E = 1500, 2501, 60000
    u, i, tu, ti, su, si = _graph(U, I, E, 5)
    m = _model("SPUIGACF", U, I, 0.0, _state("SPUIGACF", U, I, 0.0)).eval()
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    with torch.no_grad():
        Z = m.propagate(torch.from_numpy(np.stack([u, i])).to(DEV))
    whole = SampledNegEvaluator(dit, 10, 99, 3)
    hr, nd = whole(Z)
    s_whole = whole.metric_sums(Z).cpu().numpy().copy()
    n = dit.n_test_rows
    for world in (1, 2, 3, 4):
        sums = np.zeros(2)
        res = np.zeros(2)
        for r in range(world):
            lo, hi = shard_range(n, r, world)
            ev = SampledNegEvaluator(dit, 10, 99, 3, rows=(lo, hi))
            res += np.array(ev(Z))
            sums += ev.metric_sums(Z).cpu().numpy()
            assert torch.equal(ev.pi.reshape(hi - lo, 100), whole.pi.reshape(n, 100)[lo:hi])
        assert sums[0] == s_whole[0] and abs(sums[1] - s_whole[1]) < 1e-12 * max(1.0, abs(s_whole[1]))
        assert abs(res[0] - hr) < 1e-12 and abs(res[1] - nd) < 1e-12
    with pytest.raises(ValueError):
        SampledNegEvaluator(dit, 10, 99, 3, rows=(0, n + 1))


@pytest.mark.gpu
def test_cli_default_modes_parallel_in_one_process(tmp_path, monkeypatch, capsys):
    """run_Gowalla.main with the reference's default modes (NegSampling / SampledNeg): --parallel True in a lone process runs the
    one-GPU step and prints the same losses and HR/NDCG as --parallel False."""
    import run_Gowalla as R
    monkeypatch.chdir(tmp_path)
    flags = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--epochs", "2", "--eval_every", "1", "--save_every", "100",
             "--droprate", "0.2", "--batch_size", "2048"]

    def run(parallel):
        args = R.parse_args(flags + ["--parallel", parallel])
        assert (args.train_mode, args.eval_mode) == ("NegSampling", "SampledNeg")
        torch.manual_seed(args.seed)
        torch.cuda.manual_seed_all(args.seed)
        np.random.seed(args.seed)
        R.main(args)
        text = capsys.readouterr().out
        return [l.split(", time")[0] for l in text.splitlines() if l.startswith("------epoch:")] + \
            [l for l in text.splitlines() if l.startswith("epoch:") and "HR:" in l]
    a, b = run("False"), run("True")
    assert len(a) == 4 and a == b
