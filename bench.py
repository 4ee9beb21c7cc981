#!/usr/bin/env python
"""bench.py -- SPUIGACF PairSampling training step + AllNeg evaluation on synthetic Gowalla-shape data.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm (oracle port), host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + the outputs of the last timed step, DIR/<name>.npy

Exactly K steps are timed (one block, CUDA events); W >= 3 untimed steps come first.

One JSON line on stdout (rank 0).  metric/unit/config follow BASELINE.json:
  value      = propagated edges/s of the training step (steps * 2 * E / time), inputs resident in HBM,
               CUDA events, max over ranks; a "step" = sampler -> 2 propagations (independent dropout)
               -> BPR -> backward through both -> Adam (train_eval_Gowalla.py:109-139 of the reference)
  e2e        = the same through the public train_bpr-style API with the batch's train rows copied from
               pinned host memory every step and the loss read back every step
  eval       = AllNeg full-ranking users/s (device) and its own e2e (top-K lists copied to the host)
  roofline   = dominant kernel's algorithmic bytes / its live CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline = oracle port (closed-form CPU restatement) on the host cores, bounded sample
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPES = {   # SURVEY.md 8: U, I, E
    "gowalla": (29858, 40981, 1027370),
    "yelp2018": (31668, 38048, 1561406),
    "amazon-book": (52643, 91599, 2984108),
    "ml100k-shape": (943, 1682, 100000),
    "tiny": (2000, 3000, 60000),
    # BASELINE config 5: power-law scale sweep with Gowalla ratios (U = E/34.4, I = 1.37 U), SURVEY.md 8d
    "sweep-3m": (87209, 119476, 3000000),
    "sweep-10m": (290698, 398256, 10000000),
    "sweep-30m": (872093, 1194767, 30000000),
    "sweep-100m": (2906977, 3982558, 100000000),
}
HYPER = dict(lr=0.01, weight_decay=1e-6, droprate=0.2, batch=2048)   # README.md:27 of the reference


_STDOUT = sys.stdout


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def make_data(workload):
    from ngacf_b200 import hostdata
    U, I, E = SHAPES[workload]
    u, i = hostdata.synth_bipartite(U, I, E, 0)
    (tu, ti), (su, si) = hostdata.split_per_user(u, i, U, 1)
    return U, I, u, i, tu, ti, su, si


DUMP_ROWS = 65536       # --dump-outputs: larger arrays are cut to this many rows, so that the largest shapes stay under 64 MB


def write_dump(out_dir, arrays):
    """arrays: name -> numpy array, written as out_dir/<name>.npy in float32 (float64 for float64 and integer input, which holds
    ids exactly).  An array with more than DUMP_ROWS rows is cut to a fixed, seeded sample of rows (sorted), whose indices are
    written as <name>.rows.npy: the sample depends on the shape alone, so two runs with the same arguments store the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if a.ndim and a.shape[0] > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_ROWS, replace=False))
            out[name + ".rows"] = rows.astype(np.float64)
            a = a[rows]
        out[name] = a
    total = sum(a.nbytes for a in out.values())
    if total > 64 * 2 ** 20:
        raise SystemExit("--dump-outputs: %d bytes exceed the 64 MB budget" % total)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log("[bench] wrote %d arrays (%.1f MB) to %s" % (len(out), total / 2 ** 20, out_dir))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=float(p["hbm_gbs"]), bf16=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    return dict(hbm=6650.0, bf16=1400.0, source="fallback")


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name).read().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if sm:
            # "under load" = upper half of the power samples
            order = np.argsort(pw)[len(pw) // 2:]
            out.update(sm_mhz=float(np.median(np.array(sm)[order])), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=float(max(pw)))
        return out


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# --------------------------------------------------------------------------------------------------
def cpu_train_steps(workload, n_steps, warmup, budget_s, train_mode="pair"):
    import torch
    from oracle import port
    U, I, u, i, tu, ti, su, si = make_data(workload)
    torch.set_num_threads(os.cpu_count() or 1)
    g = port.build_graph(np.stack([u, i]), U, I)
    it = port.build_interactions(U, I, tu, ti, su, si)
    p = port.init_params(U, I, 2019)
    st = port.adam_init(p)
    B = HYPER["batch"]
    allpos = port.AllPositives(it) if train_mode == "neg" else None
    times = []
    t_start = time.time()
    k = 0
    while k < warmup + n_steps:
        t0 = time.time()
        lo = (k * B) % max(1, len(it.train_rows_user) - B)
        if train_mode == "neg":        # NegSampling step (8f-3): one propagation, BCE on B*5 pairs
            users, items = port.sample_negs(it, allpos, it.train_rows_user, np.asarray(ti, np.int32), lo, lo + B, 0, 0, 4, port.NEG_TAG_TRAIN)
            loss, grads, _ = port.train_neg_step_grads(p, g, users, items, port.dropout_masks(g, 0, k, HYPER["droprate"]), HYPER["droprate"])
        else:
            users, pos, neg = port.sample_pairs(it, lo, lo + B, 0, 0)
            mp = port.dropout_masks(g, 0, 2 * k, HYPER["droprate"])
            mn = port.dropout_masks(g, 0, 2 * k + 1, HYPER["droprate"])
            loss, grads, _, _ = port.train_step_grads(p, g, users, pos, neg, mp, mn, HYPER["droprate"])
        port.adam_step(p, grads, st, HYPER["lr"], HYPER["weight_decay"])
        dt = time.time() - t0
        if k >= warmup:
            times.append(dt)
        k += 1
        if time.time() - t_start > budget_s and len(times) >= 1:
            break
    return g.E, times, torch.get_num_threads()


def run_reference(args):
    """--impl reference: the reference's algorithm for this path on the CPU.  /root/reference is Python and cannot
    travel to the GPU box, so this is the oracle port (kind "port": closed-form restatement, ~16x faster than the
    reference as written, BASELINE.md section 2)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    neg = args.train_mode == "neg"
    E, times, threads = cpu_train_steps(args.workload, args.steps, min(args.warmup, 1), budget_s=150.0, train_mode=args.train_mode)
    ms = 1000.0 * float(np.mean(times))
    val = (1 if neg else 2) * E / (ms / 1000.0)
    sample = "%d of %d requested steps timed (each a full %s-shape step: %d propagation%s fwd+bwd + Adam); %d warm-up" % (
        len(times), args.steps, args.workload, 1 if neg else 2, "" if neg else "s", min(args.warmup, 1))
    line = dict(metric="spuigacf_train_propagated_edges_per_s", value=val, unit="edges/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=dict(workload=args.workload + "-shape SPUIGACF %s step" % ("NegSampling" if neg else "PairSampling"), batch=HYPER["batch"],
                            droprate=HYPER["droprate"]),
                cpu_baseline=dict(value=val, unit="edges/s", cores=threads, kind="port", sample=sample),
                e2e=dict(value=val, unit="edges/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    _STDOUT.write(json.dumps(line) + "\n")
    _STDOUT.flush()


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gowalla", choices=sorted(SHAPES))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--no-full", action="store_true", help="skip the second timing without the output-stage pruning")
    ap.add_argument("--train-mode", default="pair", choices=["pair", "neg"],
                    help="pair: PairSampling + AllNeg (the headline, SURVEY 8); neg: NegSampling + SampledNeg (8f-3, single GPU)")
    ap.add_argument("--split-bwd", action="store_true", help="dense backward as dX (on the chain) + dW/da (gradient stream)")
    ap.add_argument("--eval-mode", default="auto")
    ap.add_argument("--profile-only", action="store_true", help="run a few steps and exit (for ncu)")
    ap.add_argument("--dist", default="shard", choices=["replica", "shard"],
                    help="N>1: 'shard' = users range-partitioned, item rows all-gathered / reduce-scattered per stage (north star, strong "
                         "scaling); 'replica' = the reference's --parallel semantics (every GPU propagates the whole graph, weak scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (its loss and the updated parameters) and the last evaluation's "
                         "results to DIR/<name>.npy, to compare two builds output for output (single GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.profile_only):
        ap.error("--dump-outputs needs the timed run of this repo's CUDA path (--impl ours, no --profile-only)")
    # exactly ONE JSON line may reach stdout: anything native libraries print to fd 1 (e.g. NCCL's version banner) is
    # diverted to stderr; the JSON line is written to the saved descriptor at the end
    global _STDOUT
    sys.stdout.flush()
    _STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs is a single-GPU option")
        dist.init_process_group("nccl", device_id=dev)
    from ngacf_b200 import _lib, roofline
    from ngacf_b200.data import Interactions
    from ngacf_b200.evaluate import AllNegEvaluator
    from ngacf_b200.graph import BipartiteGraph
    from ngacf_b200.model import SPUIGACF
    from ngacf_b200.optim import FusedAdam
    from ngacf_b200.train import FusedTrainer

    W = max(args.warmup, 3)
    K = args.steps
    t0 = time.time()
    U, I, u, i, tu, ti, su, si = make_data(args.workload)
    log("[bench] synthetic %s-shape graph: U=%d I=%d E=%d (%.1fs)" % (args.workload, U, I, len(u), time.time() - t0))
    torch.manual_seed(2019)
    model = SPUIGACF(U, I, 64, [64, 64], HYPER["droprate"]).to(dev)
    adj = torch.from_numpy(np.stack([u, i])).to(dev)
    tb = time.time()
    graph = BipartiteGraph(adj, U, I)
    torch.cuda.synchronize()
    graph_build_ms = 1000 * (time.time() - tb)
    E = graph.E
    B = HYPER["batch"]
    optim = FusedAdam(model.parameters(), lr=HYPER["lr"], weight_decay=HYPER["weight_decay"])

    if world > 1 and args.train_mode == "neg":
        raise SystemExit("--train-mode neg is a single-GPU bench line (SURVEY 8f-3); the multi-GPU modes cover the PairSampling path")
    if world > 1:
        from ngacf_b200.dist import ReplicaTrainer, ShardedTrainer
        inter = Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)
        if args.dist == "shard":
            trainer = ShardedTrainer(model, inter, u, i, B, optim, sample_seed=0)
        else:
            trainer = ReplicaTrainer(model, inter, graph, B, optim, sample_seed=0)
    else:
        inter = Interactions.from_arrays(U, I, tu, ti, su, si, device=dev)
        if args.train_mode == "neg":
            from ngacf_b200.negsampling import NegSamplingTrainer
            trainer = NegSamplingTrainer(model, inter, graph, B, optim, sample_seed=0)
        else:
            trainer = FusedTrainer(model, inter, graph, B, optim, sample_seed=0, split_dense_backward=args.split_bwd)
    launches_per_step = trainer.launches_per_step(HYPER["droprate"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.profile_only:      # eager, single stream: the launch list ncu sees is the step's kernel sequence
        # ncu --profile-from-start off: only the steady-state steps (and the evaluation) between cudaProfilerStart/Stop are listed,
        # none of the one-off allocations / graph-build launches
        trainer.side = None
        for k in range(W):
            trainer._step_body(B, 0, HYPER["droprate"], model._seed(), k * B, 2 * k, False)
        ev = None
        if not args.no_eval:
            model.eval()
            ev = AllNegEvaluator(inter, args.eval_mode)
            with torch.no_grad():
                ev(model.propagate(graph))
            model.train()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for k in range(W, W + 3):
            trainer._step_body(B, 0, HYPER["droprate"], model._seed(), k * B, 2 * k, False)
        torch.cuda.synchronize()
        if ev is not None:
            model.eval()
            with torch.no_grad():
                model._eval_key = None
                ev(model.propagate(graph))
            torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return

    clocks = ClockSampler(local) if rank == 0 else None

    def timed_block(run_block):
        """One block of exactly K steps (--steps), bracketed by barrier + synchronize and timed with CUDA events (max over ranks).
        A block of ~0.1 s is noisier than a longer one: raise --steps for a steadier number."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        run_block()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---------------- device-resident timed region ----------------
    trainer.run_steps(W)
    ms_block = timed_block(lambda: trainer.run_steps(K))
    ms_step = ms_block / K
    units_per_step = trainer.units_per_step()          # propagated edges per step, all ranks
    value = units_per_step / (ms_step / 1000.0)
    if args.dump_outputs:
        # what the caller of the timed step holds after its last step: that step's loss and the updated parameters
        dumped = {"train_loss": trainer.loss.detach().reshape(1).cpu().numpy()}
        dumped.update({"param." + k: v.detach().cpu().numpy() for k, v in model.state_dict().items()})

    # ---------------- e2e: host rows in, loss out, every step ----------------
    rows_host = torch.from_numpy(np.ascontiguousarray(tu.astype(np.int32))).pin_memory()
    trainer.run_steps(2, host_rows=rows_host, read_loss=True)
    ms_e2e = timed_block(lambda: trainer.run_steps(K, host_rows=rows_host, read_loss=True))
    e2e_value = units_per_step / (ms_e2e / K / 1000.0)
    clk = clocks.stop() if clocks else {}

    # ---------------- the same step WITHOUT the output-stage pruning (N=1, PairSampling): reported next to the headline ----------------
    full_prop = None
    if world == 1 and args.train_mode == "pair" and getattr(trainer, "prune_last_stage", False) and not args.no_full:
        os.environ["NGACF_PRUNE"] = "0"
        try:
            model_f = SPUIGACF(U, I, 64, [64, 64], HYPER["droprate"]).to(dev)
            model_f.load_state_dict(model.state_dict())
            tr_f = FusedTrainer(model_f, inter, graph, B, FusedAdam(model_f.parameters(), lr=HYPER["lr"], weight_decay=HYPER["weight_decay"]),
                                sample_seed=0, split_dense_backward=args.split_bwd)
            tr_f.run_steps(W)
            bf = timed_block(lambda: tr_f.run_steps(K))
            full_prop = dict(ms_per_step=bf / K, value=units_per_step / (bf / K / 1000.0), unit="edges/s",
                             note="NGACF_PRUNE=0: the output stage is computed for every row, as the reference does (results identical up to "
                                  "the order of additions, tests/test_gpu_parity.py::test_pruned_last_stage_equals_full)")
            del tr_f, model_f
        finally:
            os.environ["NGACF_PRUNE"] = "1"

    # ---------------- per-kernel live timing (eager, one stream) -> roofline of the dominant kernel ----------------
    phases = trainer.profile_phases(5) if hasattr(trainer, "profile_phases") else None
    prof = trainer.profile_kernels(3) if phases is None else []
    hdr = {"ngacf_transform_fwd": 6, "ngacf_aggregate_fwd": 10, "ngacf_stage_bwd_prep": 4, "ngacf_stage_bwd_edges": 15, "ngacf_transform_bwd": 10,
           "ngacf_transform_bwd_dx": 7, "ngacf_transform_bwd_dw": 9, "ngacf_aggregate_fwd_active": 12, "ngacf_stage_bwd_prep_active": 8,
           "ngacf_stage_bwd_edges_active": 17}
    agg = {}
    for name, args_, ms in prof:
        key = name
        H = args_[hdr[name]] if name in hdr else 0
        if name in ("ngacf_stage_bwd_edges", "ngacf_stage_bwd_edges_active"):
            key = name + ("_users" if args_[0] == 0 else "_items")
        key = key + ("/H%d" % H if H else "")
        a = agg.setdefault(key, [0.0, 0])
        a[0] += ms
        a[1] += 1
    pk = peaks()
    n_params = sum(p.numel() for p in model.parameters())
    step_bytes = (roofline.step_bytes_compulsory(U, I, E, 2, B, 1, 5) if args.train_mode == "neg"
                  else roofline.step_bytes_compulsory(U, I, E, 2, B))
    if phases is not None:
        # partitioned step: real per-phase CUDA-event times (eager, phases back to back) and the collectives' NVLink rates
        comp = sum(p["ms"] for p in phases if p["kind"] == "compute")
        coll = [p for p in phases if p["kind"] == "collective"]
        for p in coll:      # bytes that cross NVLink per rank: (world-1)/world of the buffer for all-gather / reduce-scatter, 2x that for all-reduce
            f = 2.0 if "all-reduce" in p["name"] else 1.0
            p["nvlink_GBs_per_rank"] = f * p["bytes"] * (world - 1) / world / (p["ms"] / 1e3) / 1e9 if p["ms"] > 0 else None
        worst = max(coll, key=lambda p: p["ms"]) if coll else None
        per_gpu = step_bytes / world / (ms_step / 1e3) / 1e9
        roof = dict(bound="hbm", kernel="whole partitioned step, per GPU (the dominant KERNELS are those of the N=1 line)", achieved=per_gpu,
                    peak=pk["hbm"], unit="GB/s", frac=per_gpu / pk["hbm"], traffic=None, peak_source=pk["source"],
                    byte_model="compulsory step bytes (SURVEY 8d) / world", phases=[dict(p, ms=round(p["ms"], 4)) for p in phases],
                    compute_ms_eager=comp, collective_ms_eager=sum(p["ms"] for p in coll),
                    limiting_collective=None if worst is None else dict(name=worst["name"], us=1e3 * worst["ms"], bytes=worst["bytes"],
                                                                        nvlink_GBs_per_rank=worst["nvlink_GBs_per_rank"]),
                    step_model=dict(compulsory_bytes_per_step=step_bytes, step_ms_at_peak_one_gpu=step_bytes / (pk["hbm"] * 1e9) * 1e3))
    if phases is None:
        nsteps_prof = 3
        table = sorted(((k, v[0] / nsteps_prof, v[1] / nsteps_prof) for k, v in agg.items()), key=lambda x: -x[1])
        total_prof = sum(x[1] for x in table) if table else 0.0
        # dominant kernel = the slowest one with a fixed algorithmic-byte model (the pruned last-stage passes move a batch-dependent
        # number of bytes and are listed in `kernels` with their times only)
        top_key, top_ms_step, top_n = next(x for x in table if "_active" not in x[0])
        top_name, top_H = top_key.split("/H")[0], int(top_key.split("/H")[1]) if "/H" in top_key else 0
        n_params = sum(p.numel() for p in model.parameters())
        pk = peaks()
        gather = roofline.gather_regime(U, I) and top_name in ("ngacf_aggregate_fwd", "ngacf_stage_bwd_edges_users", "ngacf_stage_bwd_edges_items")
        top_bytes = (roofline.kernel_bytes_gather(top_name, U, I, E, top_H or 1, True) if gather
                     else roofline.kernel_bytes(top_name, U, I, E, top_H or 1, True, B, n_params))
        top_avg_ms = top_ms_step / top_n
        achieved = top_bytes / (top_avg_ms / 1000.0) / 1e9
        step_bytes = (roofline.step_bytes_compulsory(U, I, E, 2, B, 1, 5) if args.train_mode == "neg"
                      else roofline.step_bytes_compulsory(U, I, E, 2, B))
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if args.workload == "gowalla" and os.path.exists(tpath):      # DRAM bytes per launch from the committed ncu --set full capture
            traffic = json.load(open(tpath)).get(top_key, {}).get("dram_bytes_per_launch")
        roof = dict(bound="hbm", kernel=top_key, achieved=achieved, peak=pk["hbm"], unit="GB/s", frac=achieved / pk["hbm"], traffic=traffic,
                    peak_source=pk["source"], algorithmic_bytes_per_launch=top_bytes, avg_launch_ms=top_avg_ms,
                    byte_model="gather (tables > 63 MB, SURVEY 8d)" if gather else "compulsory (tables L2-resident, SURVEY 8d)",
                    share_of_step=top_ms_step / total_prof,
                    note="Gowalla-size gather tables (18 MB) are L2-resident; DRAM traffic <= algorithmic bytes (no re-reads, "
                         "profiles/ncu_traffic.json).  The gather kernels are bounded by the SM's L1TEX wavefront rate, not by L2 or HBM: a "
                         "bare 256-byte row gather of the same visits sustains 15.7 TB/s out of L2 (scripts/probe/probe_gather.cu, "
                         "profiles/r2_probe_gather.txt: ~2.4 cycles per 128-byte line per SM, L1 hits cost the same wavefronts, hot rows in "
                         "shared memory do not pay), and these kernels need 3.1-4 wavefronts per visited edge (row 2 + logit 1 + mask/edge id) "
                         "-- the compulsory byte model of SURVEY 8d cannot be reached by a kernel that must pull 2E rows through L1TEX; in the "
                         "HBM regime (sweep-10m/30m) the same kernels reach 0.9-1.06 of the measured HBM peak",
                    step_model=dict(compulsory_bytes_per_step=step_bytes, step_ms_at_peak=step_bytes / (pk["hbm"] * 1e9) * 1e3,
                                    frac_of_step_roofline=(step_bytes / (pk["hbm"] * 1e9) * 1e3) / ms_step if world == 1 else None),
                    kernels=[dict(kernel=k, ms_per_step=round(ms, 4), launches_per_step=n) for k, ms, n in table])

    # ---------------- AllNeg evaluation ----------------
    ev_out = None
    if not args.no_eval and args.train_mode == "neg":
        # SampledNeg evaluation (8f-3): 1 positive + 99 sampled negatives per test row, HR/NDCG@10, one propagation
        from ngacf_b200.negsampling import SampledNegEvaluator
        model.eval()
        sev = SampledNegEvaluator(inter, 10, 99, 0)

        def sampled_once():
            with torch.no_grad():
                model._eval_key = None
                return sev(model.propagate(graph))          # the HR/NDCG read-back is part of the call
        for _ in range(3):
            hr, nd = sampled_once()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            hr, nd = sampled_once()
        e1.record()
        torch.cuda.synchronize()
        ms_eval = e0.elapsed_time(e1) / 5
        if args.dump_outputs:
            dumped.update(eval_hr=np.array([hr], np.float64), eval_ndcg=np.array([nd], np.float64))
        ev_out = dict(metric="sampledneg_eval_rows_per_s", value=inter.n_test_rows / (ms_eval / 1000.0), unit="rows/s", ms=ms_eval,
                      rows=inter.n_test_rows, candidates_per_row=100, hr_at_10=hr, ndcg_at_10=nd,
                      e2e=dict(value=inter.n_test_rows / (ms_eval / 1000.0), unit="rows/s", d2h_bytes=16))
    elif not args.no_eval:
        model.eval()
        from ngacf_b200.dist import shard_eval_users
        ev = AllNegEvaluator(inter, args.eval_mode, users=shard_eval_users(inter.eval_users, rank, world))
        n_eval = int(inter.eval_users.numel())

        def eval_once(to_host):
            with torch.no_grad():
                model._eval_key = None            # force the propagation: it is part of the evaluation
                Z = model.propagate(graph)
                ev.rank(Z)
                res = ev.metrics()                # reads 16 sums back (the reference's result dict)
                if to_host:
                    return res, ev.top_ids.cpu()
                return res, None
        for _ in range(3):
            eval_once(False)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            res, _ = eval_once(False)
        e1.record()
        barrier()
        ms_eval = e0.elapsed_time(e1) / reps
        e0.record()
        for _ in range(reps):
            res, top_ids = eval_once(True)
        e1.record()
        barrier()
        ms_eval_e2e = e0.elapsed_time(e1) / reps
        if args.dump_outputs:
            dumped.update({"eval_" + k: np.asarray(res[k], np.float64) for k in ("precision", "recall", "ndcg", "hit_ratio")})
            dumped["eval_top_ids"] = top_ids.numpy().astype(np.float64)
        fl = roofline.eval_flops(n_eval, I)
        # live duration of the scoring entry point alone (prep + tcgen05 kernel + exact re-score), CUDA events
        _lib.PROFILE = []
        with torch.no_grad():
            ev.rank(model.propagate(graph))
        torch.cuda.synchronize()
        ev.resolve()                                          # (sets n_fallback: rank() alone leaves the flagged rows pending)
        sc_ms = [e0_.elapsed_time(e1_) for n_, a_, e0_, e1_ in _lib.PROFILE if n_.startswith("ngacf_score_topk_tc")]
        _lib.PROFILE = None
        sc_ms = float(sum(sc_ms)) if sc_ms else ms_eval
        n_local = int(ev.users.numel())
        ev_roof = dict(bound="tensor", kernel="ngacf_score_topk_tc" if ev._use_tc() else "ngacf_score_topk_exact",
                       achieved=roofline.eval_flops(n_local, I) / (sc_ms / 1000.0) / 1e12, peak=pk["bf16"], unit="TFLOP/s",
                       frac=roofline.eval_flops(n_local, I) / (sc_ms / 1000.0) / 1e12 / pk["bf16"], traffic=None, launch_ms=sc_ms,
                       note="algorithmic FLOP 2*U*I*64 (the bf16x3 split issues 3x that on the tensor pipe); K=64 makes the kernel "
                            "epilogue-bound: every accumulator is inspected once by the fused top-K (SURVEY 7 hard part 1); the chain accumulator "
                            "drained -> 12 MMAs -> accumulator full -> epilogue runs at ~2.6k cycles per 128x128 tile and CTA against 0.8k of "
                            "tensor time (DESIGN 7, scripts/probe/trace_topk.py)")
        ev_out = dict(metric="allneg_eval_users_per_s", value=n_eval / (ms_eval / 1000.0), unit="users/s", ms=ms_eval, users=n_eval,
                      e2e=dict(value=n_eval / (ms_eval_e2e / 1000.0), unit="users/s", d2h_bytes=n_eval * 20 * 4 + 128),
                      mode=("tc" if ev._use_tc() else "exact"), fallback_rows=getattr(ev, "n_fallback", 0),
                      tensor_frac_of_peak=fl / (ms_eval / 1000.0) / 1e12 / pk["bf16"],
                      recall_at_20=float(res["recall"][3]), ndcg_at_20=float(res["ndcg"][3]), roofline=ev_roof)
        model.train()

    # ---------------- CPU baseline (rank 0, N=1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        Ecpu, times, threads = cpu_train_steps(args.workload, 2, 1, budget_s=25.0, train_mode=args.train_mode)
        cpu_ms = 1000.0 * float(np.mean(times))
        cpu = dict(value=(1 if args.train_mode == "neg" else 2) * Ecpu / (cpu_ms / 1000.0), unit="edges/s", cores=threads, kind="port",
                   sample="%d full %s-shape %s training steps of the oracle port (closed form, torch CPU), 1 warm-up; %.2f s/step"
                          % (len(times), args.workload, "NegSampling" if args.train_mode == "neg" else "PairSampling", cpu_ms / 1000.0))

    if args.dump_outputs:
        write_dump(args.dump_outputs, dumped)
    if rank == 0:
        line = dict(metric="spuigacf_train_propagated_edges_per_s", value=value, unit="edges/s", n_gpus=world, steps=K, warmup=W,
                    ms_per_step=ms_step, timed_ms=ms_block,
                    higher_is_better=True, scaling="strong" if (world > 1 and args.dist == "shard") else "weak",
                    vs_baseline=None, dtype="f32",
                    data="synthetic",
                    config=dict(workload=("%s-shape SPUIGACF (U=%d I=%d E=%d d=64, 2 attention stages) " % (args.workload, U, I, E)) +
                                         ("NegSampling step: sampler (4 negatives per row) + 1 propagation (dropout %.1f) + BCE on B*5 pairs + "
                                          "backward + Adam" if args.train_mode == "neg" else
                                          "PairSampling step: sampler + 2 propagations (dropout %.1f) + BPR + backward + Adam") % HYPER["droprate"],
                                batch=B, l2="per-step working set ~%d MB > 126 MB L2, no flush" % (trainer.working_set_bytes() // 2 ** 20),
                                parallelism=trainer.parallelism(), graph_build_ms=graph_build_ms,
                                output_stage=("pruned to the batch rows (exact: the loss reads nothing else of it, SPUIGACF.py:49-52)"
                                              if getattr(trainer, "prune_last_stage", getattr(trainer, "prune", False)) else "full"),
                                full_propagation=full_prop,
                                train_rows_per_s=B / (ms_step / 1000.0) * (world if getattr(trainer, "weak", False) else 1)),
                    roofline=roof, cpu_baseline=cpu, clocks=clk,
                    e2e=dict(value=e2e_value, unit="edges/s", h2d_bytes_per_step=B * 4, d2h_bytes_per_step=4, ms_per_step=ms_e2e / K),
                    gpu_launches=launches_per_step * K, eval=ev_out)
        _STDOUT.write(json.dumps(line) + "\n")
        _STDOUT.flush()
    if world > 1:
        if hasattr(trainer, "release"):
            trainer.release()
        dist.barrier()
        sys.stderr.flush()
        os._exit(0)       # tearing NCCL down after graph-captured collectives hung on the box: leave without destroy_process_group


if __name__ == "__main__":
    main()
