"""CLI driver with the flag surface of the reference's run_Gowalla.py (:162-183) for the in-scope path
    --model SPUIGACF --adj_type ui_mat --train_mode PairSampling --eval_mode AllNeg
on the B200 kernels.  Same seeding (:191-193), checkpoint naming/format (:127-131,142-143), printed lines and
TensorBoard scalar tags (:139,149-153).  Example (the reference's README smoke test):

  python run_Gowalla.py --parallel False --gpu_id 0 --model SPUIGACF --dataset ml100k --lr 0.002 --weight_decay 0.000001 \
      --epochs 2 --droprate 0.2 --adj_type ui_mat --train_mode PairSampling --eval_mode AllNeg --eval_every 1
"""
import argparse
import ast
import math
import os
import sys
import time

import numpy as np
import torch
from torch.optim import Adam

from graphattention.BPRLoss import BPRLoss
from graphattention.SPUIGACF import SPUIGACF, SPUIMultiGACF
from ngacf_b200.data import Interactions
from ngacf_b200.hostdata import load_dataset
from train_eval_Gowalla import (diversity_report, eval_full_ranking, eval_neg_all, eval_neg_sample, list_reports, train_bpr,
                                train_neg_sample)


def prepareData(args):
    """-> train_df, test_df, train_pos_neg, test_pos_neg, userNum, itemNum, adj  (the reference's tuple; here the four
    data frames are ONE Interactions object and adj is the (2,E) index tensor of ui_mat built from ALL interactions)."""
    if args.adj_type != "ui_mat":
        raise NotImplementedError("SPUIGACF consumes --adj_type ui_mat only (run_Gowalla.py:94 passes adj.indices())")
    if (args.train_mode, args.eval_mode) not in (("PairSampling", "AllNeg"), ("NegSampling", "SampledNeg")):
        raise NotImplementedError("built: --train_mode PairSampling --eval_mode AllNeg (SURVEY.md section 8) and "
                                  "--train_mode NegSampling --eval_mode SampledNeg (8f-3), the pairs run_Gowalla.py:84-92 prepares")
    d = load_dataset(args.dataset, args.data_root, args.train_mode)
    print("userNum:{}, itemNum:{}".format(d["userNum"], d["itemNum"]))
    inter = Interactions.from_arrays(d["userNum"], d["itemNum"], d["train_u"], d["train_i"], d["test_u"], d["test_i"], device="cuda")
    adj = torch.from_numpy(np.stack([d["rt_u"], d["rt_i"]]).astype(np.int64))      # coalesced by the graph builder on the GPU
    print("lenth of traindf", len(d["train_u"]), "lenth of test_df", int(inter.eval_users.numel()) if args.eval_mode == "AllNeg" else inter.n_test_rows)
    return inter, inter, inter, inter, d["userNum"], d["itemNum"], adj


def createModels(args, userNum, itemNum):
    if args.model not in ("SPUIGACF", "SPUIMultiGACF"):
        raise NotImplementedError("--model SPUIGACF and SPUIMultiGACF are wired to the CLI.  SPUIGAGPCF exists as a class "
                                  "(graphattention.SPUIGACF.SPUIGAGPCF, needs the Laplacian as `adj`); the reference's own CLI branch "
                                  "for it reads an undefined name (run_Gowalla.py:102) and its evaluators rank 64-wide features")
    cls = SPUIGACF if args.model == "SPUIGACF" else SPUIMultiGACF
    model = cls(userNum, itemNum, embedSize=args.embedSize, layers=args.layers, droprate=args.droprate).cuda()
    lossfn = BPRLoss() if args.train_mode == "PairSampling" else torch.nn.BCEWithLogitsLoss()      # run_Gowalla.py:104-110
    optim = Adam(model.parameters(), lr=args.lr, weight_decay=args.weight_decay)
    return model, lossfn, optim


class _NullWriter:
    def add_scalar(self, *a, **k):
        pass


def _writer(args):
    comment = "_DS:{}_M:{}_E:{}_L:{}_lr:{}_wd:{}_dp:{}_rs:{}_parallel:{}".format(
        args.dataset, args.model, args.embedSize, args.layers, args.lr, args.weight_decay, args.droprate, args.seed, args.parallel)
    try:
        from torch.utils.tensorboard import SummaryWriter
        return SummaryWriter(comment=comment)
    except Exception:
        return _NullWriter()


def main(args):
    rank0 = int(os.environ.get("RANK", "0")) == 0
    summaryWriter = _writer(args) if rank0 else _NullWriter()
    train_df, test_df, train_pos_neg, test_pos_neg, userNum, itemNum, adj = prepareData(args)
    print("adj.shape", tuple(adj.shape))
    model, lossfn, optim = createModels(args, userNum, itemNum)
    os.makedirs("ckpts", exist_ok=True)
    if args.resume_from:
        checkpoint = torch.load("ckpts/{}_{}_{:03d}.pkl".format(args.model, args.dataset, args.resume_from), map_location="cuda")
        model.load_state_dict(checkpoint["model"])
        optim.load_state_dict(checkpoint["optim"])
        # the dropout stream counter resumes where the saved run stopped (one call per propagation, two per PairSampling step)
        model._call = int(checkpoint.get("dropout_calls", 0))
        print("=> loaded checkpoint '{}'".format("ckpts/{}_{:03d}.pkl".format(args.model, args.resume_from)))
    for epoch in range(args.resume_from, args.epochs):
        t0 = time.time()
        train_fn = train_bpr if args.train_mode == "PairSampling" else train_neg_sample
        train_loss = train_fn(model, args.batch_size, train_df, train_pos_neg, adj, optim, lossfn, args.parallel, epoch=epoch,
                              sample_seed=args.seed)
        summaryWriter.add_scalar("loss/train_loss", train_loss, epoch)
        print("------epoch:{}, train_loss:{:5f}, time consuming:{}s".format(epoch, train_loss, time.strftime("%H: %M: %S", time.gmtime(time.time() - t0))))
        if (epoch + 1) % args.save_every == 0 and rank0:
            # the reference's two keys (run_Gowalla.py:142-143) + the position of the dropout streams (ignored by the reference's loader)
            torch.save({"model": model.state_dict(), "optim": optim.state_dict(), "dropout_calls": int(model._call)},
                       "ckpts/{}_{}_{:03d}.pkl".format(args.model, args.dataset, epoch + 1))
        if (epoch + 1) % args.eval_every == 0:
            t0 = time.time()
            if args.eval_mode == "SampledNeg":        # run_Gowalla.py:155-160
                HR, NDCG = eval_neg_sample(model, args.batch_size, test_df, test_pos_neg, adj, 10, args.parallel, seed=args.seed)
                summaryWriter.add_scalar("metrics/HR", HR, epoch)
                summaryWriter.add_scalar("metrics/NDCG", NDCG, epoch)
                print("The time of evaluate epoch {:03d}".format(epoch) + " is: " + time.strftime("%H: %M: %S", time.gmtime(time.time() - t0)))
                print("epoch:{}, HR:{:5f}, NDCG:{:5f}".format(epoch, HR, NDCG))
                full_ranking(args, model, test_df, test_pos_neg, adj, epoch, summaryWriter, rank0)
                continue
            metrics = eval_neg_all(model, args.batch_size, test_df, test_pos_neg, adj, itemNum, args.parallel)
            print("epoch:{} metrics:{}".format(epoch, metrics))
            for i, K in enumerate([1, 5, 10, 20]):
                summaryWriter.add_scalar("metrics@{}/precision".format(K), metrics["precision"][i], epoch)
                summaryWriter.add_scalar("metrics@{}/recall".format(K), metrics["recall"][i], epoch)
                summaryWriter.add_scalar("metrics@{}/ndcg".format(K), metrics["ndcg"][i], epoch)
                summaryWriter.add_scalar("metrics@{}/hit_ratio".format(K), metrics["hit_ratio"][i], epoch)
            print("The time of evaluate epoch {:03d}".format(epoch) + " is: " + time.strftime("%H: %M: %S", time.gmtime(time.time() - t0)))
            full_ranking(args, model, test_df, test_pos_neg, adj, epoch, summaryWriter, rank0)


def full_ranking(args, model, test_df, test_pos_neg, adj, epoch, summaryWriter, rank0):
    """--eval_ks: full-ranking metrics with the standard definitions (ngacf_b200.cutoff_eval), printed by rank 0 as one line of plain
    Python values and logged as full@K/<metric>; then the same lines for the lists of each --eval_novelty_weights weight w, printed
    as `epoch:{e} novelty weight {w} ...` and logged under novelty{w}/; then those of each --eval_mmr_lambdas lambda's
    MMR-diversified lists, printed as `epoch:{e} mmr lambda {lam} ...` and logged under mmr{lam}/"""
    if not args.eval_ks:
        return
    rank_report(args, model, test_df, test_pos_neg, adj, epoch, summaryWriter, rank0, 0.0)
    for w in args.eval_novelty_weights or ():
        rank_report(args, model, test_df, test_pos_neg, adj, epoch, summaryWriter, rank0, w)
    for lam in args.eval_mmr_lambdas or ():
        rank_report(args, model, test_df, test_pos_neg, adj, epoch, summaryWriter, rank0, 0.0, lam)


def rank_report(args, model, test_df, test_pos_neg, adj, epoch, summaryWriter, rank0, w, lam=None):
    """full_ranking's lines for the lists of novelty weight w (0: the plain lists), or of MMR lambda lam (None: no re-ranking)"""
    if lam is not None:
        line, tag = "epoch:{} mmr lambda {} ".format(epoch, lam), "mmr{}/".format(lam)
    else:
        line = "epoch:{} ".format(epoch) if w == 0.0 else "epoch:{} novelty weight {} ".format(epoch, w)
        tag = "" if w == 0.0 else "novelty{}/".format(w)
    res = eval_full_ranking(model, test_df, test_pos_neg, adj, args.eval_ks, args.parallel, novelty_weight=w, mmr_lambda=lam)
    for i, K in enumerate(res["ks"]):
        for name in ("precision", "recall", "ndcg", "hit_ratio", "mrr"):
            summaryWriter.add_scalar("{}full@{}/{}".format(tag, K, name), res[name][i], epoch)
    if rank0:
        print("{}full-ranking metrics:{}".format(line, _plain(res)))
    if args.eval_beyond or args.eval_groups:
        list_lines(args, model, epoch, summaryWriter, rank0, w, lam, line, tag)
    if args.eval_diversity:
        d = diversity_report(model, novelty_weight=w, mmr_lambda=lam)
        for i, K in enumerate(d["ks"]):
            summaryWriter.add_scalar("{}diversity@{}/ild".format(tag, K), d["ild"][i], epoch)
        if rank0:
            print("{}diversity metrics:{}".format(line, _plain(d)))


def list_lines(args, model, epoch, summaryWriter, rank0, w, lam, line, tag):
    """--eval_beyond / --eval_groups: reports over the lists eval_full_ranking just ranked (every rank takes part in the all-reduce)"""
    rep = list_reports(model, args.eval_beyond, args.eval_groups, novelty_weight=w, mmr_lambda=lam)
    if rep["beyond"] is not None:
        b = rep["beyond"]
        for i, K in enumerate(b["ks"]):
            for name in ("coverage", "gini", "novelty", "arp"):
                summaryWriter.add_scalar("{}beyond@{}/{}".format(tag, K, name), b[name][i], epoch)
        if rank0:
            print("{}beyond-accuracy metrics:{}".format(line, _plain(b)))
    if rep["groups"] is not None:
        g = rep["groups"]
        for j in range(g["groups"]):
            for i, K in enumerate(g["ks"]):
                for name in ("precision", "recall", "ndcg", "hit_ratio", "mrr", "novelty", "arp"):
                    summaryWriter.add_scalar("{}group{}@{}/{}".format(tag, j, K, name), g[name][j][i], epoch)
        if rank0:
            print("{}user-group metrics:{}".format(line, _plain(g)))


def parse_novelty_weights(text):
    """'0.5,1,2' -> [0.5, 1.0, 2.0]; ValueError unless it is 1..8 distinct finite non-zero numbers"""
    try:
        ws = [float(x) for x in str(text).split(",")]
    except ValueError:
        raise ValueError("--eval_novelty_weights must be a comma-separated list of numbers, got %r" % text) from None
    if not 1 <= len(ws) <= MAX_NOVELTY_WEIGHTS:
        raise ValueError("--eval_novelty_weights takes 1..%d weights, got %d" % (MAX_NOVELTY_WEIGHTS, len(ws)))
    if not all(math.isfinite(w) and w != 0.0 for w in ws):
        raise ValueError("--eval_novelty_weights must be finite and non-zero (the plain lists are reported anyway), got %r" % text)
    if len(set(ws)) != len(ws):
        raise ValueError("--eval_novelty_weights must be distinct, got %r" % text)
    return ws


MAX_NOVELTY_WEIGHTS = 8


def parse_mmr_lambdas(text):
    """'0.5,0.8' -> [0.5, 0.8]; ValueError unless it is 1..8 distinct numbers in [0, 1)"""
    try:
        ls = [float(x) for x in str(text).split(",")]
    except ValueError:
        raise ValueError("--eval_mmr_lambdas must be a comma-separated list of numbers, got %r" % text) from None
    if not 1 <= len(ls) <= MAX_MMR_LAMBDAS:
        raise ValueError("--eval_mmr_lambdas takes 1..%d values, got %d" % (MAX_MMR_LAMBDAS, len(ls)))
    if not all(0.0 <= x < 1.0 for x in ls):
        raise ValueError("--eval_mmr_lambdas must lie in [0, 1) (1 gives the plain lists, which are reported anyway), got %r" % text)
    if len(set(ls)) != len(ls):
        raise ValueError("--eval_mmr_lambdas must be distinct, got %r" % text)
    return ls


MAX_MMR_LAMBDAS = 8


def _plain(res):
    """a metrics dict with plain Python values, for one printed line"""
    return {k: v.tolist() if hasattr(v, "tolist") else v for k, v in res.items()}


def build_parser():
    p = argparse.ArgumentParser(description="Neural Graph Attention Collaborative Filtering (B200-native SPUIGACF path)")
    p.add_argument("--dataset", type=str, default="ml100k", help="ml100k/ml1m/Gowalla/Yelp or synth-gowalla/synth-yelp2018/synth-amazon-book/synth-ml100k")
    p.add_argument("--model", type=str, default="SPUIGACF")
    p.add_argument("--adj_type", type=str, default="ui_mat")
    p.add_argument("--epochs", type=int, default=200)
    p.add_argument("--eval_every", type=int, default=10)
    p.add_argument("--save_every", type=int, default=10)
    p.add_argument("--resume_from", type=int, default=0)
    p.add_argument("--lr", type=float, default=0.001)
    p.add_argument("--weight_decay", type=float, default=0.00001)
    p.add_argument("--batch_size", type=int, default=2048)
    p.add_argument("--droprate", type=float, default=0.1)
    p.add_argument("--train_rate", type=float, default=0.7)
    p.add_argument("--seed", type=int, default=2019)
    p.add_argument("--embedSize", type=int, default=64)
    p.add_argument("--layers", type=ast.literal_eval, default=[64, 64])
    p.add_argument("--train_mode", type=str, default="NegSampling")       # the reference's defaults (run_Gowalla.py:179-180)
    p.add_argument("--eval_mode", type=str, default="SampledNeg")
    p.add_argument("--parallel", type=ast.literal_eval, default=False)
    p.add_argument("--gpu_id", type=str, default="0")
    p.add_argument("--data_root", type=str, default=None, help="directory holding 1K/u.data, Gowalla/g_train.csv, ... (default ./data)")
    p.add_argument("--eval_ks", type=str, default=None,
                   help="e.g. 20,50,100: also report full-ranking precision/recall/ndcg/hit_ratio/mrr at these cut-offs (up to 8 of 1..100) "
                        "with the standard definitions, every evaluation epoch")
    p.add_argument("--eval_beyond", type=str, default=False,
                   help="True: also report catalogue coverage, the Gini index of item exposure, novelty and average recommended popularity "
                        "of the ranked lists at the --eval_ks cut-offs")
    p.add_argument("--eval_groups", type=str, default=None,
                   help="G in 1..8: also report the --eval_ks metrics, novelty and popularity per group of users split by train degree "
                        "into G groups of about equal train interactions (NGCF section 4.3.2)")
    p.add_argument("--eval_novelty_weights", type=str, default=None,
                   help="e.g. 0.5,1,2 (1..8 distinct non-zero numbers): also rank novelty-weighted lists, by score + w * novelty(item), "
                        "and report the --eval_ks metrics (and --eval_beyond / --eval_groups) of each weight's lists")
    p.add_argument("--eval_diversity", type=str, default=False,
                   help="True: also report the intra-list diversity (mean pairwise cosine distance of the items' final features) of the "
                        "ranked lists at the --eval_ks cut-offs")
    p.add_argument("--eval_mmr_lambdas", type=str, default=None,
                   help="e.g. 0.5,0.8 (1..8 distinct values in [0, 1)): also re-rank the top 100 of each list by maximal marginal "
                        "relevance with these lambdas and report the --eval_ks metrics (and --eval_beyond / --eval_groups / "
                        "--eval_diversity) of each lambda's lists")
    return p


def parse_bool(value, flag):
    """'True' / 'False' (or a bool) -> the bool; ValueError for anything else"""
    v = value
    if isinstance(v, str):
        try:
            v = ast.literal_eval(v)
        except (ValueError, SyntaxError):
            v = None
    if not isinstance(v, bool):
        raise ValueError("%s must be True or False, got %r" % (flag, value))
    return v


def parse_args(argv=None):
    """Parses the flags and refuses unsupported combinations (ValueError) before anything is initialised -- in particular before
    --parallel True creates a process group."""
    from ngacf_b200.ops import WIDTHS
    args = build_parser().parse_args(argv)
    if args.embedSize not in WIDTHS:
        raise ValueError("--embedSize %d is not supported: the sm_100a kernels are built for embedSize %s"
                         % (args.embedSize, " and ".join(map(str, WIDTHS))))
    if args.eval_ks is not None:
        from ngacf_b200.cutoff_eval import parse_ks
        args.eval_ks = parse_ks(args.eval_ks)
    args.eval_beyond = parse_bool(args.eval_beyond, "--eval_beyond")
    args.eval_diversity = parse_bool(args.eval_diversity, "--eval_diversity")
    if args.eval_groups is not None:
        from ngacf_b200.cutoff_eval import check_groups
        try:
            G = int(args.eval_groups)
        except ValueError:
            raise ValueError("--eval_groups must be an integer in 1..8, got %r" % args.eval_groups) from None
        args.eval_groups = check_groups(G)
    if (args.eval_beyond or args.eval_groups) and not args.eval_ks:
        raise ValueError("--eval_beyond and --eval_groups report at the --eval_ks cut-offs; give --eval_ks as well")
    if args.eval_novelty_weights is not None:
        args.eval_novelty_weights = parse_novelty_weights(args.eval_novelty_weights)
        if not args.eval_ks:
            raise ValueError("--eval_novelty_weights reports at the --eval_ks cut-offs; give --eval_ks as well")
    if args.eval_diversity and not args.eval_ks:
        raise ValueError("--eval_diversity reports at the --eval_ks cut-offs; give --eval_ks as well")
    if args.eval_mmr_lambdas is not None:
        args.eval_mmr_lambdas = parse_mmr_lambdas(args.eval_mmr_lambdas)
        if not args.eval_ks:
            raise ValueError("--eval_mmr_lambdas reports at the --eval_ks cut-offs; give --eval_ks as well")
    if args.parallel and args.embedSize != 64:
        raise ValueError("--parallel True is built for --embedSize 64 only; train --embedSize %d on one GPU (--parallel False)" % args.embedSize)
    return args


def init_parallel(args):
    """--parallel True under torchrun: one process per GPU over NCCL (replaces the thread-per-GPU DataParallelModel of
    parallel.py:94-130; run_Gowalla.py:104-112).  Launch: torchrun --nproc_per_node=N run_Gowalla.py --parallel True ..."""
    if args.parallel and "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return True
    os.environ["CUDA_VISIBLE_DEVICES"] = args.gpu_id
    return False


if __name__ == "__main__":
    args = parse_args()
    print("----------------Parallel Mode is %s----------------" % ("enabled" if args.parallel else "disabled."))
    multi = init_parallel(args)
    torch.manual_seed(args.seed)
    torch.cuda.manual_seed_all(args.seed)
    np.random.seed(args.seed)
    main(args)
    if multi:
        sys.stdout.flush()
        os._exit(0)        # NCCL teardown after graph-captured collectives can hang: leave without destroy_process_group
