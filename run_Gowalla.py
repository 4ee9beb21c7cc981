"""CLI driver with the flag surface of the reference's run_Gowalla.py (:162-183) for the in-scope path
    --model SPUIGACF --adj_type ui_mat --train_mode PairSampling --eval_mode AllNeg
on the B200 kernels.  Same seeding (:191-193), checkpoint naming/format (:127-131,142-143), printed lines and
TensorBoard scalar tags (:139,149-153).  Example (the reference's README smoke test):

  python run_Gowalla.py --parallel False --gpu_id 0 --model SPUIGACF --dataset ml100k --lr 0.002 --weight_decay 0.000001 \
      --epochs 2 --droprate 0.2 --adj_type ui_mat --train_mode PairSampling --eval_mode AllNeg --eval_every 1
"""
import argparse
import ast
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
from train_eval_Gowalla import eval_neg_all, eval_neg_sample, train_bpr, train_neg_sample


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
                continue
            metrics = eval_neg_all(model, args.batch_size, test_df, test_pos_neg, adj, itemNum, args.parallel)
            print("epoch:{} metrics:{}".format(epoch, metrics))
            for i, K in enumerate([1, 5, 10, 20]):
                summaryWriter.add_scalar("metrics@{}/precision".format(K), metrics["precision"][i], epoch)
                summaryWriter.add_scalar("metrics@{}/recall".format(K), metrics["recall"][i], epoch)
                summaryWriter.add_scalar("metrics@{}/ndcg".format(K), metrics["ndcg"][i], epoch)
                summaryWriter.add_scalar("metrics@{}/hit_ratio".format(K), metrics["hit_ratio"][i], epoch)
            print("The time of evaluate epoch {:03d}".format(epoch) + " is: " + time.strftime("%H: %M: %S", time.gmtime(time.time() - t0)))


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
    return p


def parse_args(argv=None):
    """Parses the flags and refuses unsupported combinations (ValueError) before anything is initialised -- in particular before
    --parallel True creates a process group."""
    from ngacf_b200.ops import WIDTHS
    args = build_parser().parse_args(argv)
    if args.embedSize not in WIDTHS:
        raise ValueError("--embedSize %d is not supported: the sm_100a kernels are built for embedSize %s"
                         % (args.embedSize, " and ".join(map(str, WIDTHS))))
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
