"""Top-K recommendation lists from a checkpoint of run_Gowalla.py, on one GPU.

Takes run_Gowalla.py's dataset / model flags (--dataset, --model, --embedSize, --layers, --seed, --train_mode, --data_root, ...)
and loads ckpts/{model}_{dataset}_{N:03d}.pkl given by --resume_from N.  The data are loaded under the same seeds as the
training run, so the excluded train items are that run's.  Example:

  python recommend.py --dataset ml100k --model SPUIGACF --train_mode PairSampling --eval_mode AllNeg --resume_from 10 \\
      --topk 50 --users 3,17,42 --exclude train

writes recs/SPUIGACF_ml100k_010_top50.tsv: one line `user<TAB>rank<TAB>item<TAB>score` per entry, rank 1 first, scores as %.9g
(they read back to the same fp32 value).  With --similar-items all|3,17,42|@file the lists are the items most similar to those items
(cosine of the final features, the query item left out, the item pool as candidates; --users and --exclude stay at their defaults):

  python recommend.py --dataset ml100k --model SPUIGACF --train_mode PairSampling --eval_mode AllNeg --resume_from 10 \\
      --topk 10 --similar-items 3,17,42

writes recs/SPUIGACF_ml100k_010_similar10.tsv: one line `item<TAB>rank<TAB>similar_item<TAB>score` per entry.
"""
import os
import sys
import time

import numpy as np
import torch

import run_Gowalla as R
from ngacf_b200.recommend import EXCLUDE, MAX_K, Recommender


def build_parser():
    p = R.build_parser()
    p.description = "Top-K recommendation lists from a run_Gowalla.py checkpoint (one GPU)"
    p.add_argument("--topk", type=int, default=20, help="list length K, 1..%d" % MAX_K)
    p.add_argument("--users", type=str, default="eval",
                   help="eval (the AllNeg evaluation users), all, a comma-separated id list, or @FILE with one id per line")
    p.add_argument("--exclude", type=str, default="train", help="items left out of a user's list: train, all (train and test) or none")
    p.add_argument("--similar-items", type=str, default=None,
                   help="rank items like these items instead of items for users: all, a comma-separated id list, or @FILE")
    p.add_argument("--out", type=str, default=None,
                   help="output TSV (default recs/{model}_{dataset}_{N:03d}_top{K}.tsv, with --similar-items ..._similar{K}.tsv)")
    return p


def parse_ids(spec, flag="--users", words=("eval", "all")):
    """a word of `words` stays as it is; '3,17,42' and '@file' (one id per line) give an int64 array (range checked later);
    `flag` names the option in the error"""
    if spec in words:
        return spec
    if spec.startswith("@"):
        with open(spec[1:]) as f:
            tokens = [line.strip() for line in f if line.strip()]
    else:
        tokens = [t.strip() for t in spec.split(",")]
    try:
        return np.array([int(t) for t in tokens], dtype=np.int64)
    except ValueError:
        raise ValueError("%s: %r is not %s, a comma-separated list of ids or @file" % (flag, spec, ", ".join(words))) from None


def default_out(args):
    kind = "similar" if args.similar_items is not None else "top"
    return os.path.join("recs", "{}_{}_{:03d}_{}{}.tsv".format(args.model, args.dataset, args.resume_from, kind, args.topk))


def parse_args(argv=None):
    """Parses and checks the flags (ValueError) before anything touches the GPU or creates a process group."""
    from ngacf_b200.ops import check_width
    args = build_parser().parse_args(argv)
    if args.parallel:
        raise ValueError("recommend.py runs on one GPU; drop --parallel True")
    check_width(args.embedSize)
    if not 1 <= args.topk <= MAX_K:
        raise ValueError("--topk must be in 1..%d, got %d" % (MAX_K, args.topk))
    if args.exclude not in EXCLUDE:
        raise ValueError("--exclude must be one of %s, got %r" % ("/".join(EXCLUDE), args.exclude))
    if args.resume_from < 1:
        raise ValueError("--resume_from N is required: the checkpoint ckpts/{model}_{dataset}_{N:03d}.pkl to rank with")
    args.user_ids = parse_ids(args.users)
    args.item_ids = None
    if args.similar_items is not None:
        if args.users != "eval" or args.exclude != "train":
            raise ValueError("--similar-items ranks items like items: leave --users and --exclude at their defaults")
        args.item_ids = parse_ids(args.similar_items, "--similar-items", ("all",))
    if args.out is None:
        args.out = default_out(args)
    return args


def seed_all(seed):
    """run_Gowalla.py's seeding: the ml100k train/test split draws from numpy's global RNG"""
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)
    np.random.seed(seed)


def write_tsv(path, users, ids, scores):
    d = os.path.dirname(path)
    if d:
        os.makedirs(d, exist_ok=True)
    with open(path, "w") as f:
        for u, row_i, row_s in zip(users.tolist(), ids.tolist(), scores.tolist()):
            f.writelines("%d\t%d\t%d\t%.9g\n" % (u, r + 1, i, s) for r, (i, s) in enumerate(zip(row_i, row_s)) if i >= 0)


def load_model(args, userNum, itemNum):
    path = "ckpts/{}_{}_{:03d}.pkl".format(args.model, args.dataset, args.resume_from)
    if not os.path.exists(path):
        raise FileNotFoundError("checkpoint %s not found (--resume_from %d)" % (path, args.resume_from))
    model, _, _ = R.createModels(args, userNum, itemNum)
    model.load_state_dict(torch.load(path, map_location="cuda")["model"])
    return model


def similar_items(args, inter, userNum, itemNum, adj):
    """--similar-items: -> (items int64, ids int64 (n, K), scores float32 (n, K)) as numpy arrays; writes args.out"""
    items = np.arange(itemNum, dtype=np.int64) if isinstance(args.item_ids, str) else args.item_ids
    if items.size and (items.min() < 0 or items.max() >= itemNum):
        raise ValueError("--similar-items: ids must lie in [0, %d)" % itemNum)
    rec = Recommender(load_model(args, userNum, itemNum), adj, inter, "none")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ids, scores = rec.similar_items(items, args.topk)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
    write_tsv(args.out, items, ids, scores)
    print("recommend: %d items, %d most similar, %.2f ms -> %s" % (items.size, args.topk, ms, args.out))
    return items, ids, scores


def main(args):
    """-> (users int64, ids int64 (n, K), scores float32 (n, K)) as numpy arrays; writes args.out.  With --similar-items: the query
    items in place of the users"""
    seed_all(args.seed)
    inter, _, _, _, userNum, itemNum, adj = R.prepareData(args)
    if args.item_ids is not None:
        return similar_items(args, inter, userNum, itemNum, adj)
    if isinstance(args.user_ids, str):
        users = inter.eval_users.long().cpu().numpy() if args.user_ids == "eval" else np.arange(userNum, dtype=np.int64)
    else:
        users = args.user_ids
        if users.size and (users.min() < 0 or users.max() >= userNum):
            raise ValueError("--users: ids must lie in [0, %d)" % userNum)
    rec = Recommender(load_model(args, userNum, itemNum), adj, inter, args.exclude)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ids, scores = rec(users, args.topk)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
    write_tsv(args.out, users, ids, scores)
    print("recommend: %d users, top-%d, %.2f ms -> %s" % (users.size, args.topk, ms, args.out))
    return users, ids, scores


if __name__ == "__main__":
    args = parse_args()
    os.environ["CUDA_VISIBLE_DEVICES"] = args.gpu_id
    main(args)
    sys.stdout.flush()
