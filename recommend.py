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

writes recs/SPUIGACF_ml100k_010_similar10.tsv: one line `item<TAB>rank<TAB>similar_item<TAB>score` per entry.  With
--audience all|3,17,42|@file the lists are the users to show those items to (the score of the user lists, the users with any train
or test item as candidates, minus those --exclude leaves out for the item), written to ..._audience{K}.tsv as
`item<TAB>rank<TAB>user<TAB>score`; with --similar-users all|3,17,42|@file the users most similar to those users (cosine, as for
items), written to ..._similarusers{K}.tsv as `user<TAB>rank<TAB>similar_user<TAB>score`.  At most one of the three flags is given,
--users stays at its default with any of them, and --exclude too with --similar-items or --similar-users.

With --novelty-weight w (user lists only) the user lists rank by score + float32(w * novelty(item)), the item novelty of the train
split (Recommender(..., novelty_weight=w)); a positive w moves popular items down.  The scores written are those offset scores and
the default output name gains _nw{w}, e.g. recs/SPUIGACF_ml100k_010_top50_nw1.0.tsv.

With --mmr-lambda lam (user lists only, lam in [0, 1]) the user lists are diversified: the top --mmr-candidates N (default 100,
--topk..100) of each user are re-ranked by maximal marginal relevance against the cosine of the items' final features
(Recommender.diversified).  The lines keep the format, in pick order with each item's own score (so the scores are not sorted), and
the default output name gains _mmr{lam}, e.g. recs/SPUIGACF_ml100k_010_top20_mmr0.5.tsv.
"""
import os
import sys
import time

import numpy as np
import torch

import run_Gowalla as R
from ngacf_b200.cutoff_eval import check_mmr_candidates, check_mmr_lambda, check_novelty_weight
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
    p.add_argument("--audience", type=str, default=None,
                   help="rank users for these items (--exclude applies per item): all, a comma-separated id list, or @FILE")
    p.add_argument("--similar-users", type=str, default=None,
                   help="rank users like these users: all, a comma-separated id list, or @FILE")
    p.add_argument("--novelty-weight", type=float, default=0.0,
                   help="w: rank the user lists by score + w * novelty(item) (a positive w moves popular items down); 0 is the plain ranking")
    p.add_argument("--mmr-lambda", type=float, default=None,
                   help="lam in [0, 1]: diversify the user lists by maximal marginal relevance (1 keeps the ranking, 0 the least similar items)")
    p.add_argument("--mmr-candidates", type=int, default=None,
                   help="N in --topk..100: the candidates --mmr-lambda re-ranks per user (default 100)")
    p.add_argument("--out", type=str, default=None,
                   help="output TSV (default recs/{model}_{dataset}_{N:03d}_top{K}.tsv, with --similar-items ..._similar{K}.tsv, "
                        "--audience ..._audience{K}.tsv, --similar-users ..._similarusers{K}.tsv)")
    return p


# the query-list flags: (argparse dest, flag, file name tag); at most one is given
QUERY_FLAGS = (("similar_items", "--similar-items", "similar"), ("audience", "--audience", "audience"),
               ("similar_users", "--similar-users", "similarusers"))


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
    kind = next((tag for dest, _, tag in QUERY_FLAGS if getattr(args, dest) is not None), "top")
    nw = "_nw{}".format(args.novelty_weight) if args.novelty_weight != 0.0 else ""
    nw += "_mmr{}".format(args.mmr_lambda) if args.mmr_lambda is not None else ""
    return os.path.join("recs", "{}_{}_{:03d}_{}{}{}.tsv".format(args.model, args.dataset, args.resume_from, kind, args.topk, nw))


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
    given = [flag for dest, flag, _ in QUERY_FLAGS if getattr(args, dest) is not None]
    if len(given) > 1:
        raise ValueError("%s: give at most one of them" % " and ".join(given))
    args.novelty_weight = check_novelty_weight(args.novelty_weight)
    if given and args.novelty_weight != 0.0:
        raise ValueError("--novelty-weight applies to the user lists only; drop it with %s" % given[0])
    if args.mmr_lambda is not None:
        if given:
            raise ValueError("--mmr-lambda applies to the user lists only; drop it with %s" % given[0])
        try:
            args.mmr_lambda = check_mmr_lambda(args.mmr_lambda)
            args.mmr_candidates = check_mmr_candidates(100 if args.mmr_candidates is None else args.mmr_candidates, args.topk)
        except ValueError as e:
            raise ValueError("--mmr-lambda / --mmr-candidates: %s" % e) from None
    elif args.mmr_candidates is not None:
        raise ValueError("--mmr-candidates sets the candidates of --mmr-lambda; give --mmr-lambda as well")
    args.item_ids = args.audience_ids = args.similar_user_ids = None
    if args.audience is not None:
        if args.users != "eval":
            raise ValueError("--audience ranks users for items: leave --users at its default")
        args.audience_ids = parse_ids(args.audience, "--audience", ("all",))
    if args.similar_users is not None:
        if args.users != "eval" or args.exclude != "train":
            raise ValueError("--similar-users ranks users like users: leave --users and --exclude at their defaults")
        args.similar_user_ids = parse_ids(args.similar_users, "--similar-users", ("all",))
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


def query_lists(args, inter, userNum, itemNum, adj, spec, bound, flag, exclude, method, what):
    """--similar-items / --audience / --similar-users: the queries of `spec` ('all': every id in [0, bound)), ranked by
    Recommender.`method`; -> (queries int64, ids int64 (n, K), scores float32 (n, K)) as numpy arrays; writes args.out.  Ids outside
    [0, bound) are refused before the checkpoint loads; `what` % (n, K) names the lists in the report line"""
    queries = np.arange(bound, dtype=np.int64) if isinstance(spec, str) else spec
    if queries.size and (queries.min() < 0 or queries.max() >= bound):
        raise ValueError("%s: ids must lie in [0, %d)" % (flag, bound))
    rec = Recommender(load_model(args, userNum, itemNum), adj, inter, exclude)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ids, scores = getattr(rec, method)(queries, args.topk)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
    write_tsv(args.out, queries, ids, scores)
    print("recommend: %s, %.2f ms -> %s" % (what % (queries.size, args.topk), ms, args.out))
    return queries, ids, scores


def main(args):
    """-> (users int64, ids int64 (n, K), scores float32 (n, K)) as numpy arrays; writes args.out.  With --similar-items,
    --audience or --similar-users: the query ids in place of the users"""
    seed_all(args.seed)
    inter, _, _, _, userNum, itemNum, adj = R.prepareData(args)
    if args.item_ids is not None:
        return query_lists(args, inter, userNum, itemNum, adj, args.item_ids, itemNum, "--similar-items", "none", "similar_items",
                           "%d items, %d most similar")
    if args.audience_ids is not None:
        return query_lists(args, inter, userNum, itemNum, adj, args.audience_ids, itemNum, "--audience", args.exclude, "audience",
                           "%d items, audience of %d")
    if args.similar_user_ids is not None:
        return query_lists(args, inter, userNum, itemNum, adj, args.similar_user_ids, userNum, "--similar-users", "none",
                           "similar_users", "%d users, %d most similar")
    if isinstance(args.user_ids, str):
        users = inter.eval_users.long().cpu().numpy() if args.user_ids == "eval" else np.arange(userNum, dtype=np.int64)
    else:
        users = args.user_ids
        if users.size and (users.min() < 0 or users.max() >= userNum):
            raise ValueError("--users: ids must lie in [0, %d)" % userNum)
    rec = Recommender(load_model(args, userNum, itemNum), adj, inter, args.exclude)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.mmr_lambda is None:
        ids, scores = rec(users, args.topk, novelty_weight=args.novelty_weight)
    else:
        ids, scores = rec.diversified(users, args.topk, args.mmr_lambda, args.mmr_candidates, novelty_weight=args.novelty_weight)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
    write_tsv(args.out, users, ids, scores)
    nw = ", novelty weight %r" % args.novelty_weight if args.novelty_weight != 0.0 else ""
    nw += ", mmr lambda %r of %d candidates" % (args.mmr_lambda, args.mmr_candidates) if args.mmr_lambda is not None else ""
    print("recommend: %d users, top-%d%s, %.2f ms -> %s" % (users.size, args.topk, nw, ms, args.out))
    return users, ids, scores


if __name__ == "__main__":
    args = parse_args()
    os.environ["CUDA_VISIBLE_DEVICES"] = args.gpu_id
    main(args)
    sys.stdout.flush()
