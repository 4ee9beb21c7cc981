"""Full-ranking metrics at several cut-offs: ngacf_cutoff_metrics, ngacf_b200.cutoff_eval.FullRankingEvaluator,
train_eval_Gowalla.eval_full_ranking and run_Gowalla.py --eval_ks.

The oracle evaluates the definitions of ngacf_b200/cutoff_eval.py in fp64 numpy, user by user: precision h/k, recall h/|T|, NDCG
over the ideal DCG of min(|T|, k) hits, hit ratio and MRR, with the discounts 1 / np.log2(np.arange(2, K + 2))."""
import math
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DISC = 1.0 / np.log2(np.arange(2, 102))


# ------------------------------------------------------------------------------------------------
# oracle
# ------------------------------------------------------------------------------------------------
def cutoff_metrics(lists, test_sets, ks):
    """lists: (n, L) ids, -1 padded, distinct; test_sets: n arrays of test items; ks: increasing cut-offs <= L.
    -> (n, 5 len(ks)) float64, metric-major: precision at each cut-off, then recall, ndcg, hit_ratio, mrr"""
    lists = np.asarray(lists)
    nk = len(ks)
    out = np.zeros((lists.shape[0], 5 * nk))
    for j in range(lists.shape[0]):
        T = np.asarray(test_sets[j])
        hit = np.isin(lists[j], T) & (lists[j] >= 0)
        cum = np.cumsum(hit)
        first = int(np.argmax(hit)) if hit.any() else -1
        for q, k in enumerate(ks):
            h = int(cum[k - 1])
            dcg = 0.0
            for r in np.nonzero(hit[:k])[0]:        # rank order
                dcg += DISC[r]
            idcg = 0.0
            for r in range(min(T.size, k)):
                idcg += DISC[r]
            out[j, q] = h / k
            out[j, nk + q] = h / T.size if T.size else 0.0
            out[j, 2 * nk + q] = dcg / idcg if idcg > 0 else 0.0
            out[j, 3 * nk + q] = 1.0 if h > 0 else 0.0
            out[j, 4 * nk + q] = 1.0 / (first + 1) if 0 <= first < k else 0.0
    return out


def brute_force(lists, test_sets, ks):
    """the definitions, one (user, cut-off) at a time in plain Python"""
    rows = []
    for L, T in zip(np.asarray(lists).tolist(), test_sets):
        T = set(np.asarray(T).tolist())
        vals = {m: [] for m in ("p", "r", "n", "h", "m")}
        for k in ks:
            hits = [r for r in range(k) if L[r] >= 0 and L[r] in T]
            dcg = sum(1.0 / math.log2(r + 2) for r in hits)
            idcg = sum(1.0 / math.log2(r + 2) for r in range(min(len(T), k)))
            vals["p"].append(len(hits) / k)
            vals["r"].append(len(hits) / len(T))
            vals["n"].append(dcg / idcg)
            vals["h"].append(1.0 if hits else 0.0)
            vals["m"].append(1.0 / (hits[0] + 1) if hits else 0.0)
        rows.append(sum(vals.values(), []))
    return np.array(rows)


def synthetic_lists(rng, n, K_list, I=2000, max_test=300):
    """n users with 1..max_test test items (some larger than K_list) and distinct-id lists of K_list that draw about half their
    entries from the test set; some lists end in -1 padding, one is all padding"""
    test_sets, lists = [], np.full((n, K_list), -1, np.int64)
    for j in range(n):
        nt = int(rng.integers(1, max_test + 1)) if j % 4 else int(rng.integers(K_list, max_test + 1))
        T = np.sort(rng.choice(I, nt, replace=False))
        test_sets.append(T)
        length = K_list if j % 3 else int(rng.integers(0, K_list + 1))
        if j == 5:
            length = 0
        pool_hit = rng.permutation(T)
        pool_miss = rng.permutation(np.setdiff1d(np.arange(I), T))
        take_hit = min(int(rng.binomial(length, 0.5)), pool_hit.size)
        ids = np.concatenate([pool_hit[:take_hit], pool_miss[:length - take_hit]])
        lists[j, :length] = rng.permutation(ids)
    return lists, test_sets


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_oracle_equals_brute_force():
    rng = np.random.default_rng(0)
    for K_list, ks in ((100, [1, 3, 20, 37, 100]), (37, [1, 2, 36, 37]), (1, [1])):
        lists, tests = synthetic_lists(rng, 60, K_list)
        assert max(t.size for t in tests) > K_list and (lists == -1).any()
        np.testing.assert_allclose(cutoff_metrics(lists, tests, ks), brute_force(lists, tests, ks), rtol=1e-13, atol=0)


def test_oracle_shares_precision_recall_hit_ratio_with_reference_format():
    rng = np.random.default_rng(1)
    lists, tests = synthetic_lists(rng, 80, 20)
    ks = [1, 5, 10, 20]
    rows = cutoff_metrics(lists, tests, ks)
    for j in range(len(tests)):
        r = (np.isin(lists[j], tests[j]) & (lists[j] >= 0)).astype(np.float64)
        ref = port.metrics_from_hits(r, tests[j].size)
        np.testing.assert_allclose(rows[j, 0:4], ref["precision"], rtol=1e-15, atol=0)
        np.testing.assert_allclose(rows[j, 4:8], ref["recall"], rtol=1e-15, atol=0)
        np.testing.assert_array_equal(rows[j, 12:16], ref["hit_ratio"])


def test_ndcg_is_one_for_an_ideal_list_and_never_above():
    rng = np.random.default_rng(2)
    ks = [1, 3, 20, 37, 100]
    lists, tests = synthetic_lists(rng, 100, 100)
    assert (cutoff_metrics(lists, tests, ks)[:, 10:15] <= 1.0 + 1e-15).all()
    for j, T in enumerate(tests):           # the first min(|T|, 100) entries are hits
        m = min(T.size, 100)
        lists[j, :m] = rng.permutation(T)[:m]
        lists[j, m:] = -1
    nd = cutoff_metrics(lists, tests, ks)[:, 10:15]
    np.testing.assert_allclose(nd, 1.0, rtol=1e-15)


def test_discount_table_is_numpys():
    src = open(os.path.join(ROOT, "ngacf_b200", "csrc", "cutoff_metrics.cu")).read()
    body = src[src.index("c_cut_disc[NGACF_RECOMMEND_MAX_K] = {"):]
    body = body[:body.index("};")]
    vals = [float.fromhex(x) for x in re.findall(r"0x[0-9a-f.]+p[+-]\d+", body)]
    assert np.array_equal(np.array(vals), DISC)


def test_cut_off_validation_without_cuda():
    from ngacf_b200 import _lib
    from ngacf_b200.cutoff_eval import FullRankingEvaluator, check_ks, parse_ks
    assert check_ks([100, 20, 50, 20]) == [20, 50, 100] and check_ks([np.int64(7)]) == [7]
    for bad in ([], [0], [101], [1, 2, 3, 4, 5, 6, 7, 8, 9], [2.0], [True], ["5"]):
        with pytest.raises(ValueError):
            check_ks(bad)
        with pytest.raises(ValueError):
            FullRankingEvaluator(None, bad)      # refused before the interactions are touched
    assert parse_ks("100, 20,50") == [20, 50, 100]
    for bad in ("", "a", "2.5", "20,,50", "0", "101"):
        with pytest.raises(ValueError):
            parse_ks(bad)
    with pytest.raises(ValueError, match="mode"):
        FullRankingEvaluator(None, [20], mode="fast")
    with pytest.raises(_lib.NgacfError, match="top-20"):
        FullRankingEvaluator(None, [10, 50], mode="tc")


def test_cli_eval_ks_parsing(monkeypatch):
    import run_Gowalla as R
    import torch.distributed as dist
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    assert R.parse_args([]).eval_ks is None
    assert R.parse_args(["--eval_ks", "100,20,50,20"]).eval_ks == [20, 50, 100]
    assert R.parse_args(["--eval_ks", "10"]).eval_ks == [10]
    for bad in ("", "0", "101", "x", "2.5", "1,2,3,4,5,6,7,8,9"):
        with pytest.raises(ValueError):
            R.parse_args(["--parallel", "True", "--eval_ks", bad])
    assert not dist.is_initialized()


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _device_case(lists, tests):
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.int32).to(DEV).contiguous()
    ptr = np.concatenate([[0], np.cumsum([x.size for x in tests])])
    inter = SimpleNamespace(test_ptr=t(ptr), test_items=t(np.concatenate(tests)))
    return t(lists), t(np.arange(len(tests))), inter


def _run(ids, users, inter, ks, per_user=True):
    from ngacf_b200 import ops
    n = users.numel()
    sums = torch.full((5 * len(ks),), -7.0, dtype=torch.float64, device=DEV)
    rows = torch.full((n, 5 * len(ks)), -7.0, dtype=torch.float64, device=DEV) if per_user else None
    ws = torch.empty(ops.cutoff_metrics_workspace_bytes(n, len(ks)), dtype=torch.uint8, device=DEV)
    ops.cutoff_metrics(ids, users, inter, ks, sums, rows, ws)
    return sums, rows


def _close(got, ref):
    got = got.cpu().numpy() if torch.is_tensor(got) else np.asarray(got)
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-300)


@gpu
@pytest.mark.parametrize("K_list", [1, 20, 37, 100])
def test_kernel_matches_oracle_on_synthetic_lists(K_list):
    rng = np.random.default_rng(K_list)
    lists, tests = synthetic_lists(rng, 1000, K_list)
    ids, users, inter = _device_case(lists, tests)
    for n_ks in range(1, 9):
        ks = sorted(rng.choice(np.arange(1, K_list + 1), min(n_ks, K_list), replace=False).tolist())
        if n_ks == 1:
            ks = [K_list]
        ref = cutoff_metrics(lists, tests, ks)
        sums, rows = _run(ids, users, inter, ks)
        _close(rows, ref)
        _close(sums, ref.sum(0))
        if K_list == 1:
            break


@gpu
def test_c_abi_edges():
    from ngacf_b200 import _lib, ops
    lib = _lib.load()
    rng = np.random.default_rng(7)
    lists, tests = synthetic_lists(rng, 333, 100)
    ids, users, inter = _device_case(lists, tests)
    ks = [1, 10, 20, 50, 100]
    ref = cutoff_metrics(lists, tests, ks)
    n = users.numel()
    need = ops.cutoff_metrics_workspace_bytes(n, len(ks))
    ws = torch.full((need + 4096,), 0xAB, dtype=torch.uint8, device=DEV)
    sums = torch.full((5 * len(ks),), -7.0, dtype=torch.float64, device=DEV)

    def call(K_list=100, k=ks, nbytes=need, sums_p=sums.data_ptr(), per_user=None):
        ka = (__import__("ctypes").c_int32 * max(len(k), 1))(*k)
        return lib.ngacf_cutoff_metrics(ids.data_ptr(), K_list, users.data_ptr(), n, inter.test_ptr.data_ptr(), inter.test_items.data_ptr(),
                                        ka, len(k), sums_p, per_user, ws.data_ptr(), nbytes, ops._s())
    for kw, what in (({"K_list": 0}, b"list length 0"), ({"K_list": 101}, b"list length 101"), ({"k": []}, b"0 cut-offs"),
                     ({"k": list(range(1, 10))}, b"9 cut-offs"), ({"k": [5, 5]}, b"strictly increasing"),
                     ({"k": [10, 5]}, b"strictly increasing"), ({"k": [0, 5]}, b"strictly increasing"),
                     ({"K_list": 50, "k": [20, 100]}, b"1..50")):
        assert call(**kw) == -4 and what in lib.ngacf_last_error(), kw
    with pytest.raises(_lib.NgacfError, match="strictly increasing"):
        ops.cutoff_metrics(ids, users, inter, [20, 10], sums, None, ws)
    assert call(sums_p=None) == -1
    assert call(nbytes=need - 1) == -3 and b"workspace" in lib.ngacf_last_error()
    torch.cuda.synchronize()
    assert bool((ws == 0xAB).all()) and bool((sums == -7.0).all()), "a refused call wrote"
    # per_user NULL
    assert call() == 0
    torch.cuda.synchronize()
    assert bool((ws[need:] == 0xAB).all()), "ngacf_cutoff_metrics wrote past its reported workspace"
    _close(sums, ref.sum(0))
    s1, r1 = _run(ids, users, inter, ks)
    s2, r2 = _run(ids, users, inter, ks)
    assert torch.equal(s1, sums) and torch.equal(s1, s2) and torch.equal(r1, r2)
    # captured in a CUDA graph, replayed twice: the eager call's bits
    gs = torch.zeros_like(sums)
    rows = torch.zeros((n, 5 * len(ks)), dtype=torch.float64, device=DEV)
    gws = torch.empty(need, dtype=torch.uint8, device=DEV)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ops.cutoff_metrics(ids, users, inter, ks, gs, rows, gws)
    torch.cuda.current_stream().wait_stream(st)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.cutoff_metrics(ids, users, inter, ks, gs, rows, gws)
    for _ in range(2):
        gs.fill_(-1.0)
        rows.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(gs, s1) and torch.equal(rows, r1)
    # no users: zero sums
    empty = torch.empty(0, dtype=torch.int32, device=DEV)
    s0, _ = _run(ids, empty, inter, ks, per_user=False)
    assert bool((s0 == 0).all())


def _seeded_model(cls, U, I, width, seed=5):
    torch.manual_seed(seed)
    m = cls(U, I, width, [64, 64], 0.1).to(DEV)
    with torch.no_grad():            # larger embeddings than the N(0, 0.01) init, so that the scores spread
        m.uEmbd.weight.mul_(30)
        m.iEmbd.weight.mul_(30)
    return m


@pytest.fixture(scope="module")
def trained_case():
    """a split of a synthetic graph, its port interactions and seeded models' pre-ELU outputs at both widths"""
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    U, I, E = 300, 900, 9000
    u, i = port.synth_bipartite(U, I, E, 21)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 22)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    it = port.build_interactions(U, I, tu, ti, su, si)
    adj = torch.from_numpy(np.stack([u, i])).to(DEV)
    Z = {}
    for key, cls, width in (("64", SPUIGACF, 64), ("128", SPUIGACF, 128), ("multi64", SPUIMultiGACF, 64)):
        model = _seeded_model(cls, U, I, width).eval()
        with torch.no_grad():
            Z[key] = model.propagate(adj).clone()
    return SimpleNamespace(U=U, I=I, dit=dit, it=it, Z=Z)


def _oracle_for(case, Z, ks):
    """port.topk_allneg lists of every evaluated user from the final features, and the oracle rows at ks"""
    from ngacf_b200 import ops
    F = torch.empty_like(Z)
    ops.final_features(Z, F)
    F = F.cpu().numpy()
    it = case.it
    users = case.dit.eval_users.cpu().numpy()
    Fi = F[case.U:]
    K = max(ks)
    lists = np.full((users.size, K), -1, np.int64)
    tests = []
    for j, u in enumerate(users):
        top = port.topk_allneg(port.dot64_tree(np.broadcast_to(F[u], Fi.shape), Fi), it, int(u), K)
        lists[j, :top.size] = top
        tests.append(it.test_items[it.test_ptr[u]:it.test_ptr[u + 1]])
    return lists, cutoff_metrics(lists, tests, ks)


@gpu
@pytest.mark.parametrize("key,ks", [("64", [20]), ("64", [5, 50, 100]), ("128", [20]), ("128", [5, 50, 100]), ("multi64", [10, 37])])
def test_evaluator_matches_oracle(trained_case, key, ks):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    case = trained_case
    ref_lists, ref_rows = _oracle_for(case, case.Z[key], ks)
    ev = FullRankingEvaluator(case.dit, ks)
    res = ev(case.Z[key])
    assert ev.source == ("tc" if key != "128" and max(ks) <= 20 else "list")
    got = ev.top_ids.cpu().numpy()[:, :max(ks)]
    assert np.array_equal(got, ref_lists)
    _close(ev.per_user(), ref_rows)
    n = ref_rows.shape[0]
    assert res["n_users"] == n and res["ks"] == ks
    nk = len(ks)
    for q, name in enumerate(("precision", "recall", "ndcg", "hit_ratio", "mrr")):
        _close(res[name], ref_rows[:, q * nk:(q + 1) * nk].sum(0) / n)


@gpu
def test_both_sources_give_the_same_rows(trained_case):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    case = trained_case
    for ks in ([1, 5, 10, 20], [3, 7]):
        a = FullRankingEvaluator(case.dit, ks, "auto")
        b = FullRankingEvaluator(case.dit, ks, "exact")
        a.rank(case.Z["64"])
        b.rank(case.Z["64"])
        assert a.source == "tc" and b.source == "list" and b.top_ids.shape[1] == max(ks)
        assert torch.equal(a.per_user(), b.per_user())
    from ngacf_b200 import _lib
    with pytest.raises(_lib.NgacfError, match="64-wide"):
        FullRankingEvaluator(case.dit, [20], "tc").rank(case.Z["128"])


@gpu
def test_sums_equal_the_allneg_evaluators(trained_case):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    from ngacf_b200.evaluate import AllNegEvaluator
    case = trained_case
    for key in ("64", "128"):
        for mode in ("auto", "exact"):
            ae = AllNegEvaluator(case.dit, mode)
            ae(case.Z[key])
            ref = ae.sums.cpu().numpy()
            fe = FullRankingEvaluator(case.dit, [1, 5, 10, 20], mode)
            fe.rank(case.Z[key])
            s = fe.per_user().sum(0).cpu().numpy()
            for a, b in ((0, 0), (4, 4), (12, 12)):          # precision, recall, hit_ratio; the divisors differ, so the sums
                _close(s[a:a + 4], ref[b:b + 4])


@gpu
def test_shards_add_up_to_the_whole(trained_case):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    from ngacf_b200.dist import shard_eval_users
    case = trained_case
    for ks in ([5, 20], [5, 50, 100]):
        whole = FullRankingEvaluator(case.dit, ks)
        res = whole(case.Z["64"])
        rows = whole.per_user().clone()
        parts, total, n = [], 0.0, 0
        for r in range(3):
            ev = FullRankingEvaluator(case.dit, ks, users=shard_eval_users(case.dit.eval_users, r, 3))
            m = ev(case.Z["64"])
            parts.append(ev.per_user().clone())
            total = total + np.concatenate([m[k] for k in ("precision", "recall", "ndcg", "hit_ratio", "mrr")]) * m["n_users"]
            n += m["n_users"]
        assert n == res["n_users"] and torch.equal(torch.cat(parts), rows)
        _close(total / n, np.concatenate([res[k] for k in ("precision", "recall", "ndcg", "hit_ratio", "mrr")]))


def _cli_lines(R, flags, capsys):
    args = R.parse_args(flags)
    torch.manual_seed(args.seed)
    torch.cuda.manual_seed_all(args.seed)
    np.random.seed(args.seed)
    R.main(args)
    out = capsys.readouterr().out
    # wall-clock times vary between runs
    keep = [l.split(", time")[0] for l in out.splitlines() if "time of evaluate" not in l and "timeStamp" not in l]
    return keep


@gpu
def test_cli_eval_ks(tmp_path, monkeypatch, capsys):
    import ast
    import run_Gowalla as R
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--epochs", "1", "--eval_every", "1", "--save_every", "1",
            "--droprate", "0.2", "--batch_size", "2048"]
    allneg = base + ["--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--lr", "0.002", "--parallel", "False"]
    plain = _cli_lines(R, allneg, capsys)
    assert not any("full-ranking" in l for l in plain)
    withks = _cli_lines(R, allneg + ["--eval_ks", "100,5,50"], capsys)
    new = [l for l in withks if "full-ranking" in l]
    assert len(new) == 1 and [l for l in withks if "full-ranking" not in l] == plain
    assert withks.index(new[0]) == len(withks) - 1
    printed = ast.literal_eval(new[0].split("full-ranking metrics:", 1)[1])
    assert new[0].startswith("epoch:0 full-ranking metrics:") and printed["ks"] == [5, 50, 100]
    # the Python evaluator on the saved model
    args = R.parse_args(allneg)
    inter, _, _, _, U, I, adj = R.prepareData(args)
    model, _, _ = R.createModels(args, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    model.eval()
    with torch.no_grad():
        res = FullRankingEvaluator(inter, [5, 50, 100])(model.propagate(adj.to(DEV)))
    assert printed["n_users"] == res["n_users"] == int(inter.eval_users.numel())
    for k in ("precision", "recall", "ndcg", "hit_ratio", "mrr"):
        _close(printed[k], res[k])
    capsys.readouterr()          # prepareData's own lines are not part of the runs below
    # the default modes (NegSampling / SampledNeg): the line follows the HR line, --parallel True in one process prints the same
    neg = base + ["--eval_ks", "20"]
    a = _cli_lines(R, neg + ["--parallel", "False"], capsys)
    b = _cli_lines(R, neg + ["--parallel", "True"], capsys)
    assert a == b
    i = [j for j, l in enumerate(a) if "full-ranking" in l]
    assert len(i) == 1 and "HR:" in a[i[0] - 1]
