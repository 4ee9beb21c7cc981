"""Intra-list diversity and MMR-diversified lists: ngacf_list_diversity, ngacf_mmr_rerank, FullRankingEvaluator.diversity_metrics /
mmr_lambda, Recommender.diversified / list_diversity, train_eval_Gowalla.eval_full_ranking(mmr_lambda=) / diversity_report,
run_Gowalla.py --eval_diversity / --eval_mmr_lambdas and recommend.py --mmr-lambda.

The oracle computes sim(x, y) = (dot64_tree(F[U+x], F[U+y]) * rn(x)) * rn(y) in numpy float32 (each operation rounds to nearest, as
the __f*_rn intrinsics do), with rn the tree's norm as item_rnorm_kernel computes it; ILD sums in Python floats (IEEE fp64) in the
specified order, and MMR's arithmetic is numpy float32 scalars, so both reproduce the kernels bit for bit."""
import ast
import ctypes
import itertools
import math

import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu
METRICS = ("precision", "recall", "ndcg", "hit_ratio", "mrr")


# ------------------------------------------------------------------------------------------------
# oracle
# ------------------------------------------------------------------------------------------------
def rnorm(F, U, ids):
    """float32 rn of the item rows F[U + ids]: 1 / sqrt(tree sum of squares), 0 when that sum is not > 0"""
    R = np.asarray(F, np.float32)[U + np.asarray(ids, np.int64)]
    s = port.dot64_tree(R, R)
    out = np.zeros(len(s), np.float32)
    pos = s > 0
    out[pos] = np.float32(1.0) / np.sqrt(s[pos])
    return out


def sim_matrix(F, U, ids):
    """(m, m) float32: entry [a, b] = sim(ids[min(a, b)], ids[max(a, b)]) (the lower position first); the diagonal is unused"""
    ids = np.asarray(ids, np.int64)
    R = np.asarray(F, np.float32)[U + ids]
    rn = rnorm(F, U, ids)
    dots = port.dot64_tree(R[:, None, :], R[None, :, :]) if ids.size else np.zeros((0, 0), np.float32)
    upper = ((dots * rn[:, None]).astype(np.float32) * rn[None, :]).astype(np.float32)
    return np.where(np.triu(np.ones_like(upper, bool), 1), upper, upper.T)


def valid(row, I):
    return [int(i) for i in row if 0 <= int(i) < I]


def ild_row(F, U, I, row, ks):
    """ILD at each cut-off of one list, in the specified fp64 order"""
    out = []
    for k in ks:
        v = valid(list(row)[:k], I)
        m = len(v)
        if m < 2:
            out.append(0.0)
            continue
        S = sim_matrix(F, U, v)
        num = 0.0
        for b in range(1, m):
            r = 0.0
            for a in range(b):
                r += 1.0 - float(S[a, b])
            num += r
        out.append(num / (m * (m - 1) // 2))
    return out


def ild_rows(F, U, I, rows, ks):
    return np.array([ild_row(F, U, I, r, ks) for r in np.asarray(rows)], np.float64).reshape(len(rows), len(ks))


def mmr_row(F, U, I, ids, scores, K, lam):
    """MMR picks of one candidate row -> (ids int64 (K,), scores float32 (K,)), -1 / 0.0 padded"""
    pos = [c for c, i in enumerate(ids) if 0 <= int(i) < I]
    cid = np.asarray([int(ids[c]) for c in pos], np.int64)
    s = np.asarray([scores[c] for c in pos], np.float32)
    m = len(pos)
    out_i, out_s = np.full(K, -1, np.int64), np.zeros(K, np.float32)
    if m == 0:
        return out_i, out_s
    S = sim_matrix(F, U, cid)
    with np.errstate(all="ignore"):            # non-finite scores: NaN values, ranked below every number
        smax, smin = np.fmax.reduce(s), np.fmin.reduce(s)          # NaN scores skipped, as fmaxf / fminf do
        rel = ((s - smin) / (smax - smin)).astype(np.float32) if smax > smin else np.zeros(m, np.float32)
        lam32 = np.float32(lam)
        oml = np.float32(1.0) - lam32
        mx = np.zeros(m, np.float32)
        picked = np.zeros(m, bool)
        for step in range(min(K, m)):
            v = ((lam32 * rel).astype(np.float32) - (oml * mx).astype(np.float32)).astype(np.float32)
            open_ = np.flatnonzero(~picked)
            num = open_[~np.isnan(v[open_])]          # NaN values rank below every number
            p = int(num[np.argmax(v[num])]) if num.size else int(open_[0])   # first maximum: ties to the lower position
            picked[p] = True
            out_i[step], out_s[step] = cid[p], s[p]
            mx = S[p].copy() if step == 0 else np.fmax(mx, S[p])
    return out_i, out_s


def mmr_rows(F, U, I, ids, scores, K, lam):
    res = [mmr_row(F, U, I, a, b, K, lam) for a, b in zip(np.asarray(ids), np.asarray(scores))]
    return np.stack([r[0] for r in res]).reshape(-1, K), np.stack([r[1] for r in res]).reshape(-1, K)


def bits(t):
    return np.asarray(t.cpu().numpy() if torch.is_tensor(t) else t, np.float32).view(np.int32)


def _close(got, ref):
    np.testing.assert_allclose(np.asarray(got, np.float64), np.asarray(ref, np.float64), rtol=1e-12, atol=1e-300)


def random_features(rng, U, I, W):
    """random rows with all-zero items (rn = 0) and groups of duplicated items (sim ~ 1)"""
    F = rng.standard_normal((U + I, W)).astype(np.float32)
    F[U + 10:U + 20] = 0.0
    F[U + 40:U + 60] = F[U + 40]
    F[U + 70:U + 75] = F[U + 76]
    return F


def random_lists(rng, n, L, I):
    """lists of distinct ids mostly, with -1 padding, out-of-range ids, zero and duplicated item rows"""
    rows = np.stack([rng.choice(I, L, replace=False) if L <= I else rng.integers(0, I, L) for _ in range(n)]).astype(np.int64)
    for j in range(n):
        kind = j % 6
        if kind == 1:
            rows[j, rng.integers(0, L, max(1, L // 4))] = -1
        elif kind == 2:
            rows[j, rng.integers(0, L, max(1, L // 5))] = rng.choice([I, I + 7, -5, 1 << 30], max(1, L // 5))
        elif kind == 3:
            rows[j, :min(L, 12)] = np.arange(40, 40 + min(L, 12))          # duplicated rows
        elif kind == 4:
            rows[j, :min(L, 8)] = np.arange(8, 8 + min(L, 8))              # items 10..: zero rows
        elif kind == 5 and L > 3:
            rows[j, L // 2:] = -1                                          # a padded tail
    rows[0] = -1                                                            # nothing valid
    if n > 7:
        rows[7, 1:] = -1                                                    # one valid entry
    return rows


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_ild_oracle_matches_brute_force():
    rng = np.random.default_rng(1)
    U, I, W = 5, 200, 64
    F = random_features(rng, U, I, W)
    rows = random_lists(rng, 12, 37, I)
    ks = [1, 2, 5, 20, 37]
    got = ild_rows(F, U, I, rows, ks)
    for j, row in enumerate(rows):
        for q, k in enumerate(ks):
            v = valid(row[:k], I)
            pairs = list(itertools.combinations(range(len(v)), 2))
            if not pairs:
                assert got[j, q] == 0.0
                continue
            rn = rnorm(F, U, v)
            R = F[U + np.asarray(v)]
            terms = []
            for a, b in pairs:
                d = port.dot64_tree(R[a], R[b])
                terms.append(1.0 - float(np.float32(np.float32(d * rn[a]) * rn[b])))
            np.testing.assert_allclose(got[j, q], math.fsum(terms) / len(pairs), rtol=1e-12, atol=1e-15)


def test_mmr_oracle_matches_a_plain_greedy_loop():
    rng = np.random.default_rng(2)
    U, I, W = 5, 300, 64
    F = random_features(rng, U, I, W)
    for trial in range(30):
        N = int(rng.integers(1, 41))
        ids = random_lists(rng, 8, N, I)[trial % 8]
        sc = np.sort(rng.standard_normal(N).astype(np.float32))[::-1].copy()
        if trial % 5 == 0:
            sc[:] = 1.5                                                     # all equal: rel = 0
        for K in sorted({1, min(5, N), N}):
            for lam in (0.0, 0.3, 0.5, 1.0):
                oi, os_ = mmr_row(F, U, I, ids, sc, K, lam)
                # plain loop: Python lists, float32 scalars, a scan for the best (mmr, position)
                cand = [(c, int(ids[c]), np.float32(sc[c])) for c in range(N) if 0 <= ids[c] < I]
                s_list = [x[2] for x in cand]
                lo, hi = (min(s_list), max(s_list)) if cand else (0, 0)
                l32 = np.float32(lam)
                om = np.float32(1) - l32
                sel, mx = [], {}
                while len(sel) < min(K, len(cand)):
                    best = None
                    for pos, (c, i, s) in enumerate(cand):
                        if pos in sel:
                            continue
                        r = np.float32((s - lo) / (hi - lo)) if hi > lo else np.float32(0)
                        v = np.float32(l32 * r) - np.float32(om * mx.get(pos, np.float32(0)))
                        if best is None or v > best[0]:
                            best = (v, pos)
                    p = best[1]
                    sel.append(p)
                    for pos, (c, i, s) in enumerate(cand):
                        a, b = min(pos, p), max(pos, p)
                        if a == b:
                            continue
                        ia, ib = cand[a][1], cand[b][1]
                        rn = rnorm(F, U, [ia, ib])
                        sv = np.float32(np.float32(port.dot64_tree(F[U + ia], F[U + ib]) * rn[0]) * rn[1])
                        mx[pos] = sv if pos not in mx else max(mx[pos], sv)
                ref_i = [cand[p][1] for p in sel] + [-1] * (K - len(sel))
                ref_s = [cand[p][2] for p in sel] + [np.float32(0)] * (K - len(sel))
                assert oi.tolist() == ref_i, (trial, K, lam)
                assert np.array_equal(bits(os_), bits(np.asarray(ref_s, np.float32)))
                if lam == 1.0:
                    assert oi[:len(sel)].tolist() == [x[1] for x in cand][:len(sel)]


def test_python_and_cli_refusals(monkeypatch):
    import recommend as RC
    import run_Gowalla as R
    import torch.distributed as dist
    from ngacf_b200 import _lib
    from ngacf_b200.cutoff_eval import FullRankingEvaluator, check_mmr_candidates, check_mmr_lambda
    from ngacf_b200.data import Interactions
    from ngacf_b200.recommend import Recommender
    assert check_mmr_lambda(0) == 0.0 and check_mmr_lambda(1) == 1.0 and check_mmr_lambda(np.float32(0.5)) == 0.5
    for bad in (float("nan"), -0.1, 1.01, float("inf"), "0.5", None, True):
        with pytest.raises(ValueError, match="lambda"):
            check_mmr_lambda(bad)
    assert check_mmr_candidates(20, 20) == 20 and check_mmr_candidates(100, 1) == 100
    for bad in (19, 101, 50.0, True):
        with pytest.raises(ValueError, match="candidates"):
            check_mmr_candidates(bad, 20)
    it = Interactions.from_arrays(20, 30, np.arange(20) % 20, np.arange(20) % 30, np.arange(20), (np.arange(20) + 5) % 30, device="cpu")
    with pytest.raises(_lib.NgacfError, match="MMR"):
        FullRankingEvaluator(it, [10, 20], "tc", mmr_lambda=0.5)
    for bad in (float("nan"), -0.5, 2.0):
        with pytest.raises(ValueError, match="lambda"):
            FullRankingEvaluator(it, [20], "exact", mmr_lambda=bad)
    for bad in (10, 101):
        with pytest.raises(ValueError, match="candidates"):
            FullRankingEvaluator(it, [5, 20], "exact", mmr_lambda=0.5, mmr_candidates=bad)
    rec = Recommender.__new__(Recommender)
    rec.inter = None
    for kw in (dict(mmr_lambda=float("nan")), dict(mmr_lambda=1.5), dict(candidates=10), dict(candidates=101)):
        with pytest.raises(ValueError):
            rec.diversified([0], 20, **kw)
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    a = R.parse_args([])
    assert a.eval_diversity is False and a.eval_mmr_lambdas is None
    a = R.parse_args(["--eval_ks", "20", "--eval_diversity", "True", "--eval_mmr_lambdas", "0.5,0,0.8"])
    assert a.eval_diversity is True and a.eval_mmr_lambdas == [0.5, 0.0, 0.8]
    with pytest.raises(ValueError, match="--eval_diversity"):
        R.parse_args(["--parallel", "True", "--eval_diversity", "True"])
    with pytest.raises(ValueError, match="--eval_diversity"):
        R.parse_args(["--eval_ks", "20", "--eval_diversity", "yes"])
    for bad in (["--eval_mmr_lambdas", "0.5"], ["--eval_ks", "20", "--eval_mmr_lambdas", "1"],
                ["--eval_ks", "20", "--eval_mmr_lambdas", "0.5,1.0"], ["--eval_ks", "20", "--eval_mmr_lambdas", "-0.1"],
                ["--eval_ks", "20", "--eval_mmr_lambdas", "nan"], ["--eval_ks", "20", "--eval_mmr_lambdas", "0.5,0.5"],
                ["--eval_ks", "20", "--eval_mmr_lambdas", "x"], ["--eval_ks", "20", "--eval_mmr_lambdas", ""],
                ["--eval_ks", "20", "--eval_mmr_lambdas", ",".join(str(x / 10) for x in range(9))]):
        with pytest.raises(ValueError, match="--eval_mmr_lambdas"):
            R.parse_args(["--parallel", "True"] + bad)
    assert not dist.is_initialized()
    base = ["--resume_from", "7"]
    a = RC.parse_args(base + ["--mmr-lambda", "0.5"])
    assert a.mmr_lambda == 0.5 and a.mmr_candidates == 100 and a.out == "recs/SPUIGACF_ml100k_007_top20_mmr0.5.tsv"
    assert RC.parse_args(base + ["--mmr-lambda", "0.3", "--mmr-candidates", "20"]).mmr_candidates == 20
    assert RC.parse_args(base).mmr_lambda is None
    for bad in (["--mmr-lambda", "1.5"], ["--mmr-lambda", "nan"], ["--mmr-lambda", "0.5", "--mmr-candidates", "10"],
                ["--mmr-lambda", "0.5", "--mmr-candidates", "101"], ["--mmr-candidates", "50"],
                ["--mmr-lambda", "0.5", "--similar-items", "3"]):
        with pytest.raises(ValueError, match="--mmr"):
            RC.parse_args(base + bad)


# ------------------------------------------------------------------------------------------------
# GPU: the C-ABI against the oracle
# ------------------------------------------------------------------------------------------------
def _dev(a, dt=torch.int32):
    return torch.as_tensor(np.asarray(a)).to(dt).to(DEV)


def _ild(Ft, U, I, rows, ks):
    from ngacf_b200 import ops
    t = _dev(rows)
    out = torch.full((t.shape[0], len(ks)), 7.0, dtype=torch.float64, device=DEV)
    ops.list_diversity(Ft, U, I, t, ks, out)
    return out.cpu().numpy()


def _mmr(Ft, U, I, ids, sc, K, lam):
    from ngacf_b200 import ops
    ci, cs = _dev(ids), _dev(sc, torch.float32)
    oi = torch.full((ci.shape[0], K), 7, dtype=torch.int32, device=DEV)
    os_ = torch.full((ci.shape[0], K), 7.0, dtype=torch.float32, device=DEV)
    ops.mmr_rerank(Ft, U, I, ci, cs, K, lam, oi, os_)
    return oi.cpu().numpy().astype(np.int64), os_.cpu().numpy()


@pytest.fixture(scope="module")
def kernel_case():
    U, I = 7, 600
    rng = np.random.default_rng(11)
    out = dict(U=U, I=I)
    for W in (64, 128):
        F = random_features(rng, U, I, W)
        out[W] = dict(F=F, Ft=torch.from_numpy(F).to(DEV))
    return out


@gpu
@pytest.mark.parametrize("W", [64, 128])
def test_list_diversity_matches_the_oracle(kernel_case, W):
    c = kernel_case
    U, I, F, Ft = c["U"], c["I"], c[W]["F"], c[W]["Ft"]
    rng = np.random.default_rng(W)
    for L, kss in ((1, [[1]]), (20, [[20], [1, 2, 10, 20]]), (37, [[3, 37], [1, 5, 9, 13, 17, 21, 30, 37]]), (100, [[100], [10, 20, 50, 100]])):
        rows = random_lists(rng, 24, L, I)
        for ks in kss:
            got = _ild(Ft, U, I, rows, ks)
            ref = ild_rows(F, U, I, rows, ks)
            assert np.array_equal(got.view(np.int64), ref.view(np.int64)), (L, ks)
    # a two-entry list is 1 - the similar-item score of its first entry's query
    from ngacf_b200 import ops
    q = torch.tensor([3, 45, 200], dtype=torch.int32, device=DEV)
    ti, ts = torch.empty((3, 1), dtype=torch.int32, device=DEV), torch.empty((3, 1), dtype=torch.float32, device=DEV)
    ws = torch.empty(ops.similar_items_topk_workspace_bytes(W, I, 3, 1), dtype=torch.uint8, device=DEV)
    ops.similar_items_topk(Ft, U, I, q, 1, None, ti, ts, ws)
    pairs = np.stack([q.cpu().numpy(), ti[:, 0].cpu().numpy()], 1)
    got = _ild(Ft, U, I, pairs, [2])
    assert got[:, 0].tolist() == [1.0 - float(s) for s in ts[:, 0].cpu().numpy()]


@gpu
@pytest.mark.parametrize("W", [64, 128])
def test_mmr_rerank_matches_the_oracle(kernel_case, W):
    c = kernel_case
    U, I, F, Ft = c["U"], c["I"], c[W]["F"], c[W]["Ft"]
    rng = np.random.default_rng(100 + W)
    for N in (1, 20, 37, 100):
        ids = random_lists(rng, 18, N, I)
        sc = -np.sort(-rng.standard_normal((18, N)).astype(np.float32), axis=1)
        sc[1] = 0.25                                            # all equal: rel = 0
        sc[3, : N // 2] = sc[3, 0]                              # tied scores over duplicated rows: tied MMR values
        sc[4] = np.round(sc[4])
        for K in sorted({1, min(20, N), N}):
            for lam in (0.0, 0.3, 0.5, 1.0):
                gi, gs = _mmr(Ft, U, I, ids, sc, K, lam)
                ri, rs = mmr_rows(F, U, I, ids, sc, K, lam)
                assert np.array_equal(gi, ri), (N, K, lam)
                assert np.array_equal(bits(gs), bits(rs)), (N, K, lam)
                if lam == 1.0:                                  # the first K valid candidates, in order
                    for j in range(ids.shape[0]):
                        v = [(int(i), s) for i, s in zip(ids[j], sc[j]) if 0 <= i < I][:K]
                        assert gi[j, :len(v)].tolist() == [x[0] for x in v]
                        assert (gi[j, len(v):] == -1).all() and (gs[j, len(v):] == 0).all()
        perm = rng.permutation(ids.shape[0])                    # a row does not depend on the other rows of the call
        a = _mmr(Ft, U, I, ids, sc, min(20, N), 0.5)
        b = _mmr(Ft, U, I, ids[perm], sc[perm], min(20, N), 0.5)
        assert np.array_equal(a[0][perm], b[0]) and np.array_equal(bits(a[1][perm]), bits(b[1]))


@gpu
@pytest.mark.parametrize("W", [64, 128])
def test_mmr_rerank_non_finite_values(kernel_case, W):
    """scores spanning more than FLT_MAX (rel = inf / inf = NaN for the top one), NaN and infinite scores, NaN features: every row
    still picks each valid candidate once, in the oracle's order (NaN values rank below every number)"""
    c = kernel_case
    U, I = c["U"], c["I"]
    F = c[W]["F"].copy()
    F[U + 300] = np.nan                                         # NaN similarities to item 300
    Ft = torch.from_numpy(F).to(DEV)
    rng = np.random.default_rng(7)
    N = 37
    ids = np.stack([rng.choice(np.arange(200, 400), N, replace=False) for _ in range(6)]).astype(np.int64)
    ids[:, 5] = 300
    sc = -np.sort(-rng.standard_normal((6, N)).astype(np.float32), axis=1)
    sc[0, 0], sc[0, -1] = 3e38, -3e38
    sc[1, :] = np.float32(np.linspace(3e38, -3e38, N))
    sc[2, 3] = np.nan
    sc[3, 0], sc[3, 1] = np.inf, -np.inf
    sc[4, :] = np.nan
    ids[5, 10:] = -1
    for K in (N, 20, 1):
        for lam in (0.0, 0.5, 1.0):
            gi, gs = _mmr(Ft, U, I, ids, sc, K, lam)
            ri, rs = mmr_rows(F, U, I, ids, sc, K, lam)
            assert np.array_equal(gi, ri), (K, lam)
            assert np.array_equal(bits(gs), bits(rs)), (K, lam)
            if K == N:
                for j in range(ids.shape[0]):
                    v = sorted(i for i in ids[j] if 0 <= i < I)
                    assert sorted(gi[j, :len(v)].tolist()) == v and (gi[j, len(v):] == -1).all()


@gpu
def test_c_abi_refusals_and_graph_replay(kernel_case):
    from ngacf_b200 import _lib, ops
    lib = _lib.load()
    c = kernel_case
    U, I, W, F, Ft = c["U"], c["I"], 64, c[64]["F"], c[64]["Ft"]
    rng = np.random.default_rng(5)
    rows = _dev(random_lists(rng, 300, 100, I))
    sc = _dev(-np.sort(-rng.standard_normal((300, 100)).astype(np.float32), axis=1), torch.float32)
    out = torch.full((300, 3), 7.0, dtype=torch.float64, device=DEV)
    oi = torch.full((300, 20), 7, dtype=torch.int32, device=DEV)
    os_ = torch.full((300, 20), 7.0, dtype=torch.float32, device=DEV)
    s = ops._s()

    def ild(width=W, K_list=100, ks=(20, 50, 100), n=300, ids=rows.data_ptr(), r=out.data_ptr(), f=Ft.data_ptr()):
        ka = (ctypes.c_int32 * len(ks))(*ks) if ks is not None else None
        return lib.ngacf_list_diversity(f, width, U, I, ids, K_list, n, ka, len(ks) if ks is not None else 1, r, s)

    def mmr(width=W, N=100, K=20, lam=0.5, n=300, ids=rows.data_ptr(), o=oi.data_ptr()):
        return lib.ngacf_mmr_rerank(Ft.data_ptr(), width, U, I, ids, sc.data_ptr(), n, N, K, lam, o, os_.data_ptr(), s)
    for call, kw, code, what in ((ild, dict(width=96), -4, b"width 96"), (ild, dict(K_list=0), -4, b"list length 0"),
                                 (ild, dict(K_list=101), -4, b"list length 101"), (ild, dict(ks=()), -4, b"0 cut-offs"),
                                 (ild, dict(ks=tuple(range(1, 10))), -4, b"9 cut-offs"), (ild, dict(ks=(20, 20)), -4, b"cut-offs"),
                                 (ild, dict(ks=(50, 101)), -4, b"cut-offs"), (ild, dict(ks=None), -1, b"cut-off array"),
                                 (ild, dict(ids=None), -1, b"null"), (ild, dict(r=None), -1, b"null"), (ild, dict(f=None), -1, b"null"),
                                 (mmr, dict(width=32), -4, b"width 32"), (mmr, dict(N=0), -4, b"N = 0"), (mmr, dict(N=101), -4, b"N = 101"),
                                 (mmr, dict(K=0), -4, b"K = 0"), (mmr, dict(K=101), -4, b"K = 101"), (mmr, dict(N=10, K=20), -4, b"K = 20"),
                                 (mmr, dict(lam=float("nan")), -1, b"lambda"), (mmr, dict(lam=-0.01), -1, b"lambda"),
                                 (mmr, dict(lam=1.01), -1, b"lambda"), (mmr, dict(ids=None), -1, b"null"), (mmr, dict(o=None), -1, b"null")):
        assert call(**kw) == code and what in lib.ngacf_last_error(), (kw, lib.ngacf_last_error())
    assert ild(n=0) == 0 and mmr(n=0) == 0
    torch.cuda.synchronize()
    assert bool((out == 7.0).all()) and bool((oi == 7).all()) and bool((os_ == 7.0).all()), "a refused call wrote"
    with pytest.raises(_lib.NgacfError, match="lambda"):
        ops.mmr_rerank(Ft, U, I, rows, sc, 20, 1.5, oi, os_)
    with pytest.raises(_lib.NgacfError, match="CUDA"):
        ops.list_diversity(torch.from_numpy(F), U, I, rows, [20], out[:, :1])
    # captured in a CUDA graph and replayed
    ops.list_diversity(Ft, U, I, rows, [20, 50, 100], out)
    ops.mmr_rerank(Ft, U, I, rows, sc, 20, 0.5, oi, os_)
    gd, gi, gs = torch.zeros_like(out), torch.zeros_like(oi), torch.zeros_like(os_)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        ops.list_diversity(Ft, U, I, rows, [20, 50, 100], gd)
        ops.mmr_rerank(Ft, U, I, rows, sc, 20, 0.5, gi, gs)
    torch.cuda.current_stream().wait_stream(st)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.list_diversity(Ft, U, I, rows, [20, 50, 100], gd)
        ops.mmr_rerank(Ft, U, I, rows, sc, 20, 0.5, gi, gs)
    gd.zero_()
    gi.zero_()
    gs.zero_()
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(gd.view(torch.int64), out.view(torch.int64)) and torch.equal(gi, oi)
    assert torch.equal(gs.view(torch.int32), os_.view(torch.int32))
    assert np.array_equal(out[:20].cpu().numpy(), ild_rows(F, U, I, rows[:20].cpu().numpy(), [20, 50, 100]))


# ------------------------------------------------------------------------------------------------
# GPU: FullRankingEvaluator, Recommender, the call sites and the CLIs
# ------------------------------------------------------------------------------------------------
def _seeded_model(cls, U, I, width, seed=5):
    torch.manual_seed(seed)
    m = cls(U, I, width, [64, 64], 0.1).to(DEV)
    with torch.no_grad():
        m.uEmbd.weight.mul_(30)
        m.iEmbd.weight.mul_(30)
    return m


@pytest.fixture(scope="module")
def trained_case():
    """a split of a synthetic graph with a pool that leaves items out, and seeded models' pre-ELU outputs"""
    from types import SimpleNamespace
    from ngacf_b200.data import Interactions
    from ngacf_b200.model import SPUIGACF, SPUIMultiGACF
    U, I, E = 400, 1100, 14000
    u, i = port.synth_bipartite(U, I - 10, E, 31)
    (tu, ti), (su, si) = port.split_train_test(u, i, U, 32)
    dit = Interactions.from_arrays(U, I, tu, ti, su, si, device=DEV)
    adj = torch.from_numpy(np.stack([u, i])).to(DEV)
    models, Z = {}, {}
    for key, cls, width in (("64", SPUIGACF, 64), ("128", SPUIGACF, 128), ("multi64", SPUIMultiGACF, 64)):
        models[key] = _seeded_model(cls, U, I, width).eval()
        with torch.no_grad():
            Z[key] = models[key].propagate(adj).clone()
    return SimpleNamespace(U=U, I=I, dit=dit, adj=adj, models=models, Z=Z)


def _features(Z):
    from ngacf_b200 import ops
    F = torch.empty_like(Z)
    ops.final_features(Z, F)
    return F


def _oracle_candidates(case, F, users, N, exclude_sets):
    """exact top-N lists (ids, scores) by the dot64_tree score, item pool minus the user's excluded items"""
    h = case.dit.host
    in_pool = np.zeros(case.I, bool)
    in_pool[h["pool"]] = True
    items = F[case.U:]
    ids = np.full((len(users), N), -1, np.int64)
    sc = np.zeros((len(users), N), np.float32)
    for r, u in enumerate(users):
        s = port.dot64_tree(np.broadcast_to(F[u], items.shape), items)
        cand = in_pool.copy()
        cand[list(exclude_sets.get(int(u), ()))] = False
        c = np.nonzero(cand)[0]
        order = np.lexsort((c, -s[c].astype(np.float64)))[:N]
        ids[r, :order.size], sc[r, :order.size] = c[order], s[c][order]
    return ids, sc


def _train_sets(dit, users):
    h = dit.host
    return {int(u): set(h["train_items"][h["train_ptr"][u]:h["train_ptr"][u + 1]].tolist()) for u in users}


@gpu
@pytest.mark.parametrize("key,ks", [("64", [5, 20, 50]), ("128", [1, 37, 100]), ("multi64", [10, 20])])
def test_evaluator_diversity_matches_the_oracle(trained_case, key, ks):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    F = _features(c.Z[key]).cpu().numpy()
    ev = FullRankingEvaluator(c.dit, ks, "exact")
    ev.rank(c.Z[key])
    d = ev.diversity_metrics()
    n = c.dit.eval_users.numel()
    ref = ild_rows(F, c.U, c.I, ev.top_ids[:n].cpu().numpy(), ks)
    assert np.array_equal(ev._div_rows.cpu().numpy().view(np.int64), ref.view(np.int64))
    assert d["ks"] == ks and d["n_users"] == n
    _close(d["ild"], ref.sum(0) / n)
    if max(ks) <= 20 and key != "128":          # the tcgen05 lists give the same dict
        tc = FullRankingEvaluator(c.dit, ks, "tc")
        tc.rank(c.Z[key])
        assert tc.source == "tc"
        dt = tc.diversity_metrics()
        assert dt["ks"] == d["ks"] and dt["n_users"] == d["n_users"] and np.array_equal(dt["ild"], d["ild"])


@gpu
def test_shards_give_the_unsharded_sums(trained_case):
    import ngacf_b200.dist as D
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    it = c.dit
    ks = [5, 50, 100]
    whole = FullRankingEvaluator(it, ks, mmr_lambda=0.5)
    whole.rank(c.Z["64"])
    ref = whole.diversity_metrics()
    for world in range(1, 5):
        evs = [FullRankingEvaluator(it, ks, users=D.shard_eval_users(it.eval_users, r, world), mmr_lambda=0.5) for r in range(world)]
        for ev in evs:
            ev.rank(c.Z["64"])
            ev.diversity_metrics()
        assert torch.equal(torch.cat([ev.top_ids[:ev.users.numel()] for ev in evs]), whole.top_ids[:it.eval_users.numel()])
        assert torch.equal(torch.cat([ev._div_rows for ev in evs]), whole._div_rows)
        _close(sum(ev._gsums[:len(ks)] for ev in evs).cpu().numpy(), ref["ild"] * ref["n_users"])


@gpu
@pytest.mark.parametrize("key", ["64", "128"])
def test_mmr_evaluator_lists(trained_case, key):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    n = c.dit.eval_users.numel()
    for ks in ([10, 20], [5, 50, 100]):
        plain = FullRankingEvaluator(c.dit, ks, "exact")
        one = FullRankingEvaluator(c.dit, ks, mmr_lambda=1.0, mmr_candidates=100)
        rp, r1 = plain(c.Z[key]), one(c.Z[key])
        assert one.source == "mmr" and torch.equal(one.top_ids[:n], plain.top_ids[:n])
        for k in rp:
            assert np.array_equal(np.asarray(rp[k]), np.asarray(r1[k]))
        lp, l1 = plain.list_metrics(), one.list_metrics()
        for k in lp:
            assert np.array_equal(np.asarray(lp[k]), np.asarray(l1[k]))
    F = _features(c.Z[key]).cpu().numpy()
    users = c.dit.eval_users.cpu().numpy()
    sel = np.arange(0, users.size, 7)
    for N, w in ((100, 0.0), (30, 0.0), (60, 1.0)):
        ev = FullRankingEvaluator(c.dit, [10, 20], mmr_lambda=0.5, mmr_candidates=N, novelty_weight=w)
        ev.rank(c.Z[key])
        cand = _oracle_candidates(c, F, users[sel], N, _train_sets(c.dit, users[sel])) if w == 0.0 else None
        if cand is None:                        # novelty offsets: the candidates are the offset lists, checked in test_novelty_ranking
            ci, cs = ev._cand_ids[sel].cpu().numpy(), ev._cand_scores[sel].cpu().numpy()
        else:
            ci, cs = cand
            assert np.array_equal(ev._cand_ids[sel].cpu().numpy(), ci)
        ri, _ = mmr_rows(F, c.U, c.I, ci, cs, 20, 0.5)
        assert np.array_equal(ev.top_ids[sel].cpu().numpy().astype(np.int64), ri)
    g = ev.group_metrics(3)
    assert g["n_users"].sum() == n


@gpu
def test_mmr_spreads_lists_over_clusters(trained_case):
    """items in clusters of 10 near-duplicates whose scores rank whole clusters together: plain top-10 takes one cluster (two where
    train items leave gaps), MMR at 0.5 one item of each of the top clusters, and ILD and coverage both rise"""
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    g = torch.Generator().manual_seed(7)
    n_cl = c.I // 10
    # sparse non-negative centres (ELU keeps them), so clusters are nearly orthogonal; the score lives in column 0 alone
    centres = 4.0 * torch.rand((n_cl, 64), generator=g) * (torch.rand((n_cl, 64), generator=g) < 0.125)
    centres[:, 0] = 0.0
    cl = torch.arange(c.I) // 10
    Z = torch.zeros((c.U + c.I, 64))
    Z[c.U:] = centres[cl] + 0.01 * torch.rand((c.I, 64), generator=g)
    Z[c.U:, 0] = 0.2 + 0.005 * (n_cl - cl).float() + 0.0001 * torch.rand(c.I, generator=g)   # cluster 0 scores highest
    Z[:c.U, 0] = 1.0 + torch.rand(c.U, generator=g)
    Z = Z.to(DEV)
    res = {}
    for lam in (None, 0.5):
        ev = FullRankingEvaluator(c.dit, [10], "exact", mmr_lambda=lam)
        ev.rank(Z)
        res[lam] = (ev.top_ids[:c.dit.eval_users.numel()].cpu().numpy(), ev.diversity_metrics()["ild"][0], ev.list_metrics()["coverage"][0])
    plain_cl = res[None][0] // 10
    mmr_cl = res[0.5][0] // 10
    plain_n, mmr_n = np.mean([len(set(r)) for r in plain_cl]), np.mean([len(set(r)) for r in mmr_cl])
    assert plain_n < 2.5 and mmr_n > 5 and mmr_n > 2 * plain_n, (plain_n, mmr_n)
    assert res[0.5][1] > res[None][1] + 0.3 and res[0.5][2] > res[None][2]


@gpu
@pytest.mark.parametrize("key", ["64", "128", "multi64"])
def test_recommender_diversified_and_list_diversity(trained_case, key):
    from ngacf_b200.recommend import Recommender
    c = trained_case
    rec = Recommender(c.models[key], c.adj, c.dit, "train")
    F = rec.F.cpu().numpy()
    users = np.array([0, 5, 17, 17, 399])
    for K, N, lam, w in ((20, 100, 0.5, 0.0), (5, 20, 0.0, 0.0), (30, 30, 0.3, 0.0), (10, 60, 0.7, 1.0)):
        ids, sc = rec.diversified(users, K, lam, N, novelty_weight=w)
        assert ids.dtype == torch.int64 and sc.dtype == torch.float32 and ids.shape == (5, K)
        ci, cs = rec(users, N, novelty_weight=w)
        ri, rs = mmr_rows(F, c.U, c.I, ci.cpu().numpy(), cs.cpu().numpy(), K, lam)
        assert np.array_equal(ids.cpu().numpy(), ri) and np.array_equal(bits(sc), bits(rs))
        if w == 0.0:
            ci2, _ = _oracle_candidates(c, F, users, N, _train_sets(c.dit, users))
            assert np.array_equal(ci.cpu().numpy(), ci2)
    i1, s1 = rec.diversified(users, 20, 1.0)
    i0, s0 = rec(users, 20)
    assert torch.equal(i1, i0) and torch.equal(s1.view(torch.int32), s0.view(torch.int32))
    assert rec.diversified([], 5)[0].shape == (0, 5)
    lists = np.array([[3, 9, 700, -1, 9], [-1, -1, -1, -1, -1], [1, 2, 3, 4, 5]])
    got = rec.list_diversity(lists, [2, 5])
    assert got.dtype == torch.float64 and got.shape == (3, 2)
    assert np.array_equal(got.cpu().numpy(), ild_rows(F, c.U, c.I, lists, [2, 5]))
    assert np.array_equal(rec.list_diversity(torch.from_numpy(lists), [5]).cpu().numpy()[:, 0], got.cpu().numpy()[:, 1])
    for bad, ks in ((lists.astype(float), [2]), (lists[0], [2]), (lists, [6]), (np.zeros((2, 101), np.int64), [5])):
        with pytest.raises(ValueError):
            rec.list_diversity(bad, ks)


@gpu
def test_call_site_caches_one_evaluator_per_lambda(trained_case):
    import train_eval_Gowalla as T
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    model = c.models["64"]
    for attr in ("_full_evaluator", "_novelty_evaluators", "_mmr_evaluators"):
        model.__dict__.pop(attr, None)
    ks = [10, 50]
    with pytest.raises(RuntimeError, match="eval_full_ranking"):
        T.diversity_report(model, mmr_lambda=0.5)
    plain = T.eval_full_ranking(model, None, c.dit, c.adj, ks, False)
    ev0 = model._full_evaluator
    r5 = T.eval_full_ranking(model, None, c.dit, c.adj, ks, False, mmr_lambda=0.5)
    assert model._full_evaluator is ev0 and ev0.mmr_lambda is None
    ev5 = model._mmr_evaluators[(0.0, 0.5)]
    ref = FullRankingEvaluator(c.dit, ks, mmr_lambda=0.5)
    rr = ref(c.Z["64"])
    for k in METRICS:
        assert np.array_equal(r5[k], rr[k])
    d5, d0 = T.diversity_report(model, mmr_lambda=0.5), T.diversity_report(model)
    assert np.array_equal(d5["ild"], ref.diversity_metrics()["ild"]) and (d5["ild"] > d0["ild"]).all()
    rep = T.list_reports(model, True, 2, mmr_lambda=0.5)
    for k, v in ref.list_metrics().items():
        assert np.array_equal(np.asarray(rep["beyond"][k]), np.asarray(v))
    assert np.array_equal(T.eval_full_ranking(model, None, c.dit, c.adj, ks, False)["recall"], plain["recall"])
    T.eval_full_ranking(model, None, c.dit, c.adj, ks, False, mmr_lambda=0.5)
    assert model._mmr_evaluators[(0.0, 0.5)] is ev5
    with pytest.raises(ValueError):
        T.eval_full_ranking(model, None, c.dit, c.adj, ks, False, mmr_lambda=1.5)


def _cli_lines(R, flags, capsys):
    args = R.parse_args(flags)
    torch.manual_seed(args.seed)
    torch.cuda.manual_seed_all(args.seed)
    np.random.seed(args.seed)
    R.main(args)
    out = capsys.readouterr().out
    return [l.split(", time")[0] for l in out.splitlines() if "time of evaluate" not in l and "timeStamp" not in l]


@gpu
def test_run_gowalla_diversity_and_mmr_lines(tmp_path, monkeypatch, capsys):
    import run_Gowalla as R
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--epochs", "1", "--eval_every", "1", "--save_every", "1", "--droprate", "0.2",
            "--batch_size", "2048", "--eval_ks", "100,5,50", "--eval_beyond", "True", "--train_mode", "PairSampling",
            "--eval_mode", "AllNeg", "--lr", "0.002", "--parallel", "False"]
    plain = _cli_lines(R, base, capsys)
    lines = _cli_lines(R, base + ["--eval_diversity", "True", "--eval_novelty_weights", "2", "--eval_mmr_lambdas", "0.5,0"], capsys)
    assert [l for l in lines if "diversity metrics" not in l and "novelty weight" not in l and "mmr lambda" not in l] == plain
    extra = [l for l in lines if l not in plain]
    heads = [l.split(":{")[0] for l in extra]
    assert heads == ["epoch:0 diversity metrics", "epoch:0 novelty weight 2.0 full-ranking metrics",
                     "epoch:0 novelty weight 2.0 beyond-accuracy metrics", "epoch:0 novelty weight 2.0 diversity metrics"] + [
        "epoch:0 mmr lambda {} {}".format(lam, s) for lam in (0.5, 0.0)
        for s in ("full-ranking metrics", "beyond-accuracy metrics", "diversity metrics")]
    args = R.parse_args(base)
    inter, _, _, _, U, I, adj = R.prepareData(args)
    capsys.readouterr()
    model, _, _ = R.createModels(args, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    model.eval()
    with torch.no_grad():
        Z = model.propagate(adj.to(DEV))
    got = [ast.literal_eval(l.split("metrics:", 1)[1]) for l in extra]
    ev = FullRankingEvaluator(inter, [5, 50, 100])
    ev.rank(Z)
    evw = FullRankingEvaluator(inter, [5, 50, 100], novelty_weight=2.0)
    evw.rank(Z)
    refs = [ev.diversity_metrics(), evw.metrics(), evw.list_metrics(), evw.diversity_metrics()]
    for lam in (0.5, 0.0):
        e = FullRankingEvaluator(inter, [5, 50, 100], mmr_lambda=lam)
        refs += [e(Z), e.list_metrics(), e.diversity_metrics()]
    for g, r in zip(got, refs):
        assert g.keys() == r.keys()
        for k in r:
            rv = r[k].tolist() if hasattr(r[k], "tolist") else r[k]
            if k in ("ks", "n_users", "n_items", "coverage", "gini"):
                assert g[k] == rv, k
            else:
                _close(g[k], rv)


@gpu
def test_recommend_cli_mmr_lambda(tmp_path, monkeypatch, capsys):
    import recommend as RC
    import run_Gowalla as R
    from ngacf_b200.recommend import Recommender
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--lr", "0.002",
            "--droprate", "0.2", "--batch_size", "2048", "--parallel", "False"]
    args = R.parse_args(base + ["--epochs", "1", "--eval_every", "1", "--save_every", "1"])
    RC.seed_all(args.seed)
    R.main(args)
    users, ids, scores = RC.main(RC.parse_args(base + ["--resume_from", "1", "--topk", "15", "--mmr-lambda", "0.4", "--mmr-candidates", "60"]))
    assert "mmr lambda 0.4 of 60 candidates" in capsys.readouterr().out
    rows = [line.rstrip("\n").split("\t") for line in open("recs/SPUIGACF_synth-tiny_001_top15_mmr0.4.tsv")]
    a = R.parse_args(base)
    RC.seed_all(a.seed)
    inter, _, _, _, U, I, adj = R.prepareData(a)
    model, _, _ = R.createModels(a, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    rec = Recommender(model, adj, inter, "train")
    api_ids, api_sc = rec.diversified(users, 15, 0.4, 60)
    assert np.array_equal(ids, api_ids.cpu().numpy()) and np.array_equal(bits(scores), bits(api_sc))
    assert not np.array_equal(ids, rec(users, 15)[0].cpu().numpy())
    valid_ = api_ids.cpu().numpy() >= 0
    assert len(rows) == int(valid_.sum())
    assert np.array_equal(np.array([int(r[2]) for r in rows]), api_ids.cpu().numpy()[valid_])
    got_sc = np.array([np.float32(float(r[3])) for r in rows], np.float32)
    assert np.array_equal(bits(got_sc), bits(api_sc.cpu().numpy()[valid_]))
