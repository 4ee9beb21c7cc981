"""Novelty-weighted top-K lists: ngacf_recommend_topk_offset, cutoff_eval.novelty_offsets, Recommender(novelty_weight=),
FullRankingEvaluator(novelty_weight=), train_eval_Gowalla.eval_full_ranking / list_reports, run_Gowalla.py --eval_novelty_weights
and recommend.py --novelty-weight.

The oracle adds the fp32 offset to the port.dot64_tree score with one fp32 addition (numpy float32 + float32 rounds to nearest, as
__fadd_rn does) and ranks every candidate by (offset score descending, id ascending) with np.lexsort, as test_recommend's oracle
ranks the plain scores."""
import ast

import numpy as np
import pytest
import torch

from oracle import port

DEV = "cuda:0"
gpu = pytest.mark.gpu
METRICS = ("precision", "recall", "ndcg", "hit_ratio", "mrr")
DISC = 1.0 / np.log2(np.arange(2, 102))


# ------------------------------------------------------------------------------------------------
# oracle (adapted from test_recommend.py, test_cutoff_metrics.py and test_list_report.py)
# ------------------------------------------------------------------------------------------------
def score_matrix(F, U, users):
    """dot64_tree scores (n, I) of the users' rows against every item row of F (U+I, W); out-of-range users get zero rows"""
    F = np.asarray(F, np.float32)
    items = F[U:]
    return np.stack([port.dot64_tree(np.broadcast_to(F[u], items.shape), items) if 0 <= u < U else np.zeros(items.shape[0], np.float32)
                     for u in users])


def oracle_topk(S, users, U, K, excl=None, in_pool=None, off=None):
    """S: (n, I) scores of `users`; excl: dict user -> excluded item ids (None: nothing); in_pool: bool[I] (None: every item);
    off: float32[I] offsets (None: the plain scores).  -> ids int64 (n, K) (-1 padded), scores float32 (n, K) (0.0 padded)"""
    n, I = S.shape
    if off is not None:
        S = (np.asarray(S, np.float32) + np.asarray(off, np.float32)[None, :]).astype(np.float32)
    ids = np.full((n, K), -1, np.int64)
    sc = np.zeros((n, K), np.float32)
    for r, u in enumerate(users):
        if not 0 <= u < U:
            continue
        cand = np.ones(I, bool) if in_pool is None else np.asarray(in_pool, bool).copy()
        if excl is not None:
            cand[np.asarray(list(excl.get(int(u), ())), np.int64)] = False
        c = np.nonzero(cand)[0]
        s = S[r, c]
        order = np.lexsort((c, -s.astype(np.float64)))[:K]
        ids[r, :order.size] = c[order]
        sc[r, :order.size] = s[order]
    return ids, sc


def excl_sets(U, pairs):
    out = {u: set() for u in range(U)}
    for uu, ii in pairs:
        for u, i in zip(np.asarray(uu).tolist(), np.asarray(ii).tolist()):
            out[u].add(i)
    return out


def excl_csr(U, sets):
    ptr = np.zeros(U + 1, np.int64)
    items = []
    for u in range(U):
        s = sorted(sets.get(u, ()))
        ptr[u + 1] = ptr[u] + len(s)
        items += s
    return ptr, np.asarray(items, np.int64)


def novelty_table(train_items, I, n_tr):
    """nov(i) = -log2((d_i + 1) / (n_tr + 1)), d_i = distinct train users of item i (float64)"""
    d = np.bincount(np.asarray(train_items, np.int64), minlength=I).astype(np.float64)
    return -np.log2((d + 1.0) / (n_tr + 1.0)), d


def cutoff_metrics(lists, test_sets, ks):
    """(n, 5 len(ks)) float64, metric-major: precision at each cut-off, then recall, ndcg, hit_ratio, mrr"""
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
            for r in np.nonzero(hit[:k])[0]:
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


def list_rows(lists, I, ks, tables):
    """(n, len(tables) len(ks)) float64: each table's mean over the valid entries among the first k, summed in rank order"""
    lists = np.asarray(lists, np.int64)
    nv, nk = len(tables), len(ks)
    out = np.zeros((lists.shape[0], nv * nk))
    for j, row in enumerate(lists.tolist()):
        for v in range(nv):
            s, c, q = 0.0, 0, 0
            for r in range(ks[-1]):
                i = row[r]
                if 0 <= i < I:
                    s += float(tables[v][i])
                    c += 1
                if r + 1 == ks[q]:
                    out[j, v * nk + q] = s / c if c else 0.0
                    q += 1
    return out


def coverage_gini(lists, I, ks, pool):
    counts = np.zeros((len(ks), I), np.int64)
    for q, k in enumerate(ks):
        ids = np.asarray(lists)[:, :k].ravel()
        np.add.at(counts[q], ids[(ids >= 0) & (ids < I)], 1)
    c = counts[:, pool]
    n = c.shape[1]
    cov = np.array([np.count_nonzero(x) / n for x in c])
    gini = []
    for x in c:
        x = np.sort(x)
        num = int(sum((2 * (j + 1) - n - 1) * int(v) for j, v in enumerate(x)))
        den = n * int(x.sum())
        gini.append(np.float64(num) / np.float64(den) if den else 0.0)
    return cov, np.array(gini), counts


def bits(t):
    return np.asarray(t.cpu().numpy() if torch.is_tensor(t) else t, np.float32).view(np.int32)


def assert_lists(ids, sc, ref_ids, ref_sc):
    ids = ids.cpu().numpy() if torch.is_tensor(ids) else np.asarray(ids)
    assert np.array_equal(ids.astype(np.int64), ref_ids)
    assert np.array_equal(bits(sc), bits(ref_sc))


def _close(got, ref):
    np.testing.assert_allclose(np.asarray(got, np.float64), np.asarray(ref, np.float64), rtol=1e-12, atol=1e-300)


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_oracle_with_zero_offsets_is_the_plain_oracle():
    U, I = 30, 400
    rng = np.random.default_rng(1)
    F = rng.standard_normal((U + I, 64)).astype(np.float32)
    F[U + 10:U + 40] = F[U + 200]                       # exact ties across ids
    F[U + 50:U + 60] = 0.0                              # zero scores: -0.0 / +0.0
    users = np.arange(-1, U + 1)
    S = score_matrix(F, U, users)
    sets = {u: set(rng.choice(I, 20, replace=False).tolist()) for u in range(U)}
    pool = rng.random(I) < 0.8
    for K in (1, 20, 100):
        ids0, sc0 = oracle_topk(S, users, U, K, sets, pool)
        ids, sc = oracle_topk(S, users, U, K, sets, pool, np.zeros(I, np.float32))
        assert np.array_equal(ids, ids0)
        assert np.array_equal(sc, sc0)                   # -0.0 == +0.0
        assert not (bits(sc) == np.int32(-2 ** 31)).any()  # x + 0.0 is never -0.0


def test_novelty_offsets_are_the_rounded_fp64_products():
    from ngacf_b200.cutoff_eval import item_tables, novelty_offsets
    from ngacf_b200.data import Interactions
    U, I = 60, 90
    rng = np.random.default_rng(3)
    tu, ti = rng.integers(0, U, 700), rng.integers(0, I, 700)
    su, si = rng.integers(0, U, 300), rng.integers(0, I, 300)
    it = Interactions.from_arrays(U, I, tu, ti, su, si, device="cpu")
    nov, _ = novelty_table(it.host["train_items"], I, it.n_train_users)
    assert np.array_equal(item_tables(it)[0].numpy(), nov)
    for w in (1.0, 0.5, -2.25, 1e-3, 3.3, 1e30):
        off = novelty_offsets(it, w)
        assert off.dtype == torch.float32 and off.shape == (I,) and off.is_contiguous()
        assert np.array_equal(bits(off), bits(np.float32(w * nov)))
        assert novelty_offsets(it, w) is off                         # cached per weight
    assert not np.array_equal(bits(novelty_offsets(it, 0.1)), bits(np.float32(0.1 * nov.astype(np.float32))))
    for bad in (float("nan"), float("inf"), -float("inf"), "1", None, True):
        with pytest.raises(ValueError):
            novelty_offsets(it, bad)


def test_python_refusals_without_cuda():
    from ngacf_b200 import _lib
    from ngacf_b200.cutoff_eval import FullRankingEvaluator, check_novelty_weight
    from ngacf_b200.data import Interactions
    from ngacf_b200.recommend import Recommender
    assert check_novelty_weight(2) == 2.0 and check_novelty_weight(np.float32(0.5)) == 0.5 and check_novelty_weight(-0.0) == 0.0
    it = Interactions.from_arrays(20, 30, np.arange(20) % 20, np.arange(20) % 30, np.arange(20), (np.arange(20) + 5) % 30, device="cpu")
    with pytest.raises(_lib.NgacfError, match="offsets"):
        FullRankingEvaluator(it, [10, 20], "tc", novelty_weight=1.0)
    for bad in (float("nan"), float("inf"), "x", None):
        with pytest.raises(ValueError, match="novelty weight"):
            FullRankingEvaluator(it, [20], "exact", novelty_weight=bad)
    # Recommender.__call__ checks the weight before it reads any features
    rec = Recommender.__new__(Recommender)
    rec.inter = None
    with pytest.raises(ValueError, match="inter="):
        rec([0], 5, novelty_weight=1.0)
    rec.inter = it
    with pytest.raises(ValueError, match="finite"):
        rec([0], 5, novelty_weight=float("nan"))


def test_cli_refusals(monkeypatch):
    import recommend as RC
    import run_Gowalla as R
    import torch.distributed as dist
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: pytest.fail("process group created"))
    assert R.parse_args([]).eval_novelty_weights is None
    a = R.parse_args(["--eval_ks", "20", "--eval_novelty_weights", "0.5,1,-2"])
    assert a.eval_novelty_weights == [0.5, 1.0, -2.0]
    assert len(R.parse_args(["--eval_ks", "20", "--eval_novelty_weights", ",".join(str(x) for x in range(1, 9))]).eval_novelty_weights) == 8
    for bad in (["--eval_novelty_weights", "1"], ["--eval_ks", "20", "--eval_novelty_weights", "0"],
                ["--eval_ks", "20", "--eval_novelty_weights", "1,0"], ["--eval_ks", "20", "--eval_novelty_weights", "1,1.0"],
                ["--eval_ks", "20", "--eval_novelty_weights", "nan"], ["--eval_ks", "20", "--eval_novelty_weights", "inf"],
                ["--eval_ks", "20", "--eval_novelty_weights", "x"], ["--eval_ks", "20", "--eval_novelty_weights", ""],
                ["--eval_ks", "20", "--eval_novelty_weights", ",".join(str(x) for x in range(1, 10))]):
        with pytest.raises(ValueError, match="--eval_novelty_weights"):
            R.parse_args(["--parallel", "True"] + bad)
    assert not dist.is_initialized()
    base = ["--resume_from", "7"]
    assert RC.parse_args(base).novelty_weight == 0.0 and RC.parse_args(base).out == "recs/SPUIGACF_ml100k_007_top20.tsv"
    a = RC.parse_args(base + ["--novelty-weight", "1"])
    assert a.novelty_weight == 1.0 and a.out == "recs/SPUIGACF_ml100k_007_top20_nw1.0.tsv"
    assert RC.parse_args(base + ["--novelty-weight", "-0.5", "--topk", "50"]).out == "recs/SPUIGACF_ml100k_007_top50_nw-0.5.tsv"
    assert RC.parse_args(base + ["--novelty-weight", "2", "--out", "x.tsv"]).out == "x.tsv"
    for flag in ("--similar-items", "--audience", "--similar-users"):
        with pytest.raises(ValueError, match="--novelty-weight"):
            RC.parse_args(base + ["--novelty-weight", "1", flag, "3"])
        RC.parse_args(base + ["--novelty-weight", "0", flag, "3"])
    for bad in ("nan", "inf"):
        with pytest.raises(ValueError, match="finite"):
            RC.parse_args(base + ["--novelty-weight", bad])


# ------------------------------------------------------------------------------------------------
# GPU: the C-ABI against the oracle
# ------------------------------------------------------------------------------------------------
def _dev(a, dt=torch.int32):
    return None if a is None else torch.as_tensor(np.asarray(a)).to(dt).to(DEV)


def _ranker(F, U, I, users, K, off, excl_ptr=None, excl_items=None, in_pool=None):
    """ops.recommend_topk with item_offset=off (None: the plain entry point) -> (ids, scores) device tensors"""
    from ngacf_b200 import ops
    u = _dev(users)
    n = u.numel()
    ids = torch.empty((n, K), dtype=torch.int32, device=DEV)
    sc = torch.empty((n, K), dtype=torch.float32, device=DEV)
    ws = torch.empty(ops.recommend_topk_workspace_bytes(F.shape[-1], I, n, K), dtype=torch.uint8, device=DEV)
    pool = None if in_pool is None else _dev(np.asarray(in_pool, np.uint8), torch.uint8)
    ops.recommend_topk(F, U, I, u, K, _dev(excl_ptr), _dev(excl_items), pool, ids, sc, ws,
                       None if off is None else _dev(np.asarray(off, np.float32), torch.float32))
    return ids, sc


@pytest.fixture(scope="module")
def kernel_case():
    """random features at both widths over 2,400 users (one pass: at least 149 CTAs of 16 users) and 2,100 items (33 tiles, so a
    few users split the items into 4 slices), items tying in groups of 4, exclusion sets and a pool"""
    U, I = 2400, 2100
    rng = np.random.default_rng(17)
    out = dict(U=U, I=I)
    for width in (64, 128):
        base = rng.standard_normal((I // 4 + 1, width)).astype(np.float32)
        items = rng.standard_normal((I, width)).astype(np.float32)
        items[:800] = base[np.arange(800) // 4]                 # items 0..799 tie in groups of 4
        F = np.concatenate([rng.standard_normal((U, width)).astype(np.float32), items])
        out[width] = dict(F=F, Ft=torch.from_numpy(F).to(DEV))
    sets_train = {u: set(rng.choice(I, int(rng.integers(0, 60)), replace=False).tolist()) for u in range(U)}
    sets_all = {u: sets_train[u] | set(rng.choice(I, 10, replace=False).tolist()) for u in range(U)}
    sets_all[3] = set(range(I))                                 # nothing left: an all -1 row
    out["excl"] = {"none": None, "train": sets_train, "all": sets_all}
    out["pool"] = rng.random(I) < 0.85
    out["offsets"] = {
        "random": (4.0 * rng.standard_normal(I)).astype(np.float32),
        "decisive": (1e6 * rng.permutation(I)).astype(np.float32),          # the offset alone orders every row
        "ties": np.repeat(rng.choice(np.float32([-1.0, 0.0, 0.25, 1.0]), I // 4 + 1), 4)[:I].astype(np.float32),
    }
    return out


@gpu
@pytest.mark.parametrize("width", [64, 128])
@pytest.mark.parametrize("exclude", ["none", "train", "all"])
def test_offset_lists_match_the_oracle(kernel_case, width, exclude):
    from ngacf_b200 import ops
    c = kernel_case
    U, I = c["U"], c["I"]
    F, Ft = c[width]["F"], c[width]["Ft"]
    sets = c["excl"][exclude]
    ptr, items = excl_csr(U, sets) if sets is not None else (None, None)
    everyone = np.arange(U)
    sample = np.concatenate([np.arange(0, U, 16), [1, 3, U - 1]])      # oracle rows of the one-pass call
    few = [[5], [3, 9, 2000], [7, -1, 7, U, 1 << 30, 0, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20]]
    S_sample = score_matrix(F, U, sample)
    for name, off in c["offsets"].items():
        for pool in (None, c["pool"]):
            for K in (1, 20, 37, 100):
                assert ops.recommend_topk_workspace_bytes(width, I, U, K) == 0
                ids, sc = _ranker(Ft, U, I, everyone, K, off, ptr, items, pool)
                ref = oracle_topk(S_sample, sample, U, K, sets, pool, off)
                assert_lists(ids[sample], sc[sample], *ref)
                for q in few:
                    assert ops.recommend_topk_workspace_bytes(width, I, len(q), K) > 0
                    qi, qs = _ranker(Ft, U, I, q, K, off, ptr, items, pool)
                    assert_lists(qi, qs, *oracle_topk(score_matrix(F, U, q), q, U, K, sets, pool, off))
                    for r, u in enumerate(q):                  # a row does not depend on the other users of the call
                        if 0 <= u < U:
                            assert torch.equal(qi[r], ids[u]) and torch.equal(qs[r].view(torch.int32), sc[u].view(torch.int32))
                        else:
                            assert (qi[r] == -1).all() and (qs[r] == 0).all()
            if name == "decisive":        # the offset decides: rows list the candidates by offset descending
                for u in (0, 1, 2):
                    cand = np.ones(I, bool) if pool is None else pool.copy()
                    if sets is not None:
                        cand[list(sets[u])] = False
                    c_ids = np.nonzero(cand)[0]
                    expect = c_ids[np.argsort(-off[c_ids].astype(np.float64), kind="stable")][:100]
                    assert ids[u, :expect.size].cpu().numpy().tolist() == expect.tolist()
    if exclude == "all":
        assert (ids[3] == -1).all() and (sc[3] == 0).all()


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_short_rows(kernel_case, width):
    c = kernel_case
    U, I = c["U"], c["I"]
    F, Ft = c[width]["F"], c[width]["Ft"]
    rng = np.random.default_rng(width)
    pool = np.zeros(I, bool)
    pool[rng.choice(I, 12, replace=False)] = True
    sets = {0: set(range(I)), 1: set(np.nonzero(pool)[0][:5].tolist())}
    ptr, items = excl_csr(U, sets)
    off = c["offsets"]["random"]
    for users in (np.arange(U), np.array([0, 1, 2, 3])):
        ids, sc = _ranker(Ft, U, I, users, 20, off, ptr, items, pool)
        sel = np.array([0, 1, 2, 3])
        assert_lists(ids[sel], sc[sel], *oracle_topk(score_matrix(F, U, sel), sel, U, 20, sets, pool, off))
        assert (ids[0] == -1).all() and (ids[1, 7:] == -1).all() and (ids[1, :7] >= 0).all()
        assert (ids[2:, 12:] == -1).all() and (sc[2:, 12:] == 0).all() and (ids[2:, :12] >= 0).all()


@gpu
@pytest.mark.parametrize("width", [64, 128])
def test_zero_offsets_give_the_plain_lists(kernel_case, width):
    c = kernel_case
    U, I = c["U"], c["I"]
    F = c[width]["F"].copy()
    F[:50] = -np.abs(F[:50])                            # users 0..49: every product with a zero row is -0.0, so their score is
    F[U:] = np.abs(F[U:])                               # -0.0, and with non-negative other items that is their best score
    F[U + 100:U + 180] = 0.0
    Ft = torch.from_numpy(F).to(DEV)
    zero = np.zeros(I, np.float32)
    ptr, items = excl_csr(U, c["excl"]["train"])
    for users in (np.arange(U), np.array([3, 5, 8])):
        for K in (20, 100):
            pi, ps = _ranker(Ft, U, I, users, K, None, ptr, items, c["pool"])
            oi, os_ = _ranker(Ft, U, I, users, K, zero, ptr, items, c["pool"])
            assert torch.equal(pi, oi)
            pb, ob = bits(ps), bits(os_)
            assert np.array_equal(np.where(pb == np.int32(-2 ** 31), 0, pb), ob)
    ids, sc = _ranker(Ft, U, I, np.arange(50), 100, None)          # the -0.0 case was exercised
    assert (bits(sc[:, :80]) == np.int32(-2 ** 31)).all()


@gpu
def test_c_abi_edges_and_graph_replay():
    from ngacf_b200 import _lib, ops
    lib = _lib.load()
    U, I, W = 300, 2500, 64
    rng = np.random.default_rng(9)
    F = rng.standard_normal((U + I, W)).astype(np.float32)
    off = (3.0 * rng.standard_normal(I)).astype(np.float32)
    Ft, offt = torch.from_numpy(F).to(DEV), torch.from_numpy(off).to(DEV)
    users = torch.tensor([4, 8], dtype=torch.int32, device=DEV)
    out_i = torch.full((2, 100), 7, dtype=torch.int32, device=DEV)
    out_s = torch.full((2, 100), 7.0, dtype=torch.float32, device=DEV)
    need = ops.recommend_topk_workspace_bytes(W, I, 2, 100)
    assert need > 0
    buf = torch.full((need + 4096,), 0xAB, dtype=torch.uint8, device=DEV)

    def call(width=W, K=100, nbytes=need, o=offt.data_ptr(), ws=buf.data_ptr()):
        return lib.ngacf_recommend_topk_offset(Ft.data_ptr(), width, U, I, users.data_ptr(), 2, K, None, None, None, o,
                                               out_i.data_ptr(), out_s.data_ptr(), ws, nbytes, ops._s())
    for kw, code, what in ((dict(K=0), -4, b"K = 0"), (dict(K=101), -4, b"K = 101"), (dict(width=96), -4, b"width 96"),
                           (dict(o=None), -1, b"item_offset"), (dict(nbytes=need - 1), -3, b"workspace"),
                           (dict(ws=None), -3, b"workspace")):
        assert call(**kw) == code and what in lib.ngacf_last_error()
    torch.cuda.synchronize()
    assert bool((out_i == 7).all()) and bool((out_s == 7.0).all()) and bool((buf == 0xAB).all()), "a refused call wrote"
    with pytest.raises(_lib.NgacfError, match="K = 101"):
        ops.recommend_topk(Ft, U, I, users, 101, None, None, None, out_i, out_s, buf, offt)
    assert call() == 0
    torch.cuda.synchronize()
    assert bool((buf[need:] == 0xAB).all()), "ngacf_recommend_topk_offset wrote past its reported workspace"
    ref = oracle_topk(score_matrix(F, U, [4, 8]), [4, 8], U, 100, off=off)
    assert_lists(out_i, out_s, *ref)
    assert lib.ngacf_recommend_topk_offset(Ft.data_ptr(), W, U, I, users.data_ptr(), 0, 20, None, None, None, offt.data_ptr(),
                                           out_i.data_ptr(), out_s.data_ptr(), None, 0, ops._s()) == 0      # n_users == 0: no-op
    assert lib.ngacf_recommend_topk_offset(Ft.data_ptr(), W, U, I, users.data_ptr(), 0, 20, None, None, None, None, out_i.data_ptr(),
                                           out_s.data_ptr(), None, 0, ops._s()) == -1
    # captured in a CUDA graph and replayed, for both launch shapes
    for uu in (users, torch.arange(U, dtype=torch.int32, device=DEV).repeat(9)):
        n = uu.numel()
        ws = torch.empty(ops.recommend_topk_workspace_bytes(W, I, n, 100), dtype=torch.uint8, device=DEV)
        ri, rs = torch.empty((n, 100), dtype=torch.int32, device=DEV), torch.empty((n, 100), dtype=torch.float32, device=DEV)
        ops.recommend_topk(Ft, U, I, uu, 100, None, None, None, ri, rs, ws, offt)
        gi, gs = torch.full_like(ri, 7), torch.zeros_like(rs)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            ops.recommend_topk(Ft, U, I, uu, 100, None, None, None, gi, gs, ws, offt)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            ops.recommend_topk(Ft, U, I, uu, 100, None, None, None, gi, gs, ws, offt)
        gi.fill_(7)
        gs.zero_()
        g.replay()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(gi, ri) and torch.equal(gs.view(torch.int32), rs.view(torch.int32))
        if n == 2:
            assert_lists(gi, gs, *ref)


# ------------------------------------------------------------------------------------------------
# GPU: Recommender, FullRankingEvaluator, the call sites and the CLIs
# ------------------------------------------------------------------------------------------------
def _seeded_model(cls, U, I, width, seed=5):
    torch.manual_seed(seed)
    m = cls(U, I, width, [64, 64], 0.1).to(DEV)
    with torch.no_grad():            # larger embeddings than the N(0, 0.01) init, so that the scores spread
        m.uEmbd.weight.mul_(30)
        m.iEmbd.weight.mul_(30)
    return m


@pytest.fixture(scope="module")
def trained_case():
    """a split of a synthetic graph with skewed degrees, a pool that leaves items out, and seeded models' pre-ELU outputs"""
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
    nov, d = novelty_table(dit.host["train_items"], I, dit.n_train_users)
    return SimpleNamespace(U=U, I=I, dit=dit, adj=adj, models=models, Z=Z, nov=nov, d=d, split=(tu, ti, su, si))


def _features(Z):
    from ngacf_b200 import ops
    F = torch.empty_like(Z)
    ops.final_features(Z, F)
    return F


@gpu
@pytest.mark.parametrize("key", ["64", "128", "multi64"])
def test_recommender_matches_the_oracle(trained_case, key):
    from ngacf_b200.recommend import Recommender, recommend
    c = trained_case
    dit = c.dit
    in_pool = np.zeros(c.I, bool)
    in_pool[dit.host["pool"]] = True
    tu, ti, su, si = c.split
    users = np.concatenate([np.arange(c.U), [7, 7, 0]])
    for exclude, sets in (("train", excl_sets(c.U, [(tu, ti)])), ("all", excl_sets(c.U, [(tu, ti), (su, si)])), ("none", None)):
        rec = Recommender(c.models[key], c.adj, dit, exclude)
        S = score_matrix(rec.F.cpu().numpy(), c.U, users)
        for w in (1.0, -0.5, 3.7):
            off = np.float32(w * c.nov)
            for K in (1, 20, 100):
                ids, sc = rec(users, K, novelty_weight=w)
                assert ids.dtype == torch.int64 and sc.dtype == torch.float32
                assert_lists(ids, sc, *oracle_topk(S, users, c.U, K, sets, in_pool, off))
        ids0, sc0 = rec(users, 20)
        for zero in (0.0, 0, -0.0):
            ids, sc = rec(users, 20, novelty_weight=zero)
            assert torch.equal(ids, ids0) and torch.equal(sc.view(torch.int32), sc0.view(torch.int32))
    assert rec([], 5, novelty_weight=1.0)[0].shape == (0, 5)
    with pytest.raises(ValueError, match="finite"):
        rec([0], 5, novelty_weight=float("inf"))
    plain = Recommender(c.models[key], c.adj, None, "none")
    with pytest.raises(ValueError, match="inter="):
        plain([0], 5, novelty_weight=1.0)
    assert torch.equal(recommend(c.models[key], c.adj, [0, 1], 5, inter=dit)[0], Recommender(c.models[key], c.adj, dit)([0, 1], 5)[0])


def _oracle_reports(case, Z, ks, w, G):
    """oracle lists of every evaluation user for weight w, then metrics, list metrics and group metrics from them"""
    dit = case.dit
    h = dit.host
    users = dit.eval_users.cpu().numpy()
    in_pool = np.zeros(case.I, bool)
    in_pool[h["pool"]] = True
    sets = {int(u): set(h["train_items"][h["train_ptr"][u]:h["train_ptr"][u + 1]].tolist()) for u in users}
    S = score_matrix(_features(Z).cpu().numpy(), case.U, users)
    lists, _ = oracle_topk(S, users, case.U, max(ks), sets, in_pool, np.float32(w * case.nov))
    tests = [h["test_items"][h["test_ptr"][u]:h["test_ptr"][u + 1]] for u in users]
    acc = cutoff_metrics(lists, tests, ks)
    lrows = list_rows(lists, case.I, ks, [case.nov, case.d])
    cov, gini, counts = coverage_gini(lists, case.I, ks, h["pool"])
    n, nk = users.size, len(ks)
    metrics = {name: acc[:, q * nk:(q + 1) * nk].sum(0) / n for q, name in enumerate(METRICS)}
    beyond = {"coverage": cov, "gini": gini, "novelty": lrows[:, :nk].sum(0) / n, "arp": lrows[:, nk:].sum(0) / n}
    deg = np.diff(h["train_ptr"])[users]
    order = np.lexsort((users, deg))
    C = np.cumsum(deg[order]) - deg[order]
    grp = np.empty(n, np.int64)
    grp[order] = np.minimum(G - 1, (G * C) // max(int(deg.sum()), 1))
    cnt = np.maximum(np.bincount(grp, minlength=G), 1)[:, None]
    groups = {"n_users": np.bincount(grp, minlength=G)}
    for q, name in enumerate(METRICS):
        groups[name] = np.stack([acc[grp == g][:, q * nk:(q + 1) * nk].sum(0) for g in range(G)]) / cnt
    groups["novelty"] = np.stack([lrows[grp == g][:, :nk].sum(0) for g in range(G)]) / cnt
    groups["arp"] = np.stack([lrows[grp == g][:, nk:].sum(0) for g in range(G)]) / cnt
    return lists, metrics, beyond, groups, counts


@gpu
@pytest.mark.parametrize("key,ks,w", [("64", [10, 20], 1.0), ("64", [5, 50, 100], 0.5), ("128", [20], 2.0), ("128", [1, 37, 100], -1.0),
                                      ("multi64", [3, 10, 37], 1.5)])
def test_evaluator_matches_the_oracle(trained_case, key, ks, w):
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    for mode in ("auto", "exact"):
        ev = FullRankingEvaluator(c.dit, ks, mode, novelty_weight=w)
        assert ev.novelty_weight == w and ev._allneg is None
        m = ev(c.Z[key])
        assert ev.source == "list" and ev.top_ids.shape[1] == max(ks)
    lists, metrics, beyond, groups, counts = _oracle_reports(c, c.Z[key], ks, w, 3)
    n = c.dit.eval_users.numel()
    assert np.array_equal(ev.top_ids[:n].cpu().numpy().astype(np.int64), lists)
    assert m["n_users"] == n and m["ks"] == ks
    for name in METRICS:
        _close(m[name], metrics[name])
    b = ev.list_metrics()
    assert np.array_equal(ev._counts.cpu().numpy(), counts)
    assert np.array_equal(b["coverage"], beyond["coverage"]) and np.array_equal(b["gini"], beyond["gini"])
    _close(b["novelty"], beyond["novelty"])
    _close(b["arp"], beyond["arp"])
    g = ev.group_metrics(3)
    assert np.array_equal(g["n_users"], groups["n_users"])
    for name in METRICS + ("novelty", "arp"):
        _close(g[name], groups[name])


@gpu
def test_weight_zero_and_the_tc_refusal(trained_case):
    from ngacf_b200 import _lib
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    for ks in ([10, 20], [5, 50]):
        a = FullRankingEvaluator(c.dit, ks)
        b = FullRankingEvaluator(c.dit, ks, novelty_weight=0.0)
        ra, rb = a(c.Z["64"]), b(c.Z["64"])
        assert a.source == b.source and torch.equal(a.top_ids, b.top_ids)
        for k in ra:
            assert np.array_equal(np.asarray(ra[k]), np.asarray(rb[k]))
    FullRankingEvaluator(c.dit, [20], "tc", novelty_weight=0.0)
    with pytest.raises(_lib.NgacfError, match="offsets"):
        FullRankingEvaluator(c.dit, [20], "tc", novelty_weight=0.5)


@gpu
def test_a_large_weight_raises_novelty_and_coverage(trained_case):
    """features whose scores follow item popularity, as a graph model's tend to: score = 2 log2(d_i + 1) + noise, so that w = 2
    cancels the popularity term"""
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    g = torch.Generator().manual_seed(4)
    Z = 0.3 * torch.randn((c.U + c.I, 64), generator=g)
    Z[:c.U, 0] = 1.0
    Z[c.U:, 0] = torch.from_numpy(2.0 * np.log2(c.d + 1.0)).float()
    Z = Z.to(DEV)
    out = {}
    for w in (0.0, 2.0):
        ev = FullRankingEvaluator(c.dit, [20, 100], "exact", novelty_weight=w)
        ev.rank(Z)
        out[w] = ev.list_metrics()
    assert (out[2.0]["novelty"] > out[0.0]["novelty"]).all() and (out[2.0]["coverage"] > out[0.0]["coverage"]).all()
    assert (out[2.0]["arp"] < out[0.0]["arp"]).all() and (out[2.0]["gini"] < out[0.0]["gini"]).all()


@gpu
def test_shards_give_the_unsharded_sums(trained_case):
    import ngacf_b200.dist as D
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    it = c.dit
    ks = [5, 50, 100]
    whole = FullRankingEvaluator(it, ks, novelty_weight=1.5)
    whole.rank(c.Z["64"])
    whole._compute()
    whole._list_stats(True)
    for world in range(1, 5):
        evs = [FullRankingEvaluator(it, ks, users=D.shard_eval_users(it.eval_users, r, world), novelty_weight=1.5) for r in range(world)]
        for ev in evs:
            ev.rank(c.Z["64"])
            ev._compute()
            ev._list_stats(True)
        assert torch.equal(torch.cat([ev.top_ids[:ev.users.numel()] for ev in evs]), whole.top_ids[:it.eval_users.numel()])
        assert torch.equal(sum(ev._counts for ev in evs), whole._counts)
        _close(sum(ev._sums for ev in evs).cpu().numpy(), whole._sums.cpu().numpy())
        _close(sum(ev._list_rows.sum(0) for ev in evs).cpu().numpy(), whole._list_rows.sum(0).cpu().numpy())


@gpu
def test_call_site_caches_one_evaluator_per_weight(trained_case):
    import train_eval_Gowalla as T
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    c = trained_case
    model = c.models["64"]
    for attr in ("_full_evaluator", "_novelty_evaluators"):
        model.__dict__.pop(attr, None)
    ks = [10, 50]
    with pytest.raises(RuntimeError, match="eval_full_ranking"):
        T.list_reports(model, True, None, novelty_weight=2.0)
    plain = T.eval_full_ranking(model, None, c.dit, c.adj, ks, False)
    ev0 = model._full_evaluator
    r2 = T.eval_full_ranking(model, None, c.dit, c.adj, ks, False, novelty_weight=2.0)
    assert model._full_evaluator is ev0 and ev0.novelty_weight == 0.0
    ev2 = model._novelty_evaluators[2.0]
    assert ev2.novelty_weight == 2.0
    ref = FullRankingEvaluator(c.dit, ks, novelty_weight=2.0)
    rr = ref(c.Z["64"])
    for k in METRICS:
        assert np.array_equal(r2[k], rr[k])
    rep2, rep0 = T.list_reports(model, True, 2, novelty_weight=2.0), T.list_reports(model, True, 2)
    for k, v in ref.list_metrics().items():
        assert np.array_equal(np.asarray(rep2["beyond"][k]), np.asarray(v))
    assert not np.array_equal(rep2["beyond"]["novelty"], rep0["beyond"]["novelty"])
    assert np.array_equal(T.eval_full_ranking(model, None, c.dit, c.adj, ks, False)["recall"], plain["recall"])
    assert model._novelty_evaluators[2.0] is ev2
    with pytest.raises(ValueError):
        T.eval_full_ranking(model, None, c.dit, c.adj, ks, False, novelty_weight=float("nan"))


def _cli_lines(R, flags, capsys):
    args = R.parse_args(flags)
    torch.manual_seed(args.seed)
    torch.cuda.manual_seed_all(args.seed)
    np.random.seed(args.seed)
    R.main(args)
    out = capsys.readouterr().out
    return [l.split(", time")[0] for l in out.splitlines() if "time of evaluate" not in l and "timeStamp" not in l]


@gpu
def test_run_gowalla_novelty_lines(tmp_path, monkeypatch, capsys):
    import run_Gowalla as R
    from ngacf_b200.cutoff_eval import FullRankingEvaluator
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--epochs", "1", "--eval_every", "1", "--save_every", "1", "--droprate", "0.2",
            "--batch_size", "2048", "--eval_ks", "100,5,50", "--eval_beyond", "True", "--eval_groups", "3", "--train_mode", "PairSampling",
            "--eval_mode", "AllNeg", "--lr", "0.002", "--parallel", "False"]
    weights = [0.5, -2.0]
    plain = _cli_lines(R, base, capsys)
    both = _cli_lines(R, base + ["--eval_novelty_weights", "0.5,-2"], capsys)
    tagged = [l for l in both if "novelty weight" in l]
    assert [l for l in both if "novelty weight" not in l] == plain
    assert len(tagged) == 3 * len(weights) and both[-len(tagged):] == tagged
    args = R.parse_args(base)
    inter, _, _, _, U, I, adj = R.prepareData(args)
    capsys.readouterr()
    model, _, _ = R.createModels(args, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    model.eval()
    with torch.no_grad():
        Z = model.propagate(adj.to(DEV))
    for j, w in enumerate(weights):
        lines = tagged[3 * j:3 * j + 3]
        head = "epoch:0 novelty weight {} ".format(w)
        assert [l.split(":{")[0] for l in lines] == [head + s for s in ("full-ranking metrics", "beyond-accuracy metrics",
                                                                          "user-group metrics")]
        got = [ast.literal_eval(l.split("metrics:", 1)[1]) for l in lines]
        ev = FullRankingEvaluator(inter, [5, 50, 100], novelty_weight=w)
        refs = [ev(Z), ev.list_metrics(), ev.group_metrics(3)]
        for g, r in zip(got, refs):
            assert g.keys() == r.keys()
            for k in r:
                rv = r[k].tolist() if hasattr(r[k], "tolist") else r[k]
                if k in ("ks", "groups", "n_users", "n_items", "degree", "interactions", "coverage", "gini"):
                    assert g[k] == rv, (w, k)
                else:
                    _close(g[k], rv)


@gpu
def test_recommend_cli_novelty_weight(tmp_path, monkeypatch, capsys):
    import recommend as RC
    import run_Gowalla as R
    from ngacf_b200.recommend import Recommender
    monkeypatch.chdir(tmp_path)
    base = ["--dataset", "synth-tiny", "--model", "SPUIGACF", "--train_mode", "PairSampling", "--eval_mode", "AllNeg", "--lr", "0.002",
            "--droprate", "0.2", "--batch_size", "2048", "--parallel", "False"]
    args = R.parse_args(base + ["--epochs", "1", "--eval_every", "1", "--save_every", "1"])
    RC.seed_all(args.seed)
    R.main(args)
    users, ids, scores = RC.main(RC.parse_args(base + ["--resume_from", "1", "--topk", "30", "--novelty-weight", "1.5"]))
    assert "novelty weight 1.5" in capsys.readouterr().out
    rows = [line.rstrip("\n").split("\t") for line in open("recs/SPUIGACF_synth-tiny_001_top30_nw1.5.tsv")]
    a = R.parse_args(base)
    RC.seed_all(a.seed)
    inter, _, _, _, U, I, adj = R.prepareData(a)
    model, _, _ = R.createModels(a, U, I)
    model.load_state_dict(torch.load("ckpts/SPUIGACF_synth-tiny_001.pkl", map_location="cuda")["model"])
    rec = Recommender(model, adj, inter, "train")
    api_ids, api_sc = rec(users, 30, novelty_weight=1.5)
    plain_ids, _ = rec(users, 30)
    assert np.array_equal(ids, api_ids.cpu().numpy()) and np.array_equal(bits(scores), bits(api_sc))
    assert not np.array_equal(ids, plain_ids.cpu().numpy())
    valid = api_ids.cpu().numpy() >= 0
    assert len(rows) == int(valid.sum())
    got = np.array([int(r[2]) for r in rows])
    got_sc = np.array([np.float32(float(r[3])) for r in rows], np.float32)
    assert np.array_equal(got, api_ids.cpu().numpy()[valid]) and np.array_equal(bits(got_sc), bits(api_sc.cpu().numpy()[valid]))
